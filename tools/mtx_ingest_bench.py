"""Wall-clock cost of getting config 4's operand (ER 2^23, 8 non-zeros per row: 6.7e7 entries) from a .mtx file into
HBM as CSC(A) and CSR(A), on the host loaders and on the device ingest.  Development aid, not bench.py.

    python tools/mtx_ingest_bench.py [--runs 5] [--no-cli] [--dir DIR]

The operand is written in scipy.io.mmwrite's text format to a temporary directory (or DIR) and read once to warm the
page cache.  Each path is timed wall-clock from the file to a device synchronise with both operands in HBM:
  host:   osp_readcoo, then osp_coo2csr<true> and osp_coo2csr, then the two CSR arrays copied to the device
  device: osp_readcoo_device, then osp_coo2csr_result with transpose = 1 and = 0
Best and median of --runs runs.  The device path's kernels alone (no file read, no host-to-device copy) are summed
from a torch.profiler trace of one osp_readcoo_device call.  The card, its power limit and the host's core count are
printed by the same run, and the CLI (outerspace_b200/osp_spgemm_cli A.mtx A.mtx --no-transpose, i.e. config 4's
C = A*A) is timed end to end with and without --device-ingest."""
import argparse
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import outerspace_b200 as osp  # noqa: E402
from outerspace_b200 import synth  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi unavailable"
    return f"{name}, power limit / max SM clock: {q}, host cores: {os.cpu_count()}"


def stats(ts):
    return f"best {min(ts) * 1e3:9.1f} ms, median {float(np.median(ts)) * 1e3:9.1f} ms over {len(ts)} runs"


def host_path(path):
    coo, nrow, ncol = osp.readcoo(path)
    csc = osp.coo2csr(coo, ncol, transpose=True)
    csr = osp.coo2csr(coo, nrow)
    dev = [torch.from_numpy(a.view(np.uint8).reshape(-1)).to("cuda:0") for a in (csc.pos, csc.data, csr.pos, csr.data)]
    torch.cuda.synchronize()
    return dev, len(coo)


def device_path(eng, path):
    d = eng.readcoo_device(path)
    try:
        return [d.to_csr(d.ncol, transpose=True), d.to_csr(d.nrow)], d.nnz     # both synchronise before they return
    finally:
        d.free()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--no-cli", action="store_true")
    ap.add_argument("--dir", default=None)
    args = ap.parse_args()
    import scipy.io
    import scipy.sparse as sp

    print(card(), flush=True)
    with tempfile.TemporaryDirectory(dir=args.dir) as tmp:
        a, _, dims = synth.build_workload("er8m")
        m = sp.csr_matrix((a.data["val"], a.data["idx"].astype(np.int64), a.pos.astype(np.int64)), shape=(dims["rows"], dims["n_k"]))
        path = os.path.join(tmp, "er8m.mtx")
        t = time.perf_counter()
        scipy.io.mmwrite(path, m)
        del m
        size = os.path.getsize(path)
        print(f"wrote {path}: {size / 1e9:.3f} GB, {a.nnz} entries, in {time.perf_counter() - t:.1f} s", flush=True)
        with open(path, "rb") as f:                                   # warm the page cache
            while f.read(1 << 26):
                pass
        eng = osp.Engine(0)
        # the outputs of both paths, compared once outside the timed runs
        coo, nrow, ncol = osp.readcoo(path)
        want = [osp.coo2csr(coo, ncol, transpose=True), osp.coo2csr(coo, nrow)]
        del coo
        dr, n_dev = device_path(eng, path)
        for w, r in zip(want, dr):
            got = r.to_host()
            r.free()
            assert np.array_equal(got.pos, w.pos) and got.data.tobytes() == w.data.tobytes(), "the paths differ"
        del want, got
        print(f"both paths give the same CSC(A) and CSR(A) ({n_dev} entries)", flush=True)
        th, td = [], []
        for _ in range(args.runs):                                    # alternated, so drift hits both alike
            t = time.perf_counter()
            hd, _ = host_path(path)
            th.append(time.perf_counter() - t)
            del hd
            t = time.perf_counter()
            dr, _ = device_path(eng, path)
            td.append(time.perf_counter() - t)
            for r in dr:
                r.free()
        print(f"host   readcoo + coo2csr<true> + coo2csr + upload:   {stats(th)}", flush=True)
        print(f"device readcoo_device + 2 x coo2csr_result:           {stats(td)}", flush=True)
        t_read = []
        for _ in range(args.runs):
            t = time.perf_counter()
            d = eng.readcoo_device(path)
            t_read.append(time.perf_counter() - t)
            d.free()
        print(f"device readcoo_device alone (file -> triplets in HBM): {stats(t_read)}", flush=True)
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            d = eng.readcoo_device(path)
            torch.cuda.synchronize()
        d.free()
        kern = copy = 0.0
        for ev in prof.events():
            us = ev.device_time
            if ev.name.startswith("Memcpy HtoD"):
                copy += us
            elif "k_" in ev.name:
                kern += us
        print(f"device readcoo_device: kernels {kern / 1e3:.2f} ms, host-to-device copies {copy / 1e3:.2f} ms (profiler, one call)",
              flush=True)
        eng.close()
        if not args.no_cli:
            exe = os.path.join(ROOT, "outerspace_b200", "osp_spgemm_cli")
            for extra in ([], ["--device-ingest"]):
                t = time.perf_counter()
                out = subprocess.run([exe, path, path, "--no-transpose"] + extra, check=True, capture_output=True, text=True).stdout
                sec = time.perf_counter() - t
                print(f"CLI {' '.join(['--no-transpose'] + extra)}: {sec:.2f} s end to end", flush=True)
                print("    " + "\n    ".join(out.strip().splitlines()), flush=True)


if __name__ == "__main__":
    main()

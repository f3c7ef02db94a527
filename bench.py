#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 outer-product SpGEMM engine (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

One "step" = one C = A*A of the named synthetic workload: HBM-resident CSR(A), CSR(B) -> HBM-resident
CSR(C) (symbolic count + multiply + [exchange] + merge), through the C ABI (include/osp_b200.h).  Every N runs
BASELINE.json configs[3] (ER 2^23, 8 nnz/row) -- on one GPU at N=1, k-sharded over the ranks with the exchange of
the partial products at N>1 -- so the 1 -> 8 curve is one workload; the N=1 line carries a `per_config` table with
configs[0], [1], [2] and [4] at full size.  Prints ONE JSON line on rank 0.  See DESIGN.md "Measurement".

The oracle (oracle/, oracle/_ref) is used here ONLY for the `cpu_baseline` object and the
`--impl reference` arm; it is never on the measured GPU path.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "spgemm_gflops"          # 2*P / t, P = sum_k nnz(A(:,k))*nnz(B(k,:))   (SimSpGEMM.cpp:884-891 counts 1*P)
UNIT = "GFLOP/s"
L2_FLUSH_BYTES = 256 << 20        # > 126 MB L2


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------
# clocks: nvidia-smi sampled DURING the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML polled from a thread every ~2 ms
    (the timed region of config 2 is a few milliseconds long), nvidia-smi at 100 ms as the fallback."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []
        self.nvml, self.handle, self.thread, self.stop_flag = None, None, None, False
        self.sm, self.reasons_seen, self.max_sm = [], 0, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
                self.reasons_seen |= int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
            except Exception:
                try:
                    self.reasons_seen |= int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                except Exception:
                    pass
            time.sleep(0.002)

    def start(self):
        if self.nvml is not None:
            self.stop_flag = False
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=1.0)
            n = self.nvml
            bits = {"hw_slowdown": getattr(n, "nvmlClocksEventReasonHwSlowdown", 0x8),
                    "hw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                    "sw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                    "sw_power_cap": getattr(n, "nvmlClocksEventReasonSwPowerCap", 0x4)}
            reasons = sorted(k for k, b in bits.items() if self.reasons_seen & int(b))
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.max_sm,
                    "samples": len(self.sm), "reasons": reasons, "source": "nvml, 2 ms period"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi -lms 100"}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline (the ONLY users of oracle/ in this file)
# ------------------------------------------------------------------------------------------------
def cpu_reference_run(a_csr, b_csr, n_k, reps: int):
    """Times the reference's own functional path on the host: TaskProvider's constructor
    (multiplyPhase + mergePhase, SimOuterSPACE.cpp:46-132) compiled unmodified into oracle/_ref, or --
    when oracle/_ref could not be built -- the oracle restatement.  Single-threaded: the reference has
    no threading (SURVEY.md 8d).  Returns (seconds per run list, kind, products)."""
    import oracle
    from outerspace_b200 import synth
    a_csc = synth.transpose_host(a_csr, n_k)
    secs = []
    prod = oracle.flops(a_csc.pos, b_csr.pos)
    if oracle.ref_available():
        for _ in range(reps):
            secs.append(oracle.ref_taskprovider(a_csc.pos, a_csc.data, b_csr.pos, b_csr.data)["seconds"])
        return secs, "reference", prod
    for _ in range(reps):
        t0 = time.perf_counter()
        oracle.spgemm(a_csc.pos, a_csc.data, b_csr.pos, b_csr.data)
        secs.append(time.perf_counter() - t0)
    return secs, "port", prod


def workload_for(n_gpus: int, name: str | None):
    """The headline workload is the same at every N (BASELINE configs[3], the one the multi-GPU metric is quoted on and
    the largest ER config that fits one GPU): the driver's 1 -> 8 curve divides like by like.  The other configs are
    in the N=1 line's `per_config` table."""
    return name or "er8m"


WORKLOAD_DESC = {
    "mlp_fc2": "configs[0]: pruned-MLP fc2 weight 1000x1000 @1%, C=A*A",
    "er16k": "configs[1]: Erdos-Renyi 16384x16384 density 1e-3, C=A*A",
    "rmat20": "configs[2]: R-MAT scale 20, edge factor 16, C=A*A",
    "er8m": "configs[3]: Erdos-Renyi 2^23 x 2^23, 8 nnz/row, C=A*A",
    "mlp_batch": "configs[4]: activation 65536x4096 (10%) x weight^T 4096x4096 (10%)",
}
# bounded CPU samples: scale_down so that one reference run takes O(1 s)
CPU_SAMPLE_SCALE = {"mlp_fc2": 1, "er16k": 1, "rmat20": 64, "er8m": 64, "mlp_batch": 2048}


def config_of(wl: str, scale_down: int) -> dict:
    """The `config` object: identical in both arms (the driver compares them key by key)."""
    return {"workload": WORKLOAD_DESC[wl], "name": wl, "scale_down": scale_down}


def run_reference(args, rank: int, world: int) -> None:
    if rank != 0:
        return
    from outerspace_b200 import synth
    wl = workload_for(args.gpus, args.workload)
    sd = CPU_SAMPLE_SCALE[wl] * args.scale_down
    a, b, dims = synth.build_workload(wl, sd)
    secs, kind, prod = cpu_reference_run(a, b, dims["n_k"], args.warmup + args.steps)
    timed = secs[args.warmup:]
    ms = 1e3 * sum(timed) / len(timed)
    value = 2.0 * prod / (ms * 1e-3) / 1e9
    sample = f"{wl} at 1/{sd} linear scale (rows={dims['rows']}, P={prod}), one TaskProvider ctor per step; GFLOP/s is a per-product " \
             f"rate, so the sample stands for the full workload" if sd > 1 \
        else f"full {wl} (rows={dims['rows']}, P={prod}), one TaskProvider ctor per step"
    line = {
        "impl": "reference", "metric": METRIC, "value": round(value, 5), "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_of(wl, args.scale_down),
        "cpu_baseline": {"value": round(value, 5), "unit": UNIT, "cores": 1, "kind": kind, "sample": sample,
                         "host_cores_available": os.cpu_count()},
        "e2e": {"value": round(value, 5), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def kernel_table(kernel_rows):
    """kernel_rows: list over steps of [(name, ms)] -> {name: (ms per step, launches per step)} sorted by time."""
    agg, cnt = {}, {}
    for rows in kernel_rows:
        for name, ms in rows:
            agg[name] = agg.get(name, 0.0) + ms
            cnt[name] = cnt.get(name, 0) + 1
    n = max(len(kernel_rows), 1)
    return {k: (agg[k] / n, cnt[k] / n) for k in sorted(agg, key=lambda k: -agg[k])}


def kernel_algorithmic_bytes(name: str, st: dict) -> tuple[int, str]:
    """Algorithmic bytes of the named kernel over ONE step (all its launches together) when it covers the whole
    workload (DESIGN.md "Kernels": from the reference's DRAM model analyzeMultiplyTask / analyzeMergeTask,
    SimOuterSPACE.cpp:176-196)."""
    P, nnz_a, nnz_b, nnz_c = st["products"], st["nnz_a"], st["nnz_b"], st["nnz_c"]
    m, n = st["rows_c"], st["n_k"]
    if "fused" in name or "chain2" in name:
        return 8 * nnz_a + 8 * nnz_b + 16 * (n + 1) + 16 * P + 8 * nnz_c + 8 * (m + 1), \
            "fused multiply+merge: what the two phases move through HBM in the reference's model, 8nnzA + 8nnzB + 16(n+1) + 16P + 8nnzC + 8(m+1)"
    if "multiply" in name:
        return 8 * nnz_a + 8 * nnz_b + 16 * (n + 1) + 8 * P, "multiply: 8nnzA + 8nnzB + 16(n+1) + 8P"
    if "merge" in name or "long_fill" in name:
        return 8 * P + 8 * nnz_c + 8 * (m + 1), "merge: 8P + 8nnzC + 8(m+1)"
    return 16 * nnz_a + 8 * (m + n + 2), "convert/symbolic: 16nnzA + 8(m+n+2)"


def roofline_of(table: dict, st: dict, peak: float, peak_src: str, wl: str) -> dict:
    """`roofline` object for the dominant kernel of a step (by summed event time)."""
    kname = next(iter(table))
    k_ms_step, k_launches = table[kname]
    k_bytes, k_formula = kernel_algorithmic_bytes(kname, st)
    total = sum(v[0] for v in table.values()) or 1.0
    per_launch = k_bytes / max(k_launches, 1.0)
    avg_launch_ms = k_ms_step / max(k_launches, 1.0)
    achieved = per_launch / (avg_launch_ms * 1e-3) / 1e9
    out = {"bound": "hbm", "kernel": kname, "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s",
           "frac": round(achieved / peak, 4), "traffic": None, "peak_source": peak_src,
           "avg_launch_ms": round(avg_launch_ms, 5), "launches_per_step": k_launches,
           "algorithmic_bytes_per_launch": int(per_launch), "formula": k_formula,
           "share_of_kernel_time": round(k_ms_step / total, 4),
           "kernel_ms_per_step": {k: round(v[0], 5) for k, v in table.items()}}
    prof = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(prof):
        try:
            with open(prof) as f:
                tr = json.load(f).get(wl, {})
            kbase = kname.strip("() ").split("<")[0]
            if kbase in tr.get("kernels", {}):
                out["traffic"] = tr["kernels"][kbase]["dram_bytes_per_launch"]
                out["traffic_source"] = tr.get("source")
        except (OSError, ValueError, KeyError, AttributeError):
            pass
    return out


def mlp_fc2_through_mtx():
    """configs[0] the way the reference gets it: the pruned layer written by scipy.io.mmwrite(csr_matrix) like
    NN_models/util.py:61-62, read back by readcoo + coo2csr (the loader path of SimSpGEMM.cpp:55-152)."""
    import tempfile

    import scipy.io
    import scipy.sparse as sp

    import outerspace_b200 as osp
    from outerspace_b200 import synth
    a0, _, dims = synth.build_workload("mlp_fc2")
    m = sp.csr_matrix((a0.data["val"], a0.data["idx"].astype(np.int64), a0.pos.astype(np.int64)), shape=(dims["rows"], dims["n_k"]))
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "fc2_weight.mtx")
        scipy.io.mmwrite(path, m)
        coo, nrow, ncol = osp.readcoo(path)
    a = osp.coo2csr(coo, nrow)
    return a, a, dict(rows=nrow, n_k=ncol, cols=ncol)


def sampled_parity(res, a, b, dims, n_rows=48, heavy=2, row_lo=0, row_hi=None, seed=7):
    """Outside every timed region: a seeded sample of rows of C (plus the heaviest) recomputed by the oracle from
    A[rows, :] and B and compared bit for bit with the engine's rows.  The oracle is the CHECKER here, never measured."""
    import oracle
    a_pos = a.pos.astype(np.int64)
    row_hi = a.NRow() if row_hi is None else row_hi
    b_len = np.diff(b.pos.astype(np.int64))
    cs = np.concatenate([[0], np.cumsum(b_len[a.data["idx"]])])
    plen = (cs[a_pos[1:]] - cs[a_pos[:-1]])[row_lo:row_hi]
    n = min(row_hi - row_lo, res.rows)
    if n <= 0:
        return {"ok": True, "rows_checked": 0, "products_checked": 0}
    rng = np.random.default_rng(seed)
    pick = np.unique(np.concatenate([rng.integers(0, n, size=n_rows), np.argsort(plen[:n])[-heavy:]])).astype(np.int64)
    sub_pos = np.zeros(len(pick) + 1, np.uint64)
    np.cumsum(a_pos[row_lo + pick + 1] - a_pos[row_lo + pick], out=sub_pos[1:])
    sub_data = np.concatenate([a.data[a_pos[row_lo + r]:a_pos[row_lo + r + 1]] for r in pick])
    w_pos, w_data, w_prod = oracle.spgemm_rowblocks(sub_pos, sub_data, b.pos, b.data, 64)
    w_pos = np.concatenate([w_pos, np.full(len(pick) + 1 - len(w_pos), w_pos[-1], np.uint64)]).astype(np.int64)
    bad = 0
    for j, r in enumerate(pick):
        got = res.rows_to_host(int(r), int(r) + 1)
        want = w_data[w_pos[j]:w_pos[j + 1]]
        if len(got.data) != len(want) or not np.array_equal(got.data.view(np.uint64), want.view(np.uint64)):
            bad += 1
    return {"ok": bad == 0, "rows_checked": int(len(pick)), "products_checked": int(w_prod), "bad_rows": bad,
            "how": "seeded sample of rows + the heaviest, engine rows vs oracle rows, bit for bit"}


DUMP_ROWS = 4096          # rows of C in the --dump-outputs sample
DUMP_ROW_CAP = 1024       # entries kept per sampled row: at most 4096 * 1024 * (8 + 4) B = 48 MiB in all


def dump_outputs(res, out_dir: str, seed: int = 0) -> None:
    """Writes a fixed, seeded sample of C (the CSR result the caller of the timed path receives) as .npy files:
    rows.npy (the sampled row ids), row_ptr.npy ([begin, end) of each sampled row in C, so the prefix sums of every row
    before it are compared too), col_idx.npy and values.npy (the first DUMP_ROW_CAP entries of each sampled row, in
    row order).  Integers are stored as float64, exact below 2^53; values keep their float32 bits."""
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(seed)
    rows = np.sort(rng.choice(res.rows, size=min(res.rows, DUMP_ROWS), replace=False)).astype(np.int64)
    pos = res.pos_to_host().astype(np.int64)
    cols, vals = [], []
    for r in rows:
        part = res.rows_to_host(int(r), int(r) + 1).data[:DUMP_ROW_CAP]
        cols.append(part["idx"])
        vals.append(part["val"])
    out = {"rows": rows.astype(np.float64),
           "row_ptr": np.stack([pos[rows], pos[rows + 1]], 1).astype(np.float64),
           "col_idx": np.concatenate(cols or [np.zeros(0, np.uint32)]).astype(np.float64),
           "values": np.concatenate(vals or [np.zeros(0, np.float32)]).astype(np.float32)}
    for name, arr in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def measure_single(eng, torch, dev, wl, scale_down, steps, warmup, flush_l2, peak, peak_src, operands=None, dump_dir=None):
    """One workload on one GPU, HBM-resident operands: device time per step (CUDA events on the engine's stream, L2
    flushed before every step), per-kernel table, sampled-row parity.  With `dump_dir`, the result of the last timed step
    is kept and sampled there (dump_outputs) once the timed steps are over.  Returns (summary dict, operands, last stats)."""
    from outerspace_b200 import api, synth
    a, b, dims = operands if operands is not None else synth.build_workload(wl, scale_down)

    def up(x):
        return torch.from_numpy(x.view(np.uint8).reshape(-1)).to(dev)
    t = [up(a.pos), up(a.data)]
    t += t if b is a else [up(b.pos), up(b.data)]          # C = A*A: both operands are the same arrays in HBM
    stream = torch.cuda.ExternalStream(eng.stream, device=dev)

    def step(flags=0, keep=False):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        res = eng.spgemm_device(a.NRow(), t[0].data_ptr(), t[1].data_ptr(), b.NRow(), t[2].data_ptr(),
                                t[3].data_ptr(), a_is_csr=True, cols_b=dims["cols"], flags=flags, a_nnz=a.nnz, b_nnz=b.nnz)
        e1.record(stream)
        e1.synchronize()
        return res, e0.elapsed_time(e1)

    for _ in range(warmup):
        flush_l2()
        res, _ = step()
        res.free()
    torch.cuda.synchronize()
    wall0 = time.perf_counter()
    ms_steps, launches, st = [], 0, None
    for i in range(steps):
        flush_l2()
        res, ms = step()
        st = res.stats()
        launches += st["kernel_launches"]
        ms_steps.append(ms)
        if dump_dir is None or i < steps - 1:
            res.free()
    torch.cuda.synchronize()
    wall = time.perf_counter() - wall0
    if dump_dir is not None:
        dump_outputs(res, dump_dir)
        res.free()
    ms_per_step = sum(ms_steps) / len(ms_steps)
    kernel_rows = []
    for _ in range(3):
        flush_l2()
        res, _ = step(api.OSP_PROFILE_KERNELS)
        kernel_rows.append(res.kernel_times())
        res.free()
    table = kernel_table(kernel_rows)
    flush_l2()
    res, _ = step()
    par = sampled_parity(res, a, b, dims)
    res.free()
    roof = roofline_of(table, st, peak, peak_src, wl)
    alg = st["algorithmic_bytes"]
    summary = {
        "name": wl, "workload": WORKLOAD_DESC[wl], "scale_down": scale_down, "steps": steps, "ms_per_step": round(ms_per_step, 5),
        "gflops": round(2.0 * st["products"] / (ms_per_step * 1e-3) / 1e9, 3), "products": st["products"], "nnz_c": st["nnz_c"],
        "rows": st["rows_c"], "row_chunks": st["row_chunks"],
        "algorithmic_gbs": round(alg / (ms_per_step * 1e-3) / 1e9, 2), "algorithmic_frac_of_hbm_peak": round(alg / (ms_per_step * 1e-3) / 1e9 / peak, 4),
        "dominant_kernel": roof["kernel"], "dominant_kernel_frac": roof["frac"], "dominant_kernel_share": roof["share_of_kernel_time"],
        "kernel_ms_per_step": roof["kernel_ms_per_step"], "parity": par,
    }
    return summary, (a, b, dims), st, dict(ms_per_step=ms_per_step, timed_steps=len(ms_steps), wall=wall, launches=launches, roofline=roof,
                                           t=t, step=step)


def run_ours(args, rank: int, world: int, local_rank: int) -> None:
    import torch
    import torch.distributed as dist

    import outerspace_b200 as osp
    from outerspace_b200 import api, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- this engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    wl = workload_for(args.gpus, args.workload)
    peak, peak_src = peaks()
    flush_buf = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)

    def flush_l2():
        flush_buf.fill_(1)
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    per_config, parity = None, None

    if world == 1:
        eng = osp.Engine(local_rank)
        sampler.start()                               # sampled through warm-up and the timed steps (>= 50 samples)
        summary, (a, b, dims), st, m = measure_single(eng, torch, dev, wl, args.scale_down, args.steps, args.warmup, flush_l2, peak, peak_src,
                                                      dump_dir=args.dump_outputs)
        clocks = sampler.stop()
        ms_per_step, timed_steps, wall, launches, roof = m["ms_per_step"], m["timed_steps"], m["wall"], m["launches"], m["roofline"]
        parity = summary["parity"]
        # ---- the outer-product (k-slice) order of north_star, same workload and timing rules, for the record ----
        ks_ms = []
        for i in range(6):
            flush_l2()
            res, ms = m["step"](api.OSP_KSLICE_ORDER)
            res.free()
            if i >= 3:
                ks_ms.append(ms)
        kslice_ms = sum(ks_ms) / len(ks_ms)
        del m

        # ---- e2e: host CSRMatrix operands (pinned) -> osp_spgemm -> host CSRMatrix result ----
        def pinned_like(x):
            buf = torch.empty(max(x.nbytes, 8), dtype=torch.uint8, pin_memory=True)
            v = buf.numpy()[: x.nbytes].view(x.dtype)
            v[...] = x
            return buf, v
        keep = [pinned_like(x) for x in ((a.pos, a.data) if b is a else (a.pos, a.data, b.pos, b.data))]
        ha = osp.CSRMatrix(keep[0][1], keep[1][1])
        hb = ha if b is a else osp.CSRMatrix(keep[2][1], keep[3][1])       # C = A*A: the caller's one host CSRMatrix is both operands
        out_pos_buf = torch.empty((st["rows_c"] + 1) * 8, dtype=torch.uint8, pin_memory=True)
        out_dat_buf = torch.empty(max(st["nnz_c"], 1) * 8, dtype=torch.uint8, pin_memory=True)
        out_pos = out_pos_buf.numpy().view(np.uint64)
        out_dat = out_dat_buf.numpy().view(osp.ELEM)
        e2e_ms = []
        n_e2e = min(args.steps, 10)
        for i in range(2 + n_e2e):
            flush_l2()
            t0 = time.perf_counter()
            res = eng.spgemm(ha, hb, a_is_csr=True, cols_b=dims["cols"])
            res.copy_into(out_pos[: res.rows + 1], out_dat[: res.nnz])
            dt = time.perf_counter() - t0
            res.free()
            if i >= 2:
                e2e_ms.append(dt * 1e3)
        e2e_ms_step = sum(e2e_ms) / len(e2e_ms)
        h2d = int(a.pos.nbytes + a.data.nbytes + (0 if b is a else b.pos.nbytes + b.data.nbytes))   # (the engine stages aliased operands once)
        d2h = int((st["rows_c"] + 1) * 8 + st["nnz_c"] * 8)
        del keep, ha, hb, out_pos, out_dat, out_pos_buf, out_dat_buf
        products = st["products"]
        alg_bytes = st["algorithmic_bytes"]
        # ---- the other BASELINE configs at full size, fewer steps: the same measurement, one entry each ----
        if not args.no_per_config and args.scale_down == 1 and args.workload is None:
            per_config = []
            for name in ("mlp_fc2", "er16k", "rmat20", "mlp_batch"):
                try:
                    ops = mlp_fc2_through_mtx() if name == "mlp_fc2" else None
                    s2, _, _, m2 = measure_single(eng, torch, dev, name, 1, 5 if name != "rmat20" else 3, 3, flush_l2, peak, peak_src, ops)
                    del m2
                    per_config.append(s2)
                except osp.OspError as e:
                    per_config.append({"name": name, "error": str(e)})
                torch.cuda.empty_cache()
        eng.close()
    else:
        from outerspace_b200 import distributed as osd
        a, b, dims = synth.build_workload(wl, args.scale_down)
        out = osd.bench_sharded(a, b, dims, args, rank, world, local_rank, flush_l2, sampler, sampled_parity)
        ms_per_step, wall, clocks, launches, st = out["ms_per_step"], out["wall"], out["clocks"], out["launches"], out["stats"]
        timed_steps = out["timed_steps"]
        roof = roofline_of(out["kernel_table"], out["rank_stats"], peak, peak_src, wl)
        roof["formula"] += " (this rank's share)"
        e2e_ms_step, h2d, d2h = out["e2e_ms"], out["h2d"], out["d2h"]
        parity = out["parity"]
        kslice_ms = None
        products, alg_bytes = st["products"], st["algorithmic_bytes"]

    if world > 1:
        tmax = torch.tensor([ms_per_step, e2e_ms_step], dtype=torch.float64, device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms_per_step, e2e_ms_step = float(tmax[0]), float(tmax[1])
        ltot = torch.tensor([launches], dtype=torch.int64, device=dev)
        dist.all_reduce(ltot)
        launches = int(ltot[0])

    if rank == 0:
        value = 2.0 * products / (ms_per_step * 1e-3) / 1e9
        e2e_value = 2.0 * products / (e2e_ms_step * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": args.steps, "timed_steps": timed_steps,
            "warmup": args.warmup, "ms_per_step": round(ms_per_step, 5), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_of(wl, args.scale_down),
            "workload_detail": {"rows": st["rows_c"], "n_k": st["n_k"], "nnz_a": st["nnz_a"], "products": products,
                                "nnz_c": st["nnz_c"], "parallelism": "single" if world == 1 else f"k-shard{world}+alltoallv",
                                "timed_region": "HBM-resident CSR(A),CSR(B) -> HBM-resident CSR(C); CUDA events on the engine stream",
                                "l2": f"L2 flushed ({L2_FLUSH_BYTES >> 20} MiB write) before every step, outside the event pair",
                                # experimental engine paths are opt-in through the environment; a line measured with one says so
                                "opt_in": {k.lower(): os.environ.get(k, "0") not in ("", "0") for k in ("OSP_LONGROW_SWEEP", "OSP_FUSED_SHORT")}},
            "algorithmic_gbs": round(alg_bytes / (ms_per_step * 1e-3) / 1e9, 2),
            "algorithmic_frac_of_hbm_peak": round(alg_bytes / (ms_per_step * 1e-3) / 1e9 / peak, 4),
            "wall_s_timed_region": round(wall, 4),
            "phases_ms_rank0": {k: round(float(st.get("ms_" + k, 0.0)), 4) for k in ("convert", "multiply", "exchange", "merge", "total")},
            "clocks": clocks,
            "gpu_launches": int(launches),
            "parity": parity,
            "e2e": {"value": round(e2e_value, 3), "unit": UNIT, "ms_per_step": round(e2e_ms_step, 4),
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "path": "host CSRMatrix (pinned) -> osp_spgemm -> osp_result_copy to host CSRMatrix"},
            "roofline": roof,
        }
        if per_config is not None:
            line["per_config"] = per_config
        if world == 1:
            line["multiply_order"] = {"default": "row order of A (automatic)", "ms_per_step": round(ms_per_step, 5),
                                      "kslice_order_ms_per_step": round(kslice_ms, 5),
                                      "note": "OSP_KSLICE_ORDER = the reference's outer-product order incl. the device CSR->CSC task list; same bits"}
        if world == 1 and not args.no_cpu_baseline:
            sd = CPU_SAMPLE_SCALE[wl] if args.scale_down == 1 else 1
            ca, cb, cdims = (a, b, dims) if sd == 1 else synth.build_workload(wl, sd * args.scale_down)
            secs, kind, cprod = cpu_reference_run(ca, cb, cdims["n_k"], 3)
            best = min(secs)
            line["cpu_baseline"] = {
                "value": round(2.0 * cprod / best / 1e9, 5), "unit": UNIT, "cores": 1, "kind": kind,
                "sample": (f"full {wl}" if sd == 1 else f"{wl} at 1/{sd} linear scale") +
                          f" (P={cprod}), TaskProvider ctor, best of 3, {best:.3f} s",
                "host_cores_available": os.cpu_count()}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=list(WORKLOAD_DESC))
    ap.add_argument("--scale-down", type=int, default=1)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-per-config", action="store_true", help="skip the per_config table of the N=1 line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a seeded sample of the last timed step's C as DIR/<name>.npy "
                         "(single-GPU engine only: not with --gpus > 1 or --impl reference)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        args.gpus = world
    if args.dump_outputs is not None and (args.impl != "ours" or world > 1):
        ap.error("--dump-outputs samples the single-GPU engine's result: use it with --impl ours on one GPU")
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()

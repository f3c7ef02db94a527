"""bench.py's reference arm runs on the CPU: check the JSON line it prints.  On a GPU: the --dump-outputs sample."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def test_reference_arm_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "spgemm_gflops" and line["unit"] == "GFLOP/s"
    assert line["higher_is_better"] is True and line["n_gpus"] == 1 and line["steps"] == 1
    assert line["value"] > 0 and line["ms_per_step"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] == 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    # both arms run the same headline workload at every N (configs[3]); the reference arm on a stated sample of it
    assert "configs[3]" in line["config"]["workload"] and line["config"]["name"] == "er8m"
    assert set(line["config"]) == {"workload", "name", "scale_down"} and line["scaling"] == "strong"
    assert "1/64" in line["cpu_baseline"]["sample"]


@pytest.mark.gpu
def test_dump_outputs_are_the_engine_result(tmp_path):
    """--steps K times K steps; --dump-outputs: a seeded sample of the last timed step's C, float32 / float64 only, at most
    64 MB, equal bit for bit to the oracle's rows of the same seeded workload.  R-MAT at 1/128: a third of the sampled rows
    are longer than DUMP_ROW_CAP, so the truncation is checked too."""
    import bench
    from outerspace_b200 import synth
    from helpers import oracle_spgemm

    dump = tmp_path / "dump"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "rmat20", "--scale-down", "128", "--steps", "2",
                          "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(dump)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["timed_steps"] == 2
    files = sorted(os.listdir(dump))
    assert files == ["col_idx.npy", "row_ptr.npy", "rows.npy", "values.npy"]
    assert sum(os.path.getsize(dump / f) for f in files) <= 64 << 20
    got = {f[:-4]: np.load(dump / f) for f in files}
    assert all(v.dtype in (np.float32, np.float64) for v in got.values())

    a, b, dims = synth.build_workload("rmat20", 128)
    want, _ = oracle_spgemm(synth.transpose_host(a, dims["n_k"]), b)
    rows = got["rows"].astype(np.int64)
    assert 0 < len(rows) < dims["rows"] and np.all(np.diff(rows) > 0)
    pos = want.pos.astype(np.int64)
    assert np.array_equal(got["row_ptr"].astype(np.int64), np.stack([pos[rows], pos[rows + 1]], 1))
    assert np.any(pos[rows + 1] - pos[rows] > bench.DUMP_ROW_CAP)
    sel = np.concatenate([np.arange(pos[r], min(pos[r + 1], pos[r] + bench.DUMP_ROW_CAP)) for r in rows])
    assert np.array_equal(got["col_idx"].astype(np.int64), want.data["idx"][sel].astype(np.int64))
    assert np.array_equal(got["values"].view(np.uint32), want.data["val"][sel].view(np.uint32))

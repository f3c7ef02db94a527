"""The C++ host shim (include/osp_b200.hpp) keeps the reference's names: it must compile with plain g++
against the C ABI and give the same COO/CSR/CSC as the Python mirror and the oracle."""
import os
import subprocess

import numpy as np
import pytest

import oracle
import outerspace_b200 as osp
from conftest import GOLDEN, ROOT, load_npz
from helpers import reference
from test_compact import _reference_compact

BIN = os.path.join(ROOT, "tests", "cpp", "shim_host_check.bin")


def _build():
    src = os.path.join(ROOT, "tests", "cpp", "shim_host_check.cpp")
    libdir = os.path.join(ROOT, "outerspace_b200")
    osp.load_library()   # raises with the build hint when the library is missing
    subprocess.run(["g++", "-O1", "-std=c++17", "-Wall", "-Werror", "-o", BIN, src, "-L" + libdir, "-losp_b200",
                    "-Wl,-rpath," + libdir, "-Wl,-rpath-link,/usr/local/cuda/lib64"], check=True)


def _parse(lines):
    pos = np.array(lines[0].split()[1:], dtype=np.uint64)
    items = lines[1].split()[1:]
    data = np.zeros(len(items), osp.ELEM)
    for i, it in enumerate(items):
        a, b = it.split(":")
        data[i] = (int(a), float.fromhex(b))
    return pos, data


@pytest.mark.parametrize("name,sym", [("loader_corner.mtx", False), ("mlp100_fc2_weight.mtx", False)])
def test_shim_loaders_match_python_mirror_and_oracle(name, sym):
    _build()
    path = os.path.join(GOLDEN, name)
    out = subprocess.run([BIN, path] + (["sym"] if sym else []), check=True, capture_output=True, text=True).stdout.splitlines()
    nrow, ncol, nnz = (int(x) for x in out[0].split())
    coo, pr, pc = osp.readcoo(path, sym)
    assert (nrow, ncol, nnz) == (pr, pc, len(coo))
    if out[1].startswith("throw"):
        with pytest.raises(osp.DuplicateEntry):
            osp.coo2csr(coo, pr)
        return
    for k, (N, tr) in enumerate(((nrow, False), (ncol, True))):
        pos, data = _parse(out[1 + 2 * k: 3 + 2 * k])
        want = osp.coo2csr(coo, N, transpose=tr)
        assert np.array_equal(pos, want.pos) and np.array_equal(data, want.data)
        rc, opos, odata = oracle.coo2csr(coo.rows, coo.cols, coo.vals, N, transpose=tr)
        assert rc == 0 and np.array_equal(pos, opos) and np.array_equal(data, odata)
    # compact forms (csr2compact / csc2rawcompact, SimSpGEMM.cpp:154-243) through the shim = the Python mirror = the reference
    csr, csc = osp.coo2csr(coo, nrow), osp.coo2csr(coo, ncol, transpose=True)
    for k, (m, fn, raw) in enumerate(((csr, osp.csr2compact, False), (csc, osp.csc2rawcompact, True))):
        cpos = np.array(out[5 + 2 * k].split()[1:], dtype=np.uint64)
        trip = [t.split(":") for t in out[6 + 2 * k].split()[1:]]
        gpos, want = fn(m)
        assert np.array_equal(cpos, gpos)
        assert [int(t[0]) for t in trip] == list(want.rows) and [int(t[1]) for t in trip] == list(want.cols)
        assert np.array_equal(np.array([float.fromhex(t[2]) for t in trip], np.float32).view(np.uint32), want.vals.view(np.uint32))
        ref = reference(f"shim_compact_{name.split('.')[0]}_{int(raw)}", lambda impl: _reference_compact(m, raw, impl))
        assert np.array_equal(gpos, ref["gpos"]) and np.array_equal(want.rows, ref["rows"]) and np.array_equal(want.cols, ref["cols"])


@pytest.mark.gpu
def test_cli_like_reference_main():
    """osp_spgemm_cli A.mtx A.mtx = the reference's command line: C = A * A^T (matrix 2 is transposed)."""
    cli = os.path.join(ROOT, "outerspace_b200", "osp_spgemm_cli")
    assert os.path.exists(cli), "build with make -C outerspace_b200/csrc"
    path = os.path.join(GOLDEN, "mlp100_fc2_weight.mtx")
    out = subprocess.run([cli, path, path], check=True, capture_output=True, text=True).stdout
    coo, nrow, ncol = osp.readcoo(path)
    csc = osp.coo2csr(coo, ncol, transpose=True)                      # CSC(A)
    coo_t = osp.COO(coo.cols, coo.rows, coo.vals)
    csr = osp.coo2csr(coo_t, ncol)                                      # CSR(A^T)
    pos, data, prod = oracle.spgemm(csc.pos, csc.data, csr.pos, csr.data)
    h = 1469598103934665603
    for b in pos.tobytes() + data.tobytes():
        h = ((h ^ b) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    assert f"mul flops ref = {prod}" in out
    assert f"C rows = {len(pos) - 1}, nnz = {len(data)}, checksum = {h:016x}" in out, out

"""GPU suite, .mtx ingest on the device (osp_readcoo_device, osp_readcoo_buffer_device, osp_coo2csr_result): the text
goes to HBM once and is parsed there into the triplets of the host loader osp_readcoo -- the same entries in the same
order with the same float bits, as raw 32-bit words -- and the triplets become a device CSR/CSC with the bytes and the
errors of the host osp_coo2csr.  tests/test_mtx_device_sim.py runs the cases that fit the CPU emulation."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import scipy.io
import scipy.sparse as sp

import outerspace_b200 as osp
from outerspace_b200 import api, synth
from helpers import assert_bit_exact, oracle_spgemm
import test_host_loaders as hl

pytestmark = pytest.mark.gpu

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
U32 = np.uint32


# ---- the host loader, the yardstick ------------------------------------------------------------------------------------
def host_readcoo(text: bytes, sym: bool):
    """osp_readcoo_buffer: (rc, COO, nrow, ncol)."""
    lib = api.load_library()
    h = ctypes.c_void_p()
    rc = lib.osp_readcoo_buffer(ctypes.c_char_p(text), ctypes.c_uint64(len(text)), ctypes.c_int(int(sym)), ctypes.byref(h))
    if rc:
        return rc, None, 0, 0
    try:
        nrow, ncol, nnz = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_uint64()
        lib.osp_coo_dims(h, ctypes.byref(nrow), ctypes.byref(ncol), ctypes.byref(nnz))
        n = nnz.value
        coo = osp.COO(np.empty(n, U32), np.empty(n, U32), np.empty(n, np.float32))
        lib.osp_coo_copy(h, api._ptr(coo.rows), api._ptr(coo.cols), api._ptr(coo.vals))
    finally:
        lib.osp_coo_free(h)
    return 0, coo, nrow.value, ncol.value


def same_triplets(dev: "osp.DeviceCOO", want, nrow, ncol, what=""):
    got = dev.to_host()
    assert (dev.nrow, dev.ncol, dev.nnz) == (nrow, ncol, len(want)), what
    assert np.array_equal(got.rows, want.rows), f"rows differ {what}"
    assert np.array_equal(got.cols, want.cols), f"cols differ {what}"
    bad = np.nonzero(got.vals.view(U32) != want.vals.view(U32))[0]
    assert bad.size == 0, f"values differ {what} at {bad[:5]}: {got.vals[bad[:5]]} vs {want.vals[bad[:5]]}"


def check_text(engine, text: bytes, sym=None, path=None):
    """Device ingest of text (from memory, and from a file when path is given) == osp_readcoo_buffer, both sym values."""
    for s in ((False, True) if sym is None else (sym,)):
        rc, want, nrow, ncol = host_readcoo(text, s)
        assert rc == 0
        dev = engine.readcoo_buffer_device(text, sym=s)
        try:
            same_triplets(dev, want, nrow, ncol, f"(buffer, sym={s})")
        finally:
            dev.free()
        if path is not None:
            with open(path, "wb") as f:
                f.write(text)
            dev = engine.readcoo_device(path, sym=s)
            try:
                same_triplets(dev, want, nrow, ncol, f"(file, sym={s})")
            finally:
                dev.free()


# ---- texts --------------------------------------------------------------------------------------------------------------
def test_fuzz_texts_match_the_host_loader(engine, tmp_path):
    """test_host_loaders' generator: comments, blank lines, tabs, pattern entries, odd values, trailing junk."""
    path = str(tmp_path / "fuzz.mtx")
    for seed in (1, 2, 3, 4):
        hl._write(path, 1500, seed)
        with open(path, "rb") as f:
            text = f.read()
        check_text(engine, text, path=str(tmp_path / "copy.mtx"))


def test_every_odd_value(engine, tmp_path):
    body = "".join(f"{i + 1} {i + 2} {v}\n" for i, v in enumerate(hl.ODD_VALUES))
    check_text(engine, ("%%MatrixMarket\n40 40 %d\n" % len(hl.ODD_VALUES) + body).encode(), path=str(tmp_path / "odd.mtx"))


def test_line_shapes(engine, tmp_path):
    cases = [
        b"",                                                      # empty text
        b"3 3 0\n",                                               # header only
        b"3 3 0",                                                 # header without '\n'
        b"%%MatrixMarket\n% only comments\n\n   \n",              # no header at all
        b"%%MatrixMarket\r\n\r\n2 2 2\r\n1 2 0.5\r\n\r\n2 1 -1.25e1\r\n",   # CRLF
        b"4 4 3\n1 1 2\n2 3 4.5\n4 4 -1",                         # last line without '\n'
        b"4 4 3\n1 1 2\n2 3 4.5\n4 4 -1\n\n\n",                   # blank lines at the end
        b"4 4 1\n\t 2\t \t3 \t 7.25 \t\n",                        # blanks around every field
        b"4 4 2\n2 3\n1 1\n",                                     # pattern entries: value 1.0
        b"4 4 2\n2 3 1.5 trailing words\n1 1 2e\n",               # junk after the value, a dangling exponent
    ]
    for i, text in enumerate(cases):
        check_text(engine, text, path=str(tmp_path / f"shape{i}.mtx"))


def test_long_comment_and_wide_lines(engine, tmp_path):
    """A 1 MB comment before the header (longer than the header reader's chunk) and in the body, lines wider than a
    parse tile (16 KB) made of blanks, a value after kilobytes of blanks."""
    big = b"%" + b"x" * (1 << 20) + b"\n"
    text = (big + b"5 5 4\n" + big + b"1 2 3.5\n" + b" " * 40000 + b"\n" + b"2" + b" " * 20000 + b"3" + b"\t" * 17000 +
            b"0.25\n" + b" " * 33000 + b"4 5 6\n" + b"5 5 " + b" " * 70000 + b"-7.5e-3\n")
    check_text(engine, text, path=str(tmp_path / "wide.mtx"))


def test_indices_at_the_edges(engine, tmp_path):
    """0 wraps to 0xFFFFFFFF as on the host; 2^32 and 2^32 + 1 wrap as well; 19 digits are plain, 20 take the slow path;
    the mirror test compares the ids before they are narrowed (1 and 2^32 + 1 are different ids)."""
    ids = [0, 1, 2, 2 ** 32 - 1, 2 ** 32, 2 ** 32 + 1, 10 ** 18 + 7, 9999999999999999999, 18446744073709551615,
           18446744073709551616, 99999999999999999999]
    lines = [f"{a} {b} 1.5" for a in ids for b in (1, ids[(ids.index(a) + 3) % len(ids)], a)]
    lines += ["1 4294967297 2.5", "4294967297 1 3.5", "00000000000000000001 2 1"]
    check_text(engine, ("9 9 9\n" + "\n".join(lines) + "\n").encode(), path=str(tmp_path / "ids.mtx"))


def test_significant_digits_and_exponents(engine, tmp_path):
    vals = ["123456789012345", "1234567890123456", "0.123456789012345", "0.1234567890123456", "9.99999999999999e22",
            "1e22", "1e-22", "1e23", "1e-23", "12345e18", "12345e-27", "1.5e+22", "2.5E-23", "0.000000000000000000001e22",
            "100000000000000000000000", "0.0000000000000000000000001", "3.4028235e38", "3.4028236e38", "1.4e-45", "7e-46"]
    body = "".join(f"{i + 1} {i + 1} {v}\n" for i, v in enumerate(vals))
    check_text(engine, (f"30 30 {len(vals)}\n" + body).encode(), path=str(tmp_path / "digits.mtx"))


def test_nul_bytes_in_lines(engine, tmp_path):
    text = b"5 5 4\n1 2 3.5\x00junk\n2\x003 1\n3 4\x00 2\n\x00\n4 4 1.25\n"
    for sym in (False, True):
        rc, want, _, _ = host_readcoo(text, sym)
        got = None
        try:
            got = engine.readcoo_buffer_device(text, sym=sym)
            assert rc == 0
        except osp.OspError as e:
            assert e.code == rc, (e.code, rc)
        if got is not None:
            got.free()
    ok = b"5 5 2\n1 2 3.5\x00junk\n4 4 1.25\x00\n"
    check_text(engine, ok, path=str(tmp_path / "nul.mtx"))


def test_no_few_and_only_slow_lines(engine, tmp_path):
    rng = np.random.default_rng(5)
    plain = [f"{rng.integers(1, 1000)} {rng.integers(1, 1000)} {rng.standard_normal():.6g}" for _ in range(3000)]
    slow = [f"+{rng.integers(1, 1000)} {rng.integers(1, 1000)} {rng.choice(hl.ODD_VALUES)}" for _ in range(3000)]
    few = list(plain)
    for k in (0, 17, 1500, 2999):
        few[k] = slow[k]
    for i, lines in enumerate((plain, few, slow)):
        check_text(engine, ("1000 1000 3000\n" + "\n".join(lines) + "\n").encode(), path=str(tmp_path / f"slow{i}.mtx"))


# ---- errors -------------------------------------------------------------------------------------------------------------
def test_garbage_line_and_missing_file(engine, tmp_path):
    good = b"3 3 2\n1 1 2.0\n2 2 3.0\n"
    for bad in (b"3 3 2\n1 1 2.0\nfoo bar\n", b"3 3 2\n1 1 2.0\n1\n", b"% c\n3 3 2\n1 1 2.0\n-\n2 2 1\nx y\n"):
        rc, _, _, _ = host_readcoo(bad, False)
        assert rc == api.OSP_ERR_INVALID
        with pytest.raises(osp.OspError) as ei:
            engine.readcoo_buffer_device(bad)
        assert ei.value.code == api.OSP_ERR_INVALID and "line " in str(ei.value)
        check_text(engine, good)                                  # the next call is exact
    assert "line 4" in str(pytest.raises(osp.OspError, engine.readcoo_buffer_device, b"% c\n3 3 2\n1 1 2.0\n-\n2 2 1\nx y\n").value)
    with pytest.raises(osp.OspError) as ei:
        engine.readcoo_device(str(tmp_path / "does_not_exist.mtx"))
    assert ei.value.code == api.OSP_ERR_IO
    check_text(engine, good)


def test_host_coo_has_no_device_pointers(engine, tmp_path):
    p = tmp_path / "a.mtx"
    p.write_bytes(b"2 2 1\n1 1 1\n")
    lib = api.load_library()
    h = ctypes.c_void_p()
    assert lib.osp_readcoo(os.fsencode(str(p)), 0, ctypes.byref(h)) == 0
    try:
        r = ctypes.c_void_p()
        assert lib.osp_coo_device(h, ctypes.byref(r), None, None) == api.OSP_ERR_INVALID
    finally:
        lib.osp_coo_free(h)


# ---- to CSR / CSC on the device -----------------------------------------------------------------------------------------
def check_to_csr(engine, text: bytes, N_rows, N_cols):
    rc, coo, _, _ = host_readcoo(text, False)
    assert rc == 0
    dev = engine.readcoo_buffer_device(text)
    try:
        for transpose, N in ((False, N_rows), (True, N_cols)):
            rc = 0
            try:
                want = osp.coo2csr(coo, N, transpose=transpose)
            except osp.OspError as e:
                rc = e.code
            if rc:
                with pytest.raises(osp.OspError) as ei:
                    dev.to_csr(N, transpose=transpose)
                assert ei.value.code == rc, (ei.value.code, rc)
                continue
            res = dev.to_csr(N, transpose=transpose)
            got = res.to_host()
            res.free()
            assert np.array_equal(got.pos, want.pos), f"pos, transpose={transpose}"
            assert got.data.tobytes() == want.data.tobytes(), f"data, transpose={transpose}"
    finally:
        dev.free()


def test_to_csr_matches_host_coo2csr(engine):
    rng = np.random.default_rng(9)
    for trial in range(4):
        n = int(rng.integers(1, 3000))
        keys = rng.choice(300 * 200, size=n, replace=False)
        lines = "".join(f"{k // 200 + 1} {k % 200 + 1} {rng.standard_normal():.9g}\n" for k in keys)
        check_to_csr(engine, f"300 200 {n}\n{lines}".encode(), 300, 200)
    # a duplicate (233) and ids beyond N (OSP_ERR_INDEX) in either orientation, index 0 (0xFFFFFFFF) as a major id
    check_to_csr(engine, b"4 4 3\n1 2 1\n3 3 2\n1 2 5\n", 4, 4)
    check_to_csr(engine, b"4 6 2\n1 6 1\n3 3 2\n", 4, 4)
    check_to_csr(engine, b"6 4 2\n6 1 1\n3 3 2\n", 4, 4)
    check_to_csr(engine, b"4 4 2\n0 1 1\n3 3 2\n", 4, 4)
    check_to_csr(engine, b"4 4 0\n", 4, 4)
    check_to_csr(engine, b"", 0, 0)


def test_mtx_to_device_operands_to_product(engine, tmp_path):
    """.mtx -> device CSC(F1) and CSR(F2^T) -> osp_spgemm(OSP_DEVICE_POINTERS) == the host pipeline, bit for bit."""
    A = sp.random(120, 90, density=0.05, random_state=1, format="coo", dtype=np.float64)
    B = sp.random(70, 90, density=0.06, random_state=2, format="coo", dtype=np.float64)
    pa, pb = str(tmp_path / "a.mtx"), str(tmp_path / "b.mtx")
    scipy.io.mmwrite(pa, A)
    scipy.io.mmwrite(pb, B)
    # host pipeline: readcoo, transpose matrix 2, coo2csr<true>(F1), coo2csr(F2^T)
    ca, nra, nca = osp.readcoo(pa)
    cb, nrb, ncb = osp.readcoo(pb)
    cbt = osp.COO(cb.cols, cb.rows, cb.vals)
    csc = osp.coo2csr(ca, nca, transpose=True)
    csr = osp.coo2csr(cbt, ncb)
    want, _ = oracle_spgemm(csc, csr)
    da, db = engine.readcoo_device(pa), engine.readcoo_device(pb)
    ra, rb = da.to_csr(nca, transpose=True), db.to_csr(ncb, transpose=True)
    try:
        assert_bit_exact(ra.to_host(), csc, "CSC(F1)")
        assert_bit_exact(rb.to_host(), csr, "CSR(F2^T)")
        pa_, da_ = ra.device_pointers()
        pb_, db_ = rb.device_pointers()
        res = engine.spgemm_device(nca, pa_, da_, ncb, pb_, db_, a_nnz=ra.nnz, b_nnz=rb.nnz)
        got = res.to_host()
        res.free()
        assert_bit_exact(got, want, ".mtx on the device -> product")
        host = engine.spgemm(csc, csr).to_host()
        assert_bit_exact(got, host, "device ingest vs host ingest")
    finally:
        for x in (ra, rb, da, db):
            x.free()


# ---- GPU only -----------------------------------------------------------------------------------------------------------
def _mmwrite_text(n_rows, nnz_per_row, seed):
    g = synth.erdos_renyi(n_rows, n_rows, n_rows * nnz_per_row, seed=seed)
    m = sp.csr_matrix((g.data["val"], g.data["idx"], g.pos.astype(np.int64)), shape=(n_rows, n_rows))
    return m


def test_large_text_matches_the_host_loader(engine, tmp_path):
    """>= 8e6 entries (more than several 32 MB upload chunks), written like scipy.io.mmwrite, plus slow lines."""
    m = _mmwrite_text(1 << 20, 8, 3)
    path = str(tmp_path / "big.mtx")
    scipy.io.mmwrite(path, m)
    assert os.path.getsize(path) > 3 * (32 << 20)
    coo, nr, nc = osp.readcoo(path)
    assert len(coo) >= 8_000_000
    dev = engine.readcoo_device(path)
    try:
        same_triplets(dev, coo, nr, nc, "(8e6 entries)")
        for transpose, N in ((True, nc), (False, nr)):
            want = osp.coo2csr(coo, N, transpose=transpose)
            res = dev.to_csr(N, transpose=transpose)
            got = res.to_host()
            res.free()
            assert np.array_equal(got.pos, want.pos) and got.data.tobytes() == want.data.tobytes()
    finally:
        dev.free()


def test_config1_through_device_ingest(engine, tmp_path):
    """Config 1 as surveyed (the pruned MLP layer written by scipy.io.mmwrite, C = A*A) through the device ingest: the
    CSR built on the device and the product equal the host loader's and the oracle's."""
    a0, _, dims = synth.build_workload("mlp_fc2")
    m = sp.csr_matrix((a0.data["val"], a0.data["idx"].astype(np.int64), a0.pos.astype(np.int64)), shape=(dims["rows"], dims["n_k"]))
    path = str(tmp_path / "fc2_weight.mtx")
    scipy.io.mmwrite(path, m)
    coo, nrow, ncol = osp.readcoo(path)
    a_csr = osp.coo2csr(coo, nrow)
    a_csc = osp.coo2csr(coo, ncol, transpose=True)
    want, _ = oracle_spgemm(a_csc, a_csr)
    dev = engine.readcoo_device(path)
    ra = dev.to_csr(nrow)
    try:
        assert_bit_exact(ra.to_host(), a_csr, "CSR(A) built on the device")
        p, d = ra.device_pointers()
        res = engine.spgemm_device(nrow, p, d, nrow, p, d, a_is_csr=True, cols_b=ncol, a_nnz=ra.nnz, b_nnz=ra.nnz)
        got = res.to_host()
        res.free()
        assert_bit_exact(got, want, "config 1 through the device ingest")
    finally:
        ra.free()
        dev.free()


def _cli_lines(args):
    exe = os.path.join(ROOT, "outerspace_b200", "osp_spgemm_cli")
    out = subprocess.run([exe] + args, check=True, capture_output=True, text=True).stdout.splitlines()
    return [l for l in out if not l.startswith("B200 TaskProvider") and not l.startswith("ingest")]


def test_cli_device_ingest_prints_the_same(tmp_path):
    A = sp.random(400, 300, density=0.03, random_state=4, format="csr", dtype=np.float64)
    B = sp.random(250, 300, density=0.03, random_state=5, format="csr", dtype=np.float64)
    pa, pb = str(tmp_path / "a.mtx"), str(tmp_path / "b.mtx")
    scipy.io.mmwrite(pa, A)
    scipy.io.mmwrite(pb, B)
    host = _cli_lines([pa, pb])
    dev = _cli_lines([pa, pb, "--device-ingest"])
    assert any(l.startswith("mul flops ref") for l in host) and any(l.startswith("C rows") for l in host)
    assert dev == host


def test_shim_program_reads_on_the_device(tmp_path):
    """A g++-compiled program over include/osp_b200.hpp: Engine::readcoo_device + DeviceCOO::coo2csr<true> equal the
    host readcoo + coo2csr<true>."""
    src = tmp_path / "shim_mtx.cpp"
    src.write_text(r'''
#include <cstdio>
#include <fstream>
#include "osp_b200.hpp"
using namespace osp_b200;
int main(int, char **argv) {
    Engine eng(0);
    size_t NRow, NCol, DR, DC;
    std::ifstream fin(argv[1]);
    COOMatrix coo = readcoo(fin, NRow, NCol, false);
    CSRMatrix want = coo2csr<true>(coo, NCol), want_r = coo2csr(coo, NRow);
    DeviceCOO dev = eng.readcoo_device(argv[1], DR, DC, false);
    CSRMatrix got = dev.coo2csr<true>(NCol), got_r = dev.coo2csr<false>(NRow);
    bool ok = DR == NRow && DC == NCol && dev.size() == coo.size() && got.pos == want.pos && got_r.pos == want_r.pos &&
              got.data.size() == want.data.size() && got_r.data.size() == want_r.data.size();
    for (size_t i = 0; ok && i < got.data.size(); i++)
        ok = got.data[i].idx == want.data[i].idx && got.data[i].val == want.data[i].val;
    for (size_t i = 0; ok && i < got_r.data.size(); i++)
        ok = got_r.data[i].idx == want_r.data[i].idx && got_r.data[i].val == want_r.data[i].val;
    std::printf("%s %zu\n", ok ? "same" : "DIFFERENT", coo.size());
    return ok ? 0 : 1;
}
''')
    exe = tmp_path / "shim_mtx"
    lib_dir = os.path.join(ROOT, "outerspace_b200")
    subprocess.run(["g++", "-O1", "-std=c++17", "-Wall", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src),
                    "-L", lib_dir, "-losp_b200", f"-Wl,-rpath,{lib_dir}", "-Wl,-rpath-link,/usr/local/cuda/lib64"], check=True)
    A = sp.random(300, 200, density=0.05, random_state=6, format="csr", dtype=np.float64)
    path = str(tmp_path / "a.mtx")
    scipy.io.mmwrite(path, A)
    out = subprocess.run([str(exe), path], check=True, capture_output=True, text=True).stdout
    assert out.startswith("same ")

"""Host .mtx ingest (rows a4-a7 of SURVEY.md section 8a): the multi-threaded in-place parser and the counting-pass
coo2csr against the unmodified reference (`oracle/_ref`: readcoo SimSpGEMM.cpp:55-100, coo2csr<> :102-152) or, when
that is not built, the oracle port (same sscanf calls) and the recorded digest of the reference's output.  Bit-exact, every thread count, every arrival order."""
import os

import numpy as np
import pytest

import oracle
import outerspace_b200 as osp
from helpers import digest, reference

IMPL = "ref" if oracle.ref_available() else "port"


def _digest_of(outputs):
    """The reference's readcoo / coo2csr outputs (up to 1.2e4 entries here) as one digest, integers widened to 64 bits."""
    return dict(digest=digest(*(np.int64(x) if isinstance(x, int) else x for x in outputs)))

ODD_VALUES = ["nan", "inf", "-inf", "0x1.8p3", "1e", "1e+", "-0", ".5", "5.", "+3.25", "1.5abc", "1..2", "1e400", "1e-400",
              "0e99999999999", "abc", "-", ".", "1.5p3", "00012.5000", "1E5", "1e-22", "1e22", "1e23", "123456789012345",
              "1234567890123456", "0.1234567890123456789", "4.9e-324", "1.7976931348623157e308", "-1.17549435e-38"]


def _value(rng):
    k = rng.integers(0, 12)
    x = rng.standard_normal() * 10.0 ** rng.integers(-30, 30)
    if k == 0:
        return ""                                                         # pattern entry: value 1.0 (SimSpGEMM.cpp:92-93)
    if k == 1:
        return str(rng.choice(ODD_VALUES))
    if k == 2:
        return "%de%d" % (rng.integers(0, 10 ** 15), rng.integers(-25, 25))
    if k == 3:
        return "0.%s%d" % ("0" * rng.integers(0, 25), rng.integers(1, 10 ** 6))
    return ["%.8g", "%.17g", "%.3e", "%.15g", "%.6f", "%.16g", "%.9g", "%.1f"][k - 4] % x


def _write(path, n, seed):
    rng = np.random.default_rng(seed)
    lines = ["%%MatrixMarket matrix coordinate real general", "% comment", "", "   ", "  % indented comment", f"  1000000 999999 {n}  "]
    for _ in range(n):
        r, c = rng.integers(1, 10 ** 6, 2)
        sep, pre, v = rng.choice([" ", "\t", "   ", " \t "]), rng.choice(["", "", " ", "\t"]), _value(rng)
        lines.append(f"{pre}{r}{sep}{c}{sep if v else ''}{v}{rng.choice(['', ' ', '  junk']) if v else ''}")
        if rng.random() < 0.01:
            lines.append("")
        if rng.random() < 0.01:
            lines.append("% mid comment")
    with open(path, "w", newline="") as f:
        f.write("\n".join(lines) + ("\n" if seed % 2 else ""))


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("sym", [False, True])
def test_readcoo_fuzz_against_reference(tmp_path, monkeypatch, seed, sym):
    path = str(tmp_path / "fuzz.mtx")
    _write(path, 6000, seed)
    rows, cols, vals, onr, onc = oracle.readcoo(path, sym=sym, impl=IMPL)
    ref = reference(f"readcoo_fuzz_{seed}_{int(sym)}", lambda impl: _digest_of(oracle.readcoo(path, sym=sym, impl=impl)))
    assert str(ref["digest"]) == digest(rows, cols, vals, np.int64(onr), np.int64(onc)), "the reference parses differently"
    for threads in ("1", "2", "7"):
        monkeypatch.setenv("OSP_HOST_THREADS", threads)
        coo, nr, nc = osp.readcoo(path, sym=sym)
        assert (nr, nc) == (onr, onc) == (1000000, 999999)
        assert np.array_equal(coo.rows, rows) and np.array_equal(coo.cols, cols), f"indices, {threads} threads"
        bad = np.nonzero(coo.vals.view(np.uint32) != vals.view(np.uint32))[0]
        assert bad.size == 0, f"{threads} threads: values differ at {bad[:5]}: {coo.vals[bad[:5]]} vs {vals[bad[:5]]}"


def test_readcoo_refuses_garbage_and_handles_crlf(tmp_path):
    p = tmp_path / "bad.mtx"
    p.write_text("3 3 2\n1 1 2.0\nfoo bar\n")
    with pytest.raises(osp.OspError):                     # the reference pushes uninitialised indices here; we refuse
        osp.readcoo(str(p))
    q = tmp_path / "crlf.mtx"
    q.write_bytes(b"%%MatrixMarket\r\n\r\n2 2 2\r\n1 2 0.5\r\n\r\n2 1 -1.25e1\r\n")
    coo, nr, nc = osp.readcoo(str(q))
    assert (nr, nc) == (2, 2) and list(coo.rows) == [0, 1] and list(coo.cols) == [1, 0] and list(coo.vals) == [0.5, -12.5]


@pytest.mark.parametrize("order", ["row_major", "col_major", "shuffled"])
def test_coo2csr_every_arrival_order(order):
    """coo2csr picks 0, 1 or 2 counting passes from the order the triplets arrive in: the result is the reference's."""
    rng = np.random.default_rng(3)
    n, m = 700, 900
    keys = np.unique(rng.integers(0, n * m, size=20000))
    rows, cols = (keys // m).astype(np.uint32), (keys % m).astype(np.uint32)
    vals = rng.standard_normal(len(keys)).astype(np.float32)
    o = {"row_major": np.arange(len(keys)), "col_major": np.lexsort((rows, cols)), "shuffled": rng.permutation(len(keys))}[order]
    coo = osp.COO(rows[o], cols[o], vals[o])
    for transpose, N in ((False, n), (True, m)):
        got = osp.coo2csr(coo, N, transpose=transpose)
        st, pos, data = oracle.coo2csr(coo.rows, coo.cols, coo.vals, N, transpose=transpose, impl=IMPL)
        ref = reference(f"coo2csr_order_{order}_{int(transpose)}",
                        lambda impl: _digest_of(oracle.coo2csr(coo.rows, coo.cols, coo.vals, N, transpose=transpose, impl=impl)))
        assert str(ref["digest"]) == digest(np.int64(st), pos, data), "the reference builds a different CSR"
        assert st == 0 and np.array_equal(got.pos, pos) and np.array_equal(got.data.view(np.uint64), data.view(np.uint64))
    dup = osp.COO(np.append(coo.rows, coo.rows[5]), np.append(coo.cols, coo.cols[5]), np.append(coo.vals, np.float32(1)))
    for transpose, N in ((False, n), (True, m)):
        with pytest.raises(osp.DuplicateEntry):           # throw(233), SimSpGEMM.cpp:49
            osp.coo2csr(dup, N, transpose=transpose)

"""Shared helpers of the parity tests (oracle = checker, engine = product)."""
import atexit
import hashlib
import os

import numpy as np
import scipy.sparse as sp

import oracle
from outerspace_b200.formats import CSRMatrix, ELEM

REF_OUTPUTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_outputs.npz")
_RECORD = os.environ.get("OSP_RECORD_REFERENCE")      # a path: the CPU suite writes the reference outputs it meets there
_recorded = {}
_stored = None


def digest(*arrays) -> str:
    """sha256 of the arrays' bytes: stands for outputs too large to store, compared bit for bit all the same."""
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def reference(key: str, live) -> dict:
    """The unmodified reference's outputs for one seeded case.  `live(impl)` computes them (a dict of arrays) with
    impl="ref", the reference compiled into oracle/_ref; without oracle/_ref they come from tests/golden/ref_outputs.npz.

    Recording (tests/golden/make_golden.py): with OSP_RECORD_REFERENCE set, every case calls live("ref") -- or, when the
    reference sources are absent, live("port"), the in-repo code these tests pinned bit for bit to the reference on the
    same inputs -- and the suite writes the results with their source when it ends."""
    global _stored
    if _RECORD:
        impl = "ref" if oracle.ref_available() else "port"
        out = live(impl)
        _recorded.update({f"{key}__{k}": np.asarray(v) for k, v in out.items()})
        _recorded["source"] = np.asarray(impl)
        return out
    if oracle.ref_available():
        return live("ref")
    if _stored is None:
        with np.load(REF_OUTPUTS) as z:
            _stored = {k: z[k] for k in z.files}
    out = {k[len(key) + 2:]: v for k, v in _stored.items() if k.startswith(key + "__")}
    assert out, f"{REF_OUTPUTS} has no outputs for {key}"
    return out


if _RECORD:
    atexit.register(lambda: np.savez_compressed(_RECORD, **_recorded))


def pack(pos, data) -> CSRMatrix:
    return CSRMatrix(np.ascontiguousarray(pos, np.uint64), np.ascontiguousarray(data, ELEM))


def rand_sparse(rng, m, n, density, ints=False):
    mask = rng.random((m, n)) < density
    if ints:
        v = rng.integers(1, 9, size=(m, n)).astype(np.float32)
    else:
        v = (rng.standard_normal((m, n)) * 3).astype(np.float32)
        v[v == 0] = 1
    return sp.csr_matrix(np.where(mask, v, 0).astype(np.float32))


def operands(A, B):
    """scipy A, B -> (CSC(A), CSR(A), CSR(B)) in reference layout."""
    return CSRMatrix.from_scipy(sp.csc_matrix(A)), CSRMatrix.from_scipy(sp.csr_matrix(A)), CSRMatrix.from_scipy(sp.csr_matrix(B))


def oracle_spgemm(a_csc: CSRMatrix, b_csr: CSRMatrix, rows_override=0):
    pos, data, prod = oracle.spgemm(a_csc.pos, a_csc.data, b_csr.pos, b_csr.data, rows_override)
    return pack(pos, data), prod


def assert_bit_exact(got: CSRMatrix, want: CSRMatrix, what=""):
    assert got.pos.shape == want.pos.shape, f"{what}: rows {got.pos.shape} vs {want.pos.shape}"
    assert np.array_equal(got.pos, want.pos), f"{what}: row_ptr differs"
    assert np.array_equal(got.data["idx"], want.data["idx"]), f"{what}: col_idx differs"
    gv, wv = got.data["val"].view(np.uint32), want.data["val"].view(np.uint32)
    bad = np.nonzero(gv != wv)[0]
    assert bad.size == 0, f"{what}: {bad.size} values differ bitwise, first at {bad[:5]}: " \
                          f"{got.data['val'][bad[:5]]} vs {want.data['val'][bad[:5]]}"


def check_csr_invariants(c: CSRMatrix, cols: int):
    """Size-independent structural properties (SURVEY.md section 4 iii)."""
    pos = c.pos.astype(np.int64)
    assert pos[0] == 0 and pos[-1] == c.nnz
    assert np.all(np.diff(pos) >= 0), "row_ptr not monotone"
    idx = c.data["idx"].astype(np.int64)
    if c.nnz:
        assert idx.max() < cols
        d = np.diff(idx)
        starts = pos[1:-1][(pos[1:-1] > 0) & (pos[1:-1] < c.nnz)]
        interior = np.ones(c.nnz - 1, bool)
        interior[starts - 1] = False          # positions that straddle a row boundary
        assert np.all(d[interior] > 0), "columns not strictly ascending inside a row"

"""CPU suite: the oracle restatement against the committed golden fixtures (generated from the
unmodified reference by tests/golden/make_golden.py) and against the reference's outputs on seeded
inputs: the compiled reference itself when oracle/_ref is present, else their record (helpers.reference)."""
import os

import numpy as np
import pytest
import scipy.sparse as sp

import oracle
from conftest import GOLDEN, load_npz
from helpers import operands, pack, rand_sparse, reference

CASES = ["ex3x3", "rand_dups", "empty_slices", "long_row", "mlp_like_int"]


@pytest.mark.parametrize("name", CASES)
def test_port_matches_golden(name):
    g = load_npz(name)
    pos, data, prod = oracle.spgemm(g["a_csc_pos"], g["a_csc_data"], g["b_csr_pos"], g["b_csr_data"])
    assert prod == int(g["products"])
    assert np.array_equal(pos, g["c_pos"])
    assert np.array_equal(data["idx"], g["c_data"]["idx"])
    assert np.array_equal(data["val"].view(np.uint32), g["c_data"]["val"].view(np.uint32))
    # the bounded-memory variant used for the CPU baseline gives the same bits
    pos2, data2, prod2 = oracle.spgemm_rowblocks(g["a_csr_pos"], g["a_csr_data"], g["b_csr_pos"], g["b_csr_data"], 5)
    assert prod2 == prod and np.array_equal(pos2, pos) and np.array_equal(data2, data)
    assert oracle.flops(g["a_csc_pos"], g["b_csr_pos"]) == prod


def test_3x3_known_answer():
    """SURVEY.md 8a: intended rows of C = A*A for A=[[1,2,0],[0,3,4],[5,0,6]]."""
    g = load_npz("ex3x3")
    assert list(g["c_pos"]) == [0, 3, 6, 9]
    assert [(int(i), float(v)) for i, v in g["c_data"]] == [
        (0, 1.0), (1, 8.0), (2, 8.0), (0, 20.0), (1, 9.0), (2, 36.0), (0, 35.0), (1, 10.0), (2, 36.0)]
    # and the as-written (buggy) TaskProvider output the survey observed
    assert [(int(i), float(v)) for i, v in g["tp_data"]] == [
        (0, 1.0), (0, 8.0), (1, 8.0), (0, 9.0), (0, 32.0), (1, 24.0), (0, 5.0), (0, 40.0), (1, 36.0)]


def test_csr2csc_port_matches_golden():
    for name in CASES:
        g = load_npz(name)
        n_minor = len(g["a_csc_pos"]) - 1
        pos, data = oracle.csr2csc(len(g["a_csr_pos"]) - 1, n_minor, g["a_csr_pos"], g["a_csr_data"])
        assert np.array_equal(pos, g["a_csc_pos"]) and np.array_equal(data, g["a_csc_data"])


def test_loader_golden():
    g = load_npz("mlp100")
    rows, cols, vals, nrow, ncol = oracle.readcoo(os.path.join(GOLDEN, "mlp100_fc2_weight.mtx"))
    assert (nrow, ncol) == (int(g["nrow"]), int(g["ncol"]))
    assert np.array_equal(rows, g["rows"]) and np.array_equal(cols, g["cols"])
    assert np.array_equal(vals.view(np.uint32), g["vals"].view(np.uint32))
    rc, pos, data = oracle.coo2csr(rows, cols, vals, ncol, transpose=True)
    assert rc == 0 and np.array_equal(pos, g["csc_pos"]) and np.array_equal(data, g["csc_data"])
    rc, pos, data = oracle.coo2csr(rows, cols, vals, nrow)
    assert rc == 0 and np.array_equal(pos, g["csr_pos"]) and np.array_equal(data, g["csr_data"])
    for sym in (0, 1):
        g = load_npz(f"loader_corner_sym{sym}")
        rows, cols, vals, nrow, ncol = oracle.readcoo(os.path.join(GOLDEN, "loader_corner.mtx"), sym=bool(sym))
        assert (nrow, ncol) == (5, 4)
        assert np.array_equal(rows, g["rows"]) and np.array_equal(cols, g["cols"])
        assert np.array_equal(vals.view(np.uint32), g["vals"].view(np.uint32))
    # pattern entry defaults to 1.0, "-0" keeps its sign bit
    g = load_npz("loader_corner_sym0")
    assert g["vals"][1] == 1.0 and np.signbit(g["vals"][-1])


def test_duplicates_raise_233():
    rc, _, _ = oracle.coo2csr([0, 1, 1], [2, 3, 3], [1.0, 2.0, 3.0], 4)
    assert rc == 233
    rc, _, _ = oracle.coo2csr([0, 1, 1], [2, 3, 3], [1.0, 2.0, 3.0], 4, transpose=True)
    assert rc == 233


def task_sizes(a_csc, b_csr, rows_c):
    """The intended task lists: (nnz(A(:,k)), nnz(B(k,:))) of every k with both non-empty, and the ways (partial-product
    lists) of every output row.  Equal to the reference's TaskProvider on every golden case (tp_mult_sizes,
    tp_merge_ways[:, 0]); stands in for it when its outputs are recorded without the reference sources."""
    ap, bp = a_csc.pos.astype(np.int64), b_csr.pos.astype(np.int64)
    nnzc, nnzr = np.diff(ap), np.diff(bp)
    keep = (nnzc > 0) & (nnzr > 0)
    rows_of_a = a_csc.data["idx"].astype(np.int64)
    ways = np.bincount(rows_of_a[np.repeat(nnzr > 0, nnzc)], minlength=rows_c)[:rows_c]
    return np.stack([nnzc[keep], nnzr[keep]], 1).astype(np.uint32), ways.astype(np.uint32)


def _reference_product(a_csc, b_csr, pos, data, impl):
    """cscMulcsr (folded), compareCOO on the restatement's result and the TaskProvider's multiply tasks and row count."""
    if impl == "ref":
        rpos, rdata, rprod, _ = oracle.spgemm(a_csc.pos, a_csc.data, b_csr.pos, b_csr.data, impl="ref")
        tp = oracle.ref_taskprovider(a_csc.pos, a_csc.data, b_csr.pos, b_csr.data)
        return dict(pos=rpos, data=rdata, products=np.uint64(rprod), compare=oracle.ref_compare(pos, data, rpos, rdata),
                    mult_sizes=tp["mult_sizes"], tp_rows=np.uint64(len(tp["pos"])))
    rpos, rdata, rprod = oracle.spgemm(a_csc.pos, a_csc.data, b_csr.pos, b_csr.data)
    return dict(pos=rpos, data=rdata, products=np.uint64(rprod), compare=np.array_equal(pos, rpos) and np.array_equal(data, rdata),
                mult_sizes=task_sizes(a_csc, b_csr, len(rpos) - 1)[0], tp_rows=np.uint64(len(rpos)))


@pytest.mark.parametrize("seed", range(6))
def test_port_matches_compiled_reference(seed):
    rng = np.random.default_rng(1000 + seed)
    m, k, n = rng.integers(1, 80, size=3)
    A, B = rand_sparse(rng, m, k, rng.uniform(0.02, 0.5)), rand_sparse(rng, k, n, rng.uniform(0.02, 0.5))
    a_csc, a_csr, b_csr = operands(A, B)
    if a_csc.nnz == 0:
        pytest.skip("empty A")
    pos, data, prod = oracle.spgemm(a_csc.pos, a_csc.data, b_csr.pos, b_csr.data)
    ref = reference(f"spgemm_seed{seed}", lambda impl: _reference_product(a_csc, b_csr, pos, data, impl))
    rpos, rdata = ref["pos"], ref["data"]
    assert prod == int(ref["products"]) and np.array_equal(pos, rpos) and np.array_equal(data["idx"], rdata["idx"])
    assert np.array_equal(data["val"].view(np.uint32), rdata["val"].view(np.uint32))
    # the reference's own comparator accepts it too
    assert bool(ref["compare"])
    # task-size lists of the as-written TaskProvider are structural and must match the intended semantics
    nnzc = np.diff(a_csc.pos.astype(np.int64)); nnzr = np.diff(b_csr.pos.astype(np.int64))
    keep = (nnzc > 0) & (nnzr > 0)
    assert np.array_equal(ref["mult_sizes"], np.stack([nnzc[keep], nnzr[keep]], 1).astype(np.uint32))
    assert int(ref["tp_rows"]) == len(pos)          # same number of output rows: maxRowId + 1


def test_task_sizes_match_the_golden_taskprovider():
    """task_sizes (the stand-in used when recording without the reference) against the reference's stored TaskProvider."""
    for name in CASES:
        g = load_npz(name)
        mult, ways = task_sizes(pack(g["a_csc_pos"], g["a_csc_data"]), pack(g["b_csr_pos"], g["b_csr_data"]), len(g["tp_pos"]) - 1)
        assert np.array_equal(mult, g["tp_mult_sizes"]) and np.array_equal(ways, g["tp_merge_ways"][:, 0]), name


def test_coo2csr_matches_compiled_reference():
    rng = np.random.default_rng(7)
    for it in range(5):
        m, n = rng.integers(2, 60, size=2)
        A = rand_sparse(rng, m, n, 0.3).tocoo()
        perm = rng.permutation(A.nnz)
        rows, cols, vals = A.row[perm].astype(np.uint32), A.col[perm].astype(np.uint32), A.data[perm]
        if len(np.unique(rows)) < 2 or len(np.unique(cols)) < 2:
            continue                               # the reference's single-slice corner, tested in make_golden
        for tr, N in ((False, m), (True, n)):
            rc, pos, data = oracle.coo2csr(rows, cols, vals, N, transpose=tr)
            ref = reference(f"coo2csr_{it}_{int(tr)}", lambda impl: dict(zip(
                ("rc", "pos", "data"), oracle.coo2csr(rows, cols, vals, N, transpose=tr, impl=impl))))
            assert rc == int(ref["rc"]) == 0 and np.array_equal(pos, ref["pos"]) and np.array_equal(data, ref["data"])


def test_scipy_cross_check():
    """Independent check of the structure and (to tolerance) the values."""
    rng = np.random.default_rng(3)
    A, B = rand_sparse(rng, 50, 40, 0.2), rand_sparse(rng, 40, 30, 0.2)
    a_csc, _, b_csr = operands(A, B)
    pos, data, _ = oracle.spgemm(a_csc.pos, a_csc.data, b_csr.pos, b_csr.data, rows_override=50)
    C = (A @ B).tocsr(); C.sort_indices()
    assert np.array_equal(pos, C.indptr) and np.array_equal(data["idx"], C.indices)
    assert np.allclose(data["val"], C.data, rtol=1e-5, atol=1e-5)

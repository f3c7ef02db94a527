"""Compact COO (SURVEY.md 8a row a16): csr2compact / csc2rawcompact (SimSpGEMM.cpp:154-243) against the unmodified
reference functions compiled into oracle/_ref (else their recorded outputs), and the engine's product from a compact operand against the
reference's compactMulcsr (SimSpGEMM.cpp:247-263) with its partial products folded in group order.

The format conversions are host code in the reference and host code here (C ABI: osp_csr2compact,
osp_csc2rawcompact); the product is the GPU engine (tests/test_gpu_zzy_compact.py) -- the same test body runs on the
emulated engine in the CPU suite (tests/test_engine_sim.py)."""
import numpy as np
import pytest
import scipy.sparse as sp

import oracle
import outerspace_b200 as osp
from outerspace_b200 import api
from outerspace_b200.formats import COO, CSRMatrix
from helpers import assert_bit_exact, digest, operands, oracle_spgemm, rand_sparse, reference


def _cases():
    rng = np.random.default_rng(5)
    yield "random", rand_sparse(rng, 30, 40, 0.2)
    yield "ragged", sp.csr_matrix(np.triu(rng.standard_normal((25, 25)).astype(np.float32)))      # lengths 25, 24, ..., 1
    m = rand_sparse(rng, 20, 15, 0.3).tolil()
    m[0, :] = 0; m[7, :] = 0; m[19, :] = 0                                                          # empty first / middle / last slice
    yield "empty slices", sp.csr_matrix(m)
    yield "one element", sp.csr_matrix(([2.5], ([3], [1])), shape=(6, 4), dtype=np.float32)
    yield "one dense row", sp.csr_matrix(np.vstack([np.zeros((2, 9), np.float32), np.arange(1, 10, dtype=np.float32)[None, :]]))
    yield "explicit zeros", sp.csr_matrix((np.array([0.0, -0.0, 1.0], np.float32), np.array([0, 2, 1]), np.array([0, 2, 3])), shape=(2, 3))


def _reference_compact(m, raw, impl):
    """csr2compact / csc2rawcompact of the reference (impl="ref"); the C ABI's, which these tests pinned to it, otherwise."""
    if impl == "ref":
        gpos, rows, cols, vals = oracle.ref_compact(m.pos, m.data, raw=raw)
    else:
        gpos, coo = (osp.csc2rawcompact if raw else osp.csr2compact)(m)
        rows, cols, vals = coo.rows, coo.cols, coo.vals
    return dict(gpos=gpos, rows=rows, cols=cols, vals=vals)


@pytest.mark.parametrize("name,A", list(_cases()))
def test_csr2compact_and_csc2rawcompact_match_the_reference(name, A):
    for form, m in (("csr", CSRMatrix.from_scipy(sp.csr_matrix(A))), ("csc", CSRMatrix.from_scipy(sp.csc_matrix(A)))):
        for raw, fn in ((False, osp.csr2compact), (True, osp.csc2rawcompact)):
            gpos, coo = fn(m)
            ref = reference(f"compact_{name.replace(' ', '_')}_{form}_{int(raw)}", lambda impl: _reference_compact(m, raw, impl))
            assert np.array_equal(gpos, ref["gpos"]), name
            assert np.array_equal(coo.rows, ref["rows"]) and np.array_equal(coo.cols, ref["cols"]), name
            assert np.array_equal(coo.vals.view(np.uint32), ref["vals"].view(np.uint32)), name


def test_compact_of_an_empty_matrix():
    """No non-zero at all: zero groups.  (The reference indexes statNNZR[-1] there -- undefined behaviour -- so this
    corner is defined here and not compared.)"""
    m = CSRMatrix(np.zeros(5, np.uint64), np.zeros(0, api.ELEM))
    gpos, coo = osp.csr2compact(m)
    assert list(gpos) == [0] and len(coo) == 0
    gpos, coo = osp.csc2rawcompact(m)
    assert list(gpos) == [0] * 5 and len(coo) == 0


def test_compact_is_a_permutation_grouped_by_rank():
    """Structure, independent of the reference: group j = the (j+1)-th non-zero of every slice, slices ascending."""
    rng = np.random.default_rng(9)
    m = CSRMatrix.from_scipy(rand_sparse(rng, 50, 60, 0.15))
    gpos, coo = osp.csr2compact(m)
    lens = np.diff(m.pos.astype(np.int64))
    assert len(gpos) - 1 == lens.max() and gpos[-1] == m.nnz
    for j in range(len(gpos) - 1):
        rows = coo.rows[int(gpos[j]):int(gpos[j + 1])]
        want_rows = np.nonzero(lens > j)[0]
        assert np.array_equal(rows, want_rows)
        src = m.data[(m.pos[want_rows].astype(np.int64) + j)]
        assert np.array_equal(coo.cols[int(gpos[j]):int(gpos[j + 1])], src["idx"])
        assert np.array_equal(coo.vals[int(gpos[j]):int(gpos[j + 1])].view(np.uint32), src["val"].view(np.uint32))


def _reference_compact_product(gpos, coo, a_csc, b_csr, impl):
    """compactMulcsr of the reference, its partial products folded (impl="ref"); the oracle's cscMulcsr + fold, which gives
    the same bits on these inputs, otherwise.  Stored as a digest: the larger products hold ~2e5 entries."""
    if impl == "ref":
        pos, data, prod = oracle.ref_compact_spgemm(gpos, coo.rows, coo.cols, coo.vals, b_csr.pos, b_csr.data)
    else:
        c, prod = oracle_spgemm(a_csc, b_csr)
        pos, data = c.pos, c.data
    return dict(products=np.uint64(prod), digest=digest(np.asarray(pos, np.uint64), np.asarray(data, api.ELEM)))


def compact_product_check(engine):
    """compactMulcsr: A as compact COO (csr2compact of CSR(A)) times CSR(B).  The engine ingests the triplets on the
    device (coo2csr + dupcheck) and multiplies; the reference's compactMulcsr output, folded, must agree bit for bit --
    and so must the plain product from CSC(A)."""
    rng = np.random.default_rng(12)
    for m, k, n, da, db in ((40, 30, 50, 0.2, 0.2), (64, 64, 3000, 0.3, 0.05), (5, 200, 40000, 0.9, 0.02)):
        A, B = rand_sparse(rng, m, k, da), rand_sparse(rng, k, n, db)
        a_csc, a_csr, b_csr = operands(A, B)
        gpos, coo = osp.csr2compact(a_csr)
        a_back = engine.coo2csr(coo, a_csr.NRow(), n_other=k)            # the compact operand is a triplet list
        assert np.array_equal(a_back.pos, a_csr.pos) and np.array_equal(a_back.data, a_csr.data)
        res = engine.spgemm(a_back, b_csr, a_is_csr=True, cols_b=n)
        got = res.to_host(); st = res.stats(); res.free()
        want, prod = oracle_spgemm(a_csc, b_csr)
        assert st["products"] == prod
        assert_bit_exact(got, want, "compact operand vs cscMulcsr + dedup")
        ref = reference(f"compact_product_{m}x{k}x{n}", lambda impl: _reference_compact_product(gpos, coo, a_csc, b_csr, impl))
        assert int(ref["products"]) == prod
        assert digest(got.pos, got.data) == str(ref["digest"]), "compact operand vs the reference's compactMulcsr"
    # a compact operand with a repeated (row, col): compactMulcsr's dupcheck throws 233, so does the ingest
    dup = COO(np.array([0, 1, 1], np.uint32), np.array([2, 3, 3], np.uint32), np.ones(3, np.float32))
    with pytest.raises(osp.DuplicateEntry):
        engine.coo2csr(dup, 2, n_other=4)

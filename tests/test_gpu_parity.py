"""GPU suite: the CUDA path (through the C ABI) against the oracle -- bit-exact row_ptr, col_idx AND
values (the engine's merge is the deterministic k-ordered one).  Sizes here finish in seconds on the
oracle; full-size configs are covered by the property tests in test_gpu_zz_fullsize.py."""
import os

import numpy as np
import pytest
import scipy.sparse as sp

import oracle
import outerspace_b200 as osp
from outerspace_b200 import api, synth
from conftest import GOLDEN, load_npz
from helpers import assert_bit_exact, check_csr_invariants, operands, oracle_spgemm, pack, rand_sparse, reference

pytestmark = pytest.mark.gpu

CASES = ["ex3x3", "rand_dups", "empty_slices", "long_row", "mlp_like_int"]


@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("a_is_csr", [False, True])
def test_golden(engine, name, a_is_csr):
    g = load_npz(name)
    b = pack(g["b_csr_pos"], g["b_csr_data"])
    a = pack(g["a_csr_pos"], g["a_csr_data"]) if a_is_csr else pack(g["a_csc_pos"], g["a_csc_data"])
    res = engine.spgemm(a, b, a_is_csr=a_is_csr)
    got = res.to_host()
    st = res.stats()
    res.free()
    assert_bit_exact(got, pack(g["c_pos"], g["c_data"]), name)
    assert st["products"] == int(g["products"]) and st["nnz_c"] == len(g["c_data"])
    assert st["kernel_launches"] > 0


def test_mtx_pipeline_like_reference_main(engine):
    """readcoo -> coo2csr<true>/coo2csr -> TaskProvider, the call sequence of SimSpGEMM.cpp:844-893
    (with A*A instead of F1*F2^T)."""
    g = load_npz("mlp100")
    coo, nrow, ncol = osp.readcoo(os.path.join(GOLDEN, "mlp100_fc2_weight.mtx"))
    csc = osp.coo2csr(coo, ncol, transpose=True)
    csr = osp.coo2csr(coo, nrow)
    provider = osp.TaskProvider(csc, csr, engine=engine)
    assert_bit_exact(provider.mergedResult, pack(g["c_pos"], g["c_data"]), "mlp100")
    nnzc, nnzr = np.diff(csc.pos.astype(np.int64)), np.diff(csr.pos.astype(np.int64))
    keep = (nnzc > 0) & (nnzr > 0)
    assert np.array_equal(provider.getMultiplyTasks(), np.stack([nnzc[keep], nnzr[keep]], 1).astype(np.uint32))
    merge = provider.getMergeTasks()
    assert merge.shape[0] == provider.mergedResult.NRow()
    assert np.array_equal(merge[:, 1], np.diff(provider.mergedResult.pos.astype(np.int64)).astype(np.uint32))


def test_config1_as_surveyed_through_mtx(engine, tmp_path):
    """BASELINE configs[0] as SURVEY.md 8d describes it: a 1000 x 1000 layer pruned to 1 % density, written by
    scipy.io.mmwrite(csr_matrix) exactly like NN_models/util.py:61-62, read back by readcoo (SimSpGEMM.cpp:55-100),
    turned into CSC(A) / CSR(A) by coo2csr (:102-152), multiplied as A*A on the GPU, compared with the oracle."""
    import scipy.io
    a0, _, dims = synth.build_workload("mlp_fc2")
    dense = sp.csr_matrix((a0.data["val"], a0.data["idx"].astype(np.int64), a0.pos.astype(np.int64)), shape=(1000, 1000))
    path = str(tmp_path / "fc2_weight.mtx")
    scipy.io.mmwrite(path, dense)
    coo, nrow, ncol = osp.readcoo(path)
    assert (nrow, ncol) == (1000, 1000) and len(coo.rows) == 10000
    csc = osp.coo2csr(coo, ncol, transpose=True)
    csr = osp.coo2csr(coo, nrow)
    want, prod = oracle_spgemm(csc, csr)
    assert 5e4 < prod < 2e5                                   # SURVEY 8: P ~ 1e5
    for a, is_csr in ((csc, False), (csr, True)):
        res = engine.spgemm(a, csr, a_is_csr=is_csr)
        got = res.to_host()
        assert res.stats()["products"] == prod
        res.free()
        assert_bit_exact(got, want, f"config 1 through .mtx, a_is_csr={is_csr}")
        check_csr_invariants(got, 1000)
    provider = osp.TaskProvider(csc, csr, engine=engine)       # the reference's own entry point (SimOuterSPACE.cpp:859-860)
    assert_bit_exact(provider.mergedResult, want, "config 1 TaskProvider")


@pytest.mark.parametrize("seed", range(8))
def test_random_vs_oracle(engine, seed):
    rng = np.random.default_rng(seed)
    m, k, n = (int(x) for x in rng.integers(1, 300, size=3))
    A, B = rand_sparse(rng, m, k, rng.uniform(0.01, 0.3)), rand_sparse(rng, k, n, rng.uniform(0.01, 0.3))
    a_csc, a_csr, b_csr = operands(A, B)
    want, prod = oracle_spgemm(a_csc, b_csr)
    for a, is_csr, flags in ((a_csc, False, 0), (a_csr, True, 0), (a_csr, True, api.OSP_ROWWISE_ORDER),
                             (a_csr, True, api.OSP_KSLICE_ORDER)):
        res = engine.spgemm(a, b_csr, a_is_csr=is_csr, flags=flags)
        got = res.to_host()
        assert res.stats()["products"] == prod
        res.free()
        assert_bit_exact(got, want, f"seed {seed} csr={is_csr} flags={flags}")
        check_csr_invariants(got, n)


def test_task_sizes_match_reference_structure(engine):
    """The sizes the untouched timing models consume equal those of the reference's TaskProvider: its outputs stored with
    the golden cases (tests/golden/make_golden.py) and on a fresh seeded product (oracle/_ref, else their record)."""
    for name in CASES:
        g = load_npz(name)
        provider = osp.TaskProvider(pack(g["a_csc_pos"], g["a_csc_data"]), pack(g["b_csr_pos"], g["b_csr_data"]), engine=engine)
        assert np.array_equal(provider.getMultiplyTasks(), g["tp_mult_sizes"]), name
        assert np.array_equal(provider.getMergeTasks()[:, 0], g["tp_merge_ways"][:, 0]), name     # ways per output row
    rng = np.random.default_rng(5)
    A, B = rand_sparse(rng, 60, 50, 0.1), rand_sparse(rng, 50, 70, 0.1)
    a_csc, _, b_csr = operands(A, B)
    ref = reference("taskprovider_seed5", lambda impl: _reference_task_sizes(a_csc, b_csr, impl))
    provider = osp.TaskProvider(a_csc, b_csr, engine=engine)
    assert np.array_equal(provider.getMultiplyTasks(), ref["mult_sizes"])
    assert np.array_equal(provider.getMergeTasks()[:, 0], ref["merge_ways"])     # ways per output row


def _reference_task_sizes(a_csc, b_csr, impl):
    if impl == "ref":
        tp = oracle.ref_taskprovider(a_csc.pos, a_csc.data, b_csr.pos, b_csr.data)
        return dict(mult_sizes=tp["mult_sizes"], merge_ways=tp["merge_ways"][:, 0])
    from test_oracle_golden import task_sizes
    mult, ways = task_sizes(a_csc, b_csr, len(oracle_spgemm(a_csc, b_csr)[0].pos) - 1)
    return dict(mult_sizes=mult, merge_ways=ways)


def test_er_config2_scaled(engine):
    """config 2 shape at 1/4 linear scale (ER, density 1e-3): uniform short rows."""
    a, b, dims = synth.build_workload("er16k", scale_down=4)
    a_csc = synth.transpose_host(a, dims["n_k"])
    want, prod = oracle_spgemm(a_csc, b)
    res = engine.spgemm(a, b, a_is_csr=True, cols_b=dims["cols"])
    got = res.to_host(); res.free()
    assert_bit_exact(got, want, "er16k/4")


def test_rmat_small(engine):
    """config 3 shape at scale 12: skewed rows incl. rows beyond the shared-memory sort capacity."""
    a, b, dims = synth.build_workload("rmat20", scale_down=256)
    a_csc = synth.transpose_host(a, dims["n_k"])
    want, prod = oracle_spgemm(a_csc, b)
    res = engine.spgemm(a, b, a_is_csr=True)
    got = res.to_host(); st = res.stats(); res.free()
    assert st["rows_long"] > 0, "test should exercise the long-row path"
    assert_bit_exact(got, want, "rmat12")
    res = engine.spgemm(a_csc, b, a_is_csr=False)
    got = res.to_host(); res.free()
    assert_bit_exact(got, want, "rmat12 from CSC")


def test_mlp_batch_small(engine):
    """config 5 shape with a small batch: every output row is long and compresses ~40x."""
    rng = np.random.default_rng(9)
    x = synth.pruned_dense(48, 1024, 0.10, seed=1, nonneg=True)
    w = synth.pruned_dense(1024, 1024, 0.10, seed=2)
    wt = synth.transpose_host(w, 1024)
    x_csc = synth.transpose_host(x, 1024)
    want, prod = oracle_spgemm(x_csc, wt)
    for flags in (0, api.OSP_NO_FUSED_DENSE):          # fused dense rows (no bins) and multiply -> bins -> k_merge_dense
        res = engine.spgemm(x, wt, a_is_csr=True, cols_b=1024, flags=flags)
        got = res.to_host(); res.free()
        assert_bit_exact(got, want, f"mlp batch 48 flags={flags}")
    # rows with no non-zero, a column range that is not a multiple of the band width, negative zeros
    x2 = synth.pruned_dense(70, 1000, 0.15, seed=3)
    x2.data["val"][::7] *= -1.0
    w2 = synth.pruned_dense(1000, 999, 0.12, seed=4)
    b2 = w2                                     # B = w2: 1000 x 999
    want2, _ = oracle_spgemm(synth.transpose_host(x2, 1000), b2)
    for flags in (0, api.OSP_NO_FUSED_DENSE):
        res = engine.spgemm(x2, b2, a_is_csr=True, cols_b=999, flags=flags)
        got = res.to_host(); st = res.stats(); res.free()
        assert_bit_exact(got, want2, f"fused dense 70x1000x999 flags={flags}")


def _csr_from_rows(rows, n_cols, rng, explicit_zero_every=0):
    """rows: list of sorted column lists -> CSRMatrix with N(0,3) values (optionally explicit +-0.0 entries)."""
    pos = np.zeros(len(rows) + 1, dtype=np.uint64)
    pos[1:] = np.cumsum([len(r) for r in rows])
    idx = np.array([c for r in rows for c in r], dtype=np.uint32)
    assert idx.size == 0 or idx.max() < n_cols
    val = (rng.standard_normal(idx.size) * 3).astype(np.float32)
    if explicit_zero_every:
        val[::explicit_zero_every] = 0.0
        val[1::2 * explicit_zero_every] = -0.0
    return osp.CSRMatrix.from_arrays(pos, idx, val)


def _row_partials(a, b):
    blen = np.diff(b.pos.astype(np.int64))
    per_elem = blen[a.data["idx"]]
    return np.add.reduceat(np.concatenate([per_elem, [0]]), np.minimum(a.pos[:-1].astype(np.int64), per_elem.size)) * (np.diff(a.pos.astype(np.int64)) > 0)


@pytest.mark.parametrize("cols,mode,direct", [(1024, "2", "1"), (999, "2", "1"), (4096, "1", "1"), (8160, "2", "1"), (100, "2", "1"), (1024, "0", "1"),
                                              (999, "2", "0"), (4096, "2", "0")])
def test_fused_lanes_bank_aligned_rows(monkeypatch, cols, mode, direct):
    """Fused dense rows, bank-aligned kernel (osp_fusedlanes.cuh; OSP_FUSED_LANES=2 forces it, 1 = automatic, 0 = the band
    kernel): column ranges that are and are not multiples of 32, the one- and two-warp CTAs, rows of B whose columns pile
    up in one shared-memory bank (more than 32 groups: a run applied in pieces), empty rows of A and of B, rows of C beyond
    A's last row, explicit +0.0 / -0.0 entries (a column whose products are all -0.0 is still an entry), duplicates of a
    column across runs summed in k order.  direct = "1": rows of C written at the prefix of their bounds and moved into an
    exactly sized C when some row is not full (k_fl_compact); "0": rows chained by the look-back."""
    monkeypatch.setenv("OSP_FUSED_LANES", mode)
    monkeypatch.setenv("OSP_FL_DIRECT", direct)
    rng = np.random.default_rng(cols * 7 + int(mode))
    n_k = 96
    dens = 0.7 if cols <= 128 else 0.25 if cols <= 1024 else 0.06
    b_rows = []
    for k in range(n_k):
        if k % 17 == 5:
            b_rows.append([])                                                # empty row of B
        elif k % 13 == 3 and cols > 40 * 32:
            b_rows.append(sorted(int(c) for c in (rng.choice(cols // 32, 40, replace=False) * 32 + 7)))   # 40 columns in bank 7
        else:
            b_rows.append(sorted(int(c) for c in np.nonzero(rng.random(cols) < dens)[0]))
    b = _csr_from_rows(b_rows, cols, rng, explicit_zero_every=11)
    m = 37
    a_rows = []
    for i in range(m):
        if i % 9 == 4:
            a_rows.append([])                                                # empty row of A
        elif i == 7:
            a_rows.append(list(range(n_k)))                                  # every k: more than 32 runs, the empty rows of B among them
        else:
            a_rows.append(sorted(int(k) for k in np.nonzero(rng.random(n_k) < 0.5)[0]))
    a = _csr_from_rows(a_rows, n_k, rng, explicit_zero_every=13)
    want, prod = oracle_spgemm(synth.transpose_host(a, n_k), b, rows_override=m + 3)
    eng = osp.Engine(0)
    try:
        res = eng.spgemm(a, b, a_is_csr=True, rows_c=m + 3, cols_b=cols, flags=api.OSP_PROFILE_KERNELS)
        got = res.to_host(); names = [n for n, _ in res.kernel_times()]; st = res.stats(); res.free()
    finally:
        eng.close()
    assert st["products"] == prod
    if mode == "0":
        assert any("k_fused_dense" in n for n in names) and not any("k_fused_lanes" in n for n in names), names
    else:
        assert any("k_fused_lanes" in n for n in names), names
        # (the empty rows of A alone make the counts fall short of the bounds... no: their bound is 0; row 7 and the sparse rows do)
        assert any("k_fl_compact" in n for n in names) == (direct == "1" and got.nnz != sum(min(int(p), cols) for p in _row_partials(a, b))), names
    assert_bit_exact(got, want, f"fused lanes cols={cols} mode={mode} direct={direct}")
    check_csr_invariants(got, cols)


def test_fused_lanes_keeps_the_band_kernel_for_short_rows_of_b(monkeypatch):
    """Automatic mode: a B whose rows are too short to fill their quads of groups (regrouped form > 6 slots per element)
    stays with the band kernel; same bits either way."""
    monkeypatch.setenv("OSP_FUSED_LANES", "1")
    rng = np.random.default_rng(77)
    n_k, cols, m = 3000, 512, 6
    b = _csr_from_rows([sorted(int(c) for c in rng.choice(cols, 3, replace=False)) for _ in range(n_k)], cols, rng)
    a = _csr_from_rows([sorted(int(k) for k in np.nonzero(rng.random(n_k) < 0.6)[0]) for _ in range(m)], n_k, rng)
    want, prod = oracle_spgemm(synth.transpose_host(a, n_k), b)
    eng = osp.Engine(0)
    try:
        res = eng.spgemm(a, b, a_is_csr=True, cols_b=cols, flags=api.OSP_PROFILE_KERNELS)
        got = res.to_host(); names = [n for n, _ in res.kernel_times()]; res.free()
    finally:
        eng.close()
    assert any("k_fused_dense" in n for n in names) and not any("k_fused_lanes<" in n for n in names), names
    assert_bit_exact(got, want, "short rows of B")


def test_row_chunking_gives_same_bits(engine):
    rng = np.random.default_rng(21)
    A, B = rand_sparse(rng, 400, 300, 0.05), rand_sparse(rng, 300, 350, 0.05)
    a_csc, a_csr, b_csr = operands(A, B)
    want, prod = oracle_spgemm(a_csc, b_csr)
    eng = osp.Engine(0)
    try:
        eng.set_workspace_limit(64 * 1024)            # 8192 partial products per block
        res = eng.spgemm(a_csr, b_csr, a_is_csr=True)
        got = res.to_host(); st = res.stats(); res.free()
        assert st["row_chunks"] > 4
        assert_bit_exact(got, want, "chunked")
        res = eng.spgemm(a_csc, b_csr)
        got = res.to_host(); res.free()
        assert_bit_exact(got, want, "chunked from CSC")
    finally:
        eng.close()


def test_bounded_result_capacity(engine):
    """C allocated below the plan's bound (what config 3 needs at full scale, where the bound exceeds HBM): row
    blocks are admitted one by one against the capacity with the exact nnz(C) so far -- same bits; a capacity
    that cannot hold C is OSP_ERR_OOM, never a write past the allocation."""
    a, b, dims = synth.build_workload("rmat20", scale_down=256)         # skewed rows: bound well above nnz(C)
    want_pos, want_data, prod = oracle.spgemm_rowblocks(a.pos, a.data, b.pos, b.data, 4096)
    want = pack(want_pos, want_data)
    nnz_c, rows = len(want_data), len(want_pos) - 1
    cs = np.concatenate([[0], np.cumsum(np.diff(b.pos.astype(np.int64))[a.data["idx"]])])
    plen = cs[a.pos[1:].astype(np.int64)] - cs[a.pos[:-1].astype(np.int64)]      # partial products per output row
    bound = int(np.minimum(plen, dims["cols"]).sum())
    block = max(int(plen.max()), prod // 24)                            # ~24 row blocks
    cap = nnz_c + block + 64                                            # C + the last block's bound
    assert cap < bound, "the workload must leave room between nnz(C) and the plan's bound"
    eng = osp.Engine(0)
    try:
        eng.set_workspace_limit(block * 8)
        eng.set_result_limit(cap * 8)
        for is_csr, op in ((True, a), (False, synth.transpose_host(a, dims["n_k"]))):
            res = eng.spgemm(op, b, a_is_csr=is_csr, cols_b=dims["cols"])
            got = res.to_host(); st = res.stats()
            assert st["row_chunks"] > 8 and st["products"] == prod and st["nnz_c"] == nnz_c
            assert_bit_exact(got, want, f"bounded C, a_is_csr={is_csr}")
            mid = rows // 3
            part = res.rows_to_host(mid, mid + 500)                     # osp_result_copy_rows
            lo, hi = int(want_pos[mid]), int(want_pos[mid + 500])
            assert np.array_equal(part.pos, want_pos[mid:mid + 501] - want_pos[mid])
            assert np.array_equal(part.data.view(np.uint64), want_data[lo:hi].view(np.uint64))
            res.free()
        eng.set_result_limit(nnz_c * 8 // 2)                            # half of C: must fail cleanly
        with pytest.raises(osp.OspError) as ei:
            eng.spgemm(a, b, a_is_csr=True, cols_b=dims["cols"])
        assert ei.value.code == api.OSP_ERR_OOM and "does not fit" in str(ei.value)
        eng.set_result_limit(0)                                         # the engine is still usable afterwards
        res = eng.spgemm(a, b, a_is_csr=True, cols_b=dims["cols"])
        got = res.to_host(); res.free()
        assert_bit_exact(got, want, "after the failed call")
    finally:
        eng.close()


def test_edge_cases(engine):
    E = osp.ELEM
    # empty A (reference: maxRowId = 0 -> one empty output row)
    a = osp.CSRMatrix(np.zeros(5, np.uint64), np.zeros(0, E))
    b = pack([0, 1, 1, 2, 2], np.array([(0, 1.0), (3, 2.0)], E))
    for is_csr in (False, True):
        res = engine.spgemm(a, b, a_is_csr=is_csr)
        got = res.to_host(); res.free()
        assert list(got.pos) == [0, 0] and got.nnz == 0
    # empty B
    a = pack([0, 1, 2, 2, 2], np.array([(0, 1.0), (3, 2.0)], E))
    b = osp.CSRMatrix(np.zeros(5, np.uint64), np.zeros(0, E))
    res = engine.spgemm(a, b)
    got = res.to_host(); res.free()
    assert list(got.pos) == [0, 0, 0, 0, 0] and got.nnz == 0
    # 1x1
    one = pack([0, 1], np.array([(0, 3.0)], E))
    res = engine.spgemm(one, one)
    got = res.to_host(); res.free()
    assert list(got.pos) == [0, 1] and got.data[0]["idx"] == 0 and got.data[0]["val"] == 9.0
    # explicit zeros and exact cancellation stay in the structure (no numerical zero dropping)
    A = sp.csr_matrix(np.array([[1, -1], [0, 2]], np.float32)); B = sp.csr_matrix(np.array([[1, 5], [1, 0]], np.float32))
    a_csc, _, b_csr = operands(A, B)
    want, _ = oracle_spgemm(a_csc, b_csr)
    res = engine.spgemm(a_csc, b_csr)
    got = res.to_host(); res.free()
    assert_bit_exact(got, want, "cancellation")
    assert got.data["val"][0] == 0.0 and got.nnz == 3
    # explicit rows_c larger than maxRowId+1 pads empty rows
    res = engine.spgemm(a_csc, b_csr, rows_c=5)
    got = res.to_host(); res.free()
    assert got.NRow() == 5 and list(got.pos[2:]) == [3, 3, 3, 3]


def test_error_codes(engine):
    E = osp.ELEM
    a = pack([0, 1, 2], np.array([(0, 1.0), (1, 2.0)], E))
    b3 = pack([0, 1, 1, 2], np.array([(0, 1.0), (1, 2.0)], E))
    with pytest.raises(osp.OspError) as ei:                     # assert(lmat.NRow()==rmat.NRow()), SimOuterSPACE.cpp:47
        engine.spgemm(a, b3)
    assert ei.value.code == api.OSP_ERR_INVALID
    bad = pack([0, 1, 2], np.array([(0, 1.0), (7, 2.0)], E))    # k index 7 >= n_k = 2 in a CSR(A)
    b2 = pack([0, 1, 2], np.array([(0, 1.0), (1, 2.0)], E))
    with pytest.raises(osp.OspError) as ei:
        engine.spgemm(bad, b2, a_is_csr=True)
    assert ei.value.code == api.OSP_ERR_INDEX
    # engine still usable afterwards
    res = engine.spgemm(a, b2)
    assert res.to_host().nnz == 2
    res.free()


def test_operand_preconditions_are_validated(engine):
    """SURVEY 8(b): both operands "sorted ascending inside a slice, duplicate-free" (what coo2csr guarantees in the
    reference, SimSpGEMM.cpp:113-123) and every column id of B below cols_b: a violation is an error code before any
    merge kernel runs, never an out-of-bounds access; OSP_NO_VALIDATE skips the pass for callers that vouch for them."""
    E = osp.ELEM
    a = pack([0, 2, 3], np.array([(0, 1.0), (1, 2.0), (1, 3.0)], E))            # CSR(A) 2 x 2
    good = pack([0, 2, 4], np.array([(1, 1.0), (5, 2.0), (0, 3.0), (2, 4.0)], E))
    want, _ = oracle_spgemm(synth.transpose_host(a, 2), good)
    for flags in (0, api.OSP_NO_VALIDATE):
        res = engine.spgemm(a, good, a_is_csr=True, cols_b=6, flags=flags)
        assert_bit_exact(res.to_host(), want, f"valid operands, flags={flags}")
        res.free()
    unsorted_b = pack([0, 2, 4], np.array([(5, 1.0), (1, 2.0), (0, 3.0), (2, 4.0)], E))
    dup_b = pack([0, 2, 4], np.array([(1, 1.0), (1, 2.0), (0, 3.0), (2, 4.0)], E))
    unsorted_a = pack([0, 2, 3], np.array([(1, 1.0), (0, 2.0), (1, 3.0)], E))
    dup_a = pack([0, 2, 3], np.array([(1, 1.0), (1, 2.0), (1, 3.0)], E))
    bad_pos = osp.CSRMatrix(np.array([0, 3, 2], np.uint64), good.data[:2].copy())
    for aa, bb, cols, code, what in ((a, unsorted_b, 6, api.OSP_ERR_INVALID, "unsorted row of B"),
                                     (a, dup_b, 6, api.OSP_ERR_DUPLICATE, "duplicate in a row of B"),
                                     (unsorted_a, good, 6, api.OSP_ERR_INVALID, "unsorted row of A"),
                                     (dup_a, good, 6, api.OSP_ERR_DUPLICATE, "duplicate in a row of A"),
                                     (a, good, 5, api.OSP_ERR_INDEX, "column id 5 with cols_b = 5"),
                                     (a, bad_pos, 6, api.OSP_ERR_INVALID, "pos array that decreases")):
        with pytest.raises(osp.OspError) as ei:
            engine.spgemm(aa, bb, a_is_csr=True, cols_b=cols)
        assert ei.value.code == code, (what, ei.value.code, str(ei.value))
    # CSC(A) hand-over: the same checks on the column-compressed operand
    with pytest.raises(osp.OspError) as ei:
        engine.spgemm(unsorted_a, good, a_is_csr=False, cols_b=6)
    assert ei.value.code == api.OSP_ERR_INVALID
    # a last row of B that is not ascending across the slice boundary only (boundary descents are legal)
    edge = pack([0, 2, 4], np.array([(3, 1.0), (5, 2.0), (0, 3.0), (1, 4.0)], E))
    res = engine.spgemm(a, edge, a_is_csr=True, cols_b=6)
    want, _ = oracle_spgemm(synth.transpose_host(a, 2), edge)
    assert_bit_exact(res.to_host(), want, "descent across a slice boundary")
    res.free()


@pytest.mark.parametrize("name", CASES)
def test_csr2csc_device_stable(engine, name):
    """Device CSR->CSC equals coo2csr<true> of the reference (fixture made by the compiled reference)."""
    g = load_npz(name)
    a_csr = pack(g["a_csr_pos"], g["a_csr_data"])
    got = engine.csr2csc(a_csr, len(g["a_csc_pos"]) - 1)
    assert np.array_equal(got.pos, g["a_csc_pos"]) and np.array_equal(got.data, g["a_csc_data"])
    back = engine.csr2csc(got, a_csr.NRow())
    assert np.array_equal(back.pos, a_csr.pos) and np.array_equal(back.data, a_csr.data)


def test_csr2csc_random_and_duplicates(engine):
    rng = np.random.default_rng(33)
    for _ in range(4):
        m, n = (int(x) for x in rng.integers(1, 500, size=2))
        a = CSR = osp.CSRMatrix.from_scipy(rand_sparse(rng, m, n, 0.1))
        pos, data = oracle.csr2csc(m, n, a.pos, a.data)
        got = engine.csr2csc(a, n)
        assert np.array_equal(got.pos, pos) and np.array_equal(got.data, data)
    dup = pack([0, 2, 3], np.array([(1, 1.0), (1, 2.0), (0, 3.0)], osp.ELEM))
    with pytest.raises(osp.DuplicateEntry):
        engine.csr2csc(dup, 2)


def test_device_resident_operands(engine):
    """HBM-resident operands through OSP_DEVICE_POINTERS (torch only provides the allocations)."""
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(77)
    A, B = rand_sparse(rng, 200, 150, 0.05), rand_sparse(rng, 150, 180, 0.05)
    a_csc, a_csr, b_csr = operands(A, B)
    want, _ = oracle_spgemm(a_csc, b_csr)
    dev = torch.device("cuda:0")

    def up(x):
        return torch.from_numpy(x.view(np.uint8).reshape(-1).copy()).to(dev)
    t = [up(a_csr.pos), up(a_csr.data), up(b_csr.pos), up(b_csr.data)]
    torch.cuda.synchronize()
    res = engine.spgemm_device(a_csr.NRow(), t[0].data_ptr(), t[1].data_ptr(), b_csr.NRow(), t[2].data_ptr(),
                               t[3].data_ptr(), a_is_csr=True)
    got = res.to_host()
    dpos, ddata = res.device_pointers()
    assert dpos and ddata
    res.free()
    assert_bit_exact(got, want, "device operands")


def _row_lengths_case(rng, lens, cols, dup_rate):
    """A (rows x k) with one non-zero per (row, way) and B rows of chosen lengths: output row i merges
    lens[i] partial products drawn from `cols` columns, a fraction of them on repeated columns."""
    import scipy.sparse as sp
    rows = len(lens)
    ways = 6
    k = rows * ways
    a_r, a_c, b_r, b_c = [], [], [], []
    for i, L in enumerate(lens):
        cut = np.sort(rng.integers(0, L + 1, size=ways - 1))
        parts = np.diff(np.concatenate(([0], cut, [L])))
        pool = rng.choice(cols, size=max(1, int(L * (1 - dup_rate))), replace=False) if L else np.zeros(0, np.int64)
        for w, n in enumerate(parts):
            kk = i * ways + w
            a_r.append(i); a_c.append(kk)
            if n:
                c = np.unique(rng.choice(pool, size=min(int(n), pool.size), replace=False))
                b_r += [kk] * c.size; b_c += c.tolist()
    A = sp.csr_matrix((rng.standard_normal(len(a_r)).astype(np.float32) + 3, (a_r, a_c)), shape=(rows, k))
    B = sp.csr_matrix((rng.standard_normal(len(b_r)).astype(np.float32), (b_r, b_c)), shape=(k, cols))
    return A, B


@pytest.mark.parametrize("n,per_row,clustered", [(1 << 13, 8, False), (1 << 14, 6, False), (1 << 13, 10, True)])
def test_config4_shape_spread_and_clustered_columns(engine, n, per_row, clustered):
    """Config 4's shape at small scale, element-wise against the oracle: rows of C of 20-130 partial products over uniformly
    spread columns; `clustered` packs the columns of every row of B into a few dense clumps plus outliers and adds repeated
    columns, which force the k-ordered fold.  (Written for the bucket-rank merge experiment of round 2,
    profiles/r02_experiments.md; kept as a parity test of the sorting network on this shape.)  Both operand forms."""
    rng = np.random.default_rng(n + per_row)
    a = synth.erdos_renyi(n, n, per_row * n, seed=n + per_row)
    if clustered:
        cols = a.data["idx"].astype(np.int64)
        cols = np.where(rng.random(len(cols)) < 0.85, (cols % 97) + (cols // 4096) * 4096, cols)      # clumps of 97 columns + outliers
        keys = np.unique(np.repeat(np.arange(n, dtype=np.int64), np.diff(a.pos.astype(np.int64))) * n + cols)
        rows, c2 = keys // n, (keys % n).astype(np.uint32)
        pos = np.zeros(n + 1, np.uint64); np.cumsum(np.bincount(rows, minlength=n), out=pos[1:])
        a = osp.CSRMatrix.from_arrays(pos, c2, rng.standard_normal(len(c2)).astype(np.float32))
    a_csc = synth.transpose_host(a, n)
    want, prod = oracle_spgemm(a_csc, a)
    for is_csr, op in ((True, a), (False, a_csc)):
        res = engine.spgemm(op, a, a_is_csr=is_csr, cols_b=n)
        got = res.to_host(); st = res.stats(); res.free()
        assert st["products"] == prod
        assert_bit_exact(got, want, f"config-4 shape n={n} per_row={per_row} clustered={clustered} csr={is_csr}")
        check_csr_invariants(got, n)


@pytest.mark.parametrize("cols,dup_rate", [(1 << 17, 0.0), (1 << 20, 0.4), ((1 << 24) + 5, 0.2)])
def test_kway_merge_of_the_sorted_ways(engine, cols, dup_rate):
    """SURVEY 8(f) rank 4: rows of 4 097 .. 32 768 partial products made of a few long sorted ways are merged BY RANK
    (k_merge_ways, the k-way merge of merge2way / mergeHardware, SimSpGEMM.cpp:306-327, 411-441) instead of through the
    dense accumulator; rows outside that class (too short, too long) keep their kernels in the same call.  Same bits."""
    rng = np.random.default_rng(cols % 977 + int(dup_rate * 10))
    lens = [4096, 4097, 5000, 9000, 20000, 32768, 32769, 40000, 700, 12, 0, 300, 6000] * 2
    rng.shuffle(lens)
    A, B = _row_lengths_case(rng, lens, cols, dup_rate)
    a_csc, a_csr, b_csr = operands(A, B)
    want, prod = oracle_spgemm(a_csc, b_csr)
    for flags in (api.OSP_KWAY_MERGE, 0):
        res = engine.spgemm(a_csr, b_csr, a_is_csr=True, cols_b=cols, flags=flags | api.OSP_PROFILE_KERNELS)
        got = res.to_host(); names = {n for n, _ in res.kernel_times()}; res.free()
        assert any("k_merge_ways" in n for n in names) == bool(flags), names
        assert_bit_exact(got, want, f"k-way merge cols={cols} dup={dup_rate} flags={flags}")
        check_csr_invariants(got, cols)
    # in row blocks (the ways of a row never straddle a block) and through the CSC hand-over
    eng = osp.Engine(0)
    try:
        eng.set_workspace_limit(60000 * 8)
        res = eng.spgemm(a_csc, b_csr, a_is_csr=False, cols_b=cols, flags=api.OSP_KWAY_MERGE)
        got = res.to_host(); st = res.stats(); res.free()
        assert st["row_chunks"] > 1
        assert_bit_exact(got, want, "k-way merge in row blocks")
    finally:
        eng.close()


@pytest.mark.parametrize("cols,dup_rate", [(1 << 14, 0.0), (1 << 14, 0.3), (1 << 20, 0.0), (1 << 20, 0.3), ((1 << 24) + 5, 0.2)])
def test_every_row_length_class(engine, cols, dup_rate):
    """Rows of every size class of the merge chain (0, 1, 2..8, ..., 257..512, long rows) side by side in the same
    tiles; small column range = bitmap-rank variant, 2^20 = 32-bit sort keys, > 2^23 = 64-bit sort keys."""
    rng = np.random.default_rng(cols % 1000 + int(dup_rate * 10))
    lens = [0, 1, 2, 3, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64, 65, 100, 127, 128, 129, 200, 255, 256, 257, 300, 400,
            511, 512, 513, 700, 1500, 5000] * 3
    rng.shuffle(lens)
    A, B = _row_lengths_case(rng, lens, cols, dup_rate)
    a_csc, a_csr, b_csr = operands(A, B)
    want, prod = oracle_spgemm(a_csc, b_csr)
    for flags in (0, api.OSP_ROWWISE_ORDER):
        res = engine.spgemm(a_csr, b_csr, a_is_csr=True, cols_b=cols, flags=flags)
        got = res.to_host(); res.free()
        assert_bit_exact(got, want, f"length classes cols={cols} dup={dup_rate} flags={flags}")
        check_csr_invariants(got, cols)


def test_many_tiles_chain_order(engine):
    """Enough tiles for several per persistent CTA: the look-back chain, the deferred retire and the tile
    prefetch all cycle; C.pos must be the exact prefix of the survivor counts."""
    a, b, dims = synth.build_workload("er8m", scale_down=64)
    a_csc = synth.transpose_host(a, dims["n_k"])
    want, prod = oracle_spgemm(a_csc, b)
    for flags in (api.OSP_KSLICE_ORDER, api.OSP_ROWWISE_ORDER):
        res = engine.spgemm(a, b, a_is_csr=True, cols_b=dims["cols"], flags=flags)
        got = res.to_host(); st = res.stats(); res.free()
        assert st["merge_tiles"] > 2000
        assert_bit_exact(got, want, f"er8m/64 flags={flags}")


def test_coo_ingest_on_device(engine):
    """coo2csr<false/true> + dupcheck on the GPU against the host loader path (itself pinned to the reference)."""
    rng = np.random.default_rng(33)
    for m, n, nnz in ((1, 1, 1), (50, 70, 400), (3000, 2500, 200000), (20, 100000, 5000)):
        keys = rng.choice(m * n, size=min(nnz, m * n), replace=False)
        rng.shuffle(keys)
        coo = api.COO((keys // n).astype(np.uint32), (keys % n).astype(np.uint32),
                      rng.standard_normal(keys.size).astype(np.float32))
        for transpose, N in ((False, m), (True, n)):
            want = api.coo2csr(coo, N, transpose)
            got = engine.coo2csr(coo, N, transpose)
            assert_bit_exact(got, want, f"coo2csr {m}x{n} transpose={transpose}")
    # duplicates -> 233, like the reference's throw(233); out-of-range index -> OSP_ERR_INDEX
    dup = api.COO(np.array([0, 1, 1, 2], np.uint32), np.array([3, 2, 2, 0], np.uint32), np.ones(4, np.float32))
    with pytest.raises(api.DuplicateEntry):
        engine.coo2csr(dup, 3)
    bad = api.COO(np.array([0, 5], np.uint32), np.array([0, 0], np.uint32), np.ones(2, np.float32))
    with pytest.raises(api.OspError):
        engine.coo2csr(bad, 3)
    empty = api.COO(np.zeros(0, np.uint32), np.zeros(0, np.uint32), np.zeros(0, np.float32))
    got = engine.coo2csr(empty, 4)
    assert got.nnz == 0 and np.array_equal(got.pos, np.zeros(5, np.uint64))


def test_config2_full_size_bit_exact(engine):
    """BASELINE.json configs[1] at its full size (ER 16384^2, density 1e-3; P = 4.4e6): the oracle still finishes in
    a second, so the whole result is compared bit for bit, in both multiply orders."""
    a, b, dims = synth.build_workload("er16k", 1)
    a_csc = synth.transpose_host(a, dims["n_k"])
    want, prod = oracle_spgemm(a_csc, b)
    for flags in (api.OSP_KSLICE_ORDER, api.OSP_ROWWISE_ORDER):
        res = engine.spgemm(a, b, a_is_csr=True, cols_b=dims["cols"], flags=flags)
        got = res.to_host(); st = res.stats(); res.free()
        assert st["products"] == prod
        assert_bit_exact(got, want, f"er16k full flags={flags}")


def test_config4_shape_properties(engine):
    """configs[3] shape (ER, 8 nnz/row) at 1/8 linear scale, P = 6.7e7 -- too large for an element-wise oracle in a
    test, so size-independent properties: CSR invariants, nnz(C) <= P, C.pos[m] = nnz, and the checksum identity
    sum_ij C_ij = sum_k colsum_A[k] * rowsum_B[k] (float64, relative 1e-5: fp32 products and adds)."""
    a, b, dims = synth.build_workload("er8m", 8)
    res = engine.spgemm(a, b, a_is_csr=True, cols_b=dims["cols"])
    got = res.to_host(); st = res.stats(); res.free()
    check_csr_invariants(got, dims["cols"])
    assert got.nnz <= st["products"] and int(got.pos[-1]) == got.nnz and got.NRow() == dims["rows"]
    colsum_a = np.bincount(a.data["idx"], weights=a.data["val"].astype(np.float64), minlength=dims["n_k"])
    rows_b = np.repeat(np.arange(b.NRow()), np.diff(b.pos.astype(np.int64)))
    rowsum_b = np.bincount(rows_b, weights=b.data["val"].astype(np.float64), minlength=dims["n_k"])
    want_sum = float(np.dot(colsum_a, rowsum_b))
    got_sum = float(got.data["val"].astype(np.float64).sum())
    scale = float(np.dot(np.bincount(a.data["idx"], weights=np.abs(a.data["val"]).astype(np.float64), minlength=dims["n_k"]),
                         np.bincount(rows_b, weights=np.abs(b.data["val"]).astype(np.float64), minlength=dims["n_k"])))
    assert abs(got_sum - want_sum) <= 1e-5 * scale, (got_sum, want_sum, scale)
    # the per-row structure is exactly the union of the B rows selected by A's row: spot-check 64 rows
    rng = np.random.default_rng(0)
    for i in rng.integers(0, dims["rows"], size=64):
        ks = a.data["idx"][int(a.pos[i]):int(a.pos[i + 1])]
        cols = np.unique(np.concatenate([b.data["idx"][int(b.pos[k]):int(b.pos[k + 1])] for k in ks])) if ks.size else np.zeros(0, np.uint32)
        assert np.array_equal(got.data["idx"][int(got.pos[i]):int(got.pos[i + 1])], cols), f"row {i}"


def _bias_relu_host(c: "CSRMatrix", cols: int, bias):
    """numpy restatement of the step between two layers (NN_models/models.py:18-31: x = relu(fc(x))) on the engine's
    definition: out = C + bias with ONE rounded fp32 add per entry (bias alone where C has no entry), kept where > 0."""
    rows = c.NRow()
    pos = np.zeros(rows + 1, np.uint64)
    idx_all, val_all = [], []
    for i in range(rows):
        dense = np.array(bias, np.float32, copy=True) if bias is not None else np.zeros(cols, np.float32)
        lo, hi = int(c.pos[i]), int(c.pos[i + 1])
        ci, cv = c.data["idx"][lo:hi].astype(np.int64), c.data["val"][lo:hi]
        dense[ci] = (cv + np.asarray(bias, np.float32)[ci]).astype(np.float32) if bias is not None else cv
        keep = np.nonzero(dense > 0)[0]
        idx_all.append(keep.astype(np.uint32)); val_all.append(dense[keep])
        pos[i + 1] = pos[i] + keep.size
    from outerspace_b200.formats import CSRMatrix
    return CSRMatrix.from_arrays(pos, np.concatenate(idx_all) if idx_all else np.zeros(0, np.uint32),
                                 np.concatenate(val_all) if val_all else np.zeros(0, np.float32))


def test_layer_chaining_two_layers(engine):
    """act_0 -> fc1 -> relu -> fc2 -> relu with sparse activations and pruned weights, everything on the device between
    the layers (the result's device CSR is the next product's A operand); checked bit for bit against
    oracle SpGEMM + the numpy epilogue, layer by layer."""
    rng = np.random.default_rng(5)
    x = synth.pruned_dense(40, 600, 0.12, seed=11, nonneg=True)            # act_0: 40 x 600
    w1 = synth.pruned_dense(500, 600, 0.10, seed=12)                       # fc1.weight: 500 x 600
    w2 = synth.pruned_dense(300, 500, 0.15, seed=13)                       # fc2.weight: 300 x 500
    b1 = rng.standard_normal(500).astype(np.float32) * 0.5
    w1t, w2t = synth.transpose_host(w1, 600), synth.transpose_host(w2, 500)   # B = W^T in CSR: 600 x 500, 500 x 300
    # oracle chain
    c1, _ = oracle_spgemm(synth.transpose_host(x, 600), w1t, rows_override=40)
    a1 = _bias_relu_host(c1, 500, b1)
    c2, _ = oracle_spgemm(synth.transpose_host(a1, 500), w2t, rows_override=40)
    a2 = _bias_relu_host(c2, 300, None)
    # engine chain, device resident between the steps
    r1 = engine.spgemm(x, w1t, a_is_csr=True, rows_c=40, cols_b=500)
    g1 = engine.bias_relu(r1, 500, b1)
    assert_bit_exact(g1.to_host(), a1, "layer 1: relu(x W1^T + b1)")
    import torch
    dev = torch.device("cuda:0")
    tb = [torch.from_numpy(v.view(np.uint8).reshape(-1).copy()).to(dev) for v in (w2t.pos, w2t.data)]
    p_ptr, d_ptr = g1.device_pointers()
    r2 = engine.spgemm_device(40, p_ptr, d_ptr, 500, tb[0].data_ptr(), tb[1].data_ptr(), a_is_csr=True, rows_c=40, cols_b=300,
                              a_nnz=g1.nnz, b_nnz=w2t.nnz)
    g2 = engine.bias_relu(r2, 300, None)
    assert_bit_exact(g2.to_host(), a2, "layer 2: relu(a1 W2^T)")
    for r in (r1, g1, r2, g2):
        r.free()

"""The whole single-GPU engine on the CPU emulation of the CUDA execution model (tests/cusim), against the oracle.

tests/cusim/engine_sim.cpp compiles outerspace_b200/csrc/osp_engine.cu -- the C ABI, the host orchestration and every
kernel, the very sources nvcc builds for sm_100a -- with g++ against cusim.h (threads of a block = fibers, one legal
CUDA schedule) and cusim_runtime.h (device memory = host memory).  The parity tests of tests/test_gpu_parity.py that
are small enough run here UNCHANGED through the same Python binding, so host logic (planning, row blocks, capacity
admission, error paths) and kernel logic are checked bit for bit where no GPU exists; the opt-in long-row sweep
(OSP_LONGROW_SWEEP), which has not run on a B200 yet, is exercised end to end.

This is TEST INFRASTRUCTURE: the emulated library is built into a temporary directory and loaded by this module only.
The product (outerspace_b200/libosp_b200.so) has no CPU path, and an emulation cannot see data races or timing: the
`-m gpu` suite stays the gate.
"""
import os
import subprocess
import zlib

import numpy as np
import pytest
import scipy.sparse as sp

import oracle
import outerspace_b200 as osp
from outerspace_b200 import api, synth
from helpers import assert_bit_exact, check_csr_invariants, operands, oracle_spgemm, pack, rand_sparse
import test_gpu_parity as gp

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "..", "outerspace_b200", "csrc")


def _build_emulation(out, extra_defines=()):
    # CUSIM_ASAN=1 (with LD_PRELOAD=$(g++ -print-file-name=libasan.so) for the interpreter): AddressSanitizer build
    asan = ["-g", "-fsanitize=address", "-fno-omit-frame-pointer"] if os.environ.get("CUSIM_ASAN") == "1" else []
    defines = os.environ.get("CUSIM_DEFINES", "").split()      # e.g. "-DOSP_E16_FROM=3": experimental kernel variants on the emulation
    cmd = ["g++", "-O1"] + asan + defines + list(extra_defines) + ["-std=c++17", "-x", "c++", "-fPIC", "-shared", "-ffp-contract=off", "-Wall",
           "-Wno-unknown-pragmas", "-Wno-unused-function", "-I", os.path.join(HERE, "cusim"), "-I", CSRC, "-o", out,
           os.path.join(HERE, "cusim", "engine_sim.cpp"), os.path.join(CSRC, "osp_host.cpp"), "-lpthread"]
    subprocess.run(cmd, check=True)


@pytest.fixture(scope="module", autouse=True)
def emulated_library(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("cusim_engine") / "libosp_b200_cusim.so")
    _build_emulation(out)
    saved = (api._LIB_PATH, api._lib)
    api._LIB_PATH, api._lib = out, None          # this module only; restored below
    try:
        lib = api.load_library()

        yield lib
    finally:
        api._LIB_PATH, api._lib = saved


@pytest.fixture(scope="module")
def engine(emulated_library):
    eng = osp.Engine(0)
    yield eng
    eng.close()


# ---- the GPU parity tests that are small enough, unchanged --------------------------------------------------------
test_golden = gp.test_golden
test_mtx_pipeline_like_reference_main = gp.test_mtx_pipeline_like_reference_main
test_random_vs_oracle = gp.test_random_vs_oracle
test_task_sizes_match_reference_structure = gp.test_task_sizes_match_reference_structure
test_row_chunking_gives_same_bits = gp.test_row_chunking_gives_same_bits
test_edge_cases = gp.test_edge_cases
test_error_codes = gp.test_error_codes
test_operand_preconditions_are_validated = gp.test_operand_preconditions_are_validated
test_csr2csc_device_stable = gp.test_csr2csc_device_stable
test_csr2csc_random_and_duplicates = gp.test_csr2csc_random_and_duplicates
test_coo_ingest_on_device = gp.test_coo_ingest_on_device
test_er_config2_scaled = gp.test_er_config2_scaled
test_rmat_small = gp.test_rmat_small
test_mlp_batch_small = gp.test_mlp_batch_small
test_fused_lanes_bank_aligned_rows = gp.test_fused_lanes_bank_aligned_rows
test_fused_lanes_keeps_the_band_kernel_for_short_rows_of_b = gp.test_fused_lanes_keeps_the_band_kernel_for_short_rows_of_b
test_every_row_length_class = gp.test_every_row_length_class
test_kway_merge_of_the_sorted_ways = gp.test_kway_merge_of_the_sorted_ways
test_config4_shape_spread_and_clustered_columns = gp.test_config4_shape_spread_and_clustered_columns


def test_device_pointer_operands(engine):
    """OSP_DEVICE_POINTERS: operands already on the device (here: the emulated device = host memory), nothing staged."""
    rng = np.random.default_rng(77)
    A, B = rand_sparse(rng, 200, 150, 0.05), rand_sparse(rng, 150, 180, 0.05)
    a_csc, a_csr, b_csr = operands(A, B)
    want, _ = oracle_spgemm(a_csc, b_csr)
    res = engine.spgemm_device(a_csr.NRow(), a_csr.pos.ctypes.data, a_csr.data.ctypes.data, b_csr.NRow(), b_csr.pos.ctypes.data,
                               b_csr.data.ctypes.data, a_is_csr=True)
    got = res.to_host()
    assert all(res.device_pointers())
    res.free()
    assert_bit_exact(got, want, "device operands")
    # data arrays that are only 8-byte aligned (an element into a larger allocation): the validation's 128-bit loads
    # must step aside; an unsorted row behind such a pointer is still caught
    def shifted(m):
        buf = np.zeros(len(m.data) + 3, dtype=osp.ELEM)
        base = buf.ctypes.data
        off = 1 if (base // 8) % 2 == 0 else 2            # make (base + 8 * off) % 16 == 8
        buf[off:off + len(m.data)] = m.data
        return buf, base + 8 * off
    keep_a, pa = shifted(a_csr); keep_b, pb = shifted(b_csr)
    assert pa % 16 == 8 and pb % 16 == 8
    res = engine.spgemm_device(a_csr.NRow(), a_csr.pos.ctypes.data, pa, b_csr.NRow(), b_csr.pos.ctypes.data, pb, a_is_csr=True,
                               cols_b=180)
    got = res.to_host(); res.free()
    assert_bit_exact(got, want, "device operands, 8-byte aligned data")
    r = int(np.flatnonzero(np.diff(b_csr.pos.astype(np.int64)) >= 2)[0]); s0 = int(b_csr.pos[r])
    view = np.frombuffer(keep_b, dtype=osp.ELEM)          # (same memory)
    i0 = (pb - keep_b.ctypes.data) // 8 + s0
    keep_b[[i0, i0 + 1]] = keep_b[[i0 + 1, i0]]
    with pytest.raises(osp.OspError) as ei:
        engine.spgemm_device(a_csr.NRow(), a_csr.pos.ctypes.data, pa, b_csr.NRow(), b_csr.pos.ctypes.data, pb, a_is_csr=True, cols_b=180)
    assert ei.value.code == api.OSP_ERR_INVALID


# ---- value and index-range edges (tests/test_gpu_edges.py): special values through every merge kernel, the dispatch
# thresholds, the largest ids, the 32-bit copy of B.pos; the cases of 2^31 columns and more need a B200's memory ------
import test_gpu_edges as ge

test_special_values_through_each_merge_kernel = ge.test_special_values_through_each_merge_kernel
test_special_values_through_fused_dense_rows = ge.test_special_values_through_fused_dense_rows
test_oracle_and_engine_against_float64 = ge.test_oracle_and_engine_against_float64
test_nan_payload_of_device_arithmetic = ge.test_nan_payload_of_device_arithmetic
test_bias_relu_special_values = ge.test_bias_relu_special_values
test_column_range_thresholds = ge.test_column_range_thresholds
test_largest_ids_with_derived_dimensions = ge.test_largest_ids_with_derived_dimensions
engine_bpos32 = ge.engine_bpos32
test_bpos32_random_vs_oracle = ge.test_bpos32_random_vs_oracle
test_bpos32_every_row_length_class = ge.test_bpos32_every_row_length_class
test_bpos32_config4_shape = ge.test_bpos32_config4_shape
test_bpos32_row_chunking = ge.test_bpos32_row_chunking
test_bpos32_is_used_and_its_threshold = ge.test_bpos32_is_used_and_its_threshold


# ---- the device format conversions (tests/test_gpu_conversions.py): the dispatch grid three ways, duplicates in every
# bucket class, device pointers, ids up to 2^32 - 1, no output slice; the 8.6 GB accumulator and the 4e8-product R-MAT
# case need a B200 ---------------------------------------------------------------------------------------------------------
import test_gpu_conversions as gc

test_csr2csc_dispatch_grid = gc.test_csr2csc_dispatch_grid
test_coo_ingest_dispatch_grid = gc.test_coo_ingest_dispatch_grid
test_csc_hand_over_dispatch_grid = gc.test_csc_hand_over_dispatch_grid
test_csc_hand_over_of_each_merge_kernel_case = gc.test_csc_hand_over_of_each_merge_kernel_case
test_conversions_with_device_pointers = gc.test_conversions_with_device_pointers
test_coo_ids_up_to_2_32 = gc.test_coo_ids_up_to_2_32
test_conversions_into_zero_slices = gc.test_conversions_into_zero_slices


@pytest.mark.parametrize("idx_range", ge.THRESHOLDS)
def test_duplicate_in_every_bucket_class(engine, idx_range):
    """The three ranges around 2^23 through the triplets only: there the CSR input and CSC(A) have 2^23 slices, and the
    120 calls of the whole case take about four minutes per range on the emulation.  The triplets (one output slice)
    reach the same kernels with the same index range."""
    gc.duplicate_cases(engine, idx_range, through_slices=idx_range <= 131073)


@pytest.mark.parametrize("case", list(ge.FUSED_CASES))
def test_fused_dense_rows_where_nan_payloads_survive(emulated_library, tmp_path, monkeypatch, case):
    """The special values through the fused dense rows on arithmetic that keeps NaN payloads (x86, CUSIM_NAN_PAYLOADS):
    a product with the bits 0xFFFFFFFF must not be taken for k_fused_lanes' "never touched" and dropped."""
    out = str(tmp_path / "libosp_b200_cusim_payloads.so")
    _build_emulation(out, ["-DCUSIM_NAN_PAYLOADS"])
    saved = (api._LIB_PATH, api._lib)
    api._LIB_PATH, api._lib = out, None
    try:
        api.load_library()
        ge.test_special_values_through_fused_dense_rows(monkeypatch, case)
    finally:
        api._LIB_PATH, api._lib = saved


# ---- the opt-in long-row sweep (OSP_LONGROW_SWEEP), end to end: the tests a B200 will run with OSP_TEST_SWEEP=1 ------
import test_gpu_zzz_sweep as sw

test_every_row_length_class_through_the_sweep = sw.test_every_row_length_class_through_the_sweep
test_sweep_threshold_from_the_environment = sw.test_sweep_threshold_from_the_environment


def test_sweep_with_row_blocks_and_bounded_capacity():
    """Row blocks (workspace limit) and C allocated below the plan's bound: swept rows are taken block by block, the
    multiply skips their tasks in every block, the chain's carry of nnz(C) stays exact."""
    rng = np.random.default_rng(31)
    lens = [5000, 3, 0, 20000, 700, 4097, 129, 9000, 12, 6000, 300, 4500, 45, 8000] * 2
    cols = 1 << 16
    A, B = gp._row_lengths_case(rng, lens, cols, 0.3)
    a_csc, a_csr, b_csr = operands(A, B)
    want, prod = oracle_spgemm(a_csc, b_csr)
    eng = osp.Engine(0)
    try:
        eng.set_workspace_limit(25000 * 8)
        eng.set_result_limit((want.nnz + 25000 + 64) * 8)
        for flags in (api.OSP_LONGROW_SWEEP, 0):
            res = eng.spgemm(a_csr, b_csr, a_is_csr=True, cols_b=cols, flags=flags | api.OSP_PROFILE_KERNELS)
            got = res.to_host(); st = res.stats(); names = {n for n, _ in res.kernel_times()}; res.free()
            assert st["row_chunks"] > 4 and st["nnz_c"] == want.nnz
            assert any("k_long_fill" in n for n in names) == bool(flags)
            assert_bit_exact(got, want, f"row blocks, flags={flags}")
        res = eng.spgemm(a_csc, b_csr, cols_b=cols, flags=api.OSP_LONGROW_SWEEP)       # A arrives as CSC: converted on the device first
        got = res.to_host(); res.free()
        assert_bit_exact(got, want, "row blocks, sweep, CSC(A)")
    finally:
        eng.close()


def test_sweep_stays_out_where_it_does_not_apply(engine):
    """<= 16384 columns (k_merge_dense / fused dense rows own that range) and calls without a long row."""
    rng = np.random.default_rng(32)
    A, B = gp._row_lengths_case(rng, [5000, 100, 6000], 1 << 14, 0.3)
    a_csc, a_csr, b_csr = operands(A, B)
    want, _ = oracle_spgemm(a_csc, b_csr)
    res = engine.spgemm(a_csr, b_csr, a_is_csr=True, cols_b=1 << 14, flags=api.OSP_LONGROW_SWEEP | api.OSP_PROFILE_KERNELS)
    got = res.to_host(); names = {n for n, _ in res.kernel_times()}; res.free()
    assert not any("k_long_fill" in n or "k_mark_swept" in n for n in names), names
    assert_bit_exact(got, want, "small column range")
    A, B = gp._row_lengths_case(rng, [500, 100, 4096], 1 << 18, 0.3)
    a_csc, a_csr, b_csr = operands(A, B)
    want, _ = oracle_spgemm(a_csc, b_csr)
    res = engine.spgemm(a_csr, b_csr, a_is_csr=True, cols_b=1 << 18, flags=api.OSP_LONGROW_SWEEP | api.OSP_PROFILE_KERNELS)
    got = res.to_host(); names = {n for n, _ in res.kernel_times()}; res.free()
    assert not any("k_long_fill" in n for n in names), names
    assert_bit_exact(got, want, "no row above 4096 partial products")


def test_concurrent_blocks(monkeypatch):
    """CUSIM_RESIDENT=4: four blocks of every launch run at the same time on four OS threads (the emulated device has
    four SMs), so tickets interleave, the decoupled look-back chains of the scans and of the merge wait on live
    predecessors, and global atomics race for real.  Same bits."""
    monkeypatch.setenv("CUSIM_RESIDENT", "4")
    monkeypatch.setenv("CUSIM_SMS", "4")
    eng = osp.Engine(0)
    try:
        a, b, dims = synth.build_workload("er16k", scale_down=4)                 # hundreds of merge tiles through the chain
        want, _ = oracle_spgemm(synth.transpose_host(a, dims["n_k"]), b)
        for flags in (api.OSP_ROWWISE_ORDER, api.OSP_KSLICE_ORDER):
            res = eng.spgemm(a, b, a_is_csr=True, cols_b=dims["cols"], flags=flags)
            got = res.to_host(); st = res.stats(); res.free()
            assert st["merge_tiles"] > 100
            assert_bit_exact(got, want, f"er16k/4, four resident blocks, flags={flags}")
        rng = np.random.default_rng(41)
        lens = [5000, 3, 0, 20000, 700, 4097, 129, 9000, 12, 6000, 300, 4500, 45, 8000, 513, 2000] * 2
        A, B = gp._row_lengths_case(rng, lens, 1 << 17, 0.3)
        a_csc, a_csr, b_csr = operands(A, B)
        want, _ = oracle_spgemm(a_csc, b_csr)
        for flags in (0, api.OSP_LONGROW_SWEEP):
            res = eng.spgemm(a_csc, b_csr, cols_b=1 << 17, flags=flags)          # CSC(A): device conversion first
            got = res.to_host(); res.free()
            assert_bit_exact(got, want, f"long rows, four resident blocks, flags={flags}")
        csc = eng.csr2csc(a_csr, A.shape[1])
        assert np.array_equal(csc.pos, a_csc.pos) and np.array_equal(csc.data, a_csc.data)
    finally:
        eng.close()


def test_compact_operand_product(engine):
    """SURVEY 8a row a16 on the emulated engine: compactMulcsr's merged equivalent (tests/test_compact.py)."""
    from test_compact import compact_product_check
    compact_product_check(engine)


def test_sweep_row_with_more_runs_than_a_group(engine):
    """A row of A with more non-zeros than the sweep takes in one group (512): two and three groups per band, the
    group boundary inside a band, next to rows that fit one group (kept in registers)."""
    rng = np.random.default_rng(51)
    k, cols = 1400, 1 << 16
    A = sp.lil_matrix((6, k), dtype=np.float32)
    for r, n in enumerate((1300, 40, 513, 512, 0, 1024)):
        sel = rng.choice(k, size=n, replace=False)
        A[r, sel] = (rng.standard_normal(n) + 2).astype(np.float32)
    B = rand_sparse(rng, k, cols, 12.0 / cols).tolil()
    for kk in rng.choice(k, size=30, replace=False):                       # a few long rows of B: segments of many elements
        c = rng.choice(cols, size=400, replace=False)
        B[kk, c] = rng.standard_normal(400).astype(np.float32)
    a_csc, a_csr, b_csr = operands(A.tocsr(), B.tocsr())
    want, prod = oracle_spgemm(a_csc, b_csr, rows_override=6)
    res = engine.spgemm(a_csr, b_csr, a_is_csr=True, cols_b=cols, rows_c=6, flags=api.OSP_LONGROW_SWEEP | api.OSP_PROFILE_KERNELS)
    got = res.to_host(); st = res.stats(); names = {n for n, _ in res.kernel_times()}; res.free()
    assert any("k_long_fill" in n for n in names) and st["rows_long"] >= 3
    assert_bit_exact(got, want, "rows of A with up to 1300 runs")


def _live_bytes(lib):
    lib.cusim_device_bytes.restype = __import__("ctypes").c_ulonglong
    return int(lib.cusim_device_bytes())


def test_no_device_memory_is_leaked(emulated_library):
    """Every allocation of a context -- scratch, staged operands, results, including those of calls that fail half
    way -- is back when the context is destroyed (the emulated runtime counts live bytes; a real device cannot be
    asked this cheaply)."""
    before = _live_bytes(emulated_library)
    rng = np.random.default_rng(61)
    A, B = rand_sparse(rng, 60, 50, 0.2), rand_sparse(rng, 50, 70000, 0.01)
    a_csc, a_csr, b_csr = operands(A, B)
    eng = osp.Engine(0)
    r1 = eng.spgemm(a_csr, b_csr, a_is_csr=True)
    r2 = eng.spgemm(a_csc, b_csr, flags=api.OSP_LONGROW_SWEEP)
    r1.free()
    with pytest.raises(osp.OspError):                                   # k-dimension mismatch: fails before any launch
        eng.spgemm(a_csc, pack(b_csr.pos[:-3], b_csr.data[: int(b_csr.pos[-4])]))
    bad = a_csr.data.copy(); bad["idx"][0] = 10_000                     # index out of range: fails after the symbolic pass
    with pytest.raises(osp.OspError) as ei:
        eng.spgemm(pack(a_csr.pos, bad), b_csr, a_is_csr=True)
    assert ei.value.code == api.OSP_ERR_INDEX
    eng.set_result_limit(4096)                                          # C cannot fit: fails between two row blocks
    with pytest.raises(osp.OspError) as ei:
        eng.spgemm(a_csr, b_csr, a_is_csr=True, cols_b=70000)
    assert ei.value.code == api.OSP_ERR_OOM
    eng.set_result_limit(0)
    B2 = rand_sparse(rng, 50, 90, 0.3)
    r3 = eng.spgemm(a_csr, operands(A, B2)[2], a_is_csr=True, cols_b=90)
    r4 = eng.bias_relu(r3, 90, np.linspace(-1, 1, 90, dtype=np.float32))   # noqa: F841 -- left alive on purpose
    assert _live_bytes(emulated_library) > before
    eng.close()                                                         # frees r2, r3 and r4, which are still alive
    assert _live_bytes(emulated_library) == before


def test_device_out_of_memory_is_reported_not_fatal(emulated_library, monkeypatch):
    """A device too small for the call: OSP_ERR_OOM from whichever allocation fails, nothing leaked, and the context
    works again once there is room."""
    rng = np.random.default_rng(62)
    A, B = rand_sparse(rng, 300, 200, 0.2), rand_sparse(rng, 200, 400, 0.2)
    a_csc, a_csr, b_csr = operands(A, B)
    want, prod = oracle_spgemm(a_csc, b_csr)
    eng = osp.Engine(0)
    try:
        base = _live_bytes(emulated_library)
        failures = 0
        for extra_kb in (16, 64, 256, 1024, 4096, 16384):               # ever larger devices: the call fails at ever later allocations
            monkeypatch.setenv("CUSIM_DEVICE_MB", str((base + extra_kb * 1024) / (1 << 20)))
            try:
                res = eng.spgemm(a_csr, b_csr, a_is_csr=True)
            except osp.OspError as e:
                assert e.code == api.OSP_ERR_OOM, str(e)
                failures += 1
                continue
            got = res.to_host(); res.free()
            assert_bit_exact(got, want, f"device with {extra_kb} KB to spare")
        assert failures >= 2
        monkeypatch.delenv("CUSIM_DEVICE_MB")
        res = eng.spgemm(a_csr, b_csr, a_is_csr=True)
        got = res.to_host(); res.free()
        assert_bit_exact(got, want, "after the failed calls")
    finally:
        eng.close()


# ---- OSP_FUSED_SHORT (opt-in, not yet run on a B200): short-row tiles computed inside the merge chain -------------------
@pytest.fixture()
def engine_fused(emulated_library, monkeypatch):
    monkeypatch.setenv("OSP_FUSED_SHORT", "1")            # read at osp_create: every call of this context takes the fused chain
    eng = osp.Engine(0)
    yield eng
    eng.close()


def test_fused_short_rows_golden_and_random(engine_fused):
    for name in gp.CASES:
        for a_is_csr in (False, True):
            gp.test_golden(engine_fused, name, a_is_csr)
    for seed in (0, 3, 4, 7):
        gp.test_random_vs_oracle(engine_fused, seed)
    gp.test_edge_cases(engine_fused)
    gp.test_er_config2_scaled(engine_fused)
    gp.test_mtx_pipeline_like_reference_main(engine_fused)


@pytest.mark.parametrize("cols,dup_rate", [(1 << 14, 0.3), (1 << 20, 0.0), (1 << 20, 0.3), ((1 << 24) + 5, 0.2)])
def test_fused_short_rows_every_row_length_class(engine_fused, cols, dup_rate):
    """Bitmap variant, 32- and 64-bit sort keys; short rows (computed in the chain) next to medium and long rows (still
    multiplied into the bins), with and without the long-row sweep."""
    gp.test_every_row_length_class(engine_fused, cols, dup_rate)
    if (1 << 14) < cols <= (1 << 20):        # (2^24 columns = 1025 bands per swept row: slow on the emulation, covered without the fused chain)
        sw.test_every_row_length_class_through_the_sweep(engine_fused, cols, dup_rate)


def test_fused_short_rows_in_row_blocks(engine_fused):
    rng = np.random.default_rng(71)
    lens = [5000, 3, 0, 20000, 700, 4097, 129, 9000, 12, 6000, 300, 4500, 45, 8000] * 2
    A, B = gp._row_lengths_case(rng, lens, 1 << 16, 0.3)
    a_csc, a_csr, b_csr = operands(A, B)
    want, prod = oracle_spgemm(a_csc, b_csr)
    engine_fused.set_workspace_limit(25000 * 8)
    engine_fused.set_result_limit((want.nnz + 25000 + 64) * 8)
    for flags in (0, api.OSP_LONGROW_SWEEP):
        for is_csr, op in ((True, a_csr), (False, a_csc)):
            res = engine_fused.spgemm(op, b_csr, a_is_csr=is_csr, cols_b=1 << 16, flags=flags | api.OSP_PROFILE_KERNELS)
            got = res.to_host(); st = res.stats(); names = {n for n, _ in res.kernel_times()}; res.free()
            assert st["row_chunks"] > 4
            assert any("k_merge_chain_fused" in n or "k_chain2" in n for n in names), names
            if is_csr:                                   # (the CSC hand-over converts A with the default chain first)
                assert not any("k_merge_chain<" in n for n in names), names
            assert_bit_exact(got, want, f"fused short rows in row blocks, flags={flags}, csr={is_csr}")
    # a call without any long row: no multiply launch at all
    A2, B2 = rand_sparse(rng, 300, 200, 0.02), rand_sparse(rng, 200, 5000, 0.004)
    a_csc, a_csr, b_csr = operands(A2, B2)
    want, _ = oracle_spgemm(a_csc, b_csr)
    engine_fused.set_workspace_limit(1 << 30)
    engine_fused.set_result_limit(0)
    res = engine_fused.spgemm(a_csr, b_csr, a_is_csr=True, flags=api.OSP_PROFILE_KERNELS)
    got = res.to_host(); names = {n for n, _ in res.kernel_times()}; res.free()
    assert not any("k_multiply" in n for n in names), names
    assert_bit_exact(got, want, "no long row: the chain computes everything")


def test_sweep_hands_out_huge_rows_first(engine):
    """A row of more than 2^20 partial products (handed out in the first ticket pass) next to ordinary long rows."""
    rng = np.random.default_rng(81)
    k, cols = 1400, 70000
    A = sp.lil_matrix((3, k), dtype=np.float32)
    for r, n in enumerate((1400, 30, 600)):
        sel = rng.choice(k, size=n, replace=False)
        A[r, sel] = (rng.standard_normal(n) + 2).astype(np.float32)
    B = sp.random(k, cols, density=800.0 / cols, format="csr", random_state=7, dtype=np.float32,
                  data_rvs=lambda n: (rng.standard_normal(n) * 2 + 0.1).astype(np.float32))
    B.eliminate_zeros()
    a_csc, a_csr, b_csr = operands(A.tocsr(), B)
    want, prod = oracle_spgemm(a_csc, b_csr, rows_override=3)
    res = engine.spgemm(a_csr, b_csr, a_is_csr=True, cols_b=cols, rows_c=3, flags=api.OSP_LONGROW_SWEEP | api.OSP_PROFILE_KERNELS)
    got = res.to_host(); names = {n for n, _ in res.kernel_times()}; res.free()
    plen = np.diff(b_csr.pos.astype(np.int64))[a_csr.data["idx"][: int(a_csr.pos[1])]].sum()
    assert plen >= (1 << 20) and any("k_long_fill" in n for n in names)
    assert_bit_exact(got, want, "a huge row and two long ones")


def test_fused_short_rows_need_no_bins(emulated_library, monkeypatch):
    """OSP_FUSED_SHORT on a product without medium or long rows: the bins are never written, so they are not allocated
    and the workspace limit cuts no row blocks -- the same call needs many blocks on the default path."""
    rng = np.random.default_rng(91)
    A, B = rand_sparse(rng, 2000, 400, 0.01), rand_sparse(rng, 400, 30000, 0.0008)
    a_csc, a_csr, b_csr = operands(A, B)
    want, prod = oracle_spgemm(a_csc, b_csr)
    assert prod > 40000
    for fused_on in (False, True):
        if fused_on:
            monkeypatch.setenv("OSP_FUSED_SHORT", "1")
        eng = osp.Engine(0)
        try:
            eng.set_workspace_limit(4096)                                  # 512 partial products per row block
            before = _live_bytes(emulated_library)
            res = eng.spgemm(a_csr, b_csr, a_is_csr=True, cols_b=30000)
            got = res.to_host(); st = res.stats()
            grown = _live_bytes(emulated_library) - before - (st["nnz_c"] + st["rows_c"] + 1) * 8   # scratch the call added
            res.free()
            assert st["rows_medium"] == 0 and st["rows_long"] == 0
            assert (st["row_chunks"] == 1) == fused_on, st["row_chunks"]
            if fused_on:
                assert grown < prod * 8, "the bins were allocated"
            assert_bit_exact(got, want, f"fused_short={fused_on}")
        finally:
            eng.close()


# ---- the path each call takes ------------------------------------------------------------------------------------------
# Every merge path is bit-exact, so a call that drifts onto another path passes every parity test and shows only as lost
# speed.  Each case pins the kernels in launch order (OSP_PROFILE_KERNELS), the launches of the same call without
# profiling (the forked k-slice task list and the k_publish hand-overs counted too), the plan's counts and the product.
PATH_LENS = [0, 3, 40, 129, 513, 700, 4097, 5000] + [5] * 16       # short, medium and long rows; 144 rows of B
PATH_SHORT = [0, 1, 3, 40, 100, 129] * 4                          # no medium or long row
K, R = api.OSP_KSLICE_ORDER, api.OSP_ROWWISE_ORDER

# id: (environment read at osp_create, flags, operands, cols_b, workspace limit in partial products,
#      result limit as non-zeros beyond nnz(C))
PATH_CASES = {
    "cols_16384": ({}, 0, "rows", 1 << 14, 0, None),
    "cols_131072": ({}, 0, "rows", 1 << 17, 0, None),
    "cols_2_23": ({}, 0, "rows", 1 << 23, 0, None),
    "cols_above_2_23": ({}, 0, "rows", (1 << 23) + 5, 0, None),
    "csc_hand_over": ({}, 0, "rows_csc", 1 << 17, 0, None),
    "kslice": ({}, K, "rows", 1 << 17, 0, None),
    "kslice_row_blocks": ({}, K, "rows", 1 << 17, 3000, None),
    "row_blocks": ({}, R, "rows", 1 << 17, 3000, None),
    "bounded_c": ({}, 0, "rows", 1 << 17, 3000, 3064),
    "fused_lanes_full_rows": ({}, 0, "dense_full", 256, 0, None),
    "fused_lanes_compact": ({}, 0, "dense", 256, 0, None),
    "fused_lanes_chained": ({"OSP_FL_DIRECT": "0"}, 0, "dense", 256, 0, None),
    "fused_band_kernel": ({"OSP_FUSED_LANES": "0"}, 0, "dense", 256, 0, None),
    "no_fused_dense": ({}, api.OSP_NO_FUSED_DENSE, "dense", 256, 0, None),
    "longrow_sweep": ({}, api.OSP_LONGROW_SWEEP, "rows", 1 << 17, 0, None),
    "kway_merge": ({}, api.OSP_KWAY_MERGE, "rows", 1 << 17, 0, None),
    "fused_short_chain2": ({}, api.OSP_FUSED_SHORT, "rows", 1 << 17, 0, None),
    "fused_short_old": ({"OSP_FUSED_SHORT_OLD": "1"}, api.OSP_FUSED_SHORT, "rows", 1 << 17, 0, None),
    "fused_short_no_medium_rows": ({}, api.OSP_FUSED_SHORT, "short", 1 << 17, 0, None),
    "bpos32": ({"OSP_BPOS32_MIN_KB": "1"}, 0, "rows", 1 << 17, 0, None),
    "no_validate_derived_cols": ({}, api.OSP_NO_VALIDATE, "rows", 0, 0, None),
    "empty_a": ({}, 0, "empty", 1 << 17, 0, None),
}

# id: (kernels in launch order, kernel_launches, row_chunks, merge_tiles, rows_medium, rows_long)
PATH_EXPECTED = {
    "cols_16384": ([
        "k_validate_starts", "k_validate", "(k_scan<SymIn, RunOffOut>)", "k_plan<RowBinFromRuns>", "k_multiply<Src>",
        "k_merge_dense", "(k_merge_chain<uint32_t, true>)"
    ], 9, 1, 6, 1, 2),
    "cols_131072": ([
        "k_validate_starts", "k_validate", "(k_scan<SymIn, RunOffOut>)", "k_plan<RowBinFromRuns>", "k_multiply<Src>",
        "k_merge_xl", "(k_merge_chain<uint32_t, false>)"
    ], 9, 1, 7, 2, 2),
    "cols_2_23": ([
        "k_validate_starts", "k_validate", "(k_scan<SymIn, RunOffOut>)", "k_plan<RowBinFromRuns>", "k_multiply<Src>",
        "k_merge_long", "k_merge_xl", "(k_merge_chain<uint32_t, false>)"
    ], 10, 1, 7, 2, 2),
    "cols_above_2_23": ([
        "k_validate_starts", "k_validate", "(k_scan<SymIn, RunOffOut>)", "k_plan<RowBinFromRuns>", "k_multiply<Src>",
        "k_merge_long", "k_merge_xl", "(k_merge_chain<uint64_t, false>)"
    ], 10, 1, 7, 2, 2),
    "csc_hand_over": ([
        "k_validate_starts", "k_validate", "k_hist_elems", "(k_scan<U32In, U64Out>)", "k_scatter_elems",
        "k_plan<RowBinDirect>", "(k_merge_chain<uint32_t, true>)", "k_check_same", "k_validate_starts", "k_validate",
        "(k_scan<SymIn, RunOffOut>)", "k_plan<RowBinFromRuns>", "k_multiply<Src>", "k_merge_xl",
        "(k_merge_chain<uint32_t, false>)"
    ], 20, 1, 7, 2, 2),
    "kslice": ([
        "k_validate_starts", "k_validate", "(k_scan<SymIn, RunOffOut>)", "(k_scan<U32In, U32Out>)", "k_scatter_tasks",
        "k_plan<RowBinFromRuns>", "k_multiply<Src>", "k_merge_xl", "(k_merge_chain<uint32_t, false>)"
    ], 11, 1, 7, 2, 2),
    "kslice_row_blocks": ([
        "k_validate_starts", "k_validate", "(k_scan<SymIn, RunOffOut>)", "(k_scan<U32In, U32Out>)", "k_scatter_tasks",
        "k_plan<RowBinFromRuns>", "k_multiply<Src>", "k_merge_xl", "(k_merge_chain<uint32_t, false>)",
        "k_multiply<Src>", "k_merge_xl", "(k_merge_chain<uint32_t, false>)", "k_multiply<Src>", "k_merge_xl",
        "(k_merge_chain<uint32_t, false>)", "k_multiply<Src>", "k_merge_xl", "(k_merge_chain<uint32_t, false>)"
    ], 20, 4, 7, 2, 2),
    "row_blocks": ([
        "k_validate_starts", "k_validate", "(k_scan<SymIn, RunOffOut>)", "k_plan<RowBinFromRuns>", "k_multiply<Src>",
        "k_merge_xl", "(k_merge_chain<uint32_t, false>)", "k_multiply<Src>", "k_merge_xl",
        "(k_merge_chain<uint32_t, false>)", "k_multiply<Src>", "k_merge_xl", "(k_merge_chain<uint32_t, false>)",
        "k_multiply<Src>", "k_merge_xl", "(k_merge_chain<uint32_t, false>)"
    ], 18, 4, 7, 2, 2),
    "bounded_c": ([
        "k_validate_starts", "k_validate", "(k_scan<SymIn, RunOffOut>)", "k_plan<RowBinFromRuns>", "k_multiply<Src>",
        "k_merge_xl", "(k_merge_chain<uint32_t, false>)", "k_multiply<Src>", "k_merge_xl",
        "(k_merge_chain<uint32_t, false>)", "k_multiply<Src>", "k_merge_xl", "(k_merge_chain<uint32_t, false>)",
        "k_multiply<Src>", "k_merge_xl", "(k_merge_chain<uint32_t, false>)"
    ], 21, 4, 7, 2, 2),
    "fused_lanes_full_rows": ([
        "k_validate_starts", "k_validate", "(k_scan<SymIn, RunOffOut>)", "k_plan<RowBinFromRuns>", "k_fl_count",
        "k_fl_fill", "(k_scan<RowCapIn, U64Out>)", "k_fused_lanes<2>"
    ], 12, 1, 20, 5, 15),
    "fused_lanes_compact": ([
        "k_validate_starts", "k_validate", "(k_scan<SymIn, RunOffOut>)", "k_plan<RowBinFromRuns>", "k_fl_count",
        "k_fl_fill", "(k_scan<RowCapIn, U64Out>)", "k_fused_lanes<2>", "(k_scan<U32In, U64Out>)", "k_fl_compact"
    ], 14, 1, 20, 20, 0),
    "fused_lanes_chained": ([
        "k_validate_starts", "k_validate", "(k_scan<SymIn, RunOffOut>)", "k_plan<RowBinFromRuns>", "k_fl_count",
        "k_fl_fill", "k_fused_lanes<2>"
    ], 10, 1, 20, 20, 0),
    "fused_band_kernel": ([
        "k_validate_starts", "k_validate", "(k_scan<SymIn, RunOffOut>)", "k_plan<RowBinFromRuns>", "k_band_ptr",
        "k_fused_dense"
    ], 8, 1, 20, 20, 0),
    "no_fused_dense": ([
        "k_validate_starts", "k_validate", "(k_scan<SymIn, RunOffOut>)", "k_plan<RowBinFromRuns>", "k_multiply<Src>",
        "k_merge_dense", "(k_merge_chain<uint32_t, true>)"
    ], 9, 1, 20, 20, 0),
    "longrow_sweep": ([
        "k_validate_starts", "k_validate", "(k_scan<SymIn, RunOffOut>)", "k_plan<RowBinFromRuns>", "k_mark_swept",
        "k_long_bands", "k_multiply<Src>", "(k_long_fill<LR_THREADS, LR_BAND, LR_RUNS, LongRowsInBins>)", "k_merge_xl",
        "(k_merge_chain<uint32_t, false>)"
    ], 12, 1, 7, 2, 2),
    "kway_merge": ([
        "k_validate_starts", "k_validate", "(k_scan<SymIn, RunOffOut>)", "k_plan<RowBinFromRuns>", "k_multiply<Src>",
        "k_merge_ways", "k_merge_xl", "(k_merge_chain<uint32_t, false>)"
    ], 10, 1, 7, 2, 2),
    "fused_short_chain2": ([
        "k_validate_starts", "k_validate", "(k_scan<SymIn, RunOffOut>)", "k_plan<RowBinFromRuns>", "k_mark_binned",
        "k_multiply<Src>", "k_merge_xl", "(k_chain2<uint32_t, false, C2SrcProduct>)"
    ], 10, 1, 7, 2, 2),
    "fused_short_old": ([
        "k_validate_starts", "k_validate", "(k_scan<SymIn, RunOffOut>)", "k_plan<RowBinFromRuns>", "k_mark_binned",
        "k_multiply<Src>", "k_merge_xl", "(k_merge_chain_fused<uint32_t, false>)"
    ], 10, 1, 7, 2, 2),
    "fused_short_no_medium_rows": ([
        "k_validate_starts", "k_validate", "(k_scan<SymIn, RunOffOut>)", "k_plan<RowBinFromRuns>",
        "(k_chain2<uint32_t, false, C2SrcProduct>)"
    ], 7, 1, 4, 0, 0),
    "bpos32": ([
        "k_validate_starts", "k_validate", "k_narrow_pos", "(k_scan<SymIn, RunOffOut>)", "k_plan<RowBinFromRuns>",
        "k_multiply<Src>", "k_merge_xl", "(k_merge_chain<uint32_t, false>)"
    ], 10, 1, 7, 2, 2),
    "no_validate_derived_cols": ([
        "k_max_idx", "(k_scan<SymIn, RunOffOut>)", "k_plan<RowBinFromRuns>", "k_multiply<Src>", "k_merge_xl",
        "(k_merge_chain<uint32_t, false>)"
    ], 8, 1, 7, 2, 2),
    "empty_a": ([
        "k_validate_starts", "k_validate", "k_plan<RowBinFromRuns>", "(k_merge_chain<uint32_t, false>)"
    ], 6, 1, 1, 0, 0),
}

# calls that fail, each followed by an exact call on the same context.  id: (flags, operands, cols_b, workspace limit in
# partial products, result limit in bytes)
TOP = (1 << 32) - 1
FAILING_CASES = {
    "fail_index_after_kslice_fork": (K, "column_beyond_cols_b", 1 << 17, 0, 0),
    "fail_duplicate": (0, "duplicate", 1 << 17, 0, 0),
    "fail_csc_row_id_2_32_minus_1": (0, "csc_row_top", 0, 0, 0),
    "fail_column_id_2_32_minus_1": (0, "column_top", 0, 0, 0),
    "fail_admission": (0, "rows", 1 << 17, 6000, 4096),
    "fail_accumulator_limit": (0, "accumulator", TOP, 0, 0),
}

# id: (return code, osp_last_error text)
FAILING_EXPECTED = {
    "fail_index_after_kslice_fork": (api.OSP_ERR_INDEX,
        "osp_spgemm: index out of range (k of A beyond the inner dimension, or a column of B beyond cols_b)"),
    "fail_duplicate": (api.OSP_ERR_DUPLICATE,
        "osp_spgemm: duplicate (row,col) entry in operand"),
    "fail_csc_row_id_2_32_minus_1": (api.OSP_ERR_INDEX,
        "osp_spgemm: a row id of CSC(A) is 2^32 - 1; row ids must be below 2^32 - 1"),
    "fail_column_id_2_32_minus_1": (api.OSP_ERR_INDEX,
        "osp_spgemm: a column id of B is 2^32 - 1; column ids must be below 2^32 - 1"),
    "fail_admission": (api.OSP_ERR_OOM,
        "osp_spgemm: C does not fit the device: 0 non-zeros in the first 0 of 2 row blocks + a bound of 5482 for the next "
        "exceed the capacity of 512"),
    "fail_accumulator_limit": (api.OSP_ERR_UNSUPPORTED,
        "long-row accumulator does not fit: column range too large"),
}


def _failing_operands(kind, cols):
    rng = np.random.default_rng(zlib.crc32(kind.encode()))
    if kind == "csc_row_top":                          # CSC(A): row id 2^32 - 1 would give 2^32 rows
        a = osp.CSRMatrix.from_arrays(np.array([0, 1, 2], np.uint64), np.array([4, TOP], np.uint32), np.ones(2, np.float32))
        b = osp.CSRMatrix.from_arrays(np.array([0, 1, 2], np.uint64), np.array([3, 9], np.uint32), np.ones(2, np.float32))
        return a, b, False
    if kind == "accumulator":                          # a long row over 2^32 - 1 columns: its accumulator cannot fit
        a, b = ge.rows_case(rng, [3, 600, 6000], cols, lo=1 << 31)
        return a, b, True
    a, b = ge.rows_case(rng, PATH_LENS, 1 << 17)
    idx = b.data["idx"]
    if kind == "column_beyond_cols_b":
        idx[-1] = cols
    elif kind == "duplicate":
        r = int(np.flatnonzero(np.diff(b.pos.astype(np.int64)) >= 2)[0])
        idx[int(b.pos[r]) + 1] = idx[int(b.pos[r])]
    elif kind == "column_top":
        idx[-1] = TOP
    return a, b, True


def _path_operands(kind, cols):
    """(A, B, a_is_csr, oracle product) of one case."""
    rng = np.random.default_rng(zlib.crc32(kind.encode()) + cols)
    if kind in ("dense", "dense_full"):
        a = synth.pruned_dense(20, 512, 0.04, seed=1)                    # about 1500 partial products per row of C
        b = synth.pruned_dense(512, cols, 1.0 if kind == "dense_full" else 0.3, seed=2)   # every row of C full, or not
    elif kind == "empty":
        a = osp.CSRMatrix.from_arrays(np.zeros(5, np.uint64), np.zeros(0, np.uint32), np.zeros(0, np.float32))
        b = ge.rows_case(rng, [3, 7], cols)[1]
    else:
        a, b = ge.rows_case(rng, PATH_SHORT if kind == "short" else PATH_LENS, cols or (1 << 17))
    a_csc = synth.transpose_host(a, b.NRow())
    want, _ = oracle_spgemm(a_csc, b, rows_override=a.NRow())
    return (a_csc if kind == "rows_csc" else a), b, kind != "rows_csc", want


def _path_engine(monkeypatch, env, ws_elems, result_limit):
    for k, v in env.items():
        monkeypatch.setenv(k, v)                      # read at osp_create
    eng = osp.Engine(0)
    for k in env:
        monkeypatch.delenv(k)
    if ws_elems:
        eng.set_workspace_limit(ws_elems * 8)
    if result_limit:
        eng.set_result_limit(result_limit)
    return eng


@pytest.mark.parametrize("case", list(PATH_CASES) + list(FAILING_CASES))
def test_each_call_takes_its_path(emulated_library, monkeypatch, case):
    if case in FAILING_CASES:
        flags, kind, cols, ws, limit = FAILING_CASES[case]
        a, b, a_is_csr = _failing_operands(kind, cols)
        eng = _path_engine(monkeypatch, {}, ws, limit)
        try:
            with pytest.raises(osp.OspError) as ei:
                eng.spgemm(a, b, a_is_csr=a_is_csr, cols_b=cols, flags=flags)
            got_fail = (ei.value.code, str(ei.value))
            eng.set_result_limit(0)
            ok_a, ok_b, _, ok_want = _path_operands("rows", 1 << 17)
            res = eng.spgemm(ok_a, ok_b, a_is_csr=True, cols_b=1 << 17, flags=flags)       # the next call is exact
            got = res.to_host(); res.free()
        finally:
            eng.close()
        code, msg = FAILING_EXPECTED[case]
        assert got_fail == (code, f"osp error {code}: {msg}"), f"{case}: {got_fail!r}"
        assert_bit_exact(got, ok_want, f"{case}: the call after the failed one")
        return
    env, flags, kind, cols, ws, slack = PATH_CASES[case]
    a, b, a_is_csr, want = _path_operands(kind, cols)
    eng = _path_engine(monkeypatch, env, ws, (want.nnz + slack) * 8 if slack else 0)
    try:
        res = eng.spgemm(a, b, a_is_csr=a_is_csr, rows_c=a.NRow() if a_is_csr else 0, cols_b=cols,
                         flags=flags | api.OSP_PROFILE_KERNELS)
        names = [n for n, _ in res.kernel_times()]; res.free()
        res = eng.spgemm(a, b, a_is_csr=a_is_csr, rows_c=a.NRow() if a_is_csr else 0, cols_b=cols, flags=flags)
        got = res.to_host(); st = res.stats(); res.free()
    finally:
        eng.close()
    observed = (names, st["kernel_launches"], st["row_chunks"], st["merge_tiles"], st["rows_medium"], st["rows_long"])
    assert observed == PATH_EXPECTED[case], f"{case}: {observed!r}"
    assert_bit_exact(got, want, case)

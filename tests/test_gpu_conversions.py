"""GPU suite, the device format conversions: osp_csr2csc, osp_coo2csr_device and the CSC(A) hand-over of osp_spgemm
(TaskProvider(lmatCSC, rmatCSR), the reference's own boundary).  All three scatter elements into buckets (one per
output slice) and sort every bucket by its ids with the merge machinery of the product -- the merge chain in its three
key variants, k_merge_dense, k_merge_long, k_merge_xl -- with the index range (n_major, n_other, n_k) in place of the
column range; a bucket that shrank while folding held a duplicate (233).

A conversion does no arithmetic: its output must be a bit-exact permutation of its input, NaN payloads, -0.0 and
subnormals included, so conversions are compared as raw 64-bit words.  Every case of the dispatch grid names the
kernels the conversion must reach (OSP_PROFILE_KERNELS through the CSC hand-over), so a case that drifts off its kernel
fails.  tests/test_engine_sim.py runs the cases that fit the CPU emulation."""
import os
import zlib

import numpy as np
import pytest

import oracle
import outerspace_b200 as osp
from outerspace_b200 import api, synth
from helpers import assert_bit_exact, oracle_spgemm
import test_gpu_edges as ge
from test_gpu_edges import (NANS, SPECIALS, THRESHOLDS, _device_only, assert_close_to_f64, assert_same_up_to_nan,
                            inject_specials, rows_case)

pytestmark = pytest.mark.gpu

F32 = np.float32
GRID_LENS = [0, 1, 2, 8, 9, 128, 129, 512, 513, 640, 641, 4096, 4097, 5000]
DUP_LENS = [L for L in GRID_LENS if L >= 2]
COLS_B = 1000                     # columns of B in the hand-over products: C's own rows stay short


# ---- operands -----------------------------------------------------------------------------------------------------------
def bucket_matrix(rng, lens, idx_range, lo=0, ends=False):
    """CSR M, one row per bucket: bucket i holds min(lens[i], idx_range - lo) distinct ids from [lo, idx_range), with
    idx_range - 1 in every non-empty bucket (and `lo` too when `ends`).  Values: random bit patterns, SPECIALS (five NaN
    payloads, +-Inf, subnormals, -0.0) in every third element.  M is what converting its transpose must give back."""
    rows = []
    for L in lens:
        L = min(L, idx_range - lo)
        fixed = [idx_range - 1] + ([lo] if ends and L >= 2 else [])
        if L == 0:
            rows.append(np.zeros(0, np.int64))
            continue
        rest = lo + len(fixed) - 1 + rng.choice(idx_range - lo - len(fixed), size=L - len(fixed), replace=False)
        rows.append(np.sort(np.concatenate((rest, fixed))))
    pos = np.zeros(len(rows) + 1, np.uint64)
    pos[1:] = np.cumsum([r.size for r in rows])
    ids = np.concatenate(rows).astype(np.uint32)
    val = rng.integers(0, 1 << 32, size=ids.size, dtype=np.uint64).astype(np.uint32).view(F32)
    val[::3] = SPECIALS[np.arange(val[::3].size) % SPECIALS.size]
    return osp.CSRMatrix.from_arrays(pos, ids, val)


def grid_matrix(idx_range):
    rng = np.random.default_rng(idx_range % 100003)
    lens = GRID_LENS * 2 + [20000]                  # (a bucket of every id where the range is below 20000)
    rng.shuffle(lens)
    return rng, bucket_matrix(rng, lens, idx_range)


def triplets(m, rng, transpose):
    """M as shuffled triplets: (bucket, id), or (id, bucket) with transpose."""
    bucket = np.repeat(np.arange(m.NRow(), dtype=np.uint32), np.diff(m.pos.astype(np.int64)))
    perm = rng.permutation(m.nnz)
    b, i, v = bucket[perm], m.data["idx"][perm], m.data["val"][perm]
    return api.COO(i, b, v) if transpose else api.COO(b, i, v)


def sparse_b(rng, n_k, cols=COLS_B, rows=48):
    """CSR(B) (n_k x cols): a few non-empty rows, n_k - 1 among them, of 1-3 entries."""
    nz = np.unique(np.append(rng.choice(n_k, size=min(rows, n_k), replace=False), n_k - 1))
    cnt = np.zeros(n_k, np.int64)
    cnt[nz] = rng.integers(1, 4, size=nz.size)
    pos = np.zeros(n_k + 1, np.uint64)
    pos[1:] = np.cumsum(cnt)
    idx = np.concatenate([np.sort(rng.choice(cols, size=c, replace=False)) for c in cnt[nz]]).astype(np.uint32)
    return osp.CSRMatrix.from_arrays(pos, idx, rng.standard_normal(idx.size).astype(F32))


# ---- comparisons ----------------------------------------------------------------------------------------------------------
def assert_same_words(got, want_pos, want_data, what):
    """pos identical, and every element identical as a raw 64-bit word (id and value bits)."""
    assert got.pos.shape == want_pos.shape and np.array_equal(got.pos, want_pos), f"{what}: pos differs"
    g = np.ascontiguousarray(got.data).view(np.uint64)
    w = np.ascontiguousarray(want_data).view(np.uint64)
    assert g.shape == w.shape, f"{what}: {g.size} elements instead of {w.size}"
    bad = np.nonzero(g != w)[0]
    assert bad.size == 0, f"{what}: {bad.size} elements differ, first at {bad[:5]}: " \
                          f"{[hex(x) for x in g[bad[:5]]]} vs {[hex(x) for x in w[bad[:5]]]}"


def conversion_kernels(idx_range):
    """Merge kernels a conversion over idx_range must launch when it has buckets of every length class."""
    chain = ge._chain_variant(idx_range)
    if idx_range <= 16384:
        return {chain, "k_merge_dense"}
    if idx_range <= 131072:
        return {chain, "k_merge_xl"}
    return {chain, "k_merge_long", "k_merge_xl"}


def split_at_conversion(names):
    """(kernels of the CSC(A) conversion, kernels of the product): the conversion ends with its k_check_same."""
    cut = next(i for i, n in enumerate(names) if "k_check_same" in n)
    return names[:cut], names[cut + 1:]


def merge_kernels(names):
    return {n.strip("()") for n in names if "k_merge" in n}


def _spgemm_profiled(eng, a, b, **kw):
    res = eng.spgemm(a, b, flags=kw.pop("flags", 0) | api.OSP_PROFILE_KERNELS, **kw)
    got = res.to_host(); names = [n for n, _ in res.kernel_times()]; res.free()
    return got, names


def _emulated():
    return "cusim" in os.path.basename(api._LIB_PATH)


# ---- 1. the dispatch grid, three ways ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("idx_range", THRESHOLDS)
def test_csr2csc_dispatch_grid(engine, idx_range):
    """osp_csr2csc of the transpose of a matrix with buckets of every length class: the matrix, word for word."""
    rng, m = grid_matrix(idx_range)
    x = synth.transpose_host(m, idx_range)             # CSR with idx_range slices, ids = bucket ids
    pos, data = oracle.csr2csc(idx_range, m.NRow(), x.pos, x.data)
    assert_same_words(osp.CSRMatrix(pos, data), m.pos, m.data, "oracle")
    got = engine.csr2csc(x, m.NRow())
    assert_same_words(got, pos, data, f"osp_csr2csc n_major={idx_range}")


@pytest.mark.parametrize("idx_range", THRESHOLDS)
def test_coo_ingest_dispatch_grid(engine, idx_range):
    """osp_coo2csr_device of shuffled triplets, both orientations, n_other given and derived: the host coo2csr."""
    rng, m = grid_matrix(idx_range)
    for transpose in (False, True):
        coo = triplets(m, rng, transpose)
        want = api.coo2csr(coo, m.NRow(), transpose)
        assert_same_words(want, m.pos, m.data, f"host coo2csr transpose={transpose}")
        for n_other in (idx_range, 0):
            got = engine.coo2csr(coo, m.NRow(), transpose, n_other)
            assert_same_words(got, want.pos, want.data, f"coo2csr_device n_other={n_other} transpose={transpose}")


@pytest.mark.parametrize("idx_range", THRESHOLDS)
def test_csc_hand_over_dispatch_grid(engine, idx_range):
    """The rows of A are the buckets (n_k = idx_range): the conversion reaches the kernels of its range, the product
    matches the oracle and the float64 product, and is bit for bit the product of the CSR hand-over."""
    rng, a = grid_matrix(idx_range)
    a_csc = synth.transpose_host(a, idx_range)
    b = sparse_b(rng, idx_range)
    rows = a.NRow()
    got, names = _spgemm_profiled(engine, a_csc, b, rows_c=rows, cols_b=COLS_B)
    conv, _ = split_at_conversion(names)
    reached = merge_kernels(conv)
    print(f"n_k={idx_range}: conversion reached {sorted(reached)}")
    assert reached == conversion_kernels(idx_range), f"n_k={idx_range}: {conv}"
    want, _ = oracle_spgemm(a_csc, b, rows_override=rows)
    assert_same_up_to_nan(got, want, f"CSC(A) n_k={idx_range}")
    assert_close_to_f64(got, a, b, f"CSC(A) n_k={idx_range}")
    res = engine.spgemm(a, b, a_is_csr=True, rows_c=rows, cols_b=COLS_B)
    got_csr = res.to_host(); res.free()
    assert_bit_exact(got, got_csr, f"CSC(A) vs CSR(A) n_k={idx_range}")


@pytest.mark.parametrize("case", list(ge.KERNEL_CASES))
def test_csc_hand_over_of_each_merge_kernel_case(monkeypatch, case):
    """The special-value cases of test_gpu_edges, one per merge kernel, with A handed over as CSC."""
    kernel, env, flags, cols, lens = ge.KERNEL_CASES[case]
    rng = np.random.default_rng(zlib.crc32(case.encode()))
    lens = list(lens)
    rng.shuffle(lens)
    a, b = rows_case(rng, lens, cols)
    inject_specials(rng, a, b)
    a_csc = synth.transpose_host(a, b.NRow())
    want, _ = oracle_spgemm(a_csc, b)
    eng = ge._engine_with(monkeypatch, env)
    try:
        got, names = _spgemm_profiled(eng, a_csc, b, cols_b=cols, flags=flags)
    finally:
        eng.close()
    ge._reached(split_at_conversion(names)[1], kernel, case)
    assert_same_up_to_nan(got, want, case)
    assert_close_to_f64(got, a, b, case)


# ---- 2. duplicates in every bucket class ------------------------------------------------------------------------------------
def _with_duplicate(m, x, slot, val):
    """M of one bucket and its transpose x: element `slot` of the bucket (its first or last source slice) duplicated, the
    two copies valued `val`.  Returns (x with the copy in the same slice, triplets with the copies first and last in
    arrival)."""
    s = int(m.data["idx"][slot])
    data = m.data.copy()
    data["val"][slot] = val[0]
    copy = data[slot:slot + 1].copy()
    copy["val"] = val[1]
    xd = x.data.copy()
    xd["val"][int(x.pos[s])] = val[0]
    x_dup = osp.CSRMatrix(x.pos + (np.arange(x.pos.size) > s).astype(np.uint64),
                          np.insert(xd, int(x.pos[s]) + 1, np.array([(0, val[1])], osp.ELEM)))
    rest = np.delete(data, slot)
    order = np.random.default_rng(s).permutation(rest.size)
    d = np.concatenate((data[slot:slot + 1], rest[order], copy))
    coo = api.COO(np.zeros(d.size, np.uint32), d["idx"].copy(), d["val"].copy())
    return x_dup, coo


def duplicate_cases(engine, idx_range, through_slices=True):
    """One duplicated (slice, id) pair in a bucket of each length from 2 to 5000, at the first or the last source slice
    of the bucket (the copies first and last in arrival for the triplets); values that cancel (+1, -1) and two NaNs.
    osp_coo2csr_device, and with `through_slices` osp_csr2csc and the CSC hand-over (with OSP_NO_VALIDATE too, then
    from the conversion's own check), raise 233, and the next call converts exactly."""
    rng = np.random.default_rng(idx_range % 99991 + 7)
    b = sparse_b(rng, idx_range) if through_slices else None
    nan2 = np.array(NANS[:2], np.uint32).view(F32)
    for i, L in enumerate(DUP_LENS):
        m = bucket_matrix(rng, [L], idx_range, ends=True)
        x = synth.transpose_host(m, idx_range)
        first, last = 0, m.nnz - 1
        for slot, val, kind in (((first, last)[i % 2], (1.0, -1.0), "cancel"), ((last, first)[i % 2], nan2, "NaN")):
            what = f"n_major={idx_range} bucket of {L}, {kind} pair at slice {int(m.data['idx'][slot])}"
            x_dup, coo = _with_duplicate(m, x, slot, np.asarray(val, F32))
            with pytest.raises(osp.DuplicateEntry, match="duplicate"):
                engine.coo2csr(coo, 1, False, idx_range)
            clean = triplets(m, rng, False)
            assert_same_words(engine.coo2csr(clean, 1, False, idx_range), m.pos, m.data, f"{what}: the next call")
            if not through_slices:
                continue
            with pytest.raises(osp.DuplicateEntry, match="duplicate"):
                engine.csr2csc(x_dup, 1)
            with pytest.raises(osp.DuplicateEntry) as ei:
                engine.spgemm(x_dup, b, rows_c=1, cols_b=COLS_B)
            assert ei.value.code == 233 and "osp_spgemm (A)" in str(ei.value), f"{what}: {ei.value}"
            with pytest.raises(osp.DuplicateEntry) as ei:
                engine.spgemm(x_dup, b, rows_c=1, cols_b=COLS_B, flags=api.OSP_NO_VALIDATE)
            assert ei.value.code == 233 and "osp_spgemm (A)" not in str(ei.value), f"{what}: {ei.value}"
            assert_same_words(engine.csr2csc(x, 1), m.pos, m.data, f"{what}: the next call")
    if not through_slices:
        return
    want, _ = oracle_spgemm(x, b, rows_override=1)
    res = engine.spgemm(x, b, rows_c=1, cols_b=COLS_B, flags=api.OSP_NO_VALIDATE)
    got = res.to_host(); res.free()
    assert_same_up_to_nan(got, want, f"n_k={idx_range}: the product after the refused calls")


@pytest.mark.parametrize("idx_range", THRESHOLDS)
def test_duplicate_in_every_bucket_class(engine, idx_range):
    duplicate_cases(engine, idx_range)


# ---- 3. device pointers -----------------------------------------------------------------------------------------------------
class _DeviceBuffers:
    """Device allocations by torch on a GPU; host arrays on the CPU emulation, whose device memory is host memory."""

    def __init__(self):
        self.keep = []
        self.torch = None if _emulated() else pytest.importorskip("torch")

    def upload(self, arr):
        raw = np.ascontiguousarray(arr).view(np.uint8).reshape(-1).copy()
        if self.torch is None:
            buf = np.concatenate((raw, np.zeros(8, np.uint8)))         # (never an empty allocation)
        else:
            buf = self.torch.from_numpy(np.concatenate((raw, np.zeros(8, np.uint8)))).to("cuda:0")
            self.torch.cuda.synchronize()
        self.keep.append(buf)
        return buf, buf.ctypes.data if self.torch is None else buf.data_ptr()

    def empty(self, nbytes):
        return self.upload(np.full(nbytes, 0xA5, np.uint8))

    def download(self, buf, dtype, n):
        if self.torch is not None:
            self.torch.cuda.synchronize()              # (the engine's stream: an empty conversion returns unsynchronised)
        raw = buf if self.torch is None else buf.cpu().numpy()
        return raw[: n * np.dtype(dtype).itemsize].view(dtype).copy()


def test_conversions_with_device_pointers(engine):
    """osp_csr2csc and osp_coo2csr_device with OSP_DEVICE_POINTERS on a grid case (k_merge_long and k_merge_xl); n_other
    = 0 is OSP_ERR_INVALID there (the ids are on the device)."""
    idx_range = 131073
    rng, m = grid_matrix(idx_range)
    x = synth.transpose_host(m, idx_range)
    nb = m.NRow()
    dev = _DeviceBuffers()
    _, p_pos = dev.upload(x.pos)
    _, p_data = dev.upload(x.data)
    pos_out, p_pos_out = dev.empty((nb + 1) * 8)
    data_out, p_data_out = dev.empty(m.nnz * 8)
    engine.csr2csc_device(idx_range, nb, p_pos, p_data, p_pos_out, p_data_out)
    got = osp.CSRMatrix(dev.download(pos_out, np.uint64, nb + 1), dev.download(data_out, osp.ELEM, m.nnz))
    assert_same_words(got, m.pos, m.data, "osp_csr2csc, device pointers")
    for transpose in (False, True):
        coo = triplets(m, rng, transpose)
        _, pr = dev.upload(coo.rows)
        _, pc = dev.upload(coo.cols)
        _, pv = dev.upload(coo.vals)
        pos_out, p_pos_out = dev.empty((nb + 1) * 8)
        data_out, p_data_out = dev.empty(m.nnz * 8)
        engine.coo2csr_device(m.nnz, pr, pc, pv, nb, idx_range, p_pos_out, p_data_out, transpose)
        got = osp.CSRMatrix(dev.download(pos_out, np.uint64, nb + 1), dev.download(data_out, osp.ELEM, m.nnz))
        assert_same_words(got, m.pos, m.data, f"osp_coo2csr_device, device pointers, transpose={transpose}")
        with pytest.raises(osp.OspError) as ei:
            engine.coo2csr_device(m.nnz, pr, pc, pv, nb, 0, p_pos_out, p_data_out, transpose)
        assert ei.value.code == api.OSP_ERR_INVALID, str(ei.value)


# ---- 4. index edges ---------------------------------------------------------------------------------------------------------
def test_coo_ids_up_to_2_32(engine):
    """Kept ids up to 2^32 - 2 with n_other = 2^32 - 1 given, and up to 2^32 - 1 with n_other derived, in buckets of
    1 .. 4096: bit-exact.  A bucket of 5000 with n_other = 2^32 - 1 needs a long-row accumulator of 17 GB, more than
    the engine may take: OSP_ERR_UNSUPPORTED, and the context works afterwards."""
    rng = np.random.default_rng(232)
    lens = [L for L in GRID_LENS if 1 <= L <= 4096] * 2
    rng.shuffle(lens)
    cases = []
    for top, n_other in ((0xFFFFFFFE, 0xFFFFFFFF), (0xFFFFFFFF, 0)):
        m = bucket_matrix(rng, lens, top + 1, lo=1 << 31)
        assert int(m.data["idx"].max()) == top and int(m.data["idx"].min()) >= 1 << 31
        for transpose in (False, True):
            coo = triplets(m, rng, transpose)
            want = api.coo2csr(coo, m.NRow(), transpose)
            assert_same_words(want, m.pos, m.data, f"host coo2csr, largest id {top:#x}")
            got = engine.coo2csr(coo, m.NRow(), transpose, n_other)
            assert_same_words(got, m.pos, m.data, f"coo2csr_device, largest id {top:#x}, n_other={n_other}, "
                                                  f"transpose={transpose}")
            cases.append((coo, m, transpose, n_other))
    big = bucket_matrix(rng, [3, 700, 5000], 0xFFFFFFFF, lo=1 << 31)
    with pytest.raises(osp.OspError) as ei:
        engine.coo2csr(triplets(big, rng, False), big.NRow(), False, 0xFFFFFFFF)
    assert ei.value.code == api.OSP_ERR_UNSUPPORTED and "column range too large" in str(ei.value), str(ei.value)
    coo, m, transpose, n_other = cases[0]
    assert_same_words(engine.coo2csr(coo, m.NRow(), transpose, n_other), m.pos, m.data, "after the refused call")


def test_coo_bucket_through_k_merge_xl_above_2_31(engine):
    """A bucket of 5000 with n_other = 2^31 + 5: k_merge_xl with an 8.6 GB accumulator, bit-exact."""
    _device_only(engine)
    rng = np.random.default_rng(2315)
    n_other = (1 << 31) + 5
    m = bucket_matrix(rng, [5000, 1, 600, 4097], n_other, lo=n_other - 100000)
    for transpose in (False, True):
        coo = triplets(m, rng, transpose)
        got = engine.coo2csr(coo, m.NRow(), transpose, n_other)
        assert_same_words(got, m.pos, m.data, f"n_other = 2^31 + 5, transpose={transpose}")


# ---- 5. no output slice -----------------------------------------------------------------------------------------------------
def test_conversions_into_zero_slices(engine):
    """With entries and no output slice every id is out of range: OSP_ERR_INDEX, through the host- and the device-pointer
    entry points of both conversions (not success with the entries dropped).  Without entries: success, pos = [0]."""
    E = osp.ELEM
    m = osp.CSRMatrix(np.array([0, 2, 3], np.uint64), np.array([(0, 1.0), (1, 2.0), (0, 3.0)], E))
    coo = api.COO(np.array([0, 1, 1], np.uint32), np.array([0, 0, 2], np.uint32), np.array([1, 2, 3], F32))
    empty_m = osp.CSRMatrix(np.zeros(3, np.uint64), np.zeros(0, E))
    empty_coo = api.COO(np.zeros(0, np.uint32), np.zeros(0, np.uint32), np.zeros(0, F32))

    def refused(call, what):
        with pytest.raises(osp.OspError) as ei:
            call()
        assert ei.value.code == api.OSP_ERR_INDEX, f"{what}: {ei.value}"

    refused(lambda: engine.csr2csc(m, 0), "osp_csr2csc")
    for transpose in (False, True):
        for n_other in (0, 3):
            refused(lambda: engine.coo2csr(coo, 0, transpose, n_other), f"osp_coo2csr_device n_other={n_other}")
    got = engine.csr2csc(empty_m, 0)
    assert got.nnz == 0 and np.array_equal(got.pos, np.zeros(1, np.uint64))
    got = engine.coo2csr(empty_coo, 0)
    assert got.nnz == 0 and np.array_equal(got.pos, np.zeros(1, np.uint64))

    dev = _DeviceBuffers()
    _, p_pos = dev.upload(m.pos)
    _, p_data = dev.upload(m.data)
    pos_out, p_pos_out = dev.empty(8 * 4)
    _, p_data_out = dev.empty(8 * 4)
    refused(lambda: engine.csr2csc_device(2, 0, p_pos, p_data, p_pos_out, p_data_out), "osp_csr2csc, device pointers")
    _, pr = dev.upload(coo.rows)
    _, pc = dev.upload(coo.cols)
    _, pv = dev.upload(coo.vals)
    for transpose in (False, True):
        refused(lambda: engine.coo2csr_device(3, pr, pc, pv, 0, 3, p_pos_out, p_data_out, transpose),
                "osp_coo2csr_device, device pointers")
    _, p_epos = dev.upload(empty_m.pos)
    pos_out, p_pos_out = dev.empty(8)
    engine.csr2csc_device(2, 0, p_epos, p_data, p_pos_out, p_data_out)
    assert np.array_equal(dev.download(pos_out, np.uint64, 1), np.zeros(1, np.uint64))
    pos_out, p_pos_out = dev.empty(8)
    engine.coo2csr_device(0, pr, pc, pv, 0, 3, p_pos_out, p_data_out)
    assert np.array_equal(dev.download(pos_out, np.uint64, 1), np.zeros(1, np.uint64))
    got = engine.csr2csc(m, 3)                                            # the context works afterwards
    want_pos, want_data = oracle.csr2csc(2, 3, m.pos, m.data)
    assert_same_words(got, want_pos, want_data, "after the refused calls")


# ---- 6. a skewed product through the CSC hand-over ----------------------------------------------------------------------------
def test_skewed_product_through_the_csc_hand_over(engine):
    """Config 3's shape at 1/16 (R-MAT, n_k = 65536): hub rows of A beyond 4096 entries take k_merge_xl inside the
    conversion.  The conversion equals the oracle's word for word, and the product of the CSC hand-over is bit for bit the
    product of the CSR hand-over (pinned to the oracle by test_rmat_small at a smaller scale).  4e8 partial products:
    on a B200 only."""
    if _emulated():
        pytest.skip("4e8 partial products: on a B200 only")
    a, b, dims = synth.build_workload("rmat20", scale_down=16)
    n = dims["n_k"]
    assert np.diff(a.pos.astype(np.int64)).max() > 4096
    a_csc = synth.transpose_host(a, n)
    pos, data = oracle.csr2csc(n, n, a_csc.pos, a_csc.data)
    got = engine.csr2csc(a_csc, n)
    assert_same_words(got, pos, data, "osp_csr2csc of CSC(A)")
    assert_same_words(got, a.pos, a.data, "CSR(A)")
    res = engine.spgemm(a_csc, b, flags=api.OSP_PROFILE_KERNELS)
    names = [k for k, _ in res.kernel_times()]
    conv, _ = split_at_conversion(names)
    print(f"rmat16: conversion reached {sorted(merge_kernels(conv))}")
    assert "k_merge_xl" in merge_kernels(conv), conv
    got_csc = res.to_host(); res.free()
    res = engine.spgemm(a, b, a_is_csr=True)
    got_csr = res.to_host(); res.free()
    assert_bit_exact(got_csc, got_csr, "rmat16: CSC(A) vs CSR(A)")

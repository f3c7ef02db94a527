"""GPU suite, edges of the value and index ranges: special float values through every merge kernel, the column-range
thresholds of the dispatch from both sides, column ids of 2^31 and above, the 32-bit copy of B.pos.

Values: NaN sits at exactly the oracle's entries (its payload is not compared: the device returns the canonical NaN,
test_nan_payload_of_device_arithmetic), every other value is bit-identical, and nothing is dropped or added because of
its value.  Finite entries are also held against a float64 product (assert_close_to_f64), which checks the oracle and the
engine together.  Every case names the kernel it must reach (OSP_PROFILE_KERNELS), so a case that drifts off its kernel
fails instead of passing on another path.  tests/test_engine_sim.py runs the cases that fit the CPU emulation."""
import os
import zlib

import numpy as np
import pytest

import outerspace_b200 as osp
from outerspace_b200 import api, synth
from helpers import assert_bit_exact, check_csr_invariants, oracle_spgemm
import test_gpu_parity as gp

pytestmark = pytest.mark.gpu

F32 = np.float32
NANS = [0x7FC00000, 0xFFC00000, 0x7F800001, 0xFFFFFFFF, 0x7FFFFFFF]   # 0xFFFFFFFF: k_fused_lanes' "never touched"
SPECIALS = np.array(NANS + [0x7F800000, 0xFF800000,                   # +-Inf
                            0x00000001, 0x807FFFFF, 0x00400000,       # subnormals
                            0x00000000, 0x80000000,                   # +-0.0
                            0x7F7FFFFF, 0xFF7FFFFF, 0x7F000000], np.uint32).view(F32)   # near FLT_MAX
FLT_MAX = float(np.finfo(F32).max)


# ---- comparison helpers -----------------------------------------------------------------------------------------------
def assert_same_up_to_nan(got, want, what=""):
    """row_ptr and col_idx identical; NaN at exactly the same entries; every other value bit-identical (+-0.0, +-Inf)."""
    assert got.pos.shape == want.pos.shape and np.array_equal(got.pos, want.pos), f"{what}: row_ptr differs"
    assert np.array_equal(got.data["idx"], want.data["idx"]), f"{what}: col_idx differs"
    g, w = got.data["val"], want.data["val"]
    gn, wn = np.isnan(g), np.isnan(w)
    bad = np.nonzero(gn != wn)[0]
    assert bad.size == 0, f"{what}: NaN at {bad.size} other entries, first at {bad[:5]}: {g[bad[:5]]} vs {w[bad[:5]]}"
    bad = np.nonzero(g.view(np.uint32)[~gn] != w.view(np.uint32)[~wn])[0]
    assert bad.size == 0, f"{what}: {bad.size} values differ bitwise, first {g[~gn][bad[:5]]} vs {w[~wn][bad[:5]]}"


def f64_product(a, b):
    """C = A*B from CSR(A), CSR(B) in float64, entry by entry: (row, column, value, sum_k |a_ik b_kj|, partial products).
    Entries are the union of the B rows each row of A selects (explicit zeros included)."""
    apos, bpos = a.pos.astype(np.int64), b.pos.astype(np.int64)
    ak = a.data["idx"].astype(np.int64)
    arow = np.repeat(np.arange(a.NRow(), dtype=np.int64), np.diff(apos))
    cnt = np.diff(bpos)[ak]
    src = np.repeat(np.arange(ak.size), cnt)
    bp = bpos[:-1][ak][src] + np.arange(src.size) - np.repeat(np.cumsum(cnt) - cnt, cnt)
    key = (arow[src] << 32) | b.data["idx"][bp].astype(np.int64)
    uk, inv = np.unique(key, return_inverse=True)
    with np.errstate(invalid="ignore", over="ignore"):
        prod = a.data["val"][src].astype(np.float64) * b.data["val"][bp].astype(np.float64)
        val = np.bincount(inv, weights=prod, minlength=uk.size)
        mag = np.bincount(inv, weights=np.abs(prod), minlength=uk.size)
    return uk >> 32, uk & 0xFFFFFFFF, val, mag, np.bincount(inv, minlength=uk.size)


def assert_close_to_f64(got, a, b, what=""):
    """Structure = the union of the selected rows of B; every finite entry within the bound of a k-ordered recursive
    sum of separately rounded products, |c - c64| <= (n + 1) 2^-24 sum_k |a_ik b_kj| (+ (n + 1) 2^-149 for results in
    the subnormal range); an entry overflows only where sum_k |a_ik b_kj| reaches FLT_MAX; a non-finite float64 value
    is never a finite one."""
    row, col, c64, mag, n = f64_product(a, b)
    rows = np.repeat(np.arange(got.NRow(), dtype=np.int64), np.diff(got.pos.astype(np.int64)))
    assert rows.size == row.size and np.array_equal(rows, row), f"{what}: rows of C are not the union of the selected rows of B"
    assert np.array_equal(got.data["idx"].astype(np.int64), col), f"{what}: columns are not the union of the selected rows of B"
    c = got.data["val"].astype(np.float64)
    fin = np.isfinite(c)
    ok = fin & np.isfinite(c64)
    bound = (n + 1) * (2.0 ** -24 * mag + 2.0 ** -149)
    with np.errstate(invalid="ignore"):
        bad = np.nonzero(ok & ~(np.abs(c - c64) <= bound))[0]
    assert bad.size == 0, f"{what}: {bad.size} entries beyond the error bound, first {c[bad[:5]]} vs {c64[bad[:5]]}"
    bad = np.nonzero(fin & ~np.isfinite(c64))[0]
    assert bad.size == 0, f"{what}: finite where the float64 product is not: {c[bad[:5]]} vs {c64[bad[:5]]}"
    bad = np.nonzero(~fin & np.isfinite(c64) & (mag < FLT_MAX))[0]
    assert bad.size == 0, f"{what}: overflow without a partial sum that can reach FLT_MAX: {c[bad[:5]]} vs {c64[bad[:5]]}"


# ---- operands ---------------------------------------------------------------------------------------------------------
def rows_case(rng, lens, cols, lo=0, dup=0.3, ways=6):
    """CSR(A) (rows x rows*ways, one element per row and way) and CSR(B): output row i merges exactly lens[i] partial
    products, columns drawn from [lo, cols) with column cols - 1 in every non-empty row, a fraction `dup` of them repeated
    across the ways (the k-ordered fold)."""
    b_rows = []
    for L in lens:
        parts = np.diff(np.concatenate(([0], np.sort(rng.integers(0, L + 1, size=ways - 1)), [L])))
        npool = max(int(parts.max()), int(L * (1 - dup)), 1)
        pool = np.unique(np.concatenate((lo + rng.choice(cols - lo - 1, size=npool - 1, replace=False), [cols - 1])))
        while pool.size < npool:                               # (a repeat of cols - 1 drawn above)
            pool = np.unique(np.concatenate((pool, lo + rng.choice(cols - lo - 1, size=npool - pool.size, replace=False))))
        first = True
        for n in parts:
            c = rng.choice(pool, size=int(n), replace=False)
            if n and first:
                if cols - 1 not in c:
                    c[0] = cols - 1
                first = False
            b_rows.append(np.sort(c))
    rows = len(lens)
    a = osp.CSRMatrix.from_arrays(np.arange(rows + 1, dtype=np.uint64) * ways, np.arange(rows * ways, dtype=np.uint32),
                                  (rng.standard_normal(rows * ways) + 3).astype(F32))
    pos = np.zeros(len(b_rows) + 1, np.uint64)
    pos[1:] = np.cumsum([r.size for r in b_rows])
    idx = np.concatenate(b_rows).astype(np.uint32) if b_rows else np.zeros(0, np.uint32)
    b = osp.CSRMatrix.from_arrays(pos, idx, rng.standard_normal(idx.size).astype(F32))
    return a, b


def inject_specials(rng, a, b, every=37):
    """Special values in place: in row r of A (every few rows) one column whose k-ordered fold overflows (3e38, 3e38,
    -3e38: finite in any other order), one summed from subnormals only, one whose products are all -0.0, one way whose
    products of normal inputs underflow (1e-20 * 1e-20); then NaNs of five patterns, +-Inf, subnormals, +-0.0 and
    near-FLT_MAX values sprinkled over the other elements of B, and NaN, Inf (Inf * 0), -0.0 and 1e-20 over A."""
    av, bv = a.data["val"], b.data["val"]
    apos, bpos = a.pos.astype(np.int64), b.pos.astype(np.int64)
    bidx = b.data["idx"]
    keep_a = np.zeros(av.size, bool)
    keep_b = np.zeros(bv.size, bool)
    for r in range(0, a.NRow(), 2):
        ea = np.arange(apos[r], apos[r + 1])
        if ea.size == 0 or np.any(keep_a[ea]):
            continue
        ks = a.data["idx"][ea].astype(np.int64)
        pb = np.concatenate([np.arange(bpos[k], bpos[k + 1]) for k in ks])
        if pb.size == 0 or np.any(keep_b[pb]):
            continue
        owner = np.concatenate([np.full(bpos[k + 1] - bpos[k], j) for j, k in enumerate(ks)])   # element of A behind each
        cols, cnt = np.unique(bidx[pb], return_counts=True)
        av[ea] = np.abs(av[ea])
        used = set()
        three = cols[cnt >= 3]
        if three.size:
            c = three[rng.integers(three.size)]
            sel = pb[bidx[pb] == c]                                      # ascending k
            av[ea[owner[bidx[pb] == c]]] = 1.0
            bv[sel] = 1.0
            bv[sel[:3]] = [3e38, 3e38, -3e38]
            used.add(c)
        for fill in ("subnormal", "negzero"):
            free = [c for c in cols if c not in used]
            if not free:
                break
            c = free[rng.integers(len(free))]
            sel = pb[bidx[pb] == c]
            bv[sel] = (rng.integers(1, 1 << 12, size=sel.size).astype(np.uint32).view(F32) if fill == "subnormal" else -0.0)
            used.add(c)
        j = int(rng.integers(ks.size))                                   # one way: normal inputs, subnormal products
        if np.all(av[ea[j]] != 1.0):
            av[ea[j]] = 1e-20
            seg = np.arange(bpos[ks[j]], bpos[ks[j] + 1])
            seg = seg[~np.isin(bidx[seg], list(used))]
            bv[seg] = (1e-20 * np.sign(bv[seg]) + 0).astype(F32)
        keep_a[ea] = True
        keep_b[pb] = True
    free_b = np.nonzero(~keep_b)[0]
    pick = free_b[rng.random(free_b.size) < 1.0 / every]
    bv[pick] = SPECIALS[rng.integers(SPECIALS.size, size=pick.size)]
    free_a = np.nonzero(~keep_a)[0]
    pick = free_a[rng.random(free_a.size) < 0.04]
    bv_a = np.array([np.nan, np.inf, -np.inf, -0.0, 1e-20], F32)
    bv_a[0] = np.uint32(0xFFFFFFFF).view(F32)
    av[pick] = bv_a[rng.integers(bv_a.size, size=pick.size)]


def assert_case_has_every_kind(want, a, b):
    """The operands exercise what inject_specials promises: NaN, +-Inf, -0.0 and subnormal entries, and an entry
    that overflowed in k order although its float64 value is finite."""
    v = want.data["val"]
    bits = v.view(np.uint32)
    _, _, c64, _, _ = f64_product(a, b)
    kinds = {"NaN": np.isnan(v).any(), "+Inf": (v == np.inf).any(), "-Inf": (v == -np.inf).any(),
             "-0.0": (bits == 0x80000000).any(), "subnormal": (((bits & 0x7F800000) == 0) & (v != 0)).any(),
             "fold overflow": (np.isinf(v) & np.isfinite(c64) & (np.abs(c64) < FLT_MAX)).any()}
    assert all(kinds.values()), kinds


# ---- every merge kernel ----------------------------------------------------------------------------------------------
SHORT = [0, 1, 2, 3, 8, 9, 33, 64, 100, 128, 129, 200, 256, 257, 300, 511, 512] * 2
MEDIUM = [513, 640, 641, 700, 1500, 4096] * 2
LONG = [4097, 5000, 9000]
R, K = api.OSP_ROWWISE_ORDER, api.OSP_KSLICE_ORDER
# id: (kernel that must appear, environment read at osp_create, flags, cols_b, row lengths)
KERNEL_CASES = {
    "sort32": ("k_merge_chain<uint32_t, false>", {}, R, 1 << 20, SHORT + [5000]),
    "sort32_kslice": ("k_scatter_tasks", {}, K, 1 << 20, SHORT + MEDIUM),
    "sort64": ("k_merge_chain<uint64_t, false>", {}, R, (1 << 24) + 5, SHORT + [700]),
    "bitmap_rank": ("k_merge_chain<uint32_t, true>", {}, R, 1 << 14, SHORT + MEDIUM[:6]),
    "merge_long": ("k_merge_long", {}, R, 1 << 20, SHORT[:10] + MEDIUM),
    "merge_xl": ("k_merge_xl", {}, R, 1 << 20, SHORT[:10] + LONG),
    "merge_xl_medium": ("k_merge_xl", {}, K, 1 << 17, SHORT[:10] + MEDIUM + LONG),
    "merge_dense": ("k_merge_dense", {}, R | api.OSP_NO_FUSED_DENSE, 1 << 14, SHORT[:10] + MEDIUM + LONG),
    "kway": ("k_merge_ways", {}, R | api.OSP_KWAY_MERGE, 1 << 20, SHORT[:6] + [4097, 5000, 9000, 20000]),
    "long_fill": ("k_long_fill", {}, R | api.OSP_LONGROW_SWEEP, 1 << 16, SHORT[:10] + [700, 5000, 9000] * 2),
    "chain_fused": ("k_merge_chain_fused", {"OSP_FUSED_SHORT": "1", "OSP_FUSED_SHORT_OLD": "1"}, 0, 1 << 20, SHORT + MEDIUM[:4] + [5000]),
    "chain2": ("k_chain2", {"OSP_FUSED_SHORT": "1"}, 0, 1 << 20, SHORT + MEDIUM[:4] + [5000]),
    "chain2_bitmap": ("k_chain2<uint32_t, true", {"OSP_FUSED_SHORT": "1"}, 0, 1 << 14, SHORT + MEDIUM[:4]),
}
# fused dense rows (config 5's shape): id: (kernel, environment, cols)
FUSED_CASES = {
    "fused_dense": ("k_fused_dense", {"OSP_FUSED_LANES": "0"}, 999),
    "fused_lanes_direct": ("k_fused_lanes", {"OSP_FUSED_LANES": "2", "OSP_FL_DIRECT": "1"}, 999),
    "fused_lanes_chained": ("k_fused_lanes", {"OSP_FUSED_LANES": "2", "OSP_FL_DIRECT": "0"}, 256),
    "fused_lanes_auto": ("k_fused_lanes", {"OSP_FUSED_LANES": "1"}, 256),
}


def _engine_with(monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)                      # read at osp_create
    eng = osp.Engine(0)
    for k in env:
        monkeypatch.delenv(k)
    return eng


def _run(eng, a, b, **kw):
    res = eng.spgemm(a, b, a_is_csr=True, flags=kw.pop("flags", 0) | api.OSP_PROFILE_KERNELS, **kw)
    got = res.to_host(); names = [n for n, _ in res.kernel_times()]; res.free()
    return got, names


def _reached(names, kernel, what):
    hit = [n for n in names if kernel in n]
    assert hit, f"{what}: {kernel} was not launched: {names}"
    print(f"{what}: reached {hit[0]}")


@pytest.mark.parametrize("case", list(KERNEL_CASES))
def test_special_values_through_each_merge_kernel(monkeypatch, case):
    kernel, env, flags, cols, lens = KERNEL_CASES[case]
    rng = np.random.default_rng(zlib.crc32(case.encode()))
    lens = list(lens)
    rng.shuffle(lens)
    a, b = rows_case(rng, lens, cols)
    inject_specials(rng, a, b)
    want, prod = oracle_spgemm(synth.transpose_host(a, b.NRow()), b)
    assert_case_has_every_kind(want, a, b)
    eng = _engine_with(monkeypatch, env)
    try:
        got, names = _run(eng, a, b, cols_b=cols, flags=flags)
    finally:
        eng.close()
    _reached(names, kernel, case)
    assert_same_up_to_nan(got, want, case)
    assert_close_to_f64(got, a, b, case)


@pytest.mark.parametrize("case", list(FUSED_CASES))
def test_special_values_through_fused_dense_rows(monkeypatch, case):
    """k_fused_lanes marks a column never touched with the bits 0xFFFFFFFF, a NaN: a product or sum with those bits
    would be taken for "empty" and its entry dropped."""
    kernel, env, cols = FUSED_CASES[case]
    x = synth.pruned_dense(20, 512, 0.3, seed=1)
    w = synth.pruned_dense(512, cols, 0.3, seed=2)
    rng = np.random.default_rng(cols)
    inject_specials(rng, x, w)
    want, _ = oracle_spgemm(synth.transpose_host(x, 512), w)
    assert_case_has_every_kind(want, x, w)
    eng = _engine_with(monkeypatch, env)
    try:
        got, names = _run(eng, x, w, cols_b=cols)
    finally:
        eng.close()
    _reached(names, kernel, case)
    assert_same_up_to_nan(got, want, case)
    assert_close_to_f64(got, x, w, case)


@pytest.mark.parametrize("seed", range(4))
def test_oracle_and_engine_against_float64(engine, seed):
    """Random products of the parity suite (normal values): oracle and engine within the float64 bound."""
    rng = np.random.default_rng(100 + seed)
    lens = [0, 1, 7, 33, 129, 300, 513, 700, 4097][: 5 + seed]
    a, b = rows_case(rng, lens * 3, [1 << 14, 1 << 17, 1 << 20, (1 << 24) + 5][seed])
    want, _ = oracle_spgemm(synth.transpose_host(a, b.NRow()), b)
    assert_close_to_f64(want, a, b, "oracle")
    got, _ = _run(engine, a, b)
    assert_bit_exact(got, want, f"seed {seed}")


def test_nan_payload_of_device_arithmetic(engine):
    """What a B200 returns for NaN operands of the rounded multiply and add (PTX mul.rn.f32 / add.rn.f32): measured
    through the multiply (row 0 of C: NaN * 1) and the merge chain's fold (row 1: 1 * 1 + 1 * NaN).  Measured:
    every NaN result is the canonical 0x7FFFFFFF, whatever the payload and sign of the input NaN -- the CPU emulation
    (tests/cusim) returns the same.  The oracle on x86 keeps the payload; the parity tests compare NaN by position."""
    E = osp.ELEM
    n_k, cols = 4, 8
    # row 0 of C: column j = NaN_j * 1 (multiply); row 1: column j = 1 * 1 + NaN_j (add)
    a = osp.CSRMatrix(np.array([0, 1, 3], np.uint64), np.array([(0, 1.0), (1, 1.0), (2, 1.0)], E))
    nan = np.array(NANS + [0x7FC00000, 0xFFC00000, 0xFFFFFFFF], np.uint32).view(F32)
    b_rows = [(np.arange(8), nan), (np.arange(8), np.ones(8, F32)), (np.arange(8), nan), ([], [])]
    pos = np.zeros(n_k + 1, np.uint64); pos[1:] = np.cumsum([len(r[0]) for r in b_rows])
    b = osp.CSRMatrix.from_arrays(pos, np.concatenate([np.asarray(r[0], np.uint32) for r in b_rows]),
                                  np.concatenate([np.asarray(r[1], F32) for r in b_rows]))
    want, _ = oracle_spgemm(synth.transpose_host(a, n_k), b)
    for flags in (R, K):
        got, _ = _run(engine, a, b, cols_b=cols, flags=flags)
        assert_same_up_to_nan(got, want, "NaN payloads")
        bits = got.data["val"].view(np.uint32)
        print("NaN results:", [hex(x) for x in bits])
        assert np.all(bits == 0x7FFFFFFF), [hex(x) for x in bits]


# ---- osp_bias_relu ----------------------------------------------------------------------------------------------------
def test_bias_relu_special_values(engine):
    """NaN bias, NaN / -0.0 / +-Inf values of C, the widest accepted row (16384 columns, an entry at column 16383), empty
    rows of C; 16385 columns is OSP_ERR_UNSUPPORTED."""
    rng = np.random.default_rng(7)
    for cols in (16384, 999):
        a, b = rows_case(rng, [0, 30, 0, 200, 5, 0, 1, 700], cols, dup=0.2)
        inject_specials(rng, a, b, every=9)
        want_c, _ = oracle_spgemm(synth.transpose_host(a, b.NRow()), b)
        assert int(want_c.data["idx"].max()) == cols - 1 and np.any(np.diff(want_c.pos.astype(np.int64)) == 0)
        bias = rng.standard_normal(cols).astype(F32)
        bias[::5] = np.nan
        bias[1::7] = -0.0
        bias[2::11] = np.inf
        bias[cols - 1] = 0.25
        res = engine.spgemm(a, b, a_is_csr=True, cols_b=cols)
        assert_same_up_to_nan(res.to_host(), want_c, "C")
        for bb in (bias, None):
            out = engine.bias_relu(res, cols, bb)
            got = out.to_host(); out.free()
            want = gp._bias_relu_host(want_c, cols, bb)
            assert_bit_exact(got, want, f"bias_relu cols={cols} bias={bb is not None}")
        with pytest.raises(osp.OspError) as ei:
            engine.bias_relu(res, 16385, np.zeros(16385, F32))
        assert ei.value.code == api.OSP_ERR_UNSUPPORTED
        res.free()


# ---- index ranges: dispatch thresholds ---------------------------------------------------------------------------------
EDGE_LENS = [0, 1, 2, 9, 33, 128, 129, 512, 513, 640, 641, 4096, 4097, 5000]
THRESHOLDS = [16383, 16384, 16385, 131072, 131073, (1 << 23) - 1, 1 << 23, (1 << 23) + 1]


def _chain_variant(cols):
    return "k_merge_chain<uint32_t, true>" if cols <= 16384 else "k_merge_chain<uint32_t, false>" if cols <= (1 << 23) \
        else "k_merge_chain<uint64_t, false>"


@pytest.mark.parametrize("cols", THRESHOLDS)
def test_column_range_thresholds(engine, cols):
    """cols_b at each threshold of the dispatch and one either side, column cols_b - 1 in every non-empty row, rows
    at each length-class boundary; cols_b given and derived (rows of 513..640 then take a different route)."""
    rng = np.random.default_rng(cols % 1013)
    lens = EDGE_LENS * 2
    rng.shuffle(lens)
    a, b = rows_case(rng, lens, cols)
    want, _ = oracle_spgemm(synth.transpose_host(a, b.NRow()), b)
    assert int(want.data["idx"].max()) == cols - 1
    for given in (cols, 0):
        got, names = _run(engine, a, b, cols_b=given, flags=R | api.OSP_NO_FUSED_DENSE)
        _reached(names, _chain_variant(cols), f"cols={cols} given={given}")
        _reached(names, "k_merge_dense" if cols <= 16384 else "k_merge_xl", f"cols={cols} given={given}")
        if cols > 131072:
            _reached(names, "k_merge_long", f"cols={cols} given={given}")
        assert_bit_exact(got, want, f"cols={cols} cols_b given={given}")
        check_csr_invariants(got, cols)


# ---- index ranges: column ids of 2^31 and above -------------------------------------------------------------------------
def _device_only(engine):
    if "cusim" in os.path.basename(api._LIB_PATH):
        pytest.skip("accumulators of 8-17 GB: on a B200 only")


def test_column_ids_above_2_31(engine):
    """Column ids in [2^31, 2^32 - 2] with cols_b = 2^32 - 1: short and medium rows bit-exact.  A row long enough for
    k_merge_xl needs a 17 GB accumulator, beyond the sixteenth of the device it may take on a B200: OSP_ERR_UNSUPPORTED,
    and the engine works afterwards.  With cols_b = 2^31 + 5 (8.6 GB) the long row is bit-exact through k_merge_xl."""
    _device_only(engine)
    rng = np.random.default_rng(231)
    top = (1 << 32) - 1
    a, b = rows_case(rng, [0, 1, 9, 129, 512, 513, 700, 4096] * 2, top, lo=1 << 31)
    want, _ = oracle_spgemm(synth.transpose_host(a, b.NRow()), b)
    assert int(want.data["idx"].min()) >= (1 << 31) and int(want.data["idx"].max()) == top - 1
    got, names = _run(engine, a, b, cols_b=top)
    _reached(names, "k_merge_long", "2^32 - 1 columns")
    assert_bit_exact(got, want, "cols_b = 2^32 - 1, short and medium rows")
    a2, b2 = rows_case(rng, [3, 600, 6000], top, lo=1 << 31)
    with pytest.raises(osp.OspError) as ei:
        engine.spgemm(a2, b2, a_is_csr=True, cols_b=top)
    assert ei.value.code == api.OSP_ERR_UNSUPPORTED and "column range too large" in str(ei.value)
    got, _ = _run(engine, a, b, cols_b=top)
    assert_bit_exact(got, want, "after the refused call")
    cols = (1 << 31) + 5
    a3, b3 = rows_case(rng, [5, 700, 6000, 4097], cols, lo=(1 << 31) - 100000)
    want3, _ = oracle_spgemm(synth.transpose_host(a3, b3.NRow()), b3)
    got, names = _run(engine, a3, b3, cols_b=cols)
    _reached(names, "k_merge_xl", "2^31 + 5 columns")
    assert_bit_exact(got, want3, "cols_b = 2^31 + 5, long rows through k_merge_xl")
    assert_close_to_f64(got, a3, b3, "cols_b = 2^31 + 5")


def test_largest_ids_with_derived_dimensions(engine):
    """Column id 2^32 - 1 with cols_b omitted would make a column range of 2^32, row id 2^32 - 1 of CSC(A) 2^32 rows of
    C: both are OSP_ERR_INDEX (ids stay below 2^32 - 1, as with dimensions given), and the engine works afterwards.
    Column id 2^32 - 2 is the largest that is multiplied."""
    E = osp.ELEM
    a = osp.CSRMatrix(np.array([0, 2, 3], np.uint64), np.array([(0, 2.0), (1, 3.0), (1, -1.0)], E))     # CSR(A) 2 x 2
    for top, ok in ((0xFFFFFFFE, True), (0xFFFFFFFF, False)):
        b = osp.CSRMatrix(np.array([0, 2, 4], np.uint64), np.array([(5, 1.0), (top, 2.0), (7, 0.5), (top, 4.0)], E))
        if ok:
            want, _ = oracle_spgemm(synth.transpose_host(a, 2), b)
            got, _ = _run(engine, a, b)
            assert_bit_exact(got, want, "column id 2^32 - 2, cols_b derived")
            assert int(got.data["idx"][-1]) == top
            continue
        for flags in (0, api.OSP_NO_VALIDATE):
            with pytest.raises(osp.OspError) as ei:
                engine.spgemm(a, b, a_is_csr=True, flags=flags)
            assert ei.value.code == api.OSP_ERR_INDEX, str(ei.value)
    a_csc = osp.CSRMatrix(np.array([0, 2, 3], np.uint64), np.array([(0, 1.0), (0xFFFFFFFF, 2.0), (3, 1.0)], E))
    b = osp.CSRMatrix(np.array([0, 1, 2], np.uint64), np.array([(0, 1.0), (1, 2.0)], E))
    with pytest.raises(osp.OspError) as ei:
        engine.spgemm(a_csc, b)
    assert ei.value.code == api.OSP_ERR_INDEX, str(ei.value)
    got, _ = _run(engine, a, osp.CSRMatrix(np.array([0, 1, 2], np.uint64), np.array([(0, 1.0), (1, 2.0)], E)))
    assert got.nnz == 3


# ---- the 32-bit copy of B.pos (k_narrow_pos) -----------------------------------------------------------------------------
@pytest.fixture(scope="module")
def engine_bpos32():
    os.environ["OSP_BPOS32_MIN_KB"] = "1"                 # read at osp_create: every B of 127 rows or more
    try:
        eng = osp.Engine(0)
    finally:
        del os.environ["OSP_BPOS32_MIN_KB"]
    yield eng
    eng.close()


@pytest.mark.parametrize("seed", range(8))
def test_bpos32_random_vs_oracle(engine_bpos32, seed):
    gp.test_random_vs_oracle(engine_bpos32, seed)


@pytest.mark.parametrize("cols,dup_rate", [(1 << 14, 0.3), (1 << 20, 0.3), ((1 << 24) + 5, 0.2)])
def test_bpos32_every_row_length_class(engine_bpos32, cols, dup_rate):
    gp.test_every_row_length_class(engine_bpos32, cols, dup_rate)


@pytest.mark.parametrize("n,per_row,clustered", [(1 << 13, 8, False), (1 << 13, 10, True)])
def test_bpos32_config4_shape(engine_bpos32, n, per_row, clustered):
    gp.test_config4_shape_spread_and_clustered_columns(engine_bpos32, n, per_row, clustered)


def test_bpos32_many_tiles_chain_order(engine_bpos32):
    gp.test_many_tiles_chain_order(engine_bpos32)


def test_bpos32_row_chunking(engine_bpos32):
    gp.test_row_chunking_gives_same_bits(engine_bpos32)


def test_bpos32_bounded_result_capacity(engine_bpos32):
    gp.test_bounded_result_capacity(engine_bpos32)


def test_bpos32_is_used_and_its_threshold(monkeypatch):
    """k_narrow_pos runs once B.pos ((n_k + 1) * 8 bytes) reaches OSP_BPOS32_MIN_KB, not one row of B earlier; same bits."""
    rng = np.random.default_rng(32)
    eng = _engine_with(monkeypatch, {"OSP_BPOS32_MIN_KB": "4"})
    try:
        for n_k, on in ((510, False), (511, True)):               # B.pos of 4088 and 4096 bytes
            a, b = rows_case(rng, list(rng.integers(0, 700, size=n_k // 6)), 1 << 20)
            pos = np.concatenate([b.pos, np.full(n_k + 1 - b.pos.size, b.pos[-1], np.uint64)])   # empty rows up to n_k
            b = osp.CSRMatrix(pos, b.data)
            want, _ = oracle_spgemm(synth.transpose_host(a, n_k), b)
            got, names = _run(eng, a, b, cols_b=1 << 20)
            assert any("k_narrow_pos" in n for n in names) == on, (n_k, names)
            assert_bit_exact(got, want, f"n_k = {n_k}")
    finally:
        eng.close()

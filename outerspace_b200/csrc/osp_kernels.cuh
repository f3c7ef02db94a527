// osp_kernels.cuh -- sm_100a kernels of the outer-product SpGEMM engine.
//
// Phase map (reference file:line it replaces, relative to simulator/):
//   k_scan<SymIn,...>       symbolic pass: flop count SimSpGEMM.cpp:884-891 and the implicit
//                           push_back sizing of SimOuterSPACE.cpp:87-92 (+ column histogram of A)
//   k_scan<U32In,..>/k_scatter_tasks
//                           CSR->CSC conversion of A: coo2csr<true> SimSpGEMM.cpp:111-117,128-141
//   k_plan                  partitions the output rows into merge tiles and queues long rows
//   k_multiply              TaskProvider::multiplyPhase SimOuterSPACE.cpp:74-97 with the intended
//                           semantics of cscMulcsr SimSpGEMM.cpp:265-281 (true column ids)
//   k_merge_chain           TaskProvider::mergePhase SimOuterSPACE.cpp:98-132 with the intended
//   (+ k_merge_long/xl/dense  semantics of deduplicateCOO SimSpGEMM.cpp:519-535 (sum equal columns),
//    for long rows)         writing CSRMatrix mergedResult (SimOuterSPACE.cpp:140) directly, in one pass
//   k_fused_dense           multiply + merge in one kernel (dense shared-memory accumulator per output row)
//   k_multiply_peer         the multiply of the k-sharded path, storing into the owning GPU's memory
//   k_hist_*/k_scatter_*    bucket scatters of the stable conversions (osp_csr2csc, osp_coo2csr_device)
#pragma once
#include "osp_device.cuh"
#include "osp_kway.cuh"
#include <cstddef>

namespace osp {

// =====================================================================================
// Generic single-pass exclusive scan (decoupled look-back).
//   In : load(idx, valid) -> key, then value(key, valid) -> uint64 contribution (two stages so that the
//        first-level loads of all the items of a thread are in flight together).
//   Out: (idx, exclusive prefix, own contribution) for idx < n, and once (n, total, 0).
// =====================================================================================
#ifndef OSP_SCAN_BLOCK
#define OSP_SCAN_BLOCK 256
#endif
constexpr int SCAN_BLOCK = OSP_SCAN_BLOCK;
#ifndef OSP_SCAN_ITEMS
#define OSP_SCAN_ITEMS 8
#endif
constexpr int SCAN_ITEMS = OSP_SCAN_ITEMS;
constexpr int SCAN_TILE = SCAN_BLOCK * SCAN_ITEMS;

template <class In, class Out>
__global__ void __launch_bounds__(SCAN_BLOCK)
k_scan(In in, Out out, uint64_t n, uint64_t *tile_state, unsigned int *ticket) {
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_warp[SCAN_BLOCK / 32];
    __shared__ uint64_t s_tile_excl;
    if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const unsigned int lane = lane_id(), warp = threadIdx.x >> 5;
    const uint64_t wbase = uint64_t(tile) * SCAN_TILE + uint64_t(warp) * (32 * SCAN_ITEMS);

    uint64_t excl[SCAN_ITEMS], own[SCAN_ITEMS];
    uint64_t running = 0;
    // two-stage input: all the first-level loads of a thread are issued before anything depends on them
    uint64_t key[SCAN_ITEMS];
#pragma unroll
    for (int it = 0; it < SCAN_ITEMS; it++) {
        const uint64_t idx = wbase + it * 32 + lane;
        key[it] = in.load(idx, idx < n);
    }
#pragma unroll
    for (int it = 0; it < SCAN_ITEMS; it++) {
        const uint64_t idx = wbase + it * 32 + lane;
        own[it] = in.value(key[it], idx, idx < n);
    }
#pragma unroll
    for (int it = 0; it < SCAN_ITEMS; it++) {
        uint64_t x = own[it];
        uint64_t incl = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint64_t y = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += y;
        }
        excl[it] = running + incl - x;
        running += __shfl_sync(FULL, incl, 31);
    }
    if (lane == 0) s_warp[warp] = running;
    __syncthreads();
    if (warp == 0) {
        uint64_t w = lane < SCAN_BLOCK / 32 ? s_warp[lane] : 0;
        uint64_t wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint64_t y = __shfl_up_sync(FULL, wi, o);
            if (lane >= o) wi += y;
        }
        uint64_t aggregate = __shfl_sync(FULL, wi, 31);
        uint64_t tile_excl = lookback_exclusive(tile_state, tile, aggregate);
        if (lane < SCAN_BLOCK / 32) s_warp[lane] = wi - w;
        if (lane == 0) {
            s_tile_excl = tile_excl;
            uint64_t ntiles = (n + SCAN_TILE - 1) / SCAN_TILE;
            if (tile == ntiles - 1) out(n, tile_excl + aggregate, 0);
        }
    }
    __syncthreads();
    const uint64_t offset = s_tile_excl + s_warp[warp];
#pragma unroll
    for (int it = 0; it < SCAN_ITEMS; it++) {
        uint64_t idx = wbase + it * 32 + lane;
        if (idx < n) out(idx, offset + excl[it], own[it]);
    }
}

// ---- functors ---------------------------------------------------------------------------
// Symbolic pass over the non-zeros of A in row order: entry p contributes nnz(B(k_p,:)) partial
// products; the exclusive prefix is the offset of its run inside the row bins (bins are laid out
// row after row, runs inside a row in ascending k: the order in which multiplyPhase appends to
// multResults[rowId], SimOuterSPACE.cpp:91).  Side effect: column histogram of A (first step of
// the CSR->CSC conversion), skipped when col_cnt is null.
struct SymIn {
    const Elem *a;
    const uint64_t *b_pos;
    uint64_t n_k;
    uint32_t *col_cnt;
    DevScalars *sc;
    uint32_t *task_bs;     // [nnzA] offset of row k_p of B inside B's data array, or null
    const uint32_t *b_pos32;   // B.pos narrowed to 32 bits (k_narrow_pos), or null: half the footprint of the random reads
    __device__ uint64_t load(uint64_t p, bool valid) const { return valid ? a[p].idx : ~0ull; }
    __device__ uint64_t value(uint64_t k, uint64_t p, bool valid) const {
        if (!valid) return 0;
        if (k >= n_k) { atomicMax(&sc->err, 4u); return 0; }   // OSP_ERR_INDEX
        const uint64_t bs = b_pos32 ? b_pos32[k] : b_pos[k];
        const uint64_t len = (b_pos32 ? b_pos32[k + 1] : b_pos[k + 1]) - bs;
        if (task_bs) task_bs[p] = uint32_t(bs);                // the row-order multiply reads it back as a stream
        if (col_cnt) atomicAdd(&col_cnt[k], 1u);
        if (len >> TASK_LEN_BITS) { atomicMax(&sc->err, 6u); return 0; }   // OSP_ERR_UNSUPPORTED
        return len;
    }
};
// B.pos as 32-bit offsets for the symbolic pass (operands have < 2^32 non-zeros): the pass reads B.pos[k], B.pos[k+1] at the
// random k of A's elements, and an array that fits one L2 partition is served from L2 where the 64-bit one is not.
__global__ void k_narrow_pos(const uint64_t *__restrict__ pos, uint64_t n, uint32_t *__restrict__ out) {
    for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x) out[i] = uint32_t(pos[i]);
}
struct RunOffOut {
    uint64_t *run_off;   // [nnzA+1]
    DevScalars *sc;
    uint64_t n;
    __device__ void operator()(uint64_t p, uint64_t v, uint64_t) const {
        run_off[p] = v;
        if (p == n) sc->products = v;
    }
};
struct U32In {
    const uint32_t *x;
    __device__ uint64_t load(uint64_t i, bool valid) const { return valid ? x[i] : 0; }
    __device__ uint64_t value(uint64_t v, uint64_t, bool) const { return v; }
};
struct U64Out {
    uint64_t *y;
    __device__ void operator()(uint64_t i, uint64_t v, uint64_t) const { y[i] = v; }
};
struct U32Out {           // column pointers of the task list (nnzA < 2^32 is checked on the host)
    uint32_t *y;
    __device__ void operator()(uint64_t i, uint64_t v, uint64_t) const { y[i] = uint32_t(v); }
};

// =====================================================================================
// Small utility kernels
// =====================================================================================
// Hands the device scalars to the host without a copy-engine round trip and without a fence: every 8-byte word
// travels in its own 16-byte slot {word, sequence number}, written with ONE 16-byte store into mapped pinned
// memory.  The host polls until every slot carries the sequence number of this hand-over; the kernel retires at
// once, so the launches queued behind it do not wait for a system-scope fence to drain.
constexpr int PUBLISH_SLOTS = int((sizeof(DevScalars) + 7) / 8);
__global__ void k_publish(const DevScalars *d, ulonglong2 *h_slots, unsigned long long seq) {
    const unsigned long long *src = reinterpret_cast<const unsigned long long *>(d);
    if (threadIdx.x < PUBLISH_SLOTS) {
        const unsigned long long v = __ldcg(src + threadIdx.x);
#ifdef OSP_CUSIM
        h_slots[threadIdx.x] = ulonglong2{v, seq};
#else
        asm volatile("st.global.v2.u64 [%0], {%1, %2};" ::"l"(h_slots + threadIdx.x), "l"(v), "l"(seq) : "memory");
#endif
    }
}
__global__ void k_max_idx(const Elem *d, uint64_t nnz, DevScalars *sc) {
    uint32_t m = 0;
    for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < nnz; i += uint64_t(gridDim.x) * blockDim.x)
        m = max(m, d[i].idx);
    m = __reduce_max_sync(FULL, m);
    if (lane_id() == 0 && m) atomicMax(&sc->max_idx, m);
}

// Operand preconditions (SURVEY.md 8b): "both sorted ascending inside a slice, duplicate-free" -- what coo2csr guarantees
// in the reference (sort + dupcheck, SimSpGEMM.cpp:113-123) and what the merge kernels rely on (k_band_ptr's binary
// search, one-round arbitration of a duplicate-free run).  One streaming pass per operand: every position whose index
// does not exceed its predecessor's is counted, and so is every such position that opens a slice; an operand is valid
// exactly when the two counts agree.  Also: index range (idx < idx_range when given), max index of operand 1, pos[]
// monotone and within nnz.
struct ValidateOp { const uint64_t *pos; const Elem *d; uint64_t n_slices, nnz, idx_range; uint32_t *start_bits; };
// Step 1: one bit per element position that opens a (non-empty) slice -- start_bits is zeroed by the host, (nnz + 31) / 32
// words per operand -- and the pos[] checks.  The element pass then decides "descent at a slice boundary" from this bitmap
// (8 MB for 6.7e7 elements: L2-resident) instead of reading the data array a second time slice by slice, which doubled
// the kernel's DRAM traffic (ncu, config 4: 1.14 GB read for 0.60 GB of operand).
__global__ void __launch_bounds__(256)
k_validate_starts(const ValidateOp op0, const ValidateOp op1, const int n_ops, DevScalars *sc) {
    uint32_t badpos = 0;
    const uint64_t t0 = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x, nt = uint64_t(gridDim.x) * blockDim.x;
    for (int o = 0; o < n_ops; o++) {
        const ValidateOp &op = o ? op1 : op0;
        for (uint64_t r = t0; r < op.n_slices; r += nt) {
            const uint64_t s = op.pos[r], e = op.pos[r + 1];
            if (e < s || e > op.nnz) { badpos++; continue; }
            if (s < e) atomicOr(&op.start_bits[s >> 5], 1u << (s & 31));
        }
    }
    badpos = __reduce_add_sync(FULL, badpos);
    if (lane_id() == 0 && badpos) atomicAdd(&sc->v_bad_pos, (unsigned long long)badpos);
}
// Step 2: the element pass.
__global__ void __launch_bounds__(256)
k_validate(const ValidateOp op0, const ValidateOp op1, const int n_ops, DevScalars *sc) {
    uint32_t desc = 0, bdesc = 0, eq = 0, beq = 0, mx = 0;
    bool range_err = false;
    const uint64_t t0 = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x, nt = uint64_t(gridDim.x) * blockDim.x;
    for (int o = 0; o < n_ops; o++) {
        const ValidateOp &op = o ? op1 : op0;
        auto is_start = [&](uint64_t p) { return (op.start_bits[p >> 5] >> (p & 31)) & 1u; };
        // elements two at a time (one 128-bit load; data arrays are 16-byte aligned), four loads in flight per thread;
        // the predecessor of a pair's first element comes from the neighbouring lane
        const uint4 *d2 = reinterpret_cast<const uint4 *>(op.d);
        const bool aligned = (reinterpret_cast<uintptr_t>(op.d) & 15) == 0;
        const uint64_t n_pairs = aligned ? op.nnz / 2 : 0;
        for (uint64_t qw = t0 - lane_id(); qw < n_pairs; qw += 4 * nt) {      // warp-uniform bound: the shuffle below needs the whole warp
            const uint64_t q0 = qw + lane_id();
            uint4 v[4];
            uint32_t sb[4];                                                  // the 64 start bits of the warp's 32 pairs: two words, lane-selected
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const uint64_t q = q0 + u * nt;
                v[u] = q < n_pairs ? d2[q] : make_uint4(0, 0, 0, 0);
                sb[u] = q < n_pairs ? op.start_bits[q >> 4] : 0u;              // word of elements 2q, 2q + 1 (32 elements = 16 pairs per word)
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const uint64_t q = q0 + u * nt;
                const bool live = q < n_pairs;
                uint32_t prv = __shfl_up_sync(FULL, v[u].z, 1);          // second element of the pair before (lane - 1)
                if (lane_id() == 0 && live && q) prv = op.d[2 * q - 1].idx;
                if (!live) continue;
                const uint32_t c0 = v[u].x, c1 = v[u].z;
                const uint32_t b0 = (sb[u] >> ((2 * q) & 31)) & 1u, b1 = (sb[u] >> ((2 * q + 1) & 31)) & 1u;
                if (op.idx_range && (c0 >= op.idx_range || c1 >= op.idx_range)) range_err = true;
                if (o == n_ops - 1) mx = max(mx, max(c0, c1));
                if (q) { const uint32_t dn = c0 <= prv, e2 = c0 == prv; desc += dn; eq += e2; bdesc += dn & b0; beq += e2 & b0; }
                { const uint32_t dn = c1 <= c0, e2 = c1 == c0; desc += dn; eq += e2; bdesc += dn & b1; beq += e2 & b1; }
            }
        }
        for (uint64_t p = 2 * n_pairs + t0; p < op.nnz; p += nt) {          // the odd last element / an unaligned array
            const uint32_t cur = op.d[p].idx;
            if (op.idx_range && cur >= op.idx_range) range_err = true;
            if (o == n_ops - 1) mx = max(mx, cur);
            if (p) {
                const uint32_t prv = op.d[p - 1].idx, dn = cur <= prv, e2 = cur == prv, b = is_start(p);
                desc += dn; eq += e2; bdesc += dn & b; beq += e2 & b;
            }
        }
    }
    desc = __reduce_add_sync(FULL, desc); bdesc = __reduce_add_sync(FULL, bdesc);
    eq = __reduce_add_sync(FULL, eq); beq = __reduce_add_sync(FULL, beq);
    mx = __reduce_max_sync(FULL, mx);
    if (__any_sync(FULL, range_err) && lane_id() == 0) atomicMax(&sc->err, 4u);                 // OSP_ERR_INDEX
    if (lane_id() == 0) {
        if (desc) atomicAdd(&sc->v_desc, (unsigned long long)desc);
        if (bdesc) atomicAdd(&sc->v_bdesc, (unsigned long long)bdesc);
        if (eq) atomicAdd(&sc->v_eq, (unsigned long long)eq);
        if (beq) atomicAdd(&sc->v_beq, (unsigned long long)beq);
        if (mx) atomicMax(&sc->max_idx, mx);
    }
}

// =====================================================================================
// Merge plan.  Tiles are runs of consecutive output rows; row i opens a tile when
//   i == 0, i % MT_RMAX == 0, its bin start crosses a multiple of MT_CAP, or it or its
//   predecessor is longer than MT_LONG (long rows are tiles of their own).
// So a tile of short rows holds < MT_CAP + MT_LONG partial products and <= MT_RMAX rows.
// Also: row_bin[] (bin start of every row), the queues of long rows, the upper bound of nnz(C)
// and the reference's row count rule numRows = maxRowId + 1 (SimOuterSPACE.cpp:49-53).
// =====================================================================================
#ifndef OSP_CAP_SHIFT_MAX
#define OSP_CAP_SHIFT_MAX 11
#endif
#ifndef OSP_MC_THREADS
#define OSP_MC_THREADS 256
#endif
#ifndef OSP_MC_OCC
#define OSP_MC_OCC 3
#endif
constexpr int MT_CAP_SHIFT_MIN = 8, MT_CAP_SHIFT_MAX = OSP_CAP_SHIFT_MAX;
constexpr uint32_t MT_CAP = 1u << MT_CAP_SHIFT_MAX;   // partial products per tile (soft): one CTA merges a tile
constexpr uint32_t MT_LONG = 512;      // longest row sorted in registers by one warp
constexpr uint32_t MT_LONG_BM = 640;   // longest row merged by bitmap rank by one warp (small column ranges)
constexpr uint32_t MT_STAGE = MT_CAP + MT_LONG_BM;    // hard bound of a tile of short rows (shared-memory stage)
constexpr uint32_t MT_RMAX = 256;      // rows per tile (one thread per row in the tile's scans)
constexpr uint32_t MT_XL = 4096;       // longest row sorted in shared memory by one CTA

// What the producer warps of k_chain2 (osp_chain2.cuh) need to open a tile, in one 32-byte load (entries t and t + 1):
// first row, first task (non-zero of A / segment) and first partial product of the tile.
struct __align__(16) TileStart { uint32_t r0, e0; uint64_t b0; };
static_assert(sizeof(TileStart) == 16, "two tile starts are one 32-byte load");

constexpr int PLAN_BLOCK = 256;
constexpr int PLAN_ITEMS = 4;
constexpr int PLAN_TILE = PLAN_BLOCK * PLAN_ITEMS;

struct RowBinFromRuns {        // row i starts where the run of its first non-zero starts
    const uint64_t *a_pos;
    uint64_t m_a;
    const uint64_t *run_off;
    uint64_t nnz_a;
    __device__ __forceinline__ uint64_t operator()(uint64_t i) const { return run_off[i <= m_a ? a_pos[i] : nnz_a]; }
    // a row counts for numRows = maxRowId + 1 (SimOuterSPACE.cpp:49-53) when A holds a non-zero in it
    __device__ __forceinline__ bool nonempty(uint64_t i) const { return i < m_a && a_pos[i + 1] > a_pos[i]; }
    __device__ __forceinline__ uint64_t task_begin(uint64_t i) const { return i <= m_a ? a_pos[i] : nnz_a; }   // first non-zero of A of row i
};
struct RowBinDirect {
    const uint64_t *pos;
    __device__ __forceinline__ uint64_t operator()(uint64_t i) const { return pos[i]; }
    __device__ __forceinline__ bool nonempty(uint64_t i) const { return pos[i + 1] > pos[i]; }
    __device__ __forceinline__ uint64_t task_begin(uint64_t) const { return 0; }
};

template <class RB>
__global__ void __launch_bounds__(PLAN_BLOCK)
k_plan(RB rb, uint64_t rows, uint64_t cols_hint, uint64_t *row_bin, uint32_t *tile_row, uint32_t *long_list,
       uint32_t *xl_list, uint64_t *tile_state, DevScalars *sc, int ticket_slot, uint32_t long_thresh,
       uint64_t *chain_state, TileStart *tile_start = nullptr, uint32_t cap_max = MT_CAP, uint64_t cut_row = ~0ull) {
    __shared__ uint32_t s_tile;
    __shared__ uint32_t s_warp[33];
    __shared__ uint64_t s_bound[PLAN_BLOCK / 32];
    __shared__ uint32_t s_last[PLAN_BLOCK / 32];
    __shared__ uint64_t s_excl;
    if (threadIdx.x == 0) s_tile = atomicAdd(&sc->scan_ticket[ticket_slot], 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const unsigned int lane = lane_id(), warp = threadIdx.x >> 5;
    const uint64_t i0 = uint64_t(tile) * PLAN_TILE + uint64_t(threadIdx.x) * PLAN_ITEMS;
    // partial products per tile: MT_CAP, less when the whole product is small, so that there are enough
    // tiles for every persistent CTA of the merge (444 on a B200): 2^cap_shift ~ P / 1024 within [256, MT_CAP]
    const uint64_t p_all = rb(rows);
    int cap_shift = MT_CAP_SHIFT_MIN;
    while (cap_shift < MT_CAP_SHIFT_MAX && (p_all >> (cap_shift + 1)) >= 1024) cap_shift++;
    const uint64_t cap = min(1u << cap_shift, cap_max);       // (k_chain2 takes tiles that are not a power of two: shared memory)

    uint64_t s[PLAN_ITEMS + 1];
#pragma unroll
    for (int it = 0; it <= PLAN_ITEMS; it++) s[it] = rb(min(i0 + it, rows));
    uint64_t sp = i0 > 0 && i0 <= rows ? rb(i0 - 1) : 0;   // start of the previous row
    bool flag[PLAN_ITEMS];
    uint32_t nflags = 0, last = 0;
    uint64_t bound = 0;
#pragma unroll
    for (int it = 0; it < PLAN_ITEMS; it++) {
        const uint64_t i = i0 + it;
        flag[it] = false;
        if (i < rows) {
            const uint64_t len = s[it + 1] - s[it];
            const uint64_t plen = s[it] - sp;
            flag[it] = i == 0 || (i % MT_RMAX) == 0 || len > long_thresh || plen > long_thresh || (sp / cap) != (s[it] / cap) || i == cut_row;
            row_bin[i] = s[it];
            if (len > MT_XL) xl_list[atomicAdd(&sc->n_xl, 1u)] = uint32_t(i);
            else if (len > long_thresh) long_list[atomicAdd(&sc->n_long, 1u)] = uint32_t(i);
            if (rb.nonempty(i)) last = uint32_t(i + 1);
            bound += cols_hint ? min(len, cols_hint) : len;
            nflags += flag[it];
        }
        sp = s[it];
    }
    // block reductions of bound / last
    last = __reduce_max_sync(FULL, last);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) bound += __shfl_xor_sync(FULL, bound, o);
    if (lane == 0) { s_bound[warp] = bound; s_last[warp] = last; }
    uint32_t total;
    uint32_t rank = block_exclusive_scan(nflags, s_warp, total);
    if (warp == 0) {
        uint64_t b = lane < PLAN_BLOCK / 32 ? s_bound[lane] : 0;
        uint32_t l = lane < PLAN_BLOCK / 32 ? s_last[lane] : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) b += __shfl_xor_sync(FULL, b, o);
        l = __reduce_max_sync(FULL, l);
        if (lane == 0) {
            if (b) atomicAdd(&sc->cap_bound, (unsigned long long)b);
            if (l) atomicMax(&sc->last_nonempty, (unsigned long long)l);
        }
        uint64_t excl = lookback_exclusive(tile_state, tile, total);
        if (lane == 0) {
            s_excl = excl;
            const uint64_t ntiles = (rows + PLAN_TILE - 1) / PLAN_TILE;
            if (tile == ntiles - 1) {
                sc->n_tiles = uint32_t(excl + total);
                tile_row[excl + total] = uint32_t(rows);
                row_bin[rows] = rb(rows);
                if (tile_start) tile_start[excl + total] = TileStart{uint32_t(rows), uint32_t(rb.task_begin(rows)), rb(rows)};
            }
        }
    }
    __syncthreads();
    uint64_t o = s_excl + rank;
#pragma unroll
    for (int it = 0; it < PLAN_ITEMS; it++)
        if (flag[it]) {
            chain_state[o] = 0;                                                    // (look-back state of the merge chain)
            if (tile_start) tile_start[o] = TileStart{uint32_t(i0 + it), uint32_t(rb.task_begin(i0 + it)), s[it]};
            if (i0 + it == cut_row) sc->cut_tile = uint32_t(o);             // a row block of the caller starts here
            tile_row[o++] = uint32_t(i0 + it);
        }
}

// =====================================================================================
// CSR -> CSC conversion of A.  Task list in k-slice (CSC) order: every non-zero of A lands in the
// slot range of its column k together with the bin offset of its run.  The order of the tasks
// inside a column is immaterial (each task owns a distinct run), so slots are claimed with an
// atomic; `col_cnt` (the histogram built by the symbolic pass) is counted down.
// =====================================================================================
__global__ void k_scatter_tasks(const Elem *a, const uint64_t *run_off, const uint64_t *b_pos, uint64_t e0, uint64_t e1,
                                const uint32_t *col_ptr, uint32_t *col_cnt, Task *tasks, DevScalars *sc) {
    for (uint64_t p = e0 + blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; p < e1; p += uint64_t(gridDim.x) * blockDim.x) {
        const Elem e = a[p];
        const uint64_t off = run_off[p], len = run_off[p + 1] - off;
        const uint32_t c = atomicSub(&col_cnt[e.idx], 1u);
        if (len >> TASK_LEN_BITS) { atomicMax(&sc->err, 6u); continue; }     // OSP_ERR_UNSUPPORTED
        Task t;
        t.bs = uint32_t(b_pos[e.idx]); t.a = e.val; t.offlen = (off << TASK_LEN_BITS) | len;
        tasks[col_ptr[e.idx] + c - 1] = t;
    }
}

// Public stable conversion, step 1: bucket scatter of {source slice id, val} by minor index.
// One warp walks one source slice; the order inside a bucket is fixed up by the merge kernels.
__global__ void k_scatter_elems(const uint64_t *pos, const Elem *d, uint64_t n_major, uint64_t n_minor,
                                const uint64_t *pos_out, uint32_t *cursor, Elem *out, DevScalars *sc) {
    uint64_t warp = (blockIdx.x * uint64_t(blockDim.x) + threadIdx.x) >> 5;
    uint64_t nwarps = (uint64_t(gridDim.x) * blockDim.x) >> 5;
    for (uint64_t r = warp; r < n_major; r += nwarps) {
        uint64_t b = pos[r], e = pos[r + 1];
        for (uint64_t p = b + lane_id(); p < e; p += 32) {
            Elem x = d[p];
            if (x.idx >= n_minor) { atomicMax(&sc->err, 4u); continue; }
            uint32_t slot = atomicAdd(&cursor[x.idx], 1u);
            Elem y; y.idx = uint32_t(r); y.val = x.val;
            out[pos_out[x.idx] + slot] = y;
        }
    }
}
// COO ingest (coo2csr<transpose>, SimSpGEMM.cpp:102-152): the same bucket scatter from triplet arrays.
// `major` = the index that becomes the slice (row for CSR, column for CSC), `minor` the one kept in the element.
__global__ void k_hist_u32(const uint32_t *key, uint64_t nnz, uint64_t n_buckets, uint32_t *cnt, DevScalars *sc) {
    for (uint64_t p = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; p < nnz; p += uint64_t(gridDim.x) * blockDim.x) {
        const uint32_t c = key[p];
        if (c >= n_buckets) { atomicMax(&sc->err, 4u); continue; }
        atomicAdd(&cnt[c], 1u);
    }
}
__global__ void k_scatter_coo(const uint32_t *__restrict__ major, const uint32_t *__restrict__ minor, const float *__restrict__ val,
                              uint64_t nnz, uint64_t n_buckets, uint64_t n_minor, const uint64_t *__restrict__ pos_out,
                              uint32_t *cursor, Elem *__restrict__ out, DevScalars *sc) {
    for (uint64_t p = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; p < nnz; p += uint64_t(gridDim.x) * blockDim.x) {
        const uint32_t b = major[p], m = minor[p];
        if (b >= n_buckets || m >= n_minor) { atomicMax(&sc->err, 4u); continue; }
        const uint32_t slot = atomicAdd(&cursor[b], 1u);
        Elem y; y.idx = m; y.val = val[p];
        out[pos_out[b] + slot] = y;
    }
}
__global__ void k_hist_elems(const Elem *d, uint64_t nnz, uint64_t n_minor, uint32_t *cnt, DevScalars *sc) {
    for (uint64_t p = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; p < nnz; p += uint64_t(gridDim.x) * blockDim.x) {
        uint32_t c = d[p].idx;
        if (c >= n_minor) { atomicMax(&sc->err, 4u); continue; }
        atomicAdd(&cnt[c], 1u);
    }
}

// =====================================================================================
// Multiply phase (warp-flat).  A warp takes 32 tasks, scans their run lengths and then walks the
// concatenation of the 32 runs 32 partial products at a time: every lane finds the task of its
// element with a 5-step search over the scanned lengths (shuffles), reads the element of B(k,:),
// multiplies by A(i,k) and writes (col, a*b) into row i's bin.  Every lane is busy whatever the run
// lengths are, loads and stores are contiguous inside a run, and there is no per-run loop.
// Task sources: packed Task[] (k-slice order: the CSC of A) or {Elem[], run_off[]} (row order of A).
// =====================================================================================
struct TaskSrcAoS {
    const Task *t;
    __device__ __forceinline__ void load(uint64_t i, uint32_t &bs, float &a, uint64_t &off, uint32_t &len) const {
        const uint4 raw = __ldg(reinterpret_cast<const uint4 *>(t + i));   // one 128-bit load
        bs = raw.x; a = __uint_as_float(raw.y);
        const uint64_t offlen = (uint64_t(raw.w) << 32) | raw.z;
        off = offlen >> TASK_LEN_BITS;
        len = uint32_t(offlen) & ((1u << TASK_LEN_BITS) - 1);
    }
};
struct TaskSrcSoA {
    const Elem *a_data;
    const uint64_t *run_off;
    const uint32_t *task_bs;     // b_pos[k] of every task, left by the symbolic pass: a stream instead of a random lookup
    __device__ __forceinline__ void load(uint64_t i, uint32_t &bs, float &a, uint64_t &off, uint32_t &len) const {
        a = a_data[i].val; off = run_off[i];
        len = uint32_t(run_off[i + 1] - off);
        bs = task_bs[i];
    }
};
struct TaskSrcSoASwept {        // row order of A minus the tasks somebody else computes: the rows of the fused band sweep
    TaskSrcSoA src;             // (osp_longrows.cuh; bits set by k_mark_swept, skip = 1) or, with OSP_FUSED_SHORT, every
    const uint32_t *mask;       // task that is NOT marked as belonging to a long row (k_mark_binned, skip = 0)
    uint32_t skip;              // the bit value of a task that emits nothing
    __device__ __forceinline__ void load(uint64_t i, uint32_t &bs, float &a, uint64_t &off, uint32_t &len) const {
        src.load(i, bs, a, off, len);
        if (((mask[i >> 5] >> (i & 31)) & 1u) == skip) len = 0;
    }
};

// Gathered rows of B: `ld.global.L2::64B` fetches 64-byte granules where the default fetches up to a whole 128-byte line --
// a random gather of 64-byte rows moves 111 B per row from DRAM with it, 159 B without (profiles/r02_gather_probe.md).
#ifdef OSP_CUSIM
__device__ __forceinline__ Elem ld_gather(const Elem *p) { return *p; }
#else
__device__ __forceinline__ Elem ld_gather(const Elem *p) {
    Elem e; uint32_t v;
    asm volatile("ld.global.L2::64B.v2.u32 {%0, %1}, [%2];" : "=r"(e.idx), "=r"(v) : "l"(p));
    e.val = __uint_as_float(v);
    return e;
}
#endif

template <class Src>
__global__ void __launch_bounds__(256)
k_multiply(Src src, uint64_t t0, uint64_t t1, const Elem *__restrict__ b_data, Elem *__restrict__ bins, uint64_t bin_base) {
    const unsigned int lane = lane_id();
    const uint64_t warp = (blockIdx.x * uint64_t(blockDim.x) + threadIdx.x) >> 5;
    const uint64_t nwarps = (uint64_t(gridDim.x) * blockDim.x) >> 5;
    for (uint64_t base = t0 + warp * 32; base < t1; base += nwarps * 32) {
        uint32_t bs = 0, len = 0; float a = 0.f; uint64_t off = 0;
        if (base + lane < t1) src.load(base + lane, bs, a, off, len);
        const uint32_t incl = warp_inclusive_scan(len);
        const uint32_t total = __shfl_sync(FULL, incl, 31);
        const uint32_t excl = incl - len;
        const uint32_t dbs = bs - excl;                       // B index of element e of this task: dbs + e
        const uint64_t doff = off - bin_base - excl;          // bin index of element e of this task: doff + e
        for (uint32_t e0 = 0; e0 < total; e0 += 64) {          // two independent 32-element chunks per turn
            const uint32_t e[2] = {e0 + lane, e0 + 32 + lane};
            uint32_t t[2] = {0, 0};                            // number of tasks that end at or before e
#pragma unroll
            for (int step = 16; step > 0; step >>= 1) {
#pragma unroll
                for (int u = 0; u < 2; u++) {
                    const uint32_t v = __shfl_sync(FULL, incl, t[u] + step - 1);
                    if (v <= e[u]) t[u] += step;
                }
            }
            float a_t[2]; uint32_t dbs_t[2]; uint64_t doff_t[2]; Elem b[2];
#pragma unroll
            for (int u = 0; u < 2; u++) {
                a_t[u] = __shfl_sync(FULL, a, t[u] & 31);
                dbs_t[u] = __shfl_sync(FULL, dbs, t[u] & 31);
                doff_t[u] = __shfl_sync(FULL, doff, t[u] & 31);
            }
#pragma unroll
            for (int u = 0; u < 2; u++)
                if (e[u] < total) b[u] = ld_gather(b_data + uint32_t(dbs_t[u] + e[u]));    // (32-bit wrap-around: dbs = bs - excl may be "negative")
#pragma unroll
            for (int u = 0; u < 2; u++) {
                if (e[u] < total) {
                    Elem o; o.idx = b[u].idx; o.val = __fmul_rn(a_t[u], b[u].val);     // rounded on its own: no FMA
                    bins[doff_t[u] + e[u]] = o;
                }
            }
        }
    }
}

// =====================================================================================
// Merge, long rows (MT_LONG < len <= MT_XL): one CTA sorts one row's partial products by
// (col, arrival position) with a bitonic network in shared memory, left-folds equal columns in
// arrival (= k) order with separately rounded adds, and writes the compacted row back to the
// start of its bin; uniq[row] = surviving entries.  k_merge_chain copies it into C.
// Shared: uint64 keys[cap] | float vals[cap] | uint32 warp_sums[33]
// =====================================================================================
__device__ __forceinline__ void bitonic_sort_shared(uint64_t *keys, uint32_t N) {
    for (uint32_t k = 2; k <= N; k <<= 1) {
        for (uint32_t j = k >> 1; j > 0; j >>= 1) {
            for (uint32_t t = threadIdx.x; t < (N >> 1); t += blockDim.x) {
                uint32_t i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                uint32_t p = i | j;
                uint64_t x = keys[i], y = keys[p];
                bool up = (i & k) == 0;
                if ((x > y) == up) { keys[i] = y; keys[p] = x; }
            }
            __syncthreads();
        }
    }
}

// Sorted keys (col<<32 | pos) + vals[pos] -> folded, compacted row at out[0..uniq).  Returns uniq
// (valid in every thread).  When `acc` is non-null the fold of a column starts from acc[col] if its
// bit in `bits` is set (long-row accumulator) and the result goes to acc instead of `out`.
__device__ __forceinline__ uint32_t fold_sorted(const uint64_t *keys, const float *vals, uint32_t len, uint32_t N,
                                                Elem *out, uint32_t *warp_sums, float *acc, uint32_t *bits) {
    uint32_t produced = 0;
    for (uint32_t s0 = 0; s0 < N; s0 += blockDim.x) {
        uint32_t s = s0 + threadIdx.x;
        bool head = false;
        uint32_t col = 0;
        if (s < len) {
            col = uint32_t(keys[s] >> 32);
            head = (s == 0) || (uint32_t(keys[s - 1] >> 32) != col);
        }
        float sum = 0.f;
        if (head) {
            sum = vals[uint32_t(keys[s])];
            if (acc) {
                bool seen = (bits[col >> 5] >> (col & 31)) & 1u;
                if (seen) sum = __fadd_rn(acc[col], sum);
            }
            for (uint32_t u = s + 1; u < len && uint32_t(keys[u] >> 32) == col; u++)
                sum = __fadd_rn(sum, vals[uint32_t(keys[u])]);
        }
        uint32_t total;
        uint32_t rank = block_exclusive_scan(head ? 1u : 0u, warp_sums, total);
        if (head) {
            if (acc) {
                acc[col] = sum;
                atomicOr(&bits[col >> 5], 1u << (col & 31));
            } else {
                Elem o; o.idx = col; o.val = sum;
                out[produced + rank] = o;
            }
        }
        produced += total;
    }
    return produced;
}

__global__ void __launch_bounds__(256)
k_merge_long(const uint64_t *__restrict__ row_bin, uint64_t bin_base, Elem *bins, uint32_t *uniq,
             const uint32_t *long_list, const DevScalars *sc, uint64_t row_lo, uint64_t row_hi) {
    OSP_EXTERN_SMEM(smem);
    uint64_t *keys = reinterpret_cast<uint64_t *>(smem);
    float *vals = reinterpret_cast<float *>(keys + MT_XL);
    uint32_t *warp_sums = reinterpret_cast<uint32_t *>(vals + MT_XL);
    const uint32_t n_long = sc->n_long;
    for (uint32_t x = blockIdx.x; x < n_long; x += gridDim.x) {
        const uint64_t row = long_list[x];
        if (row < row_lo || row >= row_hi) continue;
        const uint64_t start = row_bin[row] - bin_base;
        const uint32_t len = uint32_t(row_bin[row + 1] - row_bin[row]), N = pow2ceil(len);
        Elem *bin = bins + start;
        for (uint32_t p = threadIdx.x; p < N; p += blockDim.x) {
            if (p < len) {
                Elem e = bin[p];
                keys[p] = (uint64_t(e.idx) << 32) | p;
                vals[p] = e.val;
            } else {
                keys[p] = ~0ull;
            }
        }
        __syncthreads();
        bitonic_sort_shared(keys, N);
        uint32_t u = fold_sorted(keys, vals, len, N, bin, warp_sums, nullptr, nullptr);
        if (threadIdx.x == 0) uniq[row] = u;
        __syncthreads();
    }
}

// Rows longer than MT_XL over a large column range: a dense per-CTA accumulator acc[cols_b] in global
// memory (one row at a time per CTA) with a presence bitmap.  The row is consumed XL_THREADS partial
// products at a time in arrival order.  Products of one chunk that hit the SAME column are serialised: every
// product enters an open-addressing table in shared memory keyed by its exact column (different columns never
// share a slot, so they never wait for each other), the lowest position of a slot goes first, so every column
// is still summed in ascending arrival (= k) order with separately rounded adds.  A chunk without a repeated
// column -- almost all of them: the runs of a row are duplicate-free -- takes one round.  No sort.  The
// accumulator is then compacted in ascending column order over the start of the row's bin and the bitmap is
// cleared.  Rows are handed out by a ticket (sc->xl_ticket, zeroed before the launch): row lengths span three
// orders of magnitude on power-law inputs, a static assignment left the longest CTA with 2-4x the mean work.
constexpr int XL_THREADS = 512;
constexpr uint32_t XL_SLOTS = 2048;                    // slots of the column table: load <= 1/4
constexpr uint32_t XL_EMPTY = 0xFFFFFFFFu;             // no column id (osp_spgemm keeps ids < 2^32 - 1, cols_b given or derived) and no thread id
__global__ void __launch_bounds__(XL_THREADS)
k_merge_xl(const uint64_t *__restrict__ row_bin, uint64_t bin_base, Elem *bins, uint32_t *uniq,
           const uint32_t *xl_list, const uint32_t *long_list, DevScalars *sc, float *acc_all, uint32_t *bits_all,
           uint64_t cols_b, uint64_t row_lo, uint64_t row_hi, uint64_t sweep_min, const uint64_t *__restrict__ kw_a_pos = nullptr) {
    __shared__ uint32_t key[XL_SLOTS];                 // column held by the slot
    __shared__ uint32_t owner[XL_SLOTS];               // lowest pending position of that column
    __shared__ uint32_t warp_sums[33];
    __shared__ uint32_t s_x;
    const uint32_t tid = threadIdx.x;
    for (uint32_t i = tid; i < XL_SLOTS; i += XL_THREADS) { key[i] = XL_EMPTY; owner[i] = XL_EMPTY; }
    const uint64_t words = (cols_b + 31) >> 5;
    float *acc = acc_all + uint64_t(blockIdx.x) * cols_b;
    uint32_t *bits = bits_all + uint64_t(blockIdx.x) * words;
    // the longest rows first, then (when the caller passes them: moderate column ranges, where compacting the
    // bitmap is cheaper than a shared-memory sort) the rows of MT_LONG .. MT_XL partial products
    const uint32_t n_xl = sc->n_xl, n_all = n_xl + (long_list ? sc->n_long : 0u);
    while (true) {
        __syncthreads();                               // the table is initialised / the previous row is finished
        if (tid == 0) {
            uint32_t x;
            while (true) {                             // next listed row of this row block
                x = atomicAdd(&sc->xl_ticket, 1u);
                if (x >= n_all) break;
                const uint64_t r = x < n_xl ? xl_list[x] : long_list[x - n_xl];
                // rows of sweep_min partial products or more belong to the fused band sweep (~0: none); rows of few long
                // ways to the k-way merge (kw_a_pos: CSR(A)'s row pointer, null when that kernel is off)
                if (r >= row_lo && r < row_hi && row_bin[r + 1] - row_bin[r] < sweep_min &&
                    !(kw_a_pos && x < n_xl && kway_takes(row_bin[r + 1] - row_bin[r], kw_a_pos[r + 1] - kw_a_pos[r]))) break;
            }
            s_x = x;
        }
        __syncthreads();
        const uint32_t x = s_x;
        if (x >= n_all) break;
        const uint64_t row = x < n_xl ? xl_list[x] : long_list[x - n_xl];
        const uint64_t len = row_bin[row + 1] - row_bin[row];
        Elem *bin = bins + (row_bin[row] - bin_base);
        Elem nxt; nxt.idx = 0; nxt.val = 0.f;
        if (tid < len) nxt = bin[tid];                                   // the next chunk is always in flight
        for (uint64_t c0 = 0; c0 < len; c0 += XL_THREADS) {
            const uint64_t p = c0 + tid;
            const bool active = p < len;
            bool pending = active;
            const Elem e = nxt;
            if (p + XL_THREADS < len) nxt = bin[p + XL_THREADS];
            uint32_t slot = 0;
            if (active) {
                slot = (e.idx * 2654435761u) >> 21;                      // 11 bits
                while (true) {
                    const uint32_t prev = atomicCAS(&key[slot], XL_EMPTY, e.idx);
                    if (prev == XL_EMPTY || prev == e.idx) break;
                    slot = (slot + 1) & (XL_SLOTS - 1);
                }
                atomicMin(&owner[slot], tid);
            }
            __syncthreads();
            while (true) {
                const bool win = pending && owner[slot] == tid;
                if (win) {
                    uint32_t *w = bits + (e.idx >> 5);
                    const uint32_t bit = 1u << (e.idx & 31);
                    const uint32_t seen = __ldcg(w);                     // the two loads go out together
                    const float old = __ldcg(acc + e.idx);
                    if (seen & bit) {
                        acc[e.idx] = __fadd_rn(old, e.val);
                    } else {
                        acc[e.idx] = e.val;
                        atomicOr(w, bit);
                    }
                    pending = false;
                }
                __syncthreads();                                         // every owner[] has been read; the adds are visible
                if (win) owner[slot] = XL_EMPTY;
                if (!__syncthreads_or(pending)) break;
                if (pending) atomicMin(&owner[slot], tid);               // next position of a repeated column
                __syncthreads();
            }
            if (active) { key[slot] = XL_EMPTY; owner[slot] = XL_EMPTY; }
            __syncthreads();
        }
        // ordered compaction of the accumulator over the (fully consumed) bin
        uint64_t produced = 0;
        for (uint64_t w0 = 0; w0 < words; w0 += XL_THREADS) {
            const uint64_t w = w0 + tid;
            uint32_t b = w < words ? __ldcg(bits + w) : 0u;
            uint32_t total;
            const uint32_t rank = block_exclusive_scan(__popc(b), warp_sums, total);
            uint64_t o = produced + rank;
            if (b) bits[w] = 0u;
            while (b) {
                const uint32_t bit = __ffs(b) - 1;
                b &= b - 1;
                const uint32_t col = uint32_t(w * 32 + bit);
                Elem r; r.idx = col; r.val = acc[col];
                bin[o++] = r;
            }
            produced += total;
        }
        if (tid == 0) uniq[row] = uint32_t(produced);
    }
}

// =====================================================================================
// Merge, long rows over a small column range (cols <= DENSE_MAX_COLS): one CTA per row folds the
// partial products into a dense accumulator in shared memory -- acc[col], seen[col] -- and then
// emits the seen columns in ascending order.  The row is consumed T partial products at a time in
// arrival order; products of one chunk that hit the same column are serialised by an arbitration
// on owner[col] (the lowest position goes first), so every column is still summed in ascending
// arrival (= k) order with separately rounded adds.  No sort, no global scratch.
// Shared: float acc[cols] | uint16 owner[cols] | uint8 seen[cols] | uint32 warp_sums[33]
// =====================================================================================
constexpr uint32_t DENSE_MAX_COLS = 16384;
constexpr int DENSE_THREADS = 512;
__host__ __device__ inline size_t dense_smem(uint64_t cols) { return size_t((cols + 15) & ~15ull) * 7 + 34 * 4; }

__global__ void __launch_bounds__(DENSE_THREADS)
k_merge_dense(const uint64_t *__restrict__ row_bin, uint64_t bin_base, Elem *bins, uint32_t *uniq,
              const uint32_t *long_list, const uint32_t *xl_list, const DevScalars *sc, uint32_t cols,
              uint64_t row_lo, uint64_t row_hi) {
    OSP_EXTERN_SMEM(smem);
    const uint32_t cpad = (cols + 15) & ~15u;
    float *acc = reinterpret_cast<float *>(smem);
    uint16_t *owner = reinterpret_cast<uint16_t *>(smem + size_t(cpad) * 4);
    unsigned char *seen = smem + size_t(cpad) * 6;
    uint32_t *warp_sums = reinterpret_cast<uint32_t *>(smem + size_t(cpad) * 7);
    const uint32_t tid = threadIdx.x;
    for (uint32_t c = tid; c < cpad; c += DENSE_THREADS) { owner[c] = 0xFFFF; seen[c] = 0; }
    __syncthreads();
    const uint32_t n_long = sc->n_long, n_all = n_long + sc->n_xl;
    for (uint32_t x = blockIdx.x; x < n_all; x += gridDim.x) {
        const uint64_t row = x < n_long ? long_list[x] : xl_list[x - n_long];
        if (row < row_lo || row >= row_hi) continue;
        const uint64_t len = row_bin[row + 1] - row_bin[row];
        Elem *bin = bins + (row_bin[row] - bin_base);
        for (uint64_t c0 = 0; c0 < len; c0 += DENSE_THREADS) {
            const uint64_t p = c0 + tid;
            bool pending = p < len;
            Elem e; e.idx = 0; e.val = 0.f;
            if (pending) e = bin[p];
            while (__syncthreads_or(pending)) {
                // the lowest pending position of every column wins this round (racing minimum, re-checked)
                bool want = pending;
                do {
                    if (want && owner[e.idx] > tid) owner[e.idx] = uint16_t(tid);
                    __syncthreads();
                    want = pending && owner[e.idx] > tid;
                } while (__syncthreads_or(want));
                if (pending && owner[e.idx] == tid) {
                    acc[e.idx] = seen[e.idx] ? __fadd_rn(acc[e.idx], e.val) : e.val;
                    seen[e.idx] = 1;
                    owner[e.idx] = 0xFFFF;
                    pending = false;
                }
            }
        }
        __syncthreads();
        // emit the seen columns in ascending order over the (fully consumed) bin
        const uint32_t per = (cols + DENSE_THREADS - 1) / DENSE_THREADS;
        const uint32_t cb = min(tid * per, cols), ce = min(cb + per, cols);
        uint32_t cnt = 0;
        for (uint32_t c = cb; c < ce; c++) cnt += seen[c];
        uint32_t total;
        uint32_t o = block_exclusive_scan(cnt, warp_sums, total);
        for (uint32_t c = cb; c < ce; c++) {
            if (seen[c]) {
                Elem r; r.idx = c; r.val = acc[c];
                bin[o++] = r;
                seen[c] = 0;
            }
        }
        if (tid == 0) uniq[row] = total;
        __syncthreads();
    }
}

// =====================================================================================
// Merge of short rows, building blocks:
//   sort_grouped        sorts (col << pb | arrival position) keys held E per lane in registers, one row per
//                       group of 2^T lanes (flip-bitonic network over VIMNMX and shuffles);
//   merge_rows_grouped  reads the rows' partial products from the shared-memory stage of their tile, sorts,
//                       left-folds equal columns in arrival (= k) order with separately rounded adds and
//                       writes the compacted rows into the tile's output stage.
// =====================================================================================
template <int V> struct ILog2 { static constexpr int value = 1 + ILog2<V / 2>::value; };
template <> struct ILog2<1> { static constexpr int value = 0; };


// Output stage of a tile: element s lives at ostage[swz(s)].  The XOR swizzle spreads the blocked writes
// of the sorted rows (lane l holds sorted positions l*E .. l*E+E-1) over all banks and keeps linear reads
// conflict-free (it permutes inside aligned groups of 16 elements = 128 B).
__device__ __forceinline__ uint32_t swz(uint32_t s) { return s ^ ((s >> 4) & 15u); }

// ---- grouped sort: several short rows per warp ------------------------------------------------------
// A row of len <= N = E << T partial products is sorted by a group of G = 1 << T lanes, E keys per lane,
// so a warp sorts 32 / G rows at once.  Bitonic network in its "flip" form: the first stage of every merge
// level compares i with i ^ (k - 1), the others i with i ^ j, and EVERY compare-exchange is ascending --
// the in-lane stages have compile-time partners and directions (two VIMNMX per pair), the cross-lane stages
// one shuffle and a min-or-max per key.  Levels up to E run inside a lane; T more levels cross lanes.
// T is a template parameter: the whole network is straight-line code, no register moves at loop edges.
#ifdef OSP_CUSIM
#define osp_smem (cusim::dyn_smem())
#else
extern __shared__ __align__(16) unsigned char osp_smem[];     // the dynamic shared memory of every kernel here
#endif
__device__ __forceinline__ uint32_t &smem_u32_at(uint32_t off) { return *reinterpret_cast<uint32_t *>(osp_smem + off); }
__device__ __forceinline__ float &smem_f32_at(uint32_t off) { return *reinterpret_cast<float *>(osp_smem + off); }
__device__ __forceinline__ uint2 &smem_u2_at(uint32_t off) { return *reinterpret_cast<uint2 *>(osp_smem + off); }

template <int E, class K>
__device__ __forceinline__ void ce_inlane(K (&x)[E], const int a, const int b) {
    const K lo = min(x[a], x[b]), hi = max(x[a], x[b]);
    x[a] = lo; x[b] = hi;
}
// Cross-lane compare-exchange: the lane keeps the smaller or the larger of its key and its partner's.
// OSP_CE_SEL=1 (experiment): compare + select instead of min-or-max under a predicate.
#ifndef OSP_CE_SEL
#define OSP_CE_SEL 0
#endif
template <class K>
__device__ __forceinline__ K ce_cross(const K x, const K y, const bool keep_min) {
#if OSP_CE_SEL
    return ((x < y) == keep_min) ? x : y;
#else
    return keep_min ? min(x, y) : max(x, y);
#endif
}
template <int E, class K>
__device__ __forceinline__ void sort_grouped(K (&x)[E], const unsigned int lig, const int T) {
#pragma unroll
    for (int k = 2; k <= E; k <<= 1) {
#pragma unroll
        for (int e = 0; e < E; e++)
            if (e < (e ^ (k - 1))) ce_inlane<E, K>(x, e, e ^ (k - 1));
#pragma unroll
        for (int j = k >> 2; j > 0; j >>= 1) {
#pragma unroll
            for (int e = 0; e < E; e++)
                if ((e & j) == 0) ce_inlane<E, K>(x, e, e | j);
        }
    }
    // The cross-lane levels are a RUNTIME loop since round 2: one body for every row class.  Fully unrolled per class the
    // merge chain was 134 KB of SASS, more than the instruction cache holds: warps sorting rows of different classes evicted
    // each other's code (ncu: no_inst 15 % of the stall samples).  The element index stays a compile-time constant, so the
    // keys never leave their registers.
#pragma unroll 1
    for (int t = 1; t <= T; t++) {
        {   // flip stage: (lane, e) <-> (lane ^ (2^t - 1), E - 1 - e); the lane whose bit t-1 is clear keeps the minima
            const bool keep_min = ((lig >> (t - 1)) & 1u) == 0;
            const int mask = (1 << t) - 1;
            K y[E];
#pragma unroll
            for (int e = 0; e < E; e++) y[e] = __shfl_xor_sync(FULL, x[E - 1 - e], mask);
#pragma unroll
            for (int e = 0; e < E; e++) x[e] = ce_cross(x[e], y[e], keep_min);
        }
#pragma unroll 1
        for (int lj = (1 << t) >> 2; lj > 0; lj >>= 1) {
            const bool keep_min = (lig & lj) == 0;
#pragma unroll
            for (int e = 0; e < E; e++) {
                const K y = __shfl_xor_sync(FULL, x[e], lj);
                x[e] = ce_cross(x[e], y, keep_min);
            }
        }
#pragma unroll
        for (int j = E >> 1; j > 0; j >>= 1) {
#pragma unroll
            for (int e = 0; e < E; e++)
                if ((e & j) == 0) ce_inlane<E, K>(x, e, e | j);
        }
    }
}

// Groups of G = 1 << T lanes merge one row each (2 <= len <= E << T; len = 0: the group idles).  `row_off`,
// `o0`, `len` are the group's own (uniform inside a group): the byte offset in shared memory of the row's
// partial products in the tile's input stage (reused as fold scratch once every input is in registers) and
// the index of the row's first element in the output stage at byte offset `ost_off`.  Returns the row's
// number of surviving entries.
// MUL (k_chain2): the stage holds the raw elements of B; element p of the row is multiplied by the float at shared-memory
// byte offset arow_off + 4 p (A(i,k) of the run it belongs to) when its value is read -- rounded on its own, no FMA.
template <int E, class K, bool MUL = false>
__device__ __forceinline__ uint32_t merge_rows_grouped(const int T, const uint32_t row_off, const uint32_t ost_off, const uint32_t o0,
                                                       const uint32_t len, const unsigned int lane, const uint32_t arow_off = 0) {
    constexpr int LE = ILog2<E>::value;
    const uint32_t G = 1u << T, PB = LE + T, N = uint32_t(E) << T;       // (T is a run-time value: one body for all classes)
    const uint32_t lig = lane & (G - 1);
    K key[E];
    {
        const uint32_t a0 = row_off + lig * 8;
#pragma unroll
        for (int e = 0; e < E; e++) {
            const uint32_t p = uint32_t(e) * G + lig;
            const K k = (K(smem_u32_at(a0 + uint32_t(e) * G * 8)) << PB) | K(p);    // past the row: harmless bytes of the stage
            key[e] = p < len ? k : ~K(0);
        }
    }
    sort_grouped<E, K>(key, lig, T);
    // lane now holds the sorted positions lig*E .. lig*E+E-1 of its group's row
    uint32_t col[E];
    float v[E];
#pragma unroll
    for (int e = 0; e < E; e++) {
        col[e] = uint32_t(key[e] >> PB);
        v[e] = smem_f32_at(row_off + 4 + (uint32_t(key[e]) & (N - 1)) * 8);       // padding keys read harmless bytes
        if (MUL) v[e] = __fmul_rn(smem_f32_at(arow_off + (uint32_t(key[e]) & (N - 1)) * 4), v[e]);
    }
    const uint32_t s0 = lig * E;
    uint32_t prev = __shfl_up_sync(FULL, col[E - 1], 1);
    const uint32_t next_first = __shfl_down_sync(FULL, col[0], 1);
    {
        bool dup = false;
        uint32_t pc = prev;
#pragma unroll
        for (int e = 0; e < E; e++) {
            dup |= s0 + e < len && s0 + e > 0 && pc == col[e];
            pc = col[e];
        }
        if (!__any_sync(FULL, dup)) {               // no duplicate column in any of the rows: sorted = merged
#pragma unroll
            for (int e = 0; e < E; e++)
                if (s0 + e < len) smem_u2_at(ost_off + swz(o0 + s0 + e) * 8) = make_uint2(col[e], __float_as_uint(v[e]));
            return len;
        }
    }
    __syncwarp();                                   // every lane has read its inputs: the rows become scratch
    uint32_t *scol = reinterpret_cast<uint32_t *>(osp_smem + row_off);
    float *sval = reinterpret_cast<float *>(osp_smem + row_off) + len;
    Elem *ostage = reinterpret_cast<Elem *>(osp_smem + ost_off);
#pragma unroll
    for (int e = 0; e < E; e++)
        if (s0 + e < len) { scol[s0 + e] = col[e]; sval[s0 + e] = v[e]; }
    __syncwarp();
    // left folds of the heads (first arrival of a column), in arrival (= k) order
    bool head[E];
    uint32_t nheads = 0;
#pragma unroll
    for (int e = 0; e < E; e++) {
        const uint32_t s = s0 + e;
        head[e] = s < len && (s == 0 || prev != col[e]);
        prev = col[e];
        if (head[e]) {
            nheads++;
            const uint32_t nxt = e + 1 < E ? col[e + 1 < E ? e + 1 : 0] : next_first;
            if (s + 1 < len && nxt == col[e]) {
                float sum = v[e];
                for (uint32_t u = s + 1; u < len && scol[u] == col[e]; u++) sum = __fadd_rn(sum, sval[u]);
                v[e] = sum;
            }
        }
    }
    uint32_t incl = nheads;                          // inclusive scan inside the group
    for (uint32_t o = 1; o < G; o <<= 1) {
        const uint32_t y = __shfl_up_sync(FULL, incl, o);
        if (lig >= o) incl += y;
    }
    const uint32_t total = __shfl_sync(FULL, incl, lane | (G - 1));
    uint32_t r = o0 + incl - nheads;
#pragma unroll
    for (int e = 0; e < E; e++) {
        if (head[e]) {
            Elem o; o.idx = col[e]; o.val = v[e];
            ostage[swz(r++)] = o;
        }
    }
    return total;
}

// ---- bitmap-rank merge of one longer row over a small column range (cols <= 32 * BM_WORDS) -------------
// No sort: every partial product sets the bit of its column in a per-warp bitmap; a prefix popcount over the
// bitmap words turns a column into its rank among the row's distinct columns (= its place in the sorted,
// folded row); the earliest arrival of a column (atomicMin over arrival positions) opens that place and the
// later arrivals are added one by one in arrival (= k) order with separately rounded adds.  S 32-element
// slots of the row live in registers, every pass works on all of them at once (independent shared-memory
// operations, five warp-level syncs per row).  ONE 16-slot instantiation serves every row up to 512 partial products
// (a 20-slot one the rare rows up to 640): slot counts fitted to the row ran up to 50 % slower on config 2 -- warps
// in different unrolled bodies thrash the instruction cache.
constexpr uint32_t BM_WORDS = 512;                         // bitmap words per warp: columns < 16384
constexpr uint32_t BM_SCRATCH = BM_WORDS * 4 + BM_WORDS * 2;   // per warp: bitmap | exclusive popcount prefix per word (u16)
__device__ __forceinline__ uint4 &smem_u4_at(uint32_t off) { return *reinterpret_cast<uint4 *>(osp_smem + off); }
__device__ __forceinline__ uint16_t &smem_u16_at(uint32_t off) { return *reinterpret_cast<uint16_t *>(osp_smem + off); }

template <int S, bool MUL = false>
__device__ __forceinline__ uint32_t merge_row_bitmap(const uint32_t row_off, const uint32_t ost_off, const uint32_t o0,
                                                     const uint32_t len, const uint32_t wpl, const uint32_t scr_off,
                                                     const unsigned int lane, const uint32_t arow_off = 0) {
    const uint32_t bm_off = scr_off, pre_off = scr_off + BM_WORDS * 4;
    // lane owns the bitmap words {4*lane + 128*q .. +3}: conflict-free 128-bit accesses
    for (uint32_t q = 0; q < wpl; q += 4) smem_u4_at(bm_off + (4 * lane + 32 * q) * 4) = make_uint4(0, 0, 0, 0);
    uint32_t col[S];
    float val[S];
#pragma unroll
    for (int s = 0; s < S; s++) {
        const uint32_t p = s * 32 + lane;
        col[s] = 0xFFFFFFFFu; val[s] = 0.f;
        if (p < len) {
            const uint2 e = smem_u2_at(row_off + p * 8); col[s] = e.x; val[s] = __uint_as_float(e.y);
            if (MUL) val[s] = __fmul_rn(smem_f32_at(arow_off + p * 4), val[s]);
        }
    }
    __syncwarp();
#pragma unroll
    for (int s = 0; s < S; s++)
        if (col[s] != 0xFFFFFFFFu) atomicOr(&smem_u32_at(bm_off + (col[s] >> 5) * 4), 1u << (col[s] & 31));
    __syncwarp();
    // exclusive prefix popcount over the words, in word order (chunk q of every lane, then chunk q+4, ...)
    uint32_t uniq = 0;
    for (uint32_t q = 0; q < wpl; q += 4) {
        const uint4 w = smem_u4_at(bm_off + (4 * lane + 32 * q) * 4);
        const uint32_t c0 = __popc(w.x), c1 = __popc(w.y), c2 = __popc(w.z), c3 = __popc(w.w);
        const uint32_t cnt = c0 + c1 + c2 + c3;
        const uint32_t incl = warp_inclusive_scan(cnt);
        const uint32_t b0 = uniq + incl - cnt;
        uint2 pk;
        pk.x = b0 | ((b0 + c0) << 16);
        pk.y = (b0 + c0 + c1) | ((b0 + c0 + c1 + c2) << 16);
        smem_u2_at(pre_off + (4 * lane + 32 * q) * 2) = pk;
        uniq += __shfl_sync(FULL, incl, 31);
    }
    // first[rank] = earliest arrival position, kept in the row's own input span (its elements are in registers)
    for (uint32_t i = lane; i < uniq; i += 32) smem_u32_at(row_off + i * 4) = 0xFFFFFFFFu;
    __syncwarp();
    uint32_t r[S];
#pragma unroll
    for (int s = 0; s < S; s++) {
        r[s] = 0;
        if (col[s] != 0xFFFFFFFFu) {
            const uint32_t w = col[s] >> 5;
            r[s] = smem_u16_at(pre_off + w * 2) + __popc(smem_u32_at(bm_off + w * 4) & ((1u << (col[s] & 31)) - 1));
            atomicMin(&smem_u32_at(row_off + r[s] * 4), uint32_t(s * 32 + lane));
        }
    }
    __syncwarp();
    uint32_t losers = 0;                              // slots of this lane that are later arrivals of their column
#pragma unroll
    for (int s = 0; s < S; s++) {
        if (col[s] != 0xFFFFFFFFu) {
            if (smem_u32_at(row_off + r[s] * 4) == uint32_t(s * 32 + lane))
                smem_u2_at(ost_off + swz(o0 + r[s]) * 8) = make_uint2(col[s], __float_as_uint(val[s]));
            else losers |= 1u << s;
        }
    }
    __syncwarp();
    if (__any_sync(FULL, losers != 0)) {              // later arrivals: slot after slot, inside a slot lowest lane first
#pragma unroll
        for (int s = 0; s < S; s++) {
            unsigned int b = __ballot_sync(FULL, (losers >> s) & 1u);
            while (b) {
                const unsigned int l = __ffs(b) - 1;
                b &= b - 1;
                if (lane == l) {
                    const uint32_t a = ost_off + swz(o0 + r[s]) * 8 + 4;
                    smem_f32_at(a) = __fadd_rn(smem_f32_at(a), val[s]);
                }
                __syncwarp();
            }
        }
    }
    return uniq;
}

// ---- TMA bulk copy (cp.async.bulk, SASS UBLKCP) and its mbarrier ---------------------------------------
#ifdef OSP_CUSIM   // tests/cusim: a bulk copy that completes at once is one legal schedule of the asynchronous one
__device__ __forceinline__ void mbar_init(uint64_t *, uint32_t) {}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *, uint32_t) {}
__device__ __forceinline__ void tma_load_1d(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *) { std::memcpy(dst_smem, src_gmem, bytes); }
__device__ __forceinline__ void mbar_wait(uint64_t *, uint32_t) {}
#else
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return uint32_t(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_1d(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!done);
}
#endif

// =====================================================================================
// Merge, the main kernel: one pass from the partial-product bins to CSR C.
// Persistent CTAs take tiles in ticket (= row) order.  A tile is a run of consecutive short rows --
// <= MT_RMAX rows, < MT_STAGE partial products, contiguous in the bins.  Per tile:
//   1. ONE TMA bulk copy (cp.async.bulk + mbarrier) pulls the tile into shared memory;
//   2. the warps take the rows one after the other: register bitonic sort by (col, arrival position),
//      k-ordered left fold of equal columns, compacted row into the tile's output stage;
//   3. a block scan of the surviving counts gives the row offsets inside the tile and the tile's aggregate,
//      published at once for the decoupled look-back across tiles;
//   4. the tile's offset in C is resolved and its output stage streams to C.data / C.pos ONE TILE LATER:
//      the chain retires tiles in order, so a tile that waited for its predecessors right after its own
//      sort would idle its CTA; deferred by one tile, the wait falls on predecessors that have had a whole
//      sort of slack, and the next tile's bulk copy is in flight underneath.  (Prefetching one tile further
//      into a second input stage was measured and dropped: it costs a resident CTA per SM and gains nothing.)
// C is written exactly once, in its final place.  Long rows are tiles of their own: merged in place
// beforehand (k_merge_long / k_merge_xl / k_merge_dense, uniq[row] survivors at the start of their bin) and
// copied here so that the chain stays in row order.
// HBM traffic = the algorithmic minimum of the merge: 8 P read + 8 nnz(C) + 8 (m+1) written.
// K = uint32_t when col << 9 fits 32 bits (cols <= 2^23), else uint64_t.
// =====================================================================================
// Rows of class c (<= 8 << c partial products) are sorted 8 keys per lane by groups of 2^c lanes, from class MC_E16_FROM on
// 16 keys per lane by groups of 2^(c-1) lanes (class 6, 257..512, has no other choice: 32 lanes x 16 keys).
#ifndef OSP_E16_FROM
#define OSP_E16_FROM 6
#endif
constexpr int MC_E16_FROM = OSP_E16_FROM;
static_assert(MC_E16_FROM >= 1 && MC_E16_FROM <= 6, "class 0 has 8 keys at most; class 6 needs 16 keys per lane");
__host__ __device__ constexpr uint32_t mc_group_bits(uint32_t c) { return c >= uint32_t(MC_E16_FROM) ? c - 1 : c; }
constexpr int MC_THREADS = OSP_MC_THREADS;
constexpr int MC_OCC = OSP_MC_OCC;                              // resident CTAs per SM (shared memory: 3 stages each)
static_assert(MT_RMAX <= MC_THREADS, "one thread per row of a tile");
constexpr uint32_t MC_STAGE_ELEMS = MT_STAGE + 16;     // + alignment shift, rounded for the swizzle groups
template <bool BM>
struct __align__(16) MergeChainSmem {
    Elem stage[MC_STAGE_ELEMS];        // input of the tile being sorted (TMA destination)
    Elem ostage[2][MC_STAGE_ELEMS];    // output of the tile being sorted / of the tile awaiting its offset
    uint32_t rstart[3][MT_RMAX + 1];   // bin start of every row relative to the tile (next, current, previous tile)
    uint32_t rout[3][MT_RMAX];         // survivors per row, then their exclusive scan
    uint32_t warp_sums[33];
    uint32_t next_batch;
    uint16_t order[MT_RMAX];           // the tile's rows grouped by size class, longest class first
    uint32_t cls_cnt[8], cls_off[8], cls_b0[9];   // per class: rows, start in order[], first batch; cls_b0[8] = batches
    uint64_t base;
    uint64_t mbar;
    uint64_t d_r0[2], d_g0[2];         // descriptors of the tiles opened ahead (written by the opening warp)
    uint32_t d_idx[2], d_R[2], d_nin[2], d_long[2];
    __align__(16) unsigned char bm_scratch[BM ? (MC_THREADS / 32) * BM_SCRATCH : 16];   // per-warp bitmaps of the bitmap-rank merge
};
struct TileDesc {                      // uniform across the CTA
    uint32_t idx;                      // position in the chain
    uint32_t R, n_in, n_out;
    uint64_t r0, g0;                   // first row, first partial product (relative to the bins pointer)
    bool is_long, last;
};

// look-back, split: publish the aggregate now, resolve the exclusive prefix later (one warp, all lanes)
__device__ __forceinline__ void lb_publish(uint64_t *state, uint32_t idx, uint64_t aggregate, uint64_t carry) {
    if (lane_id() == 0) st_relaxed_u64(state + idx, idx == 0 ? (LB_FLAG_PREFIX | (carry + aggregate)) : (LB_FLAG_AGG | aggregate));
}
__device__ __forceinline__ uint64_t lb_resolve(uint64_t *state, uint32_t idx, uint64_t aggregate, uint64_t carry) {
    if (idx == 0) return carry;
    const unsigned int lane = lane_id();
    uint64_t exclusive = 0;
    int64_t base = int64_t(idx) - 1;
    while (true) {
        const int64_t i = base - lane;
        uint64_t word = LB_FLAG_PREFIX;                  // before the chain: prefix 0 (never reached: tile 0 holds a prefix)
        if (i >= 0) {
            word = ld_relaxed_u64(state + i);
            unsigned int ns = 32;
            while ((word >> 62) == 0) {                  // predecessor still sorting: back off
                __nanosleep(ns);
                if (ns < 512) ns <<= 1;
                word = ld_relaxed_u64(state + i);
            }
        }
        const unsigned int has_prefix = __ballot_sync(FULL, (word >> 62) == 2);
        const unsigned int firstp = has_prefix ? (__ffs(has_prefix) - 1) : 31;
        uint64_t v = (lane <= firstp) ? (word & LB_VALUE_MASK) : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
        exclusive += v;
        if (has_prefix) break;
        base -= 32;
    }
    if (lane == 0) st_relaxed_u64(state + idx, LB_FLAG_PREFIX | (exclusive + aggregate));
    return exclusive;
}

// FUSED (opt-in, OSP_FUSED_SHORT; not yet run on a B200): the tiles of short rows never go through the bins.  With the
// row-order multiply a tile's partial products are the runs of consecutive tasks (run_off is the prefix the plan cut
// the tiles from), so the CTA computes them straight into its stage -- the warp-flat walk of k_multiply with
// shared-memory stores -- where the default path bulk-copies what k_multiply wrote to HBM.  Long rows (tiles of their
// own) still come merged from the bins.
struct FusedSrc {
    const uint64_t *a_pos;      // CSR(A)
    const Elem *a_data;
    const uint64_t *run_off;    // bin offset of every task's run (absolute)
    const uint32_t *task_bs;    // b_pos[k] of every task
    const Elem *b_data;
    uint64_t m_a;               // rows of A (rows beyond hold no task)
};

template <class K, bool BM, bool FUSED>
__device__ __forceinline__ void
merge_chain_body(const uint64_t *__restrict__ row_bin, const uint64_t bin_base, const Elem *__restrict__ bins,
                 const uint32_t *__restrict__ tile_row, const uint32_t t0, const uint32_t n_chain,
                 const uint32_t *__restrict__ uniq, uint64_t *tile_state, DevScalars *sc, const int carry_slot,
                 uint64_t *__restrict__ c_pos, Elem *__restrict__ c_data, const uint32_t bm_wpl, const uint32_t long_thresh,
                 const FusedSrc fs) {
    using Smem = MergeChainSmem<BM>;
    Smem &sm = *reinterpret_cast<Smem *>(osp_smem);
    const unsigned int tid = threadIdx.x, lane = lane_id(), warp = tid >> 5;
    const uint64_t carry = sc->nnz_c[carry_slot];
    if (tid == 0) mbar_init(&sm.mbar, 1);

    // Opening a tile, in three steps.  (1) ONE warp takes the ticket, reads the tile's bounds and row starts
    // (a chain of dependent global loads, ~2-3 us) and leaves the descriptor in slot `ds` -- during the sort of
    // the current tile, whose batches the other warps keep pulling.  (2) After a barrier every thread reads the
    // descriptor.  (3) One thread starts the bulk copy of the tile's partial products once the stage is free.
    auto prefetch_tile = [&](uint32_t slot, uint32_t ds) {
        uint32_t idx = 0;
        if (lane == 0) idx = atomicAdd(&sc->tile_ticket, 1u);
        idx = __shfl_sync(FULL, idx, 0);
        uint64_t r0 = 0, g0 = 0;
        uint32_t R = 0, n_in = 0, is_long = 0;
        if (idx < n_chain) {
            const uint32_t tile = t0 + idx;
            r0 = tile_row[tile];
            const uint64_t r1 = tile_row[tile + 1];
            R = uint32_t(r1 - r0);
            const uint64_t b0 = row_bin[r0], b1 = row_bin[r1];
            g0 = b0 - bin_base;
            is_long = R == 1 && b1 - b0 > long_thresh;
            n_in = is_long ? 0u : uint32_t(b1 - b0);
            if (!is_long)
                for (uint32_t j = lane; j <= R; j += 32) sm.rstart[slot][j] = uint32_t(row_bin[r0 + j] - b0);
        }
        if (lane == 0) {
            sm.d_idx[ds] = idx; sm.d_R[ds] = R; sm.d_nin[ds] = n_in; sm.d_long[ds] = is_long;
            sm.d_r0[ds] = r0; sm.d_g0[ds] = g0;
        }
    };
    auto load_desc = [&](uint32_t ds) -> TileDesc {
        TileDesc d;
        d.idx = sm.d_idx[ds]; d.R = sm.d_R[ds]; d.n_in = sm.d_nin[ds]; d.is_long = sm.d_long[ds] != 0;
        d.r0 = sm.d_r0[ds]; d.g0 = sm.d_g0[ds];
        d.last = d.idx + 1 == n_chain;
        d.n_out = 0;
        return d;
    };
    // FUSED: the tile's partial products computed into the stage by the whole CTA (tasks of rows r0 .. r0+R, 32 per
    // warp and turn, the concatenation of their runs walked 64 products at a time as in k_multiply).
    constexpr int FW = 4;                                        // independent 32-product chunks (= loads in flight per lane) per turn
    auto fill_stage = [&](const TileDesc &d) {
        if (d.idx < n_chain && !d.is_long && d.n_in) {
            const uint64_t e0 = fs.a_pos[min(d.r0, fs.m_a)], e1 = fs.a_pos[min(d.r0 + d.R, fs.m_a)];
            Elem *stage = sm.stage + uint32_t(d.g0 & 1);
            const uint64_t first = d.g0 + bin_base;              // run_off of the tile's first partial product
            for (uint64_t base = e0 + warp * 32; base < e1; base += (MC_THREADS / 32) * 32) {
                uint32_t bs = 0, len = 0, off = 0; float a = 0.f;
                if (base + lane < e1) {
                    const uint64_t i = base + lane;
                    const uint64_t ro = fs.run_off[i];
                    a = fs.a_data[i].val; off = uint32_t(ro - first);
                    len = uint32_t(fs.run_off[i + 1] - ro);
                    bs = fs.task_bs[i];
                }
                const uint32_t incl = warp_inclusive_scan(len);
                const uint32_t total = __shfl_sync(FULL, incl, 31);
                const uint32_t excl = incl - len;
                const uint32_t dbs = bs - excl, doff = off - excl;
                for (uint32_t q0 = 0; q0 < total; q0 += 32 * FW) {
                    uint32_t q[FW], t[FW];
#pragma unroll
                    for (int u = 0; u < FW; u++) { q[u] = q0 + 32 * u + lane; t[u] = 0; }
#pragma unroll
                    for (int step = 16; step > 0; step >>= 1) {
#pragma unroll
                        for (int u = 0; u < FW; u++) {
                            const uint32_t v = __shfl_sync(FULL, incl, t[u] + step - 1);
                            if (v <= q[u]) t[u] += step;
                        }
                    }
                    float a_t[FW]; uint32_t dbs_t[FW], doff_t[FW]; Elem b[FW];
#pragma unroll
                    for (int u = 0; u < FW; u++) {
                        a_t[u] = __shfl_sync(FULL, a, t[u] & 31);
                        dbs_t[u] = __shfl_sync(FULL, dbs, t[u] & 31);
                        doff_t[u] = __shfl_sync(FULL, doff, t[u] & 31);
                    }
#pragma unroll
                    for (int u = 0; u < FW; u++)
                        if (q[u] < total) b[u] = fs.b_data[dbs_t[u] + q[u]];
#pragma unroll
                    for (int u = 0; u < FW; u++)
                        if (q[u] < total) {
                            Elem o; o.idx = b[u].idx; o.val = __fmul_rn(a_t[u], b[u].val);     // rounded on its own: no FMA
                            stage[doff_t[u] + q[u]] = o;
                        }
                }
            }
        }
        __syncthreads();                                         // the stage is complete (and every warp has left the loop)
    };
    auto start_copy = [&](const TileDesc &d) {
        if (FUSED) { fill_stage(d); return; }
        if (tid == 0 && d.idx < n_chain && !d.is_long && d.n_in) {
            const uint32_t shift = uint32_t(d.g0 & 1);              // the window starts one element early when g0 is odd
            const uint32_t bytes = ((d.n_in + shift) * 8 + 15) & ~15u;
#ifndef OSP_CUSIM
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // earlier generic reads of the stage
#endif
            mbar_expect_tx(&sm.mbar, bytes);
            tma_load_1d(sm.stage, bins + (d.g0 - shift), bytes, &sm.mbar);
        }
    };
    // Resolves the offset of tile `d` in C and streams its output stage out.
    auto retire_tile = [&](const TileDesc &d, uint32_t slot, uint32_t obuf) {
        if (warp == 0) {
            const uint64_t excl = lb_resolve(tile_state, d.idx, d.n_out, carry);
            if (lane == 0) sm.base = excl;
        }
        __syncthreads();
        const uint64_t base = sm.base;
        if (tid == 0 && d.last) { c_pos[d.r0 + d.R] = base + d.n_out; sc->nnz_c[carry_slot ^ 1] = base + d.n_out; }
        if (d.is_long) {
            const Elem *src = bins + d.g0;
            uint32_t i = tid;
            for (; i + 7 * MC_THREADS < d.n_out; i += 8 * MC_THREADS) {      // eight loads in flight per thread
                Elem e[8];
#pragma unroll
                for (int u = 0; u < 8; u++) e[u] = src[i + u * MC_THREADS];
#pragma unroll
                for (int u = 0; u < 8; u++) c_data[base + i + u * MC_THREADS] = e[u];
            }
            for (; i < d.n_out; i += MC_THREADS) c_data[base + i] = src[i];
            if (tid == 0) c_pos[d.r0] = base;
            return;
        }
        const uint32_t *rout = sm.rout[slot];
        if (tid < d.R) c_pos[d.r0 + tid] = base + rout[tid];
        const Elem *ostage = sm.ostage[obuf];
        if (d.n_out == d.n_in) {                             // no duplicate column in the tile: rows are back to back
            for (uint32_t p = tid; p < d.n_out; p += MC_THREADS) c_data[base + p] = ostage[swz(p)];
        } else {
            const uint32_t *rstart = sm.rstart[slot];
            for (uint32_t j = warp; j < d.R; j += MC_THREADS / 32) {
                const uint32_t s = rstart[j], o = rout[j];
                const uint32_t u = (j + 1 < d.R ? rout[j + 1] : d.n_out) - o;
                for (uint32_t i = lane; i < u; i += 32) c_data[base + o + i] = ostage[swz(s + i)];
            }
        }
    };

    uint32_t it = 0, n_tma = 0;                            // bulk copies awaited so far (mbarrier phase parity)
    if (warp == MC_THREADS / 32 - 1) prefetch_tile(0, 0);
    __syncthreads();
    TileDesc cur = load_desc(0), prev;
    prev.idx = 0xFFFFFFFFu;
    start_copy(cur);
    while (cur.idx < n_chain) {
        const uint32_t slot = it % 3, ob = it & 1;
        if (tid == 0) sm.next_batch = 0;
        if (tid < 8) sm.cls_cnt[tid] = 0;
        __syncthreads();                                     // also: rstart[slot] is visible
        // ---- sort: stage -> ostage[ob], survivors per row ----
        if (cur.is_long) {
            cur.n_out = uniq[cur.r0];
            if (warp == MC_THREADS / 32 - 1) prefetch_tile((it + 1) % 3, (it + 1) & 1);
        } else {
            uint32_t *rstart = sm.rstart[slot], *rout = sm.rout[slot];
            Elem *ostage = sm.ostage[ob];
            const uint32_t R = cur.R;
            // size classes (while the bulk copy is in flight): class c sorts rows of <= 8 << c partial products,
            // 32 >> c rows per warp at a time (class 6: 257..512, one row per warp, 16 keys per lane; class 7: 513..640,
            // bitmap variant only)
            uint32_t my_len = 0, my_cls = 8, my_pos = 0;
            if (tid < R) {
                my_len = rstart[tid + 1] - rstart[tid];
                if (my_len <= 1) rout[tid] = my_len;            // rows of 0 / 1 partial products need no merge
                else {
                    my_cls = my_len <= 8 ? 0u : 29u - uint32_t(__clz(my_len - 1));
                    my_pos = atomicAdd(&sm.cls_cnt[my_cls], 1u);
                }
            }
            __syncthreads();
            if (tid == 0) {
                uint32_t off = 0, b = 0;
#pragma unroll
                for (int c = 7; c >= 0; c--) {
                    const uint32_t n = sm.cls_cnt[c];
                    sm.cls_off[c] = off; sm.cls_b0[c] = b;
                    off += n;
                    const uint32_t T = mc_group_bits(uint32_t(c));
                    b += c >= 6 || (BM && c == 5) ? n : (n + (32u >> T) - 1) >> (5 - T);
                }
                sm.cls_b0[8] = b;
            }
            __syncthreads();
            if (my_cls < 8) sm.order[sm.cls_off[my_cls] + my_pos] = uint16_t(tid);
            Elem *stage = sm.stage + uint32_t(cur.g0 & 1);
            const uint32_t stage_off = uint32_t(offsetof(Smem, stage)) + uint32_t(cur.g0 & 1) * 8;
            const uint32_t ost_off = uint32_t(offsetof(Smem, ostage)) + ob * uint32_t(sizeof(Elem) * MC_STAGE_ELEMS);
            if (!FUSED && cur.n_in) { mbar_wait(&sm.mbar, n_tma & 1); n_tma++; }
            if (my_len == 1) ostage[swz(rstart[tid])] = stage[rstart[tid]];
            __syncthreads();                                  // order[] is complete
            const uint32_t n_batches = sm.cls_b0[8];
            if (warp == MC_THREADS / 32 - 1) prefetch_tile((it + 1) % 3, (it + 1) & 1);   // the others start on the batches
            while (true) {
                uint32_t b = 0;
                if (lane == 0) b = atomicAdd(&sm.next_batch, 1u);
                b = __shfl_sync(FULL, b, 0);
                if (b >= n_batches) break;
                int c = 7;
                while (c > 0 && b >= sm.cls_b0[c - 1]) c--;     // cls_b0 ascends from class 6 down to class 0
                const uint32_t T = c >= 6 || (BM && c == 5) ? 5u : mc_group_bits(uint32_t(c));
                const uint32_t idx = c >= 6 || (BM && c == 5) ? b - sm.cls_b0[c] : ((b - sm.cls_b0[c]) << (5 - T)) + (lane >> T);
                const bool valid = idx < sm.cls_cnt[c];
                uint32_t j = 0, s = 0, len = 0;
                if (valid) {
                    j = sm.order[sm.cls_off[c] + idx];
                    s = rstart[j];
                    len = rstart[j + 1] - s;
                }
                const uint32_t row_off = stage_off + s * 8;
                uint32_t u;
                if (BM && c >= 5) {       // small column range: rows of > 128 partial products skip the sort
                    const uint32_t scr_off = uint32_t(offsetof(Smem, bm_scratch)) + warp * BM_SCRATCH;
                    if (c <= 6) u = merge_row_bitmap<16>(row_off, ost_off, s, len, bm_wpl, scr_off, lane);   // one hot body (instruction cache)
                    else u = merge_row_bitmap<MT_LONG_BM / 32>(row_off, ost_off, s, len, bm_wpl, scr_off, lane);   // 513..640
                } else
                if (c < MC_E16_FROM) u = merge_rows_grouped<8, K>(c, row_off, ost_off, s, len, lane);
                else u = merge_rows_grouped<16, K>(int(T), row_off, ost_off, s, len, lane);
                if (valid && (lane & ((1u << T) - 1)) == 0) rout[j] = u;
            }
            __syncthreads();
            // ---- offsets of the rows inside the tile, the tile's aggregate ----
            const uint32_t my_u = tid < R ? rout[tid] : 0u;       // MT_RMAX == MC_THREADS: one row per thread
            uint32_t n_out;
            const uint32_t my_off = block_exclusive_scan(my_u, sm.warp_sums, n_out);
            if (tid < R) rout[tid] = my_off;
            cur.n_out = n_out;
        }
        if (warp == 0) lb_publish(tile_state, cur.idx, cur.n_out, carry);
        // ---- next tile: its descriptor is ready, bulk copy into the (now free) stage ----
        __syncthreads();                                     // also: every warp is done with the stage
        const TileDesc nxt = load_desc((it + 1) & 1);
        start_copy(nxt);
        // ---- the previous tile leaves (its predecessors have had this tile's sort to publish) ----
        if (prev.idx != 0xFFFFFFFFu) retire_tile(prev, (it + 2) % 3, ob ^ 1);
        prev = cur;
        cur = nxt;
        it++;
    }
    if (prev.idx != 0xFFFFFFFFu) {
        __syncthreads();
        retire_tile(prev, (it + 2) % 3, (it & 1) ^ 1);
    }
}

template <class K, bool BM>
__global__ void __launch_bounds__(MC_THREADS, BM ? 2 : MC_OCC)
k_merge_chain(const uint64_t *__restrict__ row_bin, const uint64_t bin_base, const Elem *__restrict__ bins,
              const uint32_t *__restrict__ tile_row, const uint32_t t0, const uint32_t n_chain,
              const uint32_t *__restrict__ uniq, uint64_t *tile_state, DevScalars *sc, const int carry_slot,
              uint64_t *__restrict__ c_pos, Elem *__restrict__ c_data, const uint32_t bm_wpl, const uint32_t long_thresh) {
    merge_chain_body<K, BM, false>(row_bin, bin_base, bins, tile_row, t0, n_chain, uniq, tile_state, sc, carry_slot, c_pos, c_data, bm_wpl,
                                   long_thresh, FusedSrc{});
}

template <class K, bool BM>
__global__ void __launch_bounds__(MC_THREADS, BM ? 2 : MC_OCC)
k_merge_chain_fused(const uint64_t *__restrict__ row_bin, const uint64_t bin_base, const Elem *__restrict__ bins,
                    const uint32_t *__restrict__ tile_row, const uint32_t t0, const uint32_t n_chain,
                    const uint32_t *__restrict__ uniq, uint64_t *tile_state, DevScalars *sc, const int carry_slot,
                    uint64_t *__restrict__ c_pos, Elem *__restrict__ c_data, const uint32_t bm_wpl, const uint32_t long_thresh,
                    const FusedSrc fs) {
    merge_chain_body<K, BM, true>(row_bin, bin_base, bins, tile_row, t0, n_chain, uniq, tile_state, sc, carry_slot, c_pos, c_data, bm_wpl,
                                  long_thresh, fs);
}

// =====================================================================================
// Fused multiply + merge for products whose every row is long over a small column range (config 5: sparse
// activations x sparse weights, 4096 columns, ~1.7e5 partial products per output row).  The per-output-row
// bin IS a dense accumulator in shared memory: nothing goes through HBM between the multiply and the merge.
//   * Persistent CTAs take output rows in ticket (= row) order.  acc[col] starts at -0.0f: x + (-0) = x for
//     every x, so the first product of a column is stored exactly and no "seen" test sits on the add path.
//   * The column range is cut into one band per warp.  A warp walks the row's runs (non-zeros of A(i,:) in
//     ascending k) IN ORDER and applies, of every run, only the elements of B(k,:) inside its band -- found
//     through a per-row band index of B built once per call -- so every column is summed in ascending k with
//     separately rounded products and adds, and no two warps ever touch the same column: no barrier, no
//     arbitration while a row accumulates.
//   * Runs are taken eight at a time: (k, a) of eight runs in one coalesced load, their band bounds in one, their
//     elements in one (eight independent loads per lane), then the eight are applied one after the other.
//   * The row's surviving columns are counted, the count goes through the same decoupled look-back as the merge
//     chain, and the row streams to its final place in C.
// =====================================================================================
constexpr int FD_THREADS = 512;
constexpr int FD_WARPS = FD_THREADS / 32;
constexpr int FD_RUNS = 8;
__host__ __device__ inline size_t fused_dense_smem(uint64_t cols) { return size_t((cols + 15) & ~15ull) * 5 + 64 * 4; }

// bandptr[k * (FD_WARPS + 1) + w] = index in b_data of the first element of row k with column >= w * band
__global__ void k_band_ptr(const uint64_t *__restrict__ b_pos, const Elem *__restrict__ b_data, uint64_t n_k, uint32_t band,
                           uint32_t *__restrict__ bandptr) {
    const uint64_t t = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
    if (t >= n_k * (FD_WARPS + 1)) return;
    const uint64_t k = t / (FD_WARPS + 1);
    const uint32_t w = uint32_t(t % (FD_WARPS + 1));
    uint64_t lo = b_pos[k], hi = b_pos[k + 1];
    const uint64_t target = uint64_t(w) * band;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (b_data[mid].idx < target) lo = mid + 1; else hi = mid;
    }
    bandptr[t] = uint32_t(lo);
}

__global__ void __launch_bounds__(FD_THREADS)
k_fused_dense(const uint64_t *__restrict__ a_pos, const Elem *__restrict__ a_data, const uint64_t m_a,
              const Elem *__restrict__ b_data, const uint32_t *__restrict__ bandptr, const uint32_t cols,
              const uint64_t rows, uint64_t *tile_state, DevScalars *sc, uint64_t *__restrict__ c_pos,
              Elem *__restrict__ c_data) {
    const uint32_t cpad = (cols + 15) & ~15u;
    float *acc = reinterpret_cast<float *>(osp_smem);
    unsigned char *seen = osp_smem + size_t(cpad) * 4;
    uint32_t *warp_sums = reinterpret_cast<uint32_t *>(osp_smem + size_t(cpad) * 5);
    uint32_t *s_ticket = warp_sums + 34;
    uint64_t *s_base = reinterpret_cast<uint64_t *>(warp_sums + 36);
    const unsigned int tid = threadIdx.x, lane = lane_id(), warp = tid >> 5;
    for (uint32_t c = tid; c < cpad; c += FD_THREADS) { acc[c] = -0.0f; seen[c] = 0; }
    const uint32_t per = (cols + FD_THREADS - 1) / FD_THREADS;       // columns per thread when the row is emitted
    const uint32_t cb = min(tid * per, cols), ce = min(cb + per, cols);
    while (true) {
        __syncthreads();
        if (tid == 0) *s_ticket = atomicAdd(&sc->tile_ticket, 1u);
        __syncthreads();
        const uint64_t row = *s_ticket;
        if (row >= rows) break;
        const uint64_t p0 = row < m_a ? a_pos[row] : 0, p1 = row < m_a ? a_pos[row + 1] : 0;
        // ---- accumulate: this warp's column band of every run, runs in ascending k ----
        for (uint64_t p = p0; p < p1; p += FD_RUNS) {
            const uint32_t n_runs = uint32_t(min(uint64_t(FD_RUNS), p1 - p));
            Elem ak; ak.idx = 0; ak.val = 0.f;
            if (lane < n_runs) ak = a_data[p + lane];
            uint32_t lo = 0, hi = 0;
            if (lane < n_runs) {
                lo = bandptr[uint64_t(ak.idx) * (FD_WARPS + 1) + warp];
                hi = bandptr[uint64_t(ak.idx) * (FD_WARPS + 1) + warp + 1];
            }
            Elem be[FD_RUNS];
            uint32_t lo_u[FD_RUNS], hi_u[FD_RUNS];
            float a_u[FD_RUNS];
#pragma unroll
            for (int u = 0; u < FD_RUNS; u++) {
                lo_u[u] = __shfl_sync(FULL, lo, u);
                hi_u[u] = __shfl_sync(FULL, hi, u);
                a_u[u] = __shfl_sync(FULL, ak.val, u);
                be[u].idx = 0xFFFFFFFFu; be[u].val = 0.f;
                if (lo_u[u] + lane < hi_u[u]) be[u] = b_data[lo_u[u] + lane];
            }
#pragma unroll
            for (int u = 0; u < FD_RUNS; u++) {
                if (be[u].idx != 0xFFFFFFFFu) {
                    acc[be[u].idx] = __fadd_rn(acc[be[u].idx], __fmul_rn(a_u[u], be[u].val));
                    seen[be[u].idx] = 1;
                }
                for (uint32_t q = lo_u[u] + 32 + lane; q < hi_u[u]; q += 32) {      // bands denser than one warp width
                    const Elem b = b_data[q];
                    acc[b.idx] = __fadd_rn(acc[b.idx], __fmul_rn(a_u[u], b.val));
                    seen[b.idx] = 1;
                }
                __syncwarp();                                  // the next run may hit the same columns from other lanes
            }
        }
        __syncthreads();
        // ---- count, chain, emit ----
        uint32_t cnt = 0;
        for (uint32_t c = cb; c < ce; c++) cnt += seen[c];
        uint32_t total;
        uint32_t o = block_exclusive_scan(cnt, warp_sums, total);
        if (warp == 0) {
            lb_publish(tile_state, uint32_t(row), total, 0);
            const uint64_t excl = lb_resolve(tile_state, uint32_t(row), total, 0);
            if (lane == 0) *s_base = excl;
        }
        __syncthreads();
        const uint64_t base = *s_base;
        if (tid == 0) {
            c_pos[row] = base;
            if (row + 1 == rows) { c_pos[rows] = base + total; sc->nnz_c[1] = base + total; }
        }
        for (uint32_t c = cb; c < ce; c++) {
            if (seen[c]) {
                Elem r; r.idx = c; r.val = acc[c];
                c_data[base + o++] = r;
                seen[c] = 0;
                acc[c] = -0.0f;
            }
        }
    }
}

// =====================================================================================
// Layer chaining (SURVEY 8f rank 3): relu(C + bias) kept sparse -- what a layer of the reference's MLP applies
// between two products (x = relu(fc(x)), NN_models/models.py:18-31) -- so that act_i -> fc_i -> act_{i+1} stays
// on the device in CSR.  One row at a time per CTA, rows in ticket order: the row is densified in shared memory
// (dense[c] = bias[c], then C(i,c) + bias[c] with one rounded add where C has an entry), the entries > 0 are
// counted, the count goes through the decoupled look-back and the row streams to its final place.
// =====================================================================================
constexpr int BR_THREADS = 256;
__global__ void __launch_bounds__(BR_THREADS)
k_bias_relu(const uint64_t *__restrict__ c_pos, const Elem *__restrict__ c_data, const uint64_t rows, const uint32_t cols,
            const float *__restrict__ bias, uint64_t *tile_state, DevScalars *sc, uint64_t *__restrict__ o_pos,
            Elem *__restrict__ o_data) {
    float *dense = reinterpret_cast<float *>(osp_smem);
    uint32_t *warp_sums = reinterpret_cast<uint32_t *>(osp_smem + size_t((cols + 15) & ~15u) * 4);
    uint32_t *s_ticket = warp_sums + 34;
    uint64_t *s_base = reinterpret_cast<uint64_t *>(warp_sums + 36);
    const unsigned int tid = threadIdx.x, lane = lane_id(), warp = tid >> 5;
    const uint32_t per = (cols + BR_THREADS - 1) / BR_THREADS;
    const uint32_t cb = min(tid * per, cols), ce = min(cb + per, cols);
    while (true) {
        __syncthreads();
        if (tid == 0) *s_ticket = atomicAdd(&sc->tile_ticket, 1u);
        __syncthreads();
        const uint64_t row = *s_ticket;
        if (row >= rows) break;
        for (uint32_t c = tid; c < cols; c += BR_THREADS) dense[c] = bias ? bias[c] : 0.f;
        __syncthreads();
        const uint64_t p0 = c_pos[row], p1 = c_pos[row + 1];
        for (uint64_t p = p0 + tid; p < p1; p += BR_THREADS) {
            const Elem e = c_data[p];
            if (e.idx < cols) dense[e.idx] = bias ? __fadd_rn(e.val, bias[e.idx]) : e.val;    // columns are distinct in a row
            else atomicMax(&sc->err, 4u);
        }
        __syncthreads();
        uint32_t cnt = 0;
        for (uint32_t c = cb; c < ce; c++) cnt += dense[c] > 0.f;
        uint32_t total;
        uint32_t o = block_exclusive_scan(cnt, warp_sums, total);
        if (warp == 0) {
            lb_publish(tile_state, uint32_t(row), total, 0);
            const uint64_t excl = lb_resolve(tile_state, uint32_t(row), total, 0);
            if (lane == 0) *s_base = excl;
        }
        __syncthreads();
        const uint64_t base = *s_base;
        if (tid == 0) {
            o_pos[row] = base;
            if (row + 1 == rows) { o_pos[rows] = base + total; sc->nnz_c[1] = base + total; }
        }
        for (uint32_t c = cb; c < ce; c++) {
            const float v = dense[c];
            if (v > 0.f) { Elem r; r.idx = c; r.val = v; o_data[base + o++] = r; }
        }
    }
}

// Duplicate check of the stable conversion: a bucket that shrank while folding held a duplicate.
__global__ void k_check_same(const uint64_t *a, const uint64_t *b, uint64_t n, DevScalars *sc) {
    uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
    if (i < n && a[i] != b[i]) atomicMax(&sc->err, 233u);
}

// =====================================================================================
// k-sharded multi-GPU path (DESIGN.md "Multi-GPU"): each rank multiplies its k-range and the
// partial products travel to the owner of their output row (contiguous row blocks), where the
// segments of the G sources are regrouped row by row in ascending source (= ascending k) order.
// =====================================================================================
// Bin start of every row of the shard's product and the per-row partial-product counts the owners need.
__global__ void k_shard_rows(const uint64_t *a_pos, uint64_t m_a, const uint64_t *run_off, uint64_t nnz_a, uint64_t rows,
                             uint64_t *row_bin, uint32_t *lens, DevScalars *sc) {
    uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
    if (i > rows) return;
    const uint64_t s = run_off[i <= m_a ? a_pos[i] : nnz_a];
    row_bin[i] = s;
    if (i < rows) {
        const uint64_t e = run_off[i + 1 <= m_a ? a_pos[i + 1] : nnz_a];
        if (e - s >= (1ull << 32)) atomicMax(&sc->err, 6u);      // OSP_ERR_UNSUPPORTED
        lens[i] = uint32_t(e - s);
    }
}
__global__ void k_pick_u64(const uint64_t *src, const uint64_t *index, uint32_t n, uint64_t *dst) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[index[i]];
}
// The record a rank contributes to the call's one all-gather: words 0 .. G = the offsets of the owners' first rows in
// this rank's local row-major order (row_bin at the rows `words_in` names), then the words the host put there
// (capacities, host status), and in the last word what the device found (first error of the symbolic pass / validation).
__global__ void k_dist_record(const uint64_t *row_bin, const uint64_t *words_in, uint32_t G, uint32_t W, const DevScalars *sc,
                              uint64_t *out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W) return;
    if (i <= G) out[i] = row_bin[words_in[i]];
    else if (i + 1 == W) {
        const bool unsorted = sc->v_desc - sc->v_eq != sc->v_bdesc - sc->v_beq;
        out[i] = sc->v_bad_pos || unsorted ? 1u : sc->v_eq != sc->v_beq ? 233u : sc->err;      // OSP_ERR_INVALID / _DUPLICATE / device code
    } else out[i] = words_in[i];
}
// lens[s * RL + i] read in (i, s) order
struct TransposedIn {
    const uint32_t *lens;
    uint64_t RL;
    uint64_t G;
    __device__ uint64_t load(uint64_t j, bool valid) const { return valid ? lens[(j % G) * RL + j / G] : 0; }
    __device__ uint64_t value(uint64_t v, uint64_t, bool) const { return v; }
};
struct RowBinStrided {         // row i of the owner starts at dst_off[i * G]
    const uint64_t *off;
    uint64_t G;
    __device__ __forceinline__ uint64_t operator()(uint64_t i) const { return off[i * G]; }
    __device__ __forceinline__ bool nonempty(uint64_t i) const { return off[(i + 1) * G] > off[i * G]; }
    __device__ __forceinline__ uint64_t task_begin(uint64_t i) const { return i * G; }        // segment (row i, source 0)
};
// One warp per owned row: the row's G segments (one per source, received source-major) become one contiguous
// row in the row-major bins, sources in ascending order.  The lanes stride over the ROW's elements -- every
// lane copies whatever the segment lengths are (at G = 8 a segment is a single run of ~8 partial products) --
// and find the segment of an element by comparing its position with the scanned segment lengths.
__global__ void k_regroup(const Elem *__restrict__ recv, const uint64_t *__restrict__ src_off, const uint64_t *__restrict__ dst_off,
                          const uint32_t *__restrict__ lens, uint64_t RL, uint32_t G, Elem *__restrict__ bins, uint64_t row_lo,
                          uint64_t row_hi) {
    const unsigned int lane = lane_id();
    uint64_t warp = (blockIdx.x * uint64_t(blockDim.x) + threadIdx.x) >> 5;
    uint64_t nwarps = (uint64_t(gridDim.x) * blockDim.x) >> 5;
    for (uint64_t i = row_lo + warp; i < row_hi; i += nwarps) {
        uint32_t l = 0;
        uint64_t so = 0;
        if (lane < G) { l = lens[uint64_t(lane) * RL + i]; so = src_off[uint64_t(lane) * RL + i]; }
        const uint32_t cum = warp_inclusive_scan(l);
        const uint32_t total = __shfl_sync(FULL, cum, 31);
        const uint64_t rel = so - (cum - l);                  // source index of element p of segment s: rel_s + p
        Elem *dst = bins + dst_off[i * G];
        for (uint32_t p0 = 0; p0 < total; p0 += 32) {
            const uint32_t p = p0 + lane;
            uint32_t s = 0;
            for (uint32_t k = 0; k + 1 < G; k++) s += __shfl_sync(FULL, cum, k) <= p;
            const uint64_t src = __shfl_sync(FULL, rel, s) + p;
            if (p < total) dst[p] = recv[src];
        }
    }
}

// ---- peer-memory exchange: the multiply writes straight into the owners' memory over NVLink ------------
// Every owner holds a landing buffer made of G regions, one per source, each row-major over the owner's rows.
// A source's partial products for one owner are therefore ONE contiguous stream, at the offsets its own
// symbolic pass computed: destination = owner's region for this source + (run offset - offset of the owner's
// first row in the source's local row-major order).  The owner of a run follows from its offset alone (rows
// are owned in contiguous blocks), so the kernel needs no per-row table.
constexpr int MAX_PEERS = 16;
struct PeerDst {
    Elem *base[MAX_PEERS];           // owner's landing buffer (mapped through CUDA IPC; the own one directly)
    uint64_t bound[MAX_PEERS + 1];   // local run offset at which owner r's rows begin (bound[G] = P_local)
    int64_t delta[MAX_PEERS];        // region start inside owner r's buffer - bound[r]
    int world;
};
// The warp-flat multiply of k_multiply with every run going to the GPU that owns its output row: 8-byte stores
// over NVLink that are contiguous from run to run.  The exchange of the k-sharded path IS this kernel's store
// stream: nothing is staged or sent.
struct PeerRows { uint64_t lo[MAX_PEERS], hi[MAX_PEERS]; };      // rows of A whose runs this launch sends, per owner
__global__ void __launch_bounds__(256)
k_multiply_peer(const Elem *__restrict__ a_data, const uint64_t *__restrict__ run_off, const uint32_t *__restrict__ task_bs,
                const Elem *__restrict__ b_data, const PeerDst dst, const uint64_t *__restrict__ a_pos, const uint64_t m_a,
                const PeerRows rows, const int first_owner) {
    __shared__ Elem *s_base[MAX_PEERS];
    __shared__ uint64_t s_tb[MAX_PEERS], s_cum[MAX_PEERS + 1];
    if (threadIdx.x < MAX_PEERS) s_base[threadIdx.x] = dst.base[threadIdx.x];
    if (threadIdx.x == 0) {
        // the launch's tasks: for every owner the non-zeros of A of its rows [lo, hi), owners taken from `first_owner` on and
        // round: at any moment the G sources are writing to G different owners instead of all to the same one
        uint64_t cum = 0;
        for (int j = 0; j < dst.world; j++) {
            const int r = (first_owner + j) % dst.world;
            const uint64_t tb = a_pos[min(rows.lo[r], m_a)], te = a_pos[min(rows.hi[r], m_a)];
            s_tb[j] = tb; s_cum[j] = cum;
            cum += te - tb;
        }
        s_cum[dst.world] = cum;
    }
    __syncthreads();
    const unsigned int lane = lane_id();
    const uint64_t warp = (blockIdx.x * uint64_t(blockDim.x) + threadIdx.x) >> 5;
    const uint64_t nwarps = (uint64_t(gridDim.x) * blockDim.x) >> 5;
    const uint64_t t1 = s_cum[dst.world];
    for (uint64_t base = warp * 32; base < t1; base += nwarps * 32) {
        uint32_t bs = 0, len = 0, owner = 0; float a = 0.f; uint64_t off = 0;
        if (base + lane < t1) {
            const uint64_t f = base + lane;
            int j = 0;
            while (j + 1 < dst.world && f >= s_cum[j + 1]) j++;
            const uint64_t i = s_tb[j] + (f - s_cum[j]);
            owner = uint32_t((first_owner + j) % dst.world);
            a = a_data[i].val;
            const uint64_t o = run_off[i];
            len = uint32_t(run_off[i + 1] - o);
            bs = task_bs[i];
            off = o + uint64_t(dst.delta[owner]);
        }
        const uint32_t incl = warp_inclusive_scan(len);
        const uint32_t total = __shfl_sync(FULL, incl, 31);
        const uint32_t excl = incl - len;
        const uint32_t dbs = bs - excl;                       // B index of element e of this task: dbs + e
        const uint64_t doff = off - excl;                     // landing index of element e of this task: doff + e (mod 2^64)
        // The walk starts `shift` elements early so that every 32-lane store covers two whole 128-byte lines of the
        // owner's landing buffer (the destination of the warp's runs is one contiguous stream per owner): NVLink
        // moves full lines instead of a line and two fragments per store.
        const uint32_t shift = uint32_t(__shfl_sync(FULL, doff, 0)) & 15u;
        for (uint32_t e0 = 0; e0 < total + shift; e0 += 64) {  // two independent 32-element chunks per turn
            const uint32_t e[2] = {e0 + lane - shift, e0 + 32 + lane - shift};     // (wraps below 0 for the first lanes: >= total)
            uint32_t t[2] = {0, 0};                            // number of tasks that end at or before e
#pragma unroll
            for (int step = 16; step > 0; step >>= 1) {
#pragma unroll
                for (int u = 0; u < 2; u++) {
                    const uint32_t v = __shfl_sync(FULL, incl, t[u] + step - 1);
                    if (v <= e[u]) t[u] += step;
                }
            }
            float a_t[2]; uint32_t dbs_t[2], own_t[2]; uint64_t doff_t[2]; Elem b[2];
#pragma unroll
            for (int u = 0; u < 2; u++) {
                a_t[u] = __shfl_sync(FULL, a, t[u] & 31);
                dbs_t[u] = __shfl_sync(FULL, dbs, t[u] & 31);
                doff_t[u] = __shfl_sync(FULL, doff, t[u] & 31);
                own_t[u] = __shfl_sync(FULL, owner, t[u] & 31);
            }
#pragma unroll
            for (int u = 0; u < 2; u++)
                if (e[u] < total) b[u] = ld_gather(b_data + uint32_t(dbs_t[u] + e[u]));    // (32-bit wrap-around: dbs = bs - excl may be "negative")
#pragma unroll
            for (int u = 0; u < 2; u++) {
                if (e[u] < total) {
                    Elem o; o.idx = b[u].idx; o.val = __fmul_rn(a_t[u], b[u].val);     // rounded on its own: no FMA
                    s_base[own_t[u]][doff_t[u] + e[u]] = o;
                }
            }
        }
    }
}

}  // namespace osp

// osp_fusedlanes.cuh -- fused multiply + merge of long rows over a small column range, bank-aligned (config 5).
//
// Same job as k_fused_dense (osp_kernels.cuh): C(i,:) = sum_k A(i,k) * B(k,:) accumulated in a dense shared-memory
// row, every column summed in ascending k with separately rounded products and adds (the multiplyPhase / mergePhase
// pair of simulator/SimOuterSPACE.cpp:77-132 without ever materialising a partial product), rows of C written once.
// k_fused_dense is bound by shared-memory wavefronts (ncu, profiles/r02_ncu/
// mlp8_fused_raw.csv: L1 data pipe 85 % busy, 44 % of the shared wavefronts are bank conflicts): a warp applies ~25
// elements of a row of B at random columns of its band, so every read-modify-write of the accumulator replays ~3
// times, a `seen` byte is stored beside it, and the three shuffles + bounds per (run, band) are paid for 25 products.
//
// Here the accumulator access is conflict-free BY CONSTRUCTION:
//   * B is regrouped once per call (k_fl_count / k_fl_fill, one warp per row of B): the elements of row k are dealt
//     into groups of at most 32 in which every element sits in the lane equal to its shared-memory bank,
//     lane = col % 32.  Element j of bank b goes to group j, so row k needs max_b(multiplicity of b) groups; a slot
//     holds the value (4 bytes) and col / 32 (1 byte; cpad / 32 = empty: it points at 32 dummy floats behind the
//     row), four groups (a quad) per 32-bit word of column bytes and per 16-byte vector of values.
//     For config 5 (410 elements per row of B, 4096 columns) that is 21 groups per row, 61 % of the slots filled,
//     5 bytes per slot: the bytes read per partial product stay what the 8-byte elements cost.
//   * ONE WARP owns an output row: acc[col] lives in its 4 * cols bytes of shared memory, lane l only ever touches
//     columns = l (mod 32), i.e. bank l: no conflicts, no arbitration, and -- every column having ONE owner lane --
//     no barrier of any kind while a row accumulates; program order per lane is k order per column.
//   * A never-touched accumulator holds the bit pattern 0xFFFFFFFF, the first product of a column is stored as it is:
//     no `seen` array; the row is counted and read back by its warp (128 conflict-free words per lane for 4096 columns).
//     That pattern is a NaN, so no stored value may ever carry it: every NaN of A and B is made the canonical 0x7FFFFFFF
//     where it is loaded (fl_canonical: once per element of B per call, once per element of A per row).  IEEE arithmetic
//     then only returns an input NaN or the machine's default NaN (0x7FFFFFFF on the GPU; 0xFFC00000 on x86, where the
//     CPU emulation may run), never 0xFFFFFFFF, whatever the hardware does with NaN payloads.
//   * The loads of a run (its column-byte words and values, up to 6 quads = 24 groups) are issued while the previous
//     run is applied: two register sets, ~3.4 KB in flight per warp.
//   * Rows of C go to the prefix sum of the plan's bounds min(partial products, cols) -- no chain between the rows -- and
//     are moved into an exactly sized C only when some row is not full (below: "rows of C without a chain").
// Measured, version by version: profiles/r02_fusedlanes.md (config 5: 26.8 -> 11.2 ms per call).
// Limits: cols <= FL_MAX_COLS (one byte of col / 32 per slot); a B whose regrouped form exceeds FL_MAX_BLOWUP slots
// per element (many columns of a row in one bank) keeps the band kernel.  Selection: osp_engine.cu.
#pragma once
#include "osp_kernels.cuh"

namespace osp {

constexpr uint32_t FL_MAX_COLS = 255u * 32u;       // col / 32 and the empty marker cpad / 32 fit a byte
constexpr uint32_t FL_EMPTY = 0xFFFFFFFFu;          // accumulator not touched yet
constexpr uint32_t FL_MAX_BLOWUP = 6;               // slots per element of B beyond which the band kernel is kept
constexpr int FL_PREP_WARPS = 8;
__device__ __forceinline__ float fl_canonical(float v) { return v != v ? __uint_as_float(0x7FFFFFFFu) : v; }
#ifndef OSP_FL_QUADS
#define OSP_FL_QUADS 6                              // (8: 11.2 ms on config 5, 6: 10.8 ms -- fewer registers, less code; GPU call 23)
#endif
constexpr int FL_QUADS = OSP_FL_QUADS;              // quads (of four groups) of one run held in registers at a time

struct FlMeta {                                     // per row k of B
    uint32_t quad0;                                 // first quad of the row in vals / colb
    uint32_t groups;                                // groups of the row (its quads: (groups + 3) / 4)
};

// per warp: the accumulator row + 32 dummy floats (where the empty slots of a group land)
__host__ __device__ inline size_t fused_lanes_smem(uint64_t cols, int warps) { return (size_t((cols + 31) & ~31ull) + 32) * 4 * size_t(warps); }
__host__ __device__ inline unsigned char fused_lanes_empty_byte(uint64_t cols) { return static_cast<unsigned char>(((cols + 31) & ~31ull) >> 5); }

// Pass 1 over B: groups per row = the largest number of columns of the row that share a bank; quads are handed out
// by an atomic counter (where a row's quads lie is irrelevant to the result).
__global__ void __launch_bounds__(32 * FL_PREP_WARPS)
k_fl_count(const uint64_t *__restrict__ b_pos, const Elem *__restrict__ b_data, uint64_t n_k, FlMeta *__restrict__ meta, DevScalars *sc) {
    __shared__ uint32_t hist[FL_PREP_WARPS][32];
    const unsigned int lane = lane_id(), warp = threadIdx.x >> 5;
    for (uint64_t k = uint64_t(blockIdx.x) * FL_PREP_WARPS + warp; k < n_k; k += uint64_t(gridDim.x) * FL_PREP_WARPS) {
        hist[warp][lane] = 0;
        __syncwarp();
        const uint64_t p0 = b_pos[k], p1 = b_pos[k + 1];
        for (uint64_t p = p0 + lane; p < p1; p += 32) atomicAdd(&hist[warp][b_data[p].idx & 31u], 1u);
        __syncwarp();
        uint32_t m = hist[warp][lane];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(FULL, m, o));
        if (lane == 0) {
            const unsigned long long quads = (m + 3) >> 2;
            FlMeta mt;
            mt.quad0 = quads ? uint32_t(atomicAdd(&sc->fl_quads, quads)) : 0u;      // (the host rejects totals beyond 32 bits)
            mt.groups = m;
            meta[k] = mt;
        }
        __syncwarp();
    }
}

// Pass 2 over B: every element into its slot.  colb was preset to the byte that marks an empty slot
// (cpad / 32: the dummy floats behind an accumulator row).  Values lie lane-interleaved, the four groups of a quad side by
// side -- vals[(quad * 32 + lane) * 4 + group] -- so that a lane fetches its four values of a quad with one 16-byte load.
__global__ void __launch_bounds__(32 * FL_PREP_WARPS)
k_fl_fill(const uint64_t *__restrict__ b_pos, const Elem *__restrict__ b_data, uint64_t n_k, const FlMeta *__restrict__ meta,
          float *__restrict__ vals, uint32_t *__restrict__ colb) {
    __shared__ uint32_t hist[FL_PREP_WARPS][32];
    const unsigned int lane = lane_id(), warp = threadIdx.x >> 5;
    unsigned char *colbytes = reinterpret_cast<unsigned char *>(colb);
    for (uint64_t k = uint64_t(blockIdx.x) * FL_PREP_WARPS + warp; k < n_k; k += uint64_t(gridDim.x) * FL_PREP_WARPS) {
        hist[warp][lane] = 0;
        __syncwarp();
        const uint64_t p0 = b_pos[k], p1 = b_pos[k + 1];
        const uint64_t q0 = meta[k].quad0;
        for (uint64_t p = p0 + lane; p < p1; p += 32) {
            const Elem e = b_data[p];
            const uint32_t b = e.idx & 31u;
            const uint32_t j = atomicAdd(&hist[warp][b], 1u);      // any order inside a bank: the columns of a row are distinct
            const uint64_t slot = ((q0 + (j >> 2)) * 32 + b) * 4 + (j & 3u);
            vals[slot] = fl_canonical(e.val);
            colbytes[slot] = static_cast<unsigned char>(e.idx >> 5);
        }
        __syncwarp();
    }
}

// ---- rows of C without a chain --------------------------------------------------------------------------------------
// The plan's bound of a row, min(partial products, cols), is EXACT for a row that fills the column range -- which the rows of
// this path do more often than not (config 5: every row of C is dense).  So the rows are written at the prefix sum of
// their bounds, which is known before the multiply: no look-back, no row ever waits for the rows before it (with the
// look-back, 9 % of the warp samples were asleep waiting for the slowest of the ~1900 rows in flight, ncu r02_call19).
// If the counts then add up to the bound, C.pos = that prefix and C is final; otherwise the rows are moved left into an
// exactly sized C (k_fl_compact) behind a scan of the counts.
struct RowCapIn {          // k_scan input: bound of row i
    const uint64_t *row_bin;
    uint64_t cols;
    __device__ uint64_t load(uint64_t i, bool valid) const { return valid ? row_bin[i + 1] - row_bin[i] : 0; }
    __device__ uint64_t value(uint64_t v, uint64_t, bool) const { return v < cols ? v : cols; }
};

__global__ void __launch_bounds__(256)
k_fl_compact(const uint64_t *__restrict__ pos_bound, const uint64_t *__restrict__ pos_exact, const Elem *__restrict__ src,
             Elem *__restrict__ dst, uint64_t rows) {
    const unsigned int lane = lane_id();
    for (uint64_t row = (uint64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; row < rows; row += (uint64_t(gridDim.x) * blockDim.x) >> 5) {
        const uint64_t s0 = pos_bound[row], d0 = pos_exact[row];
        const uint32_t n = uint32_t(pos_exact[row + 1] - d0);
        for (uint32_t i = lane; i < n; i += 32) dst[d0 + i] = src[s0 + i];
    }
}

// The registers of (up to FL_QUADS quads of) one run: column-byte words, values, multiplier.
struct FlRun {
    uint32_t w[FL_QUADS];
    float4 v[FL_QUADS];
    float a;
    uint32_t groups;        // groups of this piece (<= 4 * FL_QUADS)
};

// Loads of a piece: two loads per quad and lane (4 + 16 bytes), predicated quad by quad -- no branch: with three warps per
// scheduler every unresolved branch is exposed.  Quads past `groups` stay unset (fl_apply never reads them); the unused
// groups of the last quad are loaded with it (the storage is allocated in whole quads, their column bytes say "empty").
__device__ __forceinline__ void fl_load(FlRun &r, const float4 *__restrict__ vals4, const uint32_t *__restrict__ colb, uint64_t quad0,
                                        uint32_t groups, float a, unsigned int lane) {
    r.a = a;
    r.groups = groups;
    const uint32_t *cw = colb + quad0 * 32 + lane;
    const float4 *vw = vals4 + quad0 * 32 + lane;
#pragma unroll
    for (int q = 0; q < FL_QUADS; q++) {
        if (uint32_t(4 * q) < groups) {
            r.w[q] = cw[q * 32];
            r.v[q] = vw[q * 32];
        }
    }
}

// Shared-memory accesses of the accumulator by 32-bit shared-window address: one base computed per kernel, no generic
// address arithmetic under predicates.
#ifdef OSP_CUSIM
__device__ __forceinline__ uint32_t fl_smem_base() { return 0; }
__device__ __forceinline__ uint32_t fl_lds(uint32_t addr) { return smem_u32_at(addr); }
__device__ __forceinline__ void fl_sts(uint32_t addr, uint32_t v) { smem_u32_at(addr) = v; }
__device__ __forceinline__ uint32_t fl_byte(uint32_t w, int g) { return (w >> (8 * g)) & 0xFFu; }
#else
__device__ __forceinline__ uint32_t fl_smem_base() { return uint32_t(__cvta_generic_to_shared(osp_smem)); }
__device__ __forceinline__ uint32_t fl_lds(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void fl_sts(uint32_t addr, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t fl_byte(uint32_t w, int g) { return __byte_perm(w, 0u, 0x4440u + uint32_t(g)); }
#endif

// Applies a loaded run to the warp's accumulator row; acc_lane = shared-window address of the lane's column `lane`
// (column c of the row sits 4 * c bytes into the row: (c / 32) << 7 past acc_lane for the lane c % 32).  An empty slot
// carries the column byte cpad / 32: it lands in the 32 dummy floats behind the row (one per lane, never emitted), so
// the read-modify-write needs no validity test at all.  Groups are applied FL_BLOCK at a time (all loads of the block,
// then the adds, then the stores: the real columns of a lane within one run are distinct); only the last, partly filled
// block of a run tests (uniformly) which of its groups exist.
#ifndef OSP_FL_BLOCK
#define OSP_FL_BLOCK 8
#endif
constexpr int FL_BLOCK = OSP_FL_BLOCK;
static_assert(FL_BLOCK % 4 == 0 && FL_BLOCK >= 4 && FL_BLOCK <= 16 && (4 * FL_QUADS) % FL_BLOCK == 0, "whole quads, whole blocks");
__device__ __forceinline__ float fl_f4(const float4 &v, const int g) { return g == 0 ? v.x : g == 1 ? v.y : g == 2 ? v.z : v.w; }
template <bool TAIL>
__device__ __forceinline__ void fl_block(const FlRun &r, const int b0, const uint32_t acc_lane) {
    uint32_t addr[FL_BLOCK], old[FL_BLOCK];
#pragma unroll
    for (int u = 0; u < FL_BLOCK; u++) {
        const int g = b0 + u;
        addr[u] = acc_lane + fl_byte(r.w[g >> 2], g & 3) * 128u;                // PRMT + IMAD
        old[u] = FL_EMPTY;
        if (!TAIL || uint32_t(g & ~3) < r.groups) old[u] = fl_lds(addr[u]);     // (whole quads: the missing groups of a quad are empty slots)
    }
#pragma unroll
    for (int u = 0; u < FL_BLOCK; u++) {
        const int g = b0 + u;
        const float prod = __fmul_rn(r.a, fl_f4(r.v[g >> 2], g & 3));           // rounded on its own: no FMA
        const float nv = old[u] == FL_EMPTY ? prod : __fadd_rn(__uint_as_float(old[u]), prod);
        if (!TAIL || uint32_t(g & ~3) < r.groups) fl_sts(addr[u], __float_as_uint(nv));
    }
}
__device__ __forceinline__ void fl_apply(const FlRun &r, const uint32_t acc_lane) {
#pragma unroll
    for (int b = 0; b < 4 * FL_QUADS; b += FL_BLOCK) {
        if (uint32_t(b + FL_BLOCK) <= r.groups) fl_block<false>(r, b, acc_lane);       // warp-uniform branches
        else if (uint32_t(b) < r.groups) fl_block<true>(r, b, acc_lane);
    }
}

template <int WARPS>
__global__ void __launch_bounds__(32 * WARPS)
k_fused_lanes(const uint64_t *__restrict__ a_pos, const Elem *__restrict__ a_data, const uint64_t m_a,
              const FlMeta *__restrict__ meta, const float4 *__restrict__ vals, const uint32_t *__restrict__ colb,
              const uint32_t cols, const uint64_t rows, uint64_t *tile_state, DevScalars *sc,
              uint64_t *__restrict__ c_pos, Elem *__restrict__ c_data, uint32_t *__restrict__ row_cnt) {
    const unsigned int lane = lane_id(), warp = threadIdx.x >> 5;
    const uint32_t cpad = (cols + 31) & ~31u;
    const uint32_t acc_off = warp * (cpad + 32) * 4;
    const uint32_t acc_lane = fl_smem_base() + acc_off + lane * 4;
    for (uint32_t c = 0; c < cpad; c += 32) fl_sts(acc_lane + c * 4, FL_EMPTY);
    __syncwarp();
    while (true) {
        uint32_t t = 0;
        if (lane == 0) t = atomicAdd(&sc->tile_ticket, 1u);
        const uint64_t row = __shfl_sync(FULL, t, 0);
        if (row >= rows) break;
        const uint64_t p0 = row < m_a ? a_pos[row] : 0, p1 = row < m_a ? a_pos[row + 1] : 0;
        // ---- accumulate: the runs of the row in ascending k, 32 at a time; a run longer than 4 * FL_QUADS groups in pieces ----
        for (uint64_t p = p0; p < p1; p += 32) {
            const uint32_t n_runs = uint32_t(min(uint64_t(32), p1 - p));
            Elem ak; ak.idx = 0; ak.val = 0.f;
            FlMeta mt; mt.quad0 = 0; mt.groups = 0;
            if (lane < n_runs) { ak = a_data[p + lane]; ak.val = fl_canonical(ak.val); mt = meta[ak.idx]; }
            // cursor over the pieces of the batch: (run r, first group g0 of the piece); r == n_runs: done
            uint32_t r = 0, g0 = 0, ng = __shfl_sync(FULL, mt.groups, 0);
            auto skip_empty = [&]() {                          // runs without elements (empty rows of B) have no piece
                while (r < n_runs && g0 >= ng) {
                    r++; g0 = 0;
                    ng = __shfl_sync(FULL, mt.groups, r & 31);
                }
            };
            auto load_piece = [&](FlRun &dst) {
                const uint64_t q0 = __shfl_sync(FULL, mt.quad0, r);
                const float a = __shfl_sync(FULL, ak.val, r);
                fl_load(dst, vals, colb, q0 + (g0 >> 2), min(ng - g0, uint32_t(4 * FL_QUADS)), a, lane);
                g0 += 4 * FL_QUADS;
            };
            skip_empty();
            FlRun ra, rb;
            bool have_a = r < n_runs, have_b = false;
            if (have_a) load_piece(ra);
            while (have_a) {
                skip_empty();
                have_b = r < n_runs;
                if (have_b) load_piece(rb);
                fl_apply(ra, acc_lane);
                if (!have_b) break;
                skip_empty();
                have_a = r < n_runs;
                if (have_a) load_piece(ra);
                fl_apply(rb, acc_lane);
            }
        }
        if (row_cnt) {
            // ---- no chain: the row goes to the prefix of the bounds (c_pos holds it), its count is recorded ----
            const uint64_t base = c_pos[row];
            uint32_t total = 0;
            for (uint32_t c0 = 0; c0 < cpad; c0 += 128) {
                uint32_t bits[4];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const uint32_t c = c0 + 32 * u;
                    bits[u] = FL_EMPTY;
                    if (c < cpad) { bits[u] = fl_lds(acc_lane + c * 4); fl_sts(acc_lane + c * 4, FL_EMPTY); }
                }
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const bool hit = bits[u] != FL_EMPTY;
                    const unsigned int m = __ballot_sync(FULL, hit);
                    if (hit) {
                        Elem e; e.idx = c0 + 32 * u + lane; e.val = __uint_as_float(bits[u]);
                        c_data[base + total + __popc(m & ((1u << lane) - 1u))] = e;
                    }
                    total += __popc(m);
                }
            }
            if (lane == 0) {
                row_cnt[row] = total;
                atomicAdd(&sc->nnz_c[1], static_cast<unsigned long long>(total));
            }
            __syncwarp();
        } else {
            // ---- count, chain, emit (ascending columns: word i of every lane, lanes in order) ----
            uint32_t total = 0;
            for (uint32_t c0 = 0; c0 < cpad; c0 += 128) {
                uint32_t bits[4];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    bits[u] = FL_EMPTY;
                    if (c0 + 32 * u < cpad) bits[u] = fl_lds(acc_lane + (c0 + 32 * u) * 4);
                }
#pragma unroll
                for (int u = 0; u < 4; u++) total += __popc(__ballot_sync(FULL, bits[u] != FL_EMPTY));
            }
            lb_publish(tile_state, uint32_t(row), total, 0);
            const uint64_t base = lb_resolve(tile_state, uint32_t(row), total, 0);
            if (lane == 0) {
                c_pos[row] = base;
                if (row + 1 == rows) { c_pos[rows] = base + total; sc->nnz_c[1] = base + total; }
            }
            uint64_t o = base;
            for (uint32_t c0 = 0; c0 < cpad; c0 += 128) {
                uint32_t bits[4];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const uint32_t c = c0 + 32 * u;
                    bits[u] = FL_EMPTY;
                    if (c < cpad) { bits[u] = fl_lds(acc_lane + c * 4); fl_sts(acc_lane + c * 4, FL_EMPTY); }
                }
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const bool hit = bits[u] != FL_EMPTY;
                    const unsigned int m = __ballot_sync(FULL, hit);
                    if (hit) {
                        Elem e; e.idx = c0 + 32 * u + lane; e.val = __uint_as_float(bits[u]);
                        c_data[o + __popc(m & ((1u << lane) - 1u))] = e;
                    }
                    o += __popc(m);
                }
            }
            __syncwarp();
        }
    }
}

}  // namespace osp

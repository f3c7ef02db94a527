// osp_mtx.cuh -- Matrix Market text parsed in HBM (osp_readcoo_device): the body of a .mtx file becomes the triplet
// arrays of osp_readcoo, bit for bit and in file order.
//
//   k_mtx_count_lines   '\n' per tile of MTX_TILE bytes (16-byte loads, byte-compare masks)
//   k_scan              (osp_kernels.cuh) exclusive scan of the tile counts: where each tile's newlines go
//   k_mtx_line_ends     the byte offset of every '\n' in file order; line i ends at nl[i] (the last one at the text's end)
//   k_mtx_parse         one line per thread, through the grammar the host loader uses (osp_mtx_grammar.h): 0 entries
//                       (blank or '%' line), 1 or 2 (the mirror of an off-diagonal entry when symmetric), or MTX_SLOW
//   k_mtx_slow_list     the slow lines, for the host to read with the C library (only when there are any)
//   k_mtx_slow_counts   their entry counts, back from the host
//   k_scan              exclusive scan of the per-line counts (in place): where each line's entries go
//   k_mtx_scatter       the entries of the plain lines, SoA (rows, cols, vals), and the largest row and col id
//   k_mtx_scatter_slow  the entries of the slow lines, read on the host
#pragma once
#include "osp_device.cuh"
#include "osp_mtx_grammar.h"

namespace osp {

constexpr int MTX_THREADS = 256;
constexpr int MTX_WORDS = 4;                                   // 16-byte words per thread and tile
constexpr uint64_t MTX_TILE = uint64_t(MTX_THREADS) * MTX_WORDS * 16;   // 16 KB of text per tile
constexpr uint32_t MTX_SLOW = 0xFFFFFFFFu;                     // k_mtx_parse: the line is not of the plain shape

// What the ingest kernels report (in the counters of the per-call zeroed arena).
struct MtxScalars {
    unsigned long long entries;        // entries of the plain lines
    unsigned long long n_slow;         // slow lines
    unsigned long long listed;         // k_mtx_slow_list
    unsigned int max_row, max_col;     // largest stored ids (k_mtx_scatter)
};
static_assert(sizeof(MtxScalars) % 4 == 0, "MtxScalars lives in uint32 counters");

struct MtxSlowLine { uint64_t line, begin, end; };

// Number of '\n' bytes in a 32-bit word (exact: no carry crosses a byte).
__device__ __forceinline__ uint32_t newlines_in(uint32_t w) {
    const uint32_t x = w ^ 0x0A0A0A0Au;
    const uint32_t y = ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x | 0x7F7F7F7Fu);
    return uint32_t(__popc(y));
}
__device__ __forceinline__ uint32_t newlines_in(const uint4 &w) {
    return newlines_in(w.x) + newlines_in(w.y) + newlines_in(w.z) + newlines_in(w.w);
}

// The text buffer holds n_words 16-byte words; the bytes past the text are zero.
__global__ void __launch_bounds__(MTX_THREADS)
k_mtx_count_lines(const uint4 *__restrict__ text, uint64_t n_words, uint32_t *__restrict__ tile_cnt) {
    __shared__ uint32_t s_sum;
    if (threadIdx.x == 0) s_sum = 0;
    __syncthreads();
    const uint64_t w0 = uint64_t(blockIdx.x) * (MTX_THREADS * MTX_WORDS);
    uint32_t c = 0;
#pragma unroll
    for (int it = 0; it < MTX_WORDS; it++) {
        const uint64_t w = w0 + uint64_t(it) * MTX_THREADS + threadIdx.x;
        if (w < n_words) c += newlines_in(text[w]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(FULL, c, o);
    if (lane_id() == 0) atomicAdd(&s_sum, c);
    __syncthreads();
    if (threadIdx.x == 0) tile_cnt[blockIdx.x] = s_sum;
}

// tile_off[t] = newlines before tile t (k_scan of the tile counts).
__global__ void __launch_bounds__(MTX_THREADS)
k_mtx_line_ends(const uint4 *__restrict__ text, uint64_t n_words, const uint64_t *__restrict__ tile_off, uint64_t *__restrict__ nl) {
    __shared__ uint32_t s_warp[33];
    const uint64_t w0 = uint64_t(blockIdx.x) * (MTX_THREADS * MTX_WORDS);
    uint64_t base = tile_off[blockIdx.x];
    for (int it = 0; it < MTX_WORDS; it++) {                   // 256 consecutive words per round: thread order = byte order
        const uint64_t w = w0 + uint64_t(it) * MTX_THREADS + threadIdx.x;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (w < n_words) v = text[w];
        uint32_t total = 0;
        const uint32_t excl = block_exclusive_scan(newlines_in(v), s_warp, total);
        if (total) {
            uint64_t o = base + excl;
            const uint32_t part[4] = {v.x, v.y, v.z, v.w};
            for (int k = 0; k < 4; k++)
                for (int b = 0; b < 4; b++)
                    if (((part[k] >> (8 * b)) & 0xFF) == '\n') nl[o++] = w * 16 + uint64_t(k * 4 + b);
        }
        base += total;
        __syncthreads();                                       // s_warp is reused by the next round
    }
}

// Bytes [begin, end) of line i of a text of len bytes with n_nl newlines at nl[].
__device__ __forceinline__ void mtx_line_span(const uint64_t *nl, uint64_t n_nl, uint64_t len, uint64_t i, uint64_t &begin, uint64_t &end) {
    begin = i ? nl[i - 1] + 1 : 0;
    end = i < n_nl ? nl[i] : len;
}

__global__ void __launch_bounds__(MTX_THREADS)
k_mtx_parse(const char *__restrict__ text, uint64_t len, const uint64_t *__restrict__ nl, uint64_t n_nl, int symmetric,
            uint32_t *__restrict__ cnt, MtxScalars *ms) {
    const uint64_t n_lines = n_nl + 1;
    for (uint64_t i0 = uint64_t(blockIdx.x) * MTX_THREADS; i0 < n_lines; i0 += uint64_t(gridDim.x) * MTX_THREADS) {
        const uint64_t i = i0 + threadIdx.x;
        unsigned long long entries = 0, slow = 0;
        if (i < n_lines) {
            uint64_t b, e;
            mtx_line_span(nl, n_nl, len, i, b, e);
            const char *q = text + b;
            uint64_t r = 0, c = 0;
            double v;
            const int kind = osp_mtx::plain_line(q, text + e, r, c, v);
            uint32_t n = 0;
            if (kind == osp_mtx::LINE_ENTRY) n = (symmetric && r != c) ? 2 : 1;   // ids compared before they are narrowed
            else if (kind == osp_mtx::LINE_SLOW) { n = MTX_SLOW; slow = 1; }
            cnt[i] = n;
            if (n != MTX_SLOW) entries = n;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            entries += __shfl_xor_sync(FULL, entries, o);
            slow += __shfl_xor_sync(FULL, slow, o);
        }
        if (lane_id() == 0) {
            if (entries) atomicAdd(&ms->entries, entries);
            if (slow) atomicAdd(&ms->n_slow, slow);
        }
    }
}

__global__ void k_mtx_slow_list(const uint32_t *__restrict__ cnt, const uint64_t *__restrict__ nl, uint64_t n_nl, uint64_t len,
                                MtxSlowLine *out, MtxScalars *ms) {
    const uint64_t n_lines = n_nl + 1;
    for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n_lines; i += uint64_t(gridDim.x) * blockDim.x) {
        if (cnt[i] != MTX_SLOW) continue;
        MtxSlowLine s;
        s.line = i;
        mtx_line_span(nl, n_nl, len, i, s.begin, s.end);
        out[atomicAdd(&ms->listed, 1ull)] = s;
    }
}

__global__ void k_mtx_slow_counts(const uint64_t *__restrict__ lines, const uint32_t *__restrict__ n_entries, uint64_t n_slow,
                                  uint32_t *__restrict__ cnt) {
    for (uint64_t j = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; j < n_slow; j += uint64_t(gridDim.x) * blockDim.x)
        cnt[lines[j]] = n_entries[j];
}

// off[i] = entries before line i (k_scan of the counts).
__global__ void __launch_bounds__(MTX_THREADS)
k_mtx_scatter(const char *__restrict__ text, uint64_t len, const uint64_t *__restrict__ nl, uint64_t n_nl, int symmetric,
              const uint32_t *__restrict__ off, uint32_t *__restrict__ rows, uint32_t *__restrict__ cols, float *__restrict__ vals,
              MtxScalars *ms) {
    const uint64_t n_lines = n_nl + 1;
    for (uint64_t i0 = uint64_t(blockIdx.x) * MTX_THREADS; i0 < n_lines; i0 += uint64_t(gridDim.x) * MTX_THREADS) {
        const uint64_t i = i0 + threadIdx.x;
        uint32_t mr = 0, mc = 0;
        if (i < n_lines) {
            uint64_t b, e;
            mtx_line_span(nl, n_nl, len, i, b, e);
            const char *q = text + b;
            uint64_t r = 0, c = 0;
            double v;
            if (osp_mtx::plain_line(q, text + e, r, c, v) == osp_mtx::LINE_ENTRY) {
                const uint32_t o = off[i];
                const uint32_t r32 = uint32_t(r - 1), c32 = uint32_t(c - 1);   // the host's wrap-around: id 0 -> 0xFFFFFFFF
                const float f = float(v);
                rows[o] = r32; cols[o] = c32; vals[o] = f;
                mr = r32; mc = c32;
                if (symmetric && r != c) {
                    rows[o + 1] = c32; cols[o + 1] = r32; vals[o + 1] = f;
                    mr = mc = r32 > c32 ? r32 : c32;
                }
            }
        }
        mr = __reduce_max_sync(FULL, mr);
        mc = __reduce_max_sync(FULL, mc);
        if (lane_id() == 0) {
            if (mr) atomicMax(&ms->max_row, mr);
            if (mc) atomicMax(&ms->max_col, mc);
        }
    }
}

__global__ void k_mtx_scatter_slow(const uint64_t *__restrict__ lines, const uint64_t *__restrict__ src_off, uint64_t n_slow,
                                   const uint32_t *__restrict__ s_rows, const uint32_t *__restrict__ s_cols, const float *__restrict__ s_vals,
                                   const uint32_t *__restrict__ off, uint32_t *__restrict__ rows, uint32_t *__restrict__ cols,
                                   float *__restrict__ vals) {
    for (uint64_t j = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; j < n_slow; j += uint64_t(gridDim.x) * blockDim.x) {
        const uint32_t o = off[lines[j]];
        for (uint64_t k = src_off[j]; k < src_off[j + 1]; k++) {
            const uint64_t d = o + (k - src_off[j]);
            rows[d] = s_rows[k]; cols[d] = s_cols[k]; vals[d] = s_vals[k];
        }
    }
}

}  // namespace osp

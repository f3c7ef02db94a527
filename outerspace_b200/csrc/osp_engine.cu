// osp_engine.cu -- C ABI (include/osp_b200.h) and host orchestration of the sm_100a kernels.
//
// There is no CPU fallback in this file: every entry point that computes needs a CUDA device and
// fails with OSP_ERR_NO_DEVICE / OSP_ERR_CUDA otherwise.
#include "../../include/osp_b200.h"
#include "osp_kernels.cuh"
#include "osp_longrows.cuh"
#include "osp_chain2.cuh"
#include "osp_fusedlanes.cuh"
#include "osp_mtx.cuh"
#include "osp_mtx_host.h"

#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <cerrno>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

using namespace osp;

namespace {

thread_local std::string g_last_error;

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) { cudaFree(p); p = nullptr; cap = 0; }
#ifdef OSP_CUSIM
        size_t want = bytes;                 // tests/cusim under AddressSanitizer: no head-room that would hide an overrun
#else
        size_t want = bytes + bytes / 8 + 256;
#endif
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { cudaGetLastError(); e = cudaMalloc(&p, bytes); want = bytes; }
        if (e == cudaSuccess) cap = want; else p = nullptr;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T *as() const { return static_cast<T *>(p); }
};

}  // namespace

struct osp_ctx {
    int device = 0;
    int sm_count = 148;
    size_t l2_bytes = 126u << 20;
    int chain_occ[3] = {1, 1, 1};           // resident CTAs per SM of k_merge_chain: u32 keys, u64 keys, bitmap variant
    size_t total_mem = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr;      // the CSR->CSC task list is built beside the merge plan
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    cudaEvent_t ev_half[2] = {nullptr, nullptr};      // k-sharded path: a half of the exchange has landed
    uint64_t ws_limit = 0;          // bytes of partial-product bins per row block
    uint64_t result_limit = 0;      // cap on the up-front allocation of C's data (0 = what the device can spare)
    uint64_t launches = 0;
    uint64_t call_id = 0;
    std::string err;
    DevScalars *h_sc = nullptr;     // pinned mirror
    ulonglong2 *h_slots = nullptr, *h_slots_dev = nullptr;   // mapped hand-over slots {word, sequence number} (k_publish)
    unsigned long long seq = 0;     // sequence number of the last hand-over
    // per-call zeroed arena: DevScalars | look-back states of the scans | column counters
    DevBuf arena;
    DevScalars *d_sc = nullptr;
    // operand staging (host-pointer calls) and converted operands
    DevBuf op_a_pos, op_a_data, op_b_pos, op_b_data, conv_pos, conv_data, conv_tmp, conv_chk;
    // symbolic / plan / conversion scratch
    DevBuf task_bs, run_off, row_bin, tile_row, tile_start, long_list, xl_list, uniq, col_ptr, tasks, tile_state, xl_acc, xl_bits;
    DevBuf bins;
    // fused band sweep of the long rows (opt-in, osp_longrows.cuh): task bitmap for the multiply, band index of B
    DevBuf swept, lr_bands, kw_scratch, vbits;
    DevBuf fl_meta, fl_vals, fl_colb, fl_cnt, fl_pos2;
    DevBuf bpos32;                        // B.pos narrowed to 32 bits for the symbolic pass
    // the switches of the opt-in and tuning paths, read from the environment at osp_create
    struct Switches {
        uint64_t bpos32_min = 32ull << 20;  // a B.pos of at least 32 MiB is narrowed (config 4: scan 0.848 -> 0.711 + 0.023 ms); OSP_BPOS32_MIN_KB overrides, 0 = never
        bool fused_lanes_direct = true;     // OSP_FL_DIRECT=0: rows of C chained by the look-back instead of written at the prefix of their bounds
        int fused_lanes_mode = 1;           // OSP_FUSED_LANES: 0 band kernel (k_fused_dense), 1 automatic, 2 bank-aligned kernel whatever B's regrouped size
        bool kway = false;                  // OSP_KWAY=1: rows of 4097 .. 32768 partial products in <= 64 ways go to k_merge_ways
        bool sweep = false;                 // OSP_LONGROW_SWEEP=1
        uint64_t sweep_min = 0;             // OSP_LONGROW_SWEEP_MIN: fewest partial products of a swept row (0: every xl row)
        bool fused_short = false;           // OSP_FUSED_SHORT=1: short-row tiles computed inside the merge chain
        bool chain2_old = false;            // OSP_FUSED_SHORT_OLD=1: k_merge_chain_fused instead of k_chain2 (osp_chain2.cuh)
    } sw;
    bool sweep_ok = false;                  // the device accepted the kernel's shared-memory size
    int sweep_occ = 1;                      // resident CTAs per SM of k_long_fill
    bool fused_short_ok = false;
    int chain_fused_occ[3] = {1, 1, 1};
    bool chain2_ok = false;                 // k_chain2: the warp-specialised fused chain
    int chain2_occ[3] = {1, 1, 1};
    std::vector<cudaEvent_t> events;
    size_t events_used = 0;
    // OSP_PROFILE_KERNELS: one event pair per launch
    bool profile_kernels = false;
    struct KernelMark { const char *name; cudaEvent_t e0, e1; };
    std::vector<KernelMark> marks;
    // osp_readcoo_device: two pinned chunks a file is read into while the other one is copied to the device
    char *mtx_stage[2] = {nullptr, nullptr};
    cudaEvent_t mtx_copied[2] = {nullptr, nullptr};
};

struct osp_result {
    osp_ctx *ctx = nullptr;
    uint64_t *d_pos = nullptr;
    Elem *d_data = nullptr;
    uint64_t rows = 0, nnz = 0;
    osp_stats stats;
    std::vector<std::pair<const char *, float>> kernel_ms;   // OSP_PROFILE_KERNELS
    // Event pairs behind stats.ms_* and kernel_ms, read on the first osp_result_stats / osp_result_kernels --
    // not inside the call, whose host time is part of what a caller measures.  The events belong to the
    // context and are re-recorded by its next call: after that the times stay zero.
    struct Span { float *dst; const char *name; cudaEvent_t e0, e1; };
    std::vector<Span> spans;
    uint64_t call_id = 0;
    bool timed = false;
};

namespace {

void resolve_times(osp_result *r) {
    if (r->timed) return;
    r->timed = true;
    if (r->call_id != r->ctx->call_id) return;          // the events have been reused
    for (const auto &sp : r->spans) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, sp.e0, sp.e1) != cudaSuccess) { cudaGetLastError(); continue; }
        if (sp.dst) *sp.dst += ms;
        else r->kernel_ms.emplace_back(sp.name, ms);
    }
}

int fail(osp_ctx *ctx, int code, const std::string &msg) {
    g_last_error = msg;
    if (ctx) ctx->err = msg;
    return code;
}

cudaEvent_t next_event(osp_ctx *ctx) {
    if (ctx->events_used == ctx->events.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        ctx->events.push_back(e);
    }
    cudaEvent_t e = ctx->events[ctx->events_used++];
    cudaEventRecord(e, ctx->stream);
    return e;
}

#define CU(ctx, expr)                                                                           \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess) {                                                                \
            cudaGetLastError();                                                                 \
            return fail(ctx, _e == cudaErrorMemoryAllocation ? OSP_ERR_OOM : OSP_ERR_CUDA,      \
                        std::string(#expr) + ": " + cudaGetErrorString(_e));                    \
        }                                                                                       \
    } while (0)

// The one place a kernel is launched from.  (tests/cusim runs the same call on the CPU emulation of the execution model.)
#ifdef OSP_CUSIM
#define OSP_KERNEL_LAUNCH(kernel, grid, block, smem, stream, ...) cusim::launch((grid), (block), (smem), [&] { kernel(__VA_ARGS__); })
#else
#define OSP_KERNEL_LAUNCH(kernel, grid, block, smem, stream, ...) kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)
#endif

#define LAUNCH(ctx, kernel, grid, block, smem, ...)                                             \
    do {                                                                                        \
        cudaEvent_t _m0 = nullptr;                                                              \
        if ((ctx)->profile_kernels) _m0 = next_event(ctx);                                      \
        OSP_KERNEL_LAUNCH(kernel, grid, block, smem, (ctx)->stream, __VA_ARGS__);               \
        (ctx)->launches++;                                                                      \
        CU(ctx, cudaGetLastError());                                                            \
        if (_m0) (ctx)->marks.push_back({#kernel, _m0, next_event(ctx)});                       \
    } while (0)

// The prologue of every entry point that launches kernels.
int begin_call(osp_ctx *ctx, uint32_t flags) {
    CU(ctx, cudaSetDevice(ctx->device));
    ctx->launches = 0;
    ctx->events_used = 0;
    ctx->call_id++;
    ctx->marks.clear();
    ctx->profile_kernels = flags & OSP_PROFILE_KERNELS;
    CU(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));   // side-stream work of an earlier call, also of one that failed
    return OSP_OK;
}

// Work on the side stream.  While the scope lives, ctx->stream (which LAUNCH and sync_scalars use) is stream2, behind the
// main stream's work so far unless `fork` is false.  However the scope ends, ev_join then marks the end of its work.  `on`
// false: nothing changes.  (A failed record or wait stays the last error, which the next launch's check reports.)
struct SideStream {
    osp_ctx *ctx;
    cudaStream_t main;
    SideStream(osp_ctx *c, bool on, bool fork = true) : ctx(c), main(on ? c->stream : nullptr) {
        if (!main) return;
        if (fork) {
            cudaEventRecord(ctx->ev_fork, main);
            cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork, 0);
        }
        ctx->stream = ctx->stream2;
    }
    ~SideStream() {
        if (!main) return;
        ctx->stream = main;
        cudaEventRecord(ctx->ev_join, ctx->stream2);
    }
};

// A result under construction: freed on every early return, handed out by finish_result.
struct PendingResult {
    osp_result *r;
    explicit PendingResult(osp_ctx *ctx) : r(new osp_result()) {
        r->ctx = ctx;
        std::memset(&r->stats, 0, sizeof(r->stats));
    }
    ~PendingResult() { if (r) osp_result_free(r); }
    osp_result *operator->() const { return r; }
};

// C.pos (pos_entries) and C's data (data_elems) from the stream-ordered pool; 0 allocates nothing.
int alloc_result(osp_ctx *ctx, osp_result *r, uint64_t pos_entries, uint64_t data_elems) {
    cudaError_t e = cudaSuccess;
    if (pos_entries) e = cudaMallocAsync(reinterpret_cast<void **>(&r->d_pos), pos_entries * 8, ctx->stream);
    if (e == cudaSuccess && data_elems) e = cudaMallocAsync(reinterpret_cast<void **>(&r->d_data), data_elems * 8, ctx->stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(ctx, OSP_ERR_OOM, std::string("result allocation: ") + cudaGetErrorString(e));
    }
    return OSP_OK;
}

// Hands the result out with the times of its kernels (OSP_PROFILE_KERNELS), after the spans of its stats.
int finish_result(osp_ctx *ctx, PendingResult &res, osp_result **out) {
    res->call_id = ctx->call_id;
    for (const auto &m : ctx->marks) res->spans.push_back({nullptr, m.name, m.e0, m.e1});
    ctx->profile_kernels = false;
    *out = res.r;
    res.r = nullptr;
    return OSP_OK;
}

constexpr uint64_t XL_LONG_MAX_COLS = 131072;   // up to here k_merge_xl also takes the rows of MT_LONG .. MT_XL partials
constexpr size_t LONG_SMEM = size_t(MT_XL) * 12 + 34 * 4;

unsigned int grid_for(uint64_t items, unsigned int per_block, unsigned int max_blocks) {
    uint64_t b = (items + per_block - 1) / per_block;
    if (b < 1) b = 1;
    return unsigned(std::min<uint64_t>(b, max_blocks));
}

// Device memory a call can still obtain: free memory plus what the stream-ordered pool holds but does not use.
uint64_t device_available(osp_ctx *ctx) {
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); return 0; }
    uint64_t avail = free_b;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, ctx->device) == cudaSuccess) {
        uint64_t reserved = 0, used = 0;
        if (cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &reserved) == cudaSuccess &&
            cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &used) == cudaSuccess && reserved > used)
            avail += reserved - used;
        else
            cudaGetLastError();
    }
    return avail;
}

uint64_t scan_tiles(uint64_t n) { return (n + SCAN_TILE - 1) / SCAN_TILE; }
uint64_t plan_tiles(uint64_t n) { return (n + PLAN_TILE - 1) / PLAN_TILE; }
uint64_t align16(uint64_t x) { return (x + 15) & ~15ull; }

// Layout of the per-call zeroed arena.
struct Arena {
    uint64_t *state[4] = {nullptr, nullptr, nullptr, nullptr};   // look-back states of up to four scans
    uint32_t *counters = nullptr;                       // n_counters uint32 (column histogram / cursors)
};

// One memset zeroes the device scalars, the scan states and the counters of a call.
int prepare_arena(osp_ctx *ctx, const uint64_t state_tiles[4], uint64_t n_counters, Arena &a) {
    uint64_t off = align16(sizeof(DevScalars));
    uint64_t st_off[4];
    for (int i = 0; i < 4; i++) { st_off[i] = off; off += align16(state_tiles[i] * 8); }
    uint64_t cnt_off = off;
    off += align16(n_counters * 4);
    CU(ctx, ctx->arena.reserve(off));
    CU(ctx, cudaMemsetAsync(ctx->arena.p, 0, off, ctx->stream));
    unsigned char *base = ctx->arena.as<unsigned char>();
    ctx->d_sc = reinterpret_cast<DevScalars *>(base);
    for (int i = 0; i < 4; i++) a.state[i] = reinterpret_cast<uint64_t *>(base + st_off[i]);
    a.counters = reinterpret_cast<uint32_t *>(base + cnt_off);
    return OSP_OK;
}

int sync_scalars(osp_ctx *ctx) {
    if (ctx->h_slots_dev) {
        // the scalars arrive by stores from the device; the host polls the slots' sequence numbers (a few
        // microseconds less GPU idle time than a copy + stream synchronisation at every hand-over)
        const unsigned long long seq = ++ctx->seq;
        OSP_KERNEL_LAUNCH(k_publish, 1, 32, 0, ctx->stream, ctx->d_sc, ctx->h_slots_dev, seq);
        ctx->launches++;
        CU(ctx, cudaGetLastError());
        volatile unsigned long long *slots = reinterpret_cast<volatile unsigned long long *>(ctx->h_slots);
        unsigned long long *dst = reinterpret_cast<unsigned long long *>(ctx->h_sc);
        static_assert(sizeof(DevScalars) % 8 == 0, "DevScalars is handed over in 8-byte words");
        unsigned long long spins = 0;
        for (int i = 0; i < PUBLISH_SLOTS; i++) {
            bool drained = false;
            while (slots[2 * i + 1] != seq) {
                if ((++spins & 0xFFF) == 0) {
                    cudaError_t q = cudaStreamQuery(ctx->stream);
                    if (q != cudaSuccess && q != cudaErrorNotReady) {
                        cudaGetLastError();
                        return fail(ctx, OSP_ERR_CUDA, std::string("device fault: ") + cudaGetErrorString(q));
                    }
                    if (q == cudaSuccess) {
                        // the stream has drained: the stores are done.  A slot that still lacks the sequence number after
                        // one more look was not delivered as one 16-byte write (a platform without that guarantee):
                        // take the copy engine instead of spinning for ever
                        if (drained) {
                            CU(ctx, cudaMemcpyAsync(ctx->h_sc, ctx->d_sc, sizeof(DevScalars), cudaMemcpyDeviceToHost, ctx->stream));
                            CU(ctx, cudaStreamSynchronize(ctx->stream));
                            return OSP_OK;
                        }
                        drained = true;
                    }
                }
            }
            __sync_synchronize();
            dst[i] = slots[2 * i];
        }
        return OSP_OK;
    }
    CU(ctx, cudaMemcpyAsync(ctx->h_sc, ctx->d_sc, sizeof(DevScalars), cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return OSP_OK;
}

// Buffers the plan kernel writes (sized before the plan's results are known).
int reserve_plan(osp_ctx *ctx, uint64_t rows, uint64_t max_long) {
    CU(ctx, ctx->row_bin.reserve((rows + 1) * 8));
    CU(ctx, ctx->tile_row.reserve((rows + 2) * 4));
    CU(ctx, ctx->tile_start.reserve((rows + 2) * sizeof(TileStart)));
    CU(ctx, ctx->tile_state.reserve((rows + 2) * 8));      // look-back states of the merge chain, zeroed by the plan
    CU(ctx, ctx->long_list.reserve(std::max<uint64_t>(max_long, 1) * 4));
    CU(ctx, ctx->xl_list.reserve(std::max<uint64_t>(max_long, 1) * 4));
    return OSP_OK;
}

// Longest row a warp of the merge chain takes: up to MT_LONG_BM by bitmap rank when the column range is known to be
// small at plan time, MT_LONG otherwise.  The plan and the chain must be given the same value.
uint32_t plan_long_thresh(uint64_t idx_range) { return idx_range && idx_range <= 32ull * BM_WORDS ? MT_LONG_BM : MT_LONG; }

struct MergeJob {
    uint64_t rows = 0;          // rows of the plan (c_pos has rows + 1 entries)
    uint64_t idx_range = 0;     // column ids are < idx_range
    uint32_t long_thresh = MT_LONG;   // what the plan was cut with
    uint32_t n_tiles = 0, n_long = 0, n_xl = 0;
    uint64_t *c_pos = nullptr;
    Elem *c_data = nullptr;
    uint64_t c_cap = 0;
    // fused band sweep (osp_spgemm only): rows of the xl list with >= sweep_min partial products never reached the bins
    bool sweep = false;
    uint64_t sweep_min = ~0ull;             // fewest partial products of a swept row, > MT_XL (k_merge_xl leaves those alone)
    bool sweeps_every_xl() const { return sweep && sweep_min <= MT_XL + 1; }
    const uint32_t *bandptr = nullptr;      // band index of B (k_long_bands)
    // OSP_FUSED_SHORT: the chain computes the short rows' partial products itself (k_merge_chain_fused)
    bool fused_short = false;
    bool chain2 = false;                    // ... with k_chain2 (producer warps) instead of k_merge_chain_fused
    bool kway = false;                      // k_merge_ways takes the xl rows of few long ways (needs a_pos, run_off)
    int chain_ctas_per_sm = 0;              // cap on the persistent chain's CTAs per SM (0: as many as are resident); the k-sharded
                                            // path lowers it while a peer multiply shares the SMs (the chain's CTAs take every register)
    const uint64_t *run_off = nullptr;
    const uint32_t *task_bs = nullptr;
    uint64_t m_a = 0;
    const uint64_t *a_pos = nullptr;
    const Elem *a_data = nullptr, *b_data = nullptr;
};

// Template arguments of the long-row sweep on a B200: 512 threads, a band of 16384 columns (64 KB accumulator + 32 KB
// arbitration + 2 KB bitmap), 512 runs per group: 104.6 KB per CTA, two CTAs per SM.
constexpr int LR_THREADS = 512, LR_BAND = 16384, LR_RUNS = 512;
constexpr size_t LR_SMEM = LongRowSmem<LR_BAND, LR_RUNS, true>::bytes;
constexpr uint64_t LR_MIN_PER_BAND = 64;
constexpr uint64_t LR_HUGE_ROW = 1ull << 20;           // rows from here on are started before the rest of the list

// Scratch that depends on the plan's results: look-back states of the tile chain, survivor counts of the
// long rows, the dense accumulators of the longest rows.
int reserve_merge(osp_ctx *ctx, const MergeJob &job, unsigned int &xl_ctas) {
    CU(ctx, ctx->uniq.reserve(std::max<uint64_t>(job.rows, 1) * 4));
    xl_ctas = 0;
    // with the sweep taking EVERY xl row the global accumulators are only needed for the medium rows
    const uint64_t n_acc_rows = uint64_t(job.sweeps_every_xl() ? 0u : job.n_xl) + (job.idx_range <= XL_LONG_MAX_COLS ? job.n_long : 0u);
    if (n_acc_rows && job.idx_range > DENSE_MAX_COLS) {
        const uint64_t words = (job.idx_range + 31) / 32;
        const uint64_t per_cta = job.idx_range * 4 + words * 4;
        const uint64_t budget = std::max<uint64_t>(ctx->total_mem / 16, 1ull << 28);
        const uint64_t max_ctas = budget / std::max<uint64_t>(per_cta, 1);
        if (max_ctas < 1) return fail(ctx, OSP_ERR_UNSUPPORTED, "long-row accumulator does not fit: column range too large");
        // accumulators in flight: four per SM while they are a few times L2 at most; two when they are far beyond it (config 3
        // at full size, 4 MB each: 738 ms with two, 781 with four, 988 with one -- profiles/r02_experiments.md)
        uint64_t per_sm = per_cta * uint64_t(ctx->sm_count) * 4 > 8 * uint64_t(ctx->l2_bytes) ? 2 : 4;
        if (const char *env = std::getenv("OSP_XL_CTAS_PER_SM")) { const uint64_t v = std::strtoull(env, nullptr, 10); if (v) per_sm = v; }
        xl_ctas = unsigned(std::min<uint64_t>({max_ctas, uint64_t(ctx->sm_count) * per_sm, n_acc_rows}));
        CU(ctx, ctx->xl_acc.reserve(uint64_t(xl_ctas) * job.idx_range * 4));
        CU(ctx, ctx->xl_bits.reserve(uint64_t(xl_ctas) * words * 4));
        CU(ctx, cudaMemsetAsync(ctx->xl_bits.p, 0, uint64_t(xl_ctas) * words * 4, ctx->stream));
    }
    return OSP_OK;
}

// Merges the rows [row_lo, row_hi) = tiles [t0, t1) whose partial products sit in `bins` (bin of row i at
// bins[row_bin[i] - bin_base]) into C.  `block` counts the row blocks of a call (carry of the C.pos scan).
int launch_merge(osp_ctx *ctx, const MergeJob &job, unsigned int xl_ctas, Elem *bins, uint64_t bin_base, uint32_t t0,
                 uint32_t t1, uint64_t row_lo, uint64_t row_hi, unsigned int block) {
    if (t1 <= t0 || row_hi <= row_lo) return OSP_OK;
    const uint64_t *row_bin = ctx->row_bin.as<uint64_t>();
    uint32_t *uniq = ctx->uniq.as<uint32_t>();
    // long rows first (in place, survivors counted): the chain copies them when it reaches their tile
    if (job.n_long || job.n_xl) {
        if (job.idx_range <= DENSE_MAX_COLS) {
            // small column range: every long row goes through the dense shared-memory accumulator
            const size_t sm = dense_smem(job.idx_range);
            const unsigned per_sm = unsigned(std::max<size_t>(1, std::min<size_t>(4, (200u << 10) / sm)));
            LAUNCH(ctx, k_merge_dense, std::min<unsigned>(job.n_long + job.n_xl, unsigned(ctx->sm_count) * per_sm), DENSE_THREADS,
                   sm, row_bin, bin_base, bins, uniq, ctx->long_list.as<uint32_t>(), ctx->xl_list.as<uint32_t>(), ctx->d_sc,
                   uint32_t(job.idx_range), row_lo, row_hi);
        } else {
            // moderate column ranges: the arbitration kernel takes the medium rows too (compacting a bitmap of
            // <= 4096 words beats a 4096-key shared-memory sort); huge ranges keep the sort for them
            const bool xl_takes_long = job.idx_range <= XL_LONG_MAX_COLS && xl_ctas > 0;
            if (job.n_long && !xl_takes_long)
                LAUNCH(ctx, k_merge_long, std::min<unsigned>(job.n_long, unsigned(ctx->sm_count) * 4u), 256, LONG_SMEM, row_bin,
                       bin_base, bins, uniq, ctx->long_list.as<uint32_t>(), ctx->d_sc, row_lo, row_hi);
            if (job.sweep) {
                // these rows' bins are still untouched (k_multiply skipped their tasks): computed, merged and left at
                // the start of the bin in one sweep, uniq[row] = nnz -- what the chain expects of a long row
                CU(ctx, cudaMemsetAsync(&ctx->d_sc->xl_ticket, 0, 4, ctx->stream));
                const unsigned grid = unsigned(std::min<uint64_t>(job.n_xl, uint64_t(ctx->sm_count) * ctx->sweep_occ));
                const LongRowsInBins rows{ctx->xl_list.as<uint32_t>(), ctx->d_sc, row_bin, bin_base, bins, uniq, row_lo, row_hi,
                                          job.sweep_min, LR_HUGE_ROW};
                LAUNCH(ctx, (k_long_fill<LR_THREADS, LR_BAND, LR_RUNS, LongRowsInBins>), grid, LR_THREADS, LR_SMEM, job.a_pos, job.a_data,
                       job.b_data, job.bandptr, job.idx_range, rows);
            }
            if (job.kway && job.n_xl) {
                // rows of few long sorted ways: ranks by binary search over the ways, no accumulator (osp_kway.cuh)
                CU(ctx, cudaMemsetAsync(&ctx->d_sc->kw_ticket, 0, 4, ctx->stream));
                const unsigned gridk = unsigned(std::min<uint64_t>(job.n_xl, uint64_t(ctx->sm_count) * 2));
                CU(ctx, ctx->kw_scratch.reserve(uint64_t(gridk) * KW_MAX_LEN * 8));
                LAUNCH(ctx, k_merge_ways, gridk, KW_THREADS, 0, job.a_pos, job.run_off, row_bin, bin_base, bins, uniq,
                       ctx->xl_list.as<uint32_t>(), ctx->d_sc, ctx->kw_scratch.as<Elem>(), row_lo, row_hi);
            }
            if (xl_ctas && ((job.n_xl && !job.sweeps_every_xl()) || (job.n_long && xl_takes_long))) {
                CU(ctx, cudaMemsetAsync(&ctx->d_sc->xl_ticket, 0, 4, ctx->stream));
                LAUNCH(ctx, k_merge_xl, xl_ctas, XL_THREADS, 0, row_bin, bin_base, bins, uniq, ctx->xl_list.as<uint32_t>(),
                       xl_takes_long ? ctx->long_list.as<uint32_t>() : nullptr, ctx->d_sc, ctx->xl_acc.as<float>(),
                       ctx->xl_bits.as<uint32_t>(), job.idx_range, row_lo, row_hi, job.sweep ? job.sweep_min : ~0ull,
                       job.kway ? job.a_pos : nullptr);
            }
        }
    }
    // one pass from the bins to C: tiles in row order, chained by a decoupled look-back (C.pos on the way)
    const uint32_t n_chain = t1 - t0;
    if (block > 0) {             // the first block's states were zeroed by the plan, its ticket by the arena memset
        CU(ctx, cudaMemsetAsync(ctx->tile_state.p, 0, uint64_t(n_chain) * 8, ctx->stream));
        CU(ctx, cudaMemsetAsync(&ctx->d_sc->tile_ticket, 0, 4, ctx->stream));
    }
    const int carry_slot = int(block & 1);
    // small column range: rows of more than 128 partial products are merged by bitmap rank instead of a sort
    const uint32_t bm_words = job.idx_range <= 32ull * BM_WORDS ? uint32_t((job.idx_range + 31) / 32) : 0u;
    const uint32_t bm_wpl = (((bm_words + 31) / 32) + 3) & ~3u;           // bitmap words per lane, a multiple of 4
#define MC_ARGS row_bin, bin_base, bins, ctx->tile_row.as<uint32_t>(), t0, n_chain, uniq, ctx->tile_state.as<uint64_t>(), ctx->d_sc, \
                carry_slot, job.c_pos, job.c_data, bm_wpl, job.long_thresh
    const int variant = bm_words ? 2 : job.idx_range <= (1ull << 23) ? 0 : 1;
    if (job.fused_short && job.chain2) {
        const C2SrcProduct src{job.a_data, job.run_off, job.task_bs, job.b_data};
        const TileStart *tiles = ctx->tile_start.as<TileStart>();
        const unsigned int grid2 = std::min<unsigned>(n_chain, unsigned(ctx->sm_count) * unsigned(ctx->chain2_occ[variant == 2 && job.long_thresh != MT_LONG_BM ? 0 : variant]));
#define C2_ARGS tiles, row_bin, bin_base, bins, t0, n_chain, uniq, ctx->tile_state.as<uint64_t>(), ctx->d_sc, carry_slot, job.c_pos, job.c_data, \
                bm_wpl, job.long_thresh, src
        // the bitmap variant needs the smaller tiles the plan cuts when it knows the column range up front
        const int v2 = variant == 2 && job.long_thresh != MT_LONG_BM ? 0 : variant;
        if (v2 == 2) LAUNCH(ctx, (k_chain2<uint32_t, true, C2SrcProduct>), grid2, C2_THREADS, sizeof(Chain2Smem<true>), C2_ARGS);
        else if (v2 == 0) LAUNCH(ctx, (k_chain2<uint32_t, false, C2SrcProduct>), grid2, C2_THREADS, sizeof(Chain2Smem<false>), C2_ARGS);
        else LAUNCH(ctx, (k_chain2<uint64_t, false, C2SrcProduct>), grid2, C2_THREADS, sizeof(Chain2Smem<false>), C2_ARGS);
#undef C2_ARGS
        return OSP_OK;
    }
    if (job.fused_short) {
        const FusedSrc fs{job.a_pos, job.a_data, job.run_off, job.task_bs, job.b_data, job.m_a};
        const unsigned int gridf = std::min<unsigned>(n_chain, unsigned(ctx->sm_count) * unsigned(ctx->chain_fused_occ[variant]));
        if (variant == 2) LAUNCH(ctx, (k_merge_chain_fused<uint32_t, true>), gridf, MC_THREADS, sizeof(MergeChainSmem<true>), MC_ARGS, fs);
        else if (variant == 0) LAUNCH(ctx, (k_merge_chain_fused<uint32_t, false>), gridf, MC_THREADS, sizeof(MergeChainSmem<false>), MC_ARGS, fs);
        else LAUNCH(ctx, (k_merge_chain_fused<uint64_t, false>), gridf, MC_THREADS, sizeof(MergeChainSmem<false>), MC_ARGS, fs);
        return OSP_OK;
    }
    const int occ = job.chain_ctas_per_sm > 0 ? std::min(job.chain_ctas_per_sm, ctx->chain_occ[variant]) : ctx->chain_occ[variant];
    const unsigned int grid = std::min<unsigned>(n_chain, unsigned(ctx->sm_count) * unsigned(occ));   // persistent CTAs
    if (variant == 2) LAUNCH(ctx, (k_merge_chain<uint32_t, true>), grid, MC_THREADS, sizeof(MergeChainSmem<true>), MC_ARGS);
    else if (variant == 0) LAUNCH(ctx, (k_merge_chain<uint32_t, false>), grid, MC_THREADS, sizeof(MergeChainSmem<false>), MC_ARGS);
    else LAUNCH(ctx, (k_merge_chain<uint64_t, false>), grid, MC_THREADS, sizeof(MergeChainSmem<false>), MC_ARGS);
#undef MC_ARGS
    return OSP_OK;
}

// Stable transposition on the device (all pointers are device pointers): histogram -> scan ->
// bucket scatter -> per-bucket sort by source slice id (the merge machinery; a bucket that shrinks
// while folding held a duplicate (row, col): the reference's dupcheck, SimSpGEMM.cpp:43-53).
// With `coo` set the source is a triplet list instead of a compressed matrix (COO ingest): n_minor buckets keyed
// by coo->major, elements {coo->minor < n_major, val} -- the same machinery, the same duplicate check.
struct CooSrc { const uint32_t *major, *minor; const float *val; };
int csr2csc_device(osp_ctx *ctx, uint64_t n_major, uint64_t n_minor, const uint64_t *d_pos, const Elem *d_data,
                   uint64_t nnz, uint64_t *d_pos_out, Elem *d_data_out, const CooSrc *coo = nullptr) {
    if (nnz >= (1ull << 32)) return fail(ctx, OSP_ERR_UNSUPPORTED, "operands with >= 2^32 non-zeros are not supported");
    // no output slice: every id of a non-empty operand is out of range (DESIGN section 2, divergence iii)
    if (n_minor == 0 && nnz) return fail(ctx, OSP_ERR_INDEX, "index out of range in operand: there is no output slice");
    if (nnz == 0) {
        CU(ctx, cudaMemsetAsync(d_pos_out, 0, (n_minor + 1) * 8, ctx->stream));
        return OSP_OK;
    }
    Arena ar;
    const uint64_t st[4] = {scan_tiles(n_minor), plan_tiles(n_minor), 0, 0};
    int rc = prepare_arena(ctx, st, n_minor, ar);
    if (rc) return rc;
    uint32_t *cnt = ar.counters;
    if (coo) LAUNCH(ctx, k_hist_u32, grid_for(nnz, 256, unsigned(ctx->sm_count) * 16u), 256, 0, coo->major, nnz, n_minor, cnt, ctx->d_sc);
    else LAUNCH(ctx, k_hist_elems, grid_for(nnz, 256, unsigned(ctx->sm_count) * 16u), 256, 0, d_data, nnz, n_minor, cnt, ctx->d_sc);
    LAUNCH(ctx, (k_scan<U32In, U64Out>), unsigned(st[0]), SCAN_BLOCK, 0, U32In{cnt}, U64Out{d_pos_out}, n_minor, ar.state[0],
           &ctx->d_sc->scan_ticket[0]);
    CU(ctx, cudaMemsetAsync(cnt, 0, n_minor * 4, ctx->stream));
    CU(ctx, ctx->conv_tmp.reserve(nnz * 8 + 16));
    if (coo)
        LAUNCH(ctx, k_scatter_coo, grid_for(nnz, 256, unsigned(ctx->sm_count) * 16u), 256, 0, coo->major, coo->minor, coo->val, nnz,
               n_minor, n_major, d_pos_out, cnt, ctx->conv_tmp.as<Elem>(), ctx->d_sc);
    else
        LAUNCH(ctx, k_scatter_elems, grid_for(n_major, 8, unsigned(ctx->sm_count) * 16u), 256, 0, d_pos, d_data, n_major, n_minor,
               d_pos_out, cnt, ctx->conv_tmp.as<Elem>(), ctx->d_sc);
    rc = reserve_plan(ctx, n_minor, std::min(n_minor, nnz));
    if (rc) return rc;
    LAUNCH(ctx, k_plan<RowBinDirect>, unsigned(st[1]), PLAN_BLOCK, 0, RowBinDirect{d_pos_out}, n_minor, n_major,
           ctx->row_bin.as<uint64_t>(), ctx->tile_row.as<uint32_t>(), ctx->long_list.as<uint32_t>(),
           ctx->xl_list.as<uint32_t>(), ar.state[1], ctx->d_sc, 1, plan_long_thresh(std::max<uint64_t>(n_major, 1)), ctx->tile_state.as<uint64_t>());
    rc = sync_scalars(ctx);
    if (rc) return rc;
    if (ctx->h_sc->err) return fail(ctx, OSP_ERR_INDEX, "index out of range in operand");
    MergeJob job;
    job.rows = n_minor; job.idx_range = std::max<uint64_t>(n_major, 1); job.long_thresh = plan_long_thresh(job.idx_range);
    job.n_tiles = ctx->h_sc->n_tiles; job.n_long = ctx->h_sc->n_long; job.n_xl = ctx->h_sc->n_xl;
    CU(ctx, ctx->conv_chk.reserve((n_minor + 1) * 8));
    job.c_pos = ctx->conv_chk.as<uint64_t>(); job.c_data = d_data_out; job.c_cap = nnz;
    unsigned int xl_ctas = 0;
    rc = reserve_merge(ctx, job, xl_ctas);
    if (rc) return rc;
    rc = launch_merge(ctx, job, xl_ctas, ctx->conv_tmp.as<Elem>(), 0, 0, job.n_tiles, 0, n_minor, 0);
    if (rc) return rc;
    LAUNCH(ctx, k_check_same, grid_for(n_minor + 1, 256, 1u << 30), 256, 0, d_pos_out, job.c_pos, n_minor + 1, ctx->d_sc);
    rc = sync_scalars(ctx);
    if (rc) return rc;
    if (ctx->h_sc->err == 233) return fail(ctx, OSP_ERR_DUPLICATE, "duplicate (row,col) entry in operand");
    if (ctx->h_sc->err) return fail(ctx, OSP_ERR_INDEX, "index out of range in operand");
    return OSP_OK;
}

// Operands of a call as device pointers (host operands are staged into the context's buffers).
struct Operands {
    const uint64_t *a_pos = nullptr, *b_pos = nullptr;
    const Elem *a_data = nullptr, *b_data = nullptr;
    uint64_t nnz_a = 0, nnz_b = 0;
    float ms_h2d = 0.f;
};

int stage_operands(osp_ctx *ctx, const osp_spgemm_args *args, Operands &op) {
    const uint64_t n_k = args->n_k;
    if (args->flags & OSP_DEVICE_POINTERS) {
        op.a_pos = args->a_pos; op.b_pos = args->b_pos;
        op.a_data = static_cast<const Elem *>(args->a_data);
        op.b_data = static_cast<const Elem *>(args->b_data);
        if (args->a_nnz && args->b_nnz) {
            op.nnz_a = args->a_nnz;
            op.nnz_b = args->b_nnz;
        } else {
            CU(ctx, cudaMemcpyAsync(&ctx->h_sc->products, op.a_pos + args->a_slices, 8, cudaMemcpyDeviceToHost, ctx->stream));
            CU(ctx, cudaMemcpyAsync(&ctx->h_sc->cap_bound, op.b_pos + n_k, 8, cudaMemcpyDeviceToHost, ctx->stream));
            CU(ctx, cudaStreamSynchronize(ctx->stream));
            op.nnz_a = ctx->h_sc->products;
            op.nnz_b = ctx->h_sc->cap_bound;
        }
    } else {
        op.nnz_a = args->a_pos[args->a_slices];
        op.nnz_b = args->b_pos[n_k];
        // C = A*A on the caller's one CSRMatrix (the same arrays as both operands): staged once
        const bool same = args->b_pos == args->a_pos && args->b_data == args->a_data && args->a_slices == n_k;
        CU(ctx, ctx->op_a_pos.reserve((args->a_slices + 1) * 8));
        CU(ctx, ctx->op_a_data.reserve(std::max<uint64_t>(op.nnz_a, 1) * 8));
        if (!same) {
            CU(ctx, ctx->op_b_pos.reserve((n_k + 1) * 8));
            CU(ctx, ctx->op_b_data.reserve(std::max<uint64_t>(op.nnz_b, 1) * 8));
        }
        cudaEvent_t e0 = next_event(ctx);
        CU(ctx, cudaMemcpyAsync(ctx->op_a_pos.p, args->a_pos, (args->a_slices + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
        if (!same) CU(ctx, cudaMemcpyAsync(ctx->op_b_pos.p, args->b_pos, (n_k + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
        if (op.nnz_a && args->a_data)
            CU(ctx, cudaMemcpyAsync(ctx->op_a_data.p, args->a_data, op.nnz_a * 8, cudaMemcpyHostToDevice, ctx->stream));
        if (!same && op.nnz_b && args->b_data)
            CU(ctx, cudaMemcpyAsync(ctx->op_b_data.p, args->b_data, op.nnz_b * 8, cudaMemcpyHostToDevice, ctx->stream));
        cudaEvent_t e1 = next_event(ctx);
        CU(ctx, cudaEventSynchronize(e1));
        cudaEventElapsedTime(&op.ms_h2d, e0, e1);
        op.a_pos = ctx->op_a_pos.as<uint64_t>(); op.a_data = ctx->op_a_data.as<Elem>();
        op.b_pos = same ? op.a_pos : ctx->op_b_pos.as<uint64_t>();
        op.b_data = same ? op.a_data : ctx->op_b_data.as<Elem>();
    }
    if ((op.nnz_a && !args->a_data) || (op.nnz_b && !args->b_data))
        return fail(ctx, OSP_ERR_INVALID, "osp_spgemm: NULL data array");
    if (op.nnz_a >= (1ull << 32) || op.nnz_b >= (1ull << 32))
        return fail(ctx, OSP_ERR_UNSUPPORTED, "operands with >= 2^32 non-zeros are not supported");
    return OSP_OK;
}

template <class Src>
int launch_multiply(osp_ctx *ctx, Src src, uint64_t t0, uint64_t t1, uint64_t products, const Elem *b_data, Elem *bins,
                    uint64_t bin_base) {
    uint64_t n = t1 - t0;
    if (!n || !products) return OSP_OK;
    unsigned int grid = grid_for(n, 256, unsigned(ctx->sm_count) * 32u);
    LAUNCH(ctx, k_multiply<Src>, grid, 256, 0, src, t0, t1, b_data, bins, bin_base);
    return OSP_OK;
}

// Operand preconditions (k_validate): launched into the current arena; check_operands() reads the verdict after the next
// hand-over of the device scalars.
int launch_validate(osp_ctx *ctx, ValidateOp op0, ValidateOp op1, int n_ops) {
    // one bit per element position (does it open a slice?), both operands back to back in ctx->vbits
    const uint64_t w0 = (op0.nnz + 31) / 32 + 1, w1 = n_ops > 1 ? (op1.nnz + 31) / 32 + 1 : 0;
    CU(ctx, ctx->vbits.reserve((w0 + w1) * 4));
    CU(ctx, cudaMemsetAsync(ctx->vbits.p, 0, (w0 + w1) * 4, ctx->stream));
    op0.start_bits = ctx->vbits.as<uint32_t>();
    op1.start_bits = ctx->vbits.as<uint32_t>() + (n_ops > 1 ? w0 : 0);
    const uint64_t slices = std::max<uint64_t>({op0.n_slices, n_ops > 1 ? op1.n_slices : 0, 1});
    const uint64_t elems = std::max<uint64_t>({op0.nnz, n_ops > 1 ? op1.nnz : 0, 1});
    LAUNCH(ctx, k_validate_starts, grid_for(slices, 512, unsigned(ctx->sm_count) * 8u), 256, 0, op0, op1, n_ops, ctx->d_sc);
    LAUNCH(ctx, k_validate, grid_for(elems, 1024, unsigned(ctx->sm_count) * 8u), 256, 0, op0, op1, n_ops, ctx->d_sc);
    return OSP_OK;
}
int check_operands(osp_ctx *ctx, const char *who) {
    const DevScalars &h = *ctx->h_sc;
    if (h.v_bad_pos) return fail(ctx, OSP_ERR_INVALID, std::string(who) + ": a pos array decreases or points past its data array");
    if (h.v_desc - h.v_eq != h.v_bdesc - h.v_beq)
        return fail(ctx, OSP_ERR_INVALID, std::string(who) + ": the indices of a slice are not ascending (operands must be sorted inside every slice, "
                                                             "as coo2csr leaves them, SimSpGEMM.cpp:113-120)");
    if (h.v_eq != h.v_beq) return fail(ctx, OSP_ERR_DUPLICATE, std::string(who) + ": duplicate (row,col) entry in operand");
    return OSP_OK;
}

// ---- osp_spgemm, stage by stage ---------------------------------------------------------------------------------------

// The paths of a call.  Set by choose_paths and choose_long_row_paths only, apart from the row-order override of a
// blocked call (cut_row_blocks).
struct Paths {
    bool rowwise = false;                   // tasks in row order of A; else the outer-product order with a CSR->CSC task list
    bool fused = false;                     // fused dense rows: no partial product reaches HBM
    bool fused_short = false;               // OSP_FUSED_SHORT: short rows computed inside the merge chain ...
    bool chain2 = false;                    // ... by k_chain2 (else k_merge_chain_fused)
    bool sweep = false;                     // long rows computed and merged by the band sweep (k_long_fill)
    bool kway = false;                      // long rows of few long ways merged by k_merge_ways
};

// The paths that are settled before the symbolic pass.
Paths choose_paths(const osp_ctx *ctx, const osp_spgemm_args *args, uint64_t nnz_a, uint64_t nnz_b, uint64_t m_a) {
    const uint32_t f = args->flags;
    Paths p;
    // ---- multiply order.  The outer-product (k-slice) order of the reference streams B once and scatters 8-byte
    // partial products over the bins; row order of A writes the bins as ONE stream, gathers the rows of B and needs
    // no CSR->CSC task list.  Measured (profiles/README.md): row order wins on every config -- config 2 (bins
    // L2-resident) 0.141 vs 0.161 ms per call, config 4 9.1 vs 16.6 ms -- so it is the automatic choice;
    // OSP_KSLICE_ORDER selects the outer-product order (same bins, same bits).
    p.rowwise = (f & OSP_ROWWISE_ORDER) || !(f & OSP_KSLICE_ORDER);
    // ---- fused dense rows: when the column range is small and the rows are expected to be long (config 5), the
    // per-row bin is a dense accumulator in shared memory and no partial product ever reaches HBM.
    if (args->cols_b && args->cols_b <= DENSE_MAX_COLS && !(f & OSP_NO_FUSED_DENSE) && nnz_a && nnz_b && args->n_k) {
        const double p_est = double(nnz_a) * double(nnz_b) / double(args->n_k);
        p.fused = p_est / double(std::max<uint64_t>(m_a, 1)) >= 1024.0;
        if (p.fused) p.rowwise = true;
    }
    // ---- OSP_FUSED_SHORT: no bins for the tiles of short rows; the multiply only serves the long rows.  Decided before the
    // plan: the bitmap variant of k_chain2 takes smaller tiles (shared memory)
    p.fused_short = ctx->fused_short_ok && ((f & OSP_FUSED_SHORT) || ctx->sw.fused_short) && !(f & OSP_KSLICE_ORDER) && p.rowwise &&
                    !p.fused && nnz_a > 0;
    p.chain2 = p.fused_short && ctx->chain2_ok && !ctx->sw.chain2_old;
    return p;
}

// The long-row paths, which need the plan's count of xl rows.
void choose_long_row_paths(const osp_ctx *ctx, uint32_t flags, const MergeJob &job, uint64_t lr_index_bytes, Paths &p) {
    const bool applies = !(flags & OSP_KSLICE_ORDER) && p.rowwise && !p.fused && job.n_xl > 0 && job.idx_range > DENSE_MAX_COLS;
    // ---- fused band sweep of the long rows (opt-in).  The band index of B (4 bytes per row of B and band) must fit a
    // sixteenth of the device, else the call stays on the default path.
    p.sweep = applies && ctx->sweep_ok && ((flags & OSP_LONGROW_SWEEP) || ctx->sw.sweep) &&
              lr_index_bytes <= std::max<uint64_t>(ctx->total_mem / 16, 256ull << 20);
    // ---- k-way merge of the long rows made of few long ways (opt-in until measured).  Needs the row-order bins (ways =
    // runs of consecutive tasks).
    p.kway = applies && !p.sweep && ((flags & OSP_KWAY_MERGE) || ctx->sw.kway);
}

// One osp_spgemm call: its operands and what the stages learn about them.
struct SpgemmCall {
    const osp_spgemm_args *args = nullptr;
    bool validate = true;
    Operands op;                            // A is re-pointed at its row-compressed form by the CSC(A) hand-over
    uint64_t n_k = 0, m_a = 0;
    uint64_t m_plan = 0;                    // rows the plan covers: every row of A, and every row the caller asked for
    uint64_t cols_b = 0;                    // as given; derived from B at the hand-over when it was not
    uint64_t rows_c = 0, P = 0, cap_bound = 0;
    Paths paths;
    bool forked = false;                    // the k-slice task list runs on the side stream
    Arena ar;
    uint64_t st[4] = {0, 0, 0, 0};          // tiles of the arena's scans
    uint64_t *run_off = nullptr;
    uint32_t *task_bs = nullptr;
    MergeJob job;
    unsigned int xl_ctas = 0;
    uint64_t lr_bands = 0;                  // bands of the long-row sweep

    bool masked() const { return paths.sweep || paths.fused_short; }     // the multiply reads a task bitmap
    // OSP_FUSED_SHORT without a single medium or long row: nothing is ever written to the bins, so they cost no memory
    // and the workspace limit cuts no row blocks (a bounded C still does)
    bool no_bins() const { return paths.fused_short && job.n_xl + job.n_long == 0; }
    uint64_t lr_index_bytes() const { return std::max<uint64_t>(n_k, 1) * (lr_bands + 1) * 4; }
};

// CSC(A) -> CSR(A) on the device: the bins are offset in k order per row.  Rows of A = max row id + 1 (SimOuterSPACE.cpp:49-53).
int convert_a(osp_ctx *ctx, SpgemmCall &c) {
    const osp_spgemm_args *args = c.args;
    Arena ar0;
    const uint64_t st0[4] = {0, 0, 0, 0};
    int rc = prepare_arena(ctx, st0, 0, ar0);
    if (rc) return rc;
    if (c.validate) {             // also leaves the largest row id in max_idx
        const ValidateOp opa{c.op.a_pos, c.op.a_data, args->a_slices, c.op.nnz_a, args->rows_c, nullptr};
        rc = launch_validate(ctx, opa, opa, 1);
        if (rc) return rc;
    } else if (c.op.nnz_a)
        LAUNCH(ctx, k_max_idx, grid_for(c.op.nnz_a, 1024, unsigned(ctx->sm_count) * 8u), 256, 0, c.op.a_data, c.op.nnz_a, ctx->d_sc);
    rc = sync_scalars(ctx);
    if (rc) return rc;
    if (c.validate) {
        if (ctx->h_sc->err) return fail(ctx, OSP_ERR_INDEX, "osp_spgemm: rows_c is smaller than the largest row id of A + 1");
        rc = check_operands(ctx, "osp_spgemm (A)");
        if (rc) return rc;
    }
    c.m_a = uint64_t(ctx->h_sc->max_idx) + 1;
    if (c.m_a >= (1ull << 32))        // the rows of C are uint32 ids, rows_c < 2^32: row id 2^32 - 1 has no room
        return fail(ctx, OSP_ERR_INDEX, "osp_spgemm: a row id of CSC(A) is 2^32 - 1; row ids must be below 2^32 - 1");
    CU(ctx, ctx->conv_pos.reserve((c.m_a + 1) * 8));
    CU(ctx, ctx->conv_data.reserve(std::max<uint64_t>(c.op.nnz_a, 1) * 8));
    rc = csr2csc_device(ctx, c.n_k, c.m_a, c.op.a_pos, c.op.a_data, c.op.nnz_a, ctx->conv_pos.as<uint64_t>(), ctx->conv_data.as<Elem>());
    if (rc) return rc;
    c.op.a_pos = ctx->conv_pos.as<uint64_t>();
    c.op.a_data = ctx->conv_data.as<Elem>();
    return OSP_OK;
}

// Symbolic pass, k-slice task list and merge plan: launched back to back.
int launch_symbolic_and_plan(osp_ctx *ctx, SpgemmCall &c) {
    const Operands &op = c.op;
    const uint64_t nnz_a = op.nnz_a, nnz_b = op.nnz_b, n_k = c.n_k;
    c.st[0] = scan_tiles(std::max<uint64_t>(nnz_a, 1));
    c.st[1] = plan_tiles(c.m_plan);
    c.st[2] = scan_tiles(std::max<uint64_t>(n_k, 1));
    c.st[3] = c.paths.fused ? scan_tiles(c.m_plan + 1) : 0;       // prefix of the row bounds / counts (osp_fusedlanes.cuh)
    int rc = prepare_arena(ctx, c.st, c.paths.rowwise ? 0 : n_k, c.ar);
    if (rc) return rc;
    if (c.validate) {
        // B: ascending, duplicate-free rows, column ids below cols_b (or their maximum when cols_b is to be derived);
        // A in row-compressed form: ascending rows (k < n_k is the symbolic pass's check).  A converted on the device a
        // moment ago is sorted by construction; A == B (C = A*A on the same arrays) is read once.
        const bool a_is_csr = c.args->flags & OSP_A_IS_CSR;
        const ValidateOp opb{op.b_pos, op.b_data, n_k, nnz_b, c.cols_b, nullptr};
        const ValidateOp opa{op.a_pos, op.a_data, c.m_a, nnz_a, 0, nullptr};
        const bool same = a_is_csr && op.a_pos == op.b_pos && op.a_data == op.b_data && c.m_a == n_k;
        rc = a_is_csr && !same ? launch_validate(ctx, opa, opb, 2) : launch_validate(ctx, opb, opb, 1);
        if (rc) return rc;
    } else if (!c.cols_b && nnz_b)
        LAUNCH(ctx, k_max_idx, grid_for(nnz_b, 1024, unsigned(ctx->sm_count) * 8u), 256, 0, op.b_data, nnz_b, ctx->d_sc);
    CU(ctx, ctx->run_off.reserve((nnz_a + 1) * 8));
    CU(ctx, ctx->task_bs.reserve(std::max<uint64_t>(nnz_a, 1) * 4));
    c.run_off = ctx->run_off.as<uint64_t>();
    c.task_bs = ctx->task_bs.as<uint32_t>();
    uint32_t *col_cnt = c.paths.rowwise ? nullptr : c.ar.counters;
    if (nnz_a) {
        const uint32_t *b_pos32 = nullptr;
        if (ctx->sw.bpos32_min && (n_k + 1) * 8 >= ctx->sw.bpos32_min && nnz_b < (1ull << 32)) {
            // B.pos beyond what the L2 keeps under the pass's streams: a 32-bit copy for its random reads
            CU(ctx, ctx->bpos32.reserve((n_k + 1) * 4));
            LAUNCH(ctx, k_narrow_pos, grid_for(n_k + 1, 256, unsigned(ctx->sm_count) * 8u), 256, 0, op.b_pos, n_k + 1, ctx->bpos32.as<uint32_t>());
            b_pos32 = ctx->bpos32.as<uint32_t>();
        }
        LAUNCH(ctx, (k_scan<SymIn, RunOffOut>), unsigned(c.st[0]), SCAN_BLOCK, 0, SymIn{op.a_data, op.b_pos, n_k, col_cnt, ctx->d_sc, c.task_bs, b_pos32},
               RunOffOut{c.run_off, ctx->d_sc, nnz_a}, nnz_a, c.ar.state[0], &ctx->d_sc->scan_ticket[0]);
    } else {
        CU(ctx, cudaMemsetAsync(c.run_off, 0, 8, ctx->stream));
    }
    if (!c.paths.rowwise && nnz_a) {
        // CSR->CSC task list on the side stream: it needs only the symbolic pass, not the plan, and the host round trip
        // of the hand-over waits for the plan alone; the multiply joins it
        CU(ctx, ctx->col_ptr.reserve((n_k + 1) * 4));
        CU(ctx, ctx->tasks.reserve(nnz_a * sizeof(Task)));
        c.forked = !ctx->profile_kernels;         // (per-kernel event pairs assume one stream)
        SideStream side(ctx, c.forked);
        LAUNCH(ctx, (k_scan<U32In, U32Out>), unsigned(c.st[2]), SCAN_BLOCK, 0, U32In{col_cnt}, U32Out{ctx->col_ptr.as<uint32_t>()},
               n_k, c.ar.state[2], &ctx->d_sc->scan_ticket[2]);
        LAUNCH(ctx, k_scatter_tasks, grid_for(nnz_a, 256, unsigned(ctx->sm_count) * 16u), 256, 0, op.a_data, c.run_off, op.b_pos,
               uint64_t(0), nnz_a, ctx->col_ptr.as<uint32_t>(), col_cnt, ctx->tasks.as<Task>(), ctx->d_sc);
    }
    rc = reserve_plan(ctx, c.m_plan, std::min(c.m_plan, std::max<uint64_t>(nnz_a, 1)));
    if (rc) return rc;
    const uint32_t cap_max = !c.paths.chain2 ? MT_CAP : plan_long_thresh(c.cols_b) == MT_LONG_BM ? C2_CAP_BM : C2_CAP;
    LAUNCH(ctx, k_plan<RowBinFromRuns>, unsigned(c.st[1]), PLAN_BLOCK, 0, RowBinFromRuns{op.a_pos, c.m_a, c.run_off, nnz_a}, c.m_plan,
           c.cols_b, ctx->row_bin.as<uint64_t>(), ctx->tile_row.as<uint32_t>(), ctx->long_list.as<uint32_t>(),
           ctx->xl_list.as<uint32_t>(), c.ar.state[1], ctx->d_sc, 1, plan_long_thresh(c.cols_b), ctx->tile_state.as<uint64_t>(),
           ctx->tile_start.as<TileStart>(), cap_max);
    return OSP_OK;
}

// The one mid-pipeline hand-over: the verdict on the operands, the sizes of the bins and of C, the merge job.
int take_hand_over(osp_ctx *ctx, SpgemmCall &c) {
    int rc = sync_scalars(ctx);
    if (rc) return rc;
    const DevScalars &h = *ctx->h_sc;
    if (c.validate && h.v_bad_pos) return check_operands(ctx, "osp_spgemm");     // (a broken pos array also looks like a huge row)
    if (h.err == 6) return fail(ctx, OSP_ERR_UNSUPPORTED, "osp_spgemm: a row of B holds >= 2^24 non-zeros");
    if (h.err) return fail(ctx, OSP_ERR_INDEX, "osp_spgemm: index out of range (k of A beyond the inner dimension, or a column of B beyond cols_b)");
    if (c.validate) {
        rc = check_operands(ctx, "osp_spgemm");
        if (rc) return rc;
    }
    c.P = h.products;
    if (c.P >> 40) return fail(ctx, OSP_ERR_UNSUPPORTED, "osp_spgemm: more than 2^40 partial products");
    if (!c.cols_b) c.cols_b = uint64_t(h.max_idx) + 1;
    if (c.cols_b >= (1ull << 32))       // as for a given cols_b (< 2^32): column ids stay below 2^32 - 1, the kernels' "no column"
        return fail(ctx, OSP_ERR_INDEX, "osp_spgemm: a column id of B is 2^32 - 1; column ids must be below 2^32 - 1");
    // reference rule numRows = max row id of A + 1 (SimOuterSPACE.cpp:49-53): the last row of A holding a
    // non-zero, whether or not it meets a non-empty row of B
    c.rows_c = c.args->rows_c ? c.args->rows_c : std::max<uint64_t>(h.last_nonempty, 1);
    if (c.rows_c < h.last_nonempty) return fail(ctx, OSP_ERR_INDEX, "osp_spgemm: rows_c is smaller than the largest row id of A + 1");
    // the merge job of the plan, the long-row paths, the merge scratch
    MergeJob &job = c.job;
    job.rows = c.m_plan; job.idx_range = std::max<uint64_t>(c.cols_b, 1); job.long_thresh = plan_long_thresh(c.args->cols_b);
    job.n_tiles = h.n_tiles; job.n_long = h.n_long; job.n_xl = h.n_xl;
    c.lr_bands = (job.idx_range + LR_BAND - 1) / LR_BAND;
    choose_long_row_paths(ctx, c.args->flags, job, c.lr_index_bytes(), c.paths);
    if (c.paths.sweep) {
        // the swept rows' tasks are flagged for the multiply, which emits nothing for them; k_long_fill computes and merges
        // them straight into the start of their bins (launch_merge).  Only rows of the xl list are ever swept, and only
        // where a band sees enough of the row to pay for its barriers: a row must bring LR_MIN_PER_BAND partial products
        // per band on average (16 M columns = 1024 bands: rows from 65 536 partial products), shorter rows stay with
        // k_multiply + k_merge_xl.  (Unmeasured starting point.)
        job.sweep = true;
        job.sweep_min = std::max<uint64_t>({ctx->sw.sweep_min, MT_XL + 1, LR_MIN_PER_BAND * c.lr_bands});
        job.a_pos = c.op.a_pos; job.a_data = c.op.a_data; job.b_data = c.op.b_data;
    }
    if (c.paths.kway) {           // the multiply writes these rows' bins as usual, k_merge_ways replaces k_merge_xl for them
        job.kway = true;
        job.a_pos = c.op.a_pos; job.run_off = c.run_off;
    }
    if (c.paths.fused_short) {
        job.fused_short = true; job.chain2 = c.paths.chain2;
        job.run_off = c.run_off; job.task_bs = c.task_bs; job.m_a = c.m_a;
        job.a_pos = c.op.a_pos; job.a_data = c.op.a_data; job.b_data = c.op.b_data;
    }
    c.cap_bound = std::max<uint64_t>(c.args->cols_b ? h.cap_bound : std::min<uint64_t>(h.cap_bound, c.P), 1);
    return reserve_merge(ctx, job, c.xl_ctas);
}

// The task bitmap the multiply reads (long-row sweep, fused short rows), and the sweep's band index of B.
int launch_task_bitmap(osp_ctx *ctx, SpgemmCall &c) {
    if (!c.masked()) return OSP_OK;
    const MergeJob &job = c.job;
    const uint64_t words = (c.op.nnz_a + 31) / 32 + 1;
    CU(ctx, ctx->swept.reserve(words * 4));
    CU(ctx, cudaMemsetAsync(ctx->swept.p, 0, words * 4, ctx->stream));
    if (c.paths.fused_short) {
        // marked = goes to the bins: medium rows, and the xl rows the sweep leaves alone
        if (job.n_xl + job.n_long)
            LAUNCH(ctx, k_mark_binned, grid_for(uint64_t(job.n_xl + job.n_long) * 32, 256, unsigned(ctx->sm_count) * 8u), 256, 0, c.op.a_pos,
                   ctx->xl_list.as<uint32_t>(), ctx->long_list.as<uint32_t>(), ctx->d_sc, ctx->row_bin.as<uint64_t>(),
                   c.paths.sweep ? job.sweep_min : ~0ull, ctx->swept.as<uint32_t>());
    } else {
        // marked = swept: computed by k_long_fill, not by the multiply
        LAUNCH(ctx, k_mark_swept, grid_for(uint64_t(job.n_xl) * 32, 256, unsigned(ctx->sm_count) * 8u), 256, 0, c.op.a_pos,
               ctx->xl_list.as<uint32_t>(), ctx->d_sc, ctx->row_bin.as<uint64_t>(), job.sweep_min, ctx->swept.as<uint32_t>());
    }
    if (c.paths.sweep) {
        CU(ctx, ctx->lr_bands.reserve(c.lr_index_bytes()));
        LAUNCH(ctx, k_long_bands, grid_for(c.n_k * (c.lr_bands + 1), 256, 1u << 30), 256, 0, c.op.b_pos, c.op.b_data, c.n_k,
               uint32_t(LR_BAND), uint32_t(c.lr_bands), ctx->lr_bands.as<uint32_t>());
        c.job.bandptr = ctx->lr_bands.as<uint32_t>();
    }
    return OSP_OK;
}

struct Capacity {
    bool bounded = false;       // C is allocated below the plan's bound: every row block is admitted against c_cap
    uint64_t c_cap = 0;         // elements of C allocated up front
    uint64_t block_limit = 0;   // partial products of a row block
};

// ---- capacity of C.  The plan only knows the bound sum_i min(len_i, cols) of nnz(C).  On skewed inputs the bound
// is far above nnz(C) and can exceed the device (config 3 at full scale: 154 GB of bound next to 167 GB of partial
// products): then C gets what the device can spare, the call runs in small row blocks, and every block is admitted
// against that capacity with the exact nnz(C) of the blocks before it (carried by the merge chain anyway).
Capacity c_capacity(osp_ctx *ctx, const SpgemmCall &c) {
    const uint64_t limit_elems = std::max<uint64_t>(ctx->ws_limit / 8, 1);
    Capacity cap{false, c.cap_bound, limit_elems};
    if (c.paths.fused) return cap;
    const uint64_t P_bins = c.no_bins() ? 0 : c.P;
    if (ctx->result_limit) {
        cap.bounded = c.cap_bound * 8 > ctx->result_limit;
        if (cap.bounded) cap.c_cap = std::max<uint64_t>(ctx->result_limit / 8, 1);
    } else if ((c.cap_bound + std::min(P_bins, limit_elems)) * 8 > ctx->total_mem / 4) {      // small calls never ask the driver
        const uint64_t slack = (1ull << 30) + ctx->total_mem / 64;
        const uint64_t avail = device_available(ctx);
        auto bins_extra = [&](uint64_t elems) { const uint64_t b = std::min(P_bins, elems) * 8 + 16; return b > ctx->bins.cap ? b + b / 8 : 0; };
        if (c.cap_bound * 8 + bins_extra(limit_elems) + slack > avail) {
            cap.bounded = true;
            cap.block_limit = std::min<uint64_t>(limit_elems, std::max<uint64_t>(ctx->total_mem / 128, 1ull << 20));   // 1/16 of the device per block
            const uint64_t rest = bins_extra(cap.block_limit) + slack;
            cap.c_cap = std::min<uint64_t>(c.cap_bound, avail > rest ? (avail - rest) / 8 : 1);
        }
    }
    return cap;
}

// Where a row block starts: its first tile, row, bin offset and element of A.  A call of n blocks has n + 1 of them.
struct Block {
    uint32_t tile;
    uint64_t row, bin, elem;
};

// ---- row blocks, and the bins of the largest.  `h_row_bin` is the host copy of the bin offsets (blocked calls only).
int cut_row_blocks(osp_ctx *ctx, SpgemmCall &c, const Capacity &cap, std::vector<Block> &blocks, std::vector<uint64_t> &h_row_bin) {
    const uint32_t n_tiles = c.job.n_tiles;
    if (c.paths.fused || ((c.no_bins() ? 0 : c.P) <= cap.block_limit && !cap.bounded)) {
        blocks = {{0, 0, 0, 0}, {n_tiles, c.m_plan, c.paths.fused ? 0 : c.P, c.op.nnz_a}};
    } else {
        // blocks are row ranges: their tasks are taken in row order of A, whatever order the call asked for
        c.paths.rowwise = true;
        std::vector<uint32_t> h_tile_row(n_tiles + 1);
        std::vector<uint64_t> h_a_pos(c.m_a + 1);
        h_row_bin.resize(c.m_plan + 1);
        CU(ctx, cudaMemcpyAsync(h_tile_row.data(), ctx->tile_row.p, (n_tiles + 1) * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(ctx, cudaMemcpyAsync(h_row_bin.data(), ctx->row_bin.p, (c.m_plan + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(ctx, cudaMemcpyAsync(h_a_pos.data(), c.op.a_pos, (c.m_a + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        auto push = [&](uint32_t t) {
            const uint64_t r = h_tile_row[t];
            blocks.push_back({t, r, h_row_bin[r], h_a_pos[std::min(r, c.m_a)]});
        };
        push(0);
        uint32_t t = 0;
        while (t < n_tiles) {
            const uint64_t start = h_row_bin[h_tile_row[t]];
            uint32_t u = t + 1;
            while (u < n_tiles && h_row_bin[h_tile_row[u + 1]] - start <= cap.block_limit) u++;
            push(u);
            t = u;
        }
    }
    uint64_t max_block = 0;
    for (size_t b = 0; b + 1 < blocks.size(); b++) max_block = std::max(max_block, blocks[b + 1].bin - blocks[b].bin);
    CU(ctx, ctx->bins.reserve(std::max<uint64_t>(c.no_bins() ? 0 : max_block, 1) * 8 + 16));
    return OSP_OK;
}

// Fused dense rows, bank-aligned variant (osp_fusedlanes.cuh): B regrouped so that a warp's accumulator accesses never
// conflict.  Kept off when the regrouped B would be much larger than B (many columns of a row in one bank, or rows of B
// too short to fill a quad of groups): `ran` stays false.  OSP_FUSED_LANES=0: band kernel, =2: bank-aligned whatever the size.
int fused_rows_lanes(osp_ctx *ctx, SpgemmCall &c, osp_result *res, std::vector<cudaEvent_t> &ev_blocks, bool &ran) {
    ran = false;
    if (c.cols_b > FL_MAX_COLS || ctx->sw.fused_lanes_mode == 0) return OSP_OK;
    const Operands &op = c.op;
    MergeJob &job = c.job;
    const uint64_t n_k = c.n_k, m_plan = c.m_plan, cols_b = c.cols_b;
    CU(ctx, ctx->fl_meta.reserve(std::max<uint64_t>(n_k, 1) * sizeof(FlMeta)));
    FlMeta *meta = ctx->fl_meta.as<FlMeta>();
    const unsigned prep_grid = grid_for(n_k, FL_PREP_WARPS, unsigned(ctx->sm_count) * 8u);
    LAUNCH(ctx, k_fl_count, prep_grid, 32 * FL_PREP_WARPS, 0, op.b_pos, op.b_data, n_k, meta, ctx->d_sc);
    int rc = sync_scalars(ctx);
    if (rc) return rc;
    const uint64_t quads = ctx->h_sc->fl_quads;
    if (quads >= (1ull << 32) || (ctx->sw.fused_lanes_mode != 2 && quads * 128 > uint64_t(FL_MAX_BLOWUP) * op.nnz_b)) return OSP_OK;
    CU(ctx, ctx->fl_vals.reserve(std::max<uint64_t>(quads, 1) * 128 * 4));
    CU(ctx, ctx->fl_colb.reserve(std::max<uint64_t>(quads, 1) * 32 * 4));
    float *vals = ctx->fl_vals.as<float>();
    const float4 *vals4 = ctx->fl_vals.as<float4>();
    uint32_t *colb = ctx->fl_colb.as<uint32_t>();
    CU(ctx, cudaMemsetAsync(colb, fused_lanes_empty_byte(cols_b), std::max<uint64_t>(quads, 1) * 32 * 4, ctx->stream));   // every slot empty
    CU(ctx, cudaMemsetAsync(vals, 0, std::max<uint64_t>(quads, 1) * 128 * 4, ctx->stream));                                  // (the unused slots of a quad are loaded with it)
    LAUNCH(ctx, k_fl_fill, prep_grid, 32 * FL_PREP_WARPS, 0, op.b_pos, op.b_data, n_k, meta, vals, colb);
    CU(ctx, cudaMemsetAsync(ctx->tile_state.p, 0, (m_plan + 1) * 8, ctx->stream));
    CU(ctx, cudaMemsetAsync(&ctx->d_sc->tile_ticket, 0, 4, ctx->stream));
    ev_blocks.push_back(next_event(ctx));
    const int warps = fused_lanes_smem(cols_b, 2) <= 14336 ? 2 : 1;     // narrow rows: two per CTA (32 CTAs per SM at most)
    const size_t sm = fused_lanes_smem(cols_b, warps);
    int occ = 1;
    if (warps == 2) { CU(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_fused_lanes<2>, 64, sm)); }
    else { CU(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_fused_lanes<1>, 32, sm)); }
    const unsigned grid = unsigned(std::min<uint64_t>((m_plan + warps - 1) / warps, uint64_t(ctx->sm_count) * std::max(occ, 1)));
    // rows of C at the prefix of their bounds (no chain); C was allocated at the bound
    const bool direct = ctx->sw.fused_lanes_direct && job.c_cap >= c.cap_bound;
    uint32_t *row_cnt = nullptr;
    if (direct) {
        CU(ctx, ctx->fl_cnt.reserve(m_plan * 4));
        row_cnt = ctx->fl_cnt.as<uint32_t>();
        LAUNCH(ctx, (k_scan<RowCapIn, U64Out>), unsigned(c.st[3]), SCAN_BLOCK, 0, RowCapIn{ctx->row_bin.as<uint64_t>(), cols_b},
               U64Out{job.c_pos}, m_plan, c.ar.state[3], &ctx->d_sc->scan_ticket[3]);
    }
    if (warps == 2) {
        LAUNCH(ctx, k_fused_lanes<2>, grid, 64, sm, op.a_pos, op.a_data, c.m_a, meta, vals4, colb, uint32_t(cols_b), m_plan,
               ctx->tile_state.as<uint64_t>(), ctx->d_sc, job.c_pos, job.c_data, row_cnt);
    } else {
        LAUNCH(ctx, k_fused_lanes<1>, grid, 32, sm, op.a_pos, op.a_data, c.m_a, meta, vals4, colb, uint32_t(cols_b), m_plan,
               ctx->tile_state.as<uint64_t>(), ctx->d_sc, job.c_pos, job.c_data, row_cnt);
    }
    if (direct) {
        rc = sync_scalars(ctx);
        if (rc) return rc;
        const uint64_t nnz = ctx->h_sc->nnz_c[1];
        if (nnz != c.cap_bound) {
            // some row is not full: exact C.pos from the counts, rows moved into an exactly sized C
            CU(ctx, ctx->fl_pos2.reserve((m_plan + 1) * 8));
            uint64_t *pos2 = ctx->fl_pos2.as<uint64_t>();
            CU(ctx, cudaMemsetAsync(c.ar.state[3], 0, c.st[3] * 8, ctx->stream));
            CU(ctx, cudaMemsetAsync(&ctx->d_sc->scan_ticket[3], 0, 4, ctx->stream));
            LAUNCH(ctx, (k_scan<U32In, U64Out>), unsigned(c.st[3]), SCAN_BLOCK, 0, U32In{row_cnt}, U64Out{pos2}, m_plan, c.ar.state[3],
                   &ctx->d_sc->scan_ticket[3]);
            Elem *c2 = nullptr;
            if (cudaError_t e = cudaMallocAsync(reinterpret_cast<void **>(&c2), std::max<uint64_t>(nnz, 1) * 8, ctx->stream); e != cudaSuccess) {
                cudaGetLastError();
                return fail(ctx, OSP_ERR_OOM, std::string("result allocation (exact size): ") + cudaGetErrorString(e));
            }
            LAUNCH(ctx, k_fl_compact, grid_for(m_plan * 32, 256, unsigned(ctx->sm_count) * 16u), 256, 0, job.c_pos, pos2, job.c_data, c2, m_plan);
            CU(ctx, cudaMemcpyAsync(job.c_pos, pos2, (m_plan + 1) * 8, cudaMemcpyDeviceToDevice, ctx->stream));
            CU(ctx, cudaFreeAsync(res->d_data, ctx->stream));
            res->d_data = c2; job.c_data = c2; job.c_cap = std::max<uint64_t>(nnz, 1);
        }
    }
    ev_blocks.push_back(next_event(ctx));
    ran = true;
    return OSP_OK;
}

// Fused dense rows, band kernel (k_fused_dense).
int fused_rows_band(osp_ctx *ctx, SpgemmCall &c, std::vector<cudaEvent_t> &ev_blocks) {
    const Operands &op = c.op;
    const uint64_t n_k = c.n_k, m_plan = c.m_plan, cols_b = c.cols_b;
    const uint32_t band = uint32_t((cols_b + FD_WARPS - 1) / FD_WARPS);
    CU(ctx, ctx->tasks.reserve(n_k * (FD_WARPS + 1) * 4));                  // the band index of B
    uint32_t *bandptr = ctx->tasks.as<uint32_t>();
    LAUNCH(ctx, k_band_ptr, grid_for(n_k * (FD_WARPS + 1), 256, 1u << 30), 256, 0, op.b_pos, op.b_data, n_k, band, bandptr);
    CU(ctx, cudaMemsetAsync(ctx->tile_state.p, 0, (m_plan + 1) * 8, ctx->stream));
    CU(ctx, cudaMemsetAsync(&ctx->d_sc->tile_ticket, 0, 4, ctx->stream));
    ev_blocks.push_back(next_event(ctx));
    const size_t sm = fused_dense_smem(cols_b);
    int occ = 1;
    CU(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_fused_dense, FD_THREADS, sm));
    const unsigned grid = unsigned(std::min<uint64_t>(m_plan, uint64_t(ctx->sm_count) * std::max(occ, 1)));
    LAUNCH(ctx, k_fused_dense, grid, FD_THREADS, sm, op.a_pos, op.a_data, c.m_a, op.b_data, bandptr, uint32_t(cols_b), m_plan,
           ctx->tile_state.as<uint64_t>(), ctx->d_sc, c.job.c_pos, c.job.c_data);
    ev_blocks.push_back(next_event(ctx));
    return OSP_OK;
}

// Multiply into the bins and merge into C, row block by row block.
int run_blocks(osp_ctx *ctx, SpgemmCall &c, const Capacity &cap, const std::vector<Block> &blocks, const std::vector<uint64_t> &h_row_bin,
               cudaEvent_t ev_sym, std::vector<cudaEvent_t> &ev_blocks) {
    const size_t n_blocks = blocks.size() - 1;
    const Operands &op = c.op;
    const MergeJob &job = c.job;
    Elem *bins = ctx->bins.as<Elem>();
    for (size_t b = 0; b < n_blocks; b++) {
        const Block &lo = blocks[b], &hi = blocks[b + 1];
        const uint64_t p_block = hi.bin - lo.bin;
        int rc;
        if (cap.bounded) {
            // admit the block: nnz(C) of the blocks before it (exact) + this block's bound must fit C's capacity
            uint64_t carry = 0, bound_b = 0;
            if (b > 0) {
                rc = sync_scalars(ctx);
                if (rc) return rc;
                carry = ctx->h_sc->nnz_c[b & 1];
            }
            for (uint64_t r = lo.row; r < hi.row; r++) bound_b += std::min<uint64_t>(h_row_bin[r + 1] - h_row_bin[r], job.idx_range);
            if (carry + bound_b > cap.c_cap)
                return fail(ctx, OSP_ERR_OOM, "osp_spgemm: C does not fit the device: " + std::to_string(carry) + " non-zeros in the first " +
                                 std::to_string(b) + " of " + std::to_string(n_blocks) + " row blocks + a bound of " + std::to_string(bound_b) +
                                 " for the next exceed the capacity of " + std::to_string(cap.c_cap));
        }
        ev_blocks.push_back(b == 0 ? ev_sym : next_event(ctx));     // nothing is recorded between the hand-over and the multiply
        if (c.forked && b == 0) CU(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
        if (c.paths.rowwise && c.no_bins())
            rc = OSP_OK;                                                  // every tile is computed inside the chain
        else if (c.paths.rowwise && c.masked())
            rc = launch_multiply(ctx, TaskSrcSoASwept{TaskSrcSoA{op.a_data, c.run_off, c.task_bs}, ctx->swept.as<uint32_t>(), c.paths.fused_short ? 0u : 1u},
                                 lo.elem, hi.elem, p_block, op.b_data, bins, lo.bin);
        else if (c.paths.rowwise) rc = launch_multiply(ctx, TaskSrcSoA{op.a_data, c.run_off, c.task_bs}, lo.elem, hi.elem, p_block, op.b_data, bins, lo.bin);
        else rc = launch_multiply(ctx, TaskSrcAoS{ctx->tasks.as<Task>()}, 0, op.nnz_a, p_block, op.b_data, bins, lo.bin);
        if (rc) return rc;
        ev_blocks.push_back(next_event(ctx));
        rc = launch_merge(ctx, job, c.xl_ctas, bins, lo.bin, lo.tile, hi.tile, lo.row, hi.row, unsigned(b));
        if (rc) return rc;
        ev_blocks.push_back(next_event(ctx));
    }
    return OSP_OK;
}


// ---- .mtx text -> triplets in HBM (osp_readcoo_device, osp_mtx.cuh) ------------------------------------------------
// The text of a file or of the caller's memory.
struct MtxSource {
    const char *mem = nullptr;
    int fd = -1;
    uint64_t size = 0;
    bool read(uint64_t off, uint64_t n, char *dst) const {      // exactly n bytes at off
        if (mem) { std::memcpy(dst, mem + off, n); return true; }
        while (n) {
            const ssize_t k = pread(fd, dst, n, off_t(off));
            if (k < 0 && errno == EINTR) continue;
            if (k <= 0) return false;
            dst += k; off += uint64_t(k); n -= uint64_t(k);
        }
        return true;
    }
};

// The header as osp_readcoo_buffer finds it: the first line that is neither blank nor a comment.  Read a megabyte at a
// time until that line is complete, however long the comment block before it.  body = offset of the line after it,
// lines = lines up to there.
int mtx_header(osp_ctx *ctx, const MtxSource &src, uint64_t hdr[3], uint64_t &body, uint64_t &lines) {
    std::string buf;                  // text from buf_off on
    uint64_t buf_off = 0, at = 0;
    bool seen = false;
    body = lines = 0;
    while (at < src.size && !seen) {
        uint64_t nl;
        for (;;) {
            const size_t rel = buf.find('\n', size_t(at - buf_off));
            if (rel != std::string::npos) { nl = buf_off + rel; break; }
            const uint64_t have = buf_off + buf.size();
            if (have == src.size) { nl = src.size; break; }
            const uint64_t n = std::min<uint64_t>(1u << 20, src.size - have);
            const size_t old = buf.size();
            buf.resize(old + n);
            if (!src.read(have, n, &buf[old])) return fail(ctx, OSP_ERR_IO, "osp_readcoo_device: read error");
        }
        const std::string line = buf.substr(size_t(at - buf_off), size_t(nl - at));
        at = std::min<uint64_t>(nl + 1, src.size);
        lines++;
        seen = osp_mtx::header_line(line, hdr);
        buf.erase(0, size_t(at - buf_off));
        buf_off = at;
    }
    body = at;
    return OSP_OK;
}

// Scratch of one call from the stream-ordered pool, released however the call returns.
struct DevTemp {
    osp_ctx *ctx;
    void *p = nullptr;
    explicit DevTemp(osp_ctx *c) : ctx(c) {}
    ~DevTemp() { if (p) cudaFreeAsync(p, ctx->stream); }
    template <class T> T *as(uint64_t byte_off = 0) const { return reinterpret_cast<T *>(static_cast<char *>(p) + byte_off); }
};
int temp_alloc(osp_ctx *ctx, DevTemp &t, uint64_t bytes, const char *what) {
    const cudaError_t e = cudaMallocAsync(&t.p, std::max<uint64_t>(bytes, 16), ctx->stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        t.p = nullptr;
        return fail(ctx, OSP_ERR_OOM, std::string("osp_readcoo_device: ") + what + ": " + cudaGetErrorString(e));
    }
    return OSP_OK;
}

int read_scalars(osp_ctx *ctx, const MtxScalars *d, MtxScalars &h) {
    CU(ctx, cudaMemcpyAsync(&h, d, sizeof(MtxScalars), cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return OSP_OK;
}

// The body [body, src.size) into HBM: the caller's memory in one copy; a file through two pinned chunks, one filled by
// pread while the other is copied.
constexpr uint64_t MTX_STAGE_BYTES = 32ull << 20;
int upload_text(osp_ctx *ctx, const MtxSource &src, uint64_t body, uint64_t len, char *d_text) {
    if (src.mem) {
        CU(ctx, cudaMemcpyAsync(d_text, src.mem + body, len, cudaMemcpyHostToDevice, ctx->stream));
        return OSP_OK;
    }
    for (int i = 0; i < 2; i++) {
        if (!ctx->mtx_stage[i]) CU(ctx, cudaMallocHost(reinterpret_cast<void **>(&ctx->mtx_stage[i]), MTX_STAGE_BYTES));
        if (!ctx->mtx_copied[i]) CU(ctx, cudaEventCreateWithFlags(&ctx->mtx_copied[i], cudaEventDisableTiming));
    }
    for (uint64_t off = 0, k = 0; off < len; k++) {
        const uint64_t n = std::min(MTX_STAGE_BYTES, len - off);
        char *stage = ctx->mtx_stage[k & 1];
        CU(ctx, cudaEventSynchronize(ctx->mtx_copied[k & 1]));           // the copy out of this chunk is done
        if (!src.read(body + off, n, stage)) return fail(ctx, OSP_ERR_IO, "osp_readcoo_device: read error");
        CU(ctx, cudaMemcpyAsync(d_text + off, stage, n, cudaMemcpyHostToDevice, ctx->stream));
        CU(ctx, cudaEventRecord(ctx->mtx_copied[k & 1], ctx->stream));
        off += n;
    }
    return OSP_OK;
}

struct CooGuard {
    osp_coo *c;
    ~CooGuard() { if (c) osp_coo_free(c); }
};

// The triplets of osp_readcoo_buffer(text of src), bit for bit, built in HBM.
int mtx_ingest_impl(osp_ctx *ctx, const MtxSource &src, int symmetric, osp_coo **out) {
    uint64_t hdr[3] = {0, 0, 0}, body = 0, lines_before = 0;
    int rc = mtx_header(ctx, src, hdr, body, lines_before);
    if (rc) return rc;
    CooGuard guard{new osp_coo()};
    osp_coo *c = guard.c;
    c->ctx = ctx;
    c->nrow = hdr[0]; c->ncol = hdr[1]; c->nnz_header = hdr[2];
    const uint64_t len = src.size - body;
    if (len == 0) {
        *out = c;
        guard.c = nullptr;
        return OSP_OK;
    }
    // ---- the text, zero-padded to whole 16-byte words ----
    const uint64_t n_words = (len + 15) / 16, n_tiles = (len + MTX_TILE - 1) / MTX_TILE;
    DevTemp d_text(ctx), d_tiles(ctx), d_lines(ctx), d_slow(ctx);
    if ((rc = temp_alloc(ctx, d_text, n_words * 16, "text"))) return rc;
    if ((rc = upload_text(ctx, src, body, len, d_text.as<char>()))) return rc;
    if (n_words * 16 > len) CU(ctx, cudaMemsetAsync(d_text.as<char>(len), 0, n_words * 16 - len, ctx->stream));
    // ---- newlines: count per tile, scan, positions ----
    if ((rc = temp_alloc(ctx, d_tiles, n_tiles * 4 + (n_tiles + 1) * 8 + 16, "tile counts"))) return rc;
    uint32_t *tile_cnt = d_tiles.as<uint32_t>();
    uint64_t *tile_off = d_tiles.as<uint64_t>(align16(n_tiles * 4));
    Arena ar;
    const uint64_t st_tiles[4] = {scan_tiles(n_tiles), 0, 0, 0};
    if ((rc = prepare_arena(ctx, st_tiles, 0, ar))) return rc;
    LAUNCH(ctx, k_mtx_count_lines, unsigned(n_tiles), MTX_THREADS, 0, d_text.as<uint4>(), n_words, tile_cnt);
    LAUNCH(ctx, (k_scan<U32In, U64Out>), unsigned(scan_tiles(n_tiles)), SCAN_BLOCK, 0, U32In{tile_cnt}, U64Out{tile_off}, n_tiles,
           ar.state[0], &ctx->d_sc->scan_ticket[0]);
    uint64_t n_nl = 0;
    CU(ctx, cudaMemcpyAsync(&n_nl, tile_off + n_tiles, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    const uint64_t n_lines = n_nl + 1;                 // the last line ends at the end of the text (it may be empty)
    // per line: where it ends (8 bytes) and its entry count, then offset (4 bytes)
    if ((rc = temp_alloc(ctx, d_lines, align16(n_nl * 8) + (n_lines + 1) * 4, "line scratch"))) return rc;
    uint64_t *nl = d_lines.as<uint64_t>();
    uint32_t *cnt = d_lines.as<uint32_t>(align16(n_nl * 8));
    LAUNCH(ctx, k_mtx_line_ends, unsigned(n_tiles), MTX_THREADS, 0, d_text.as<uint4>(), n_words, tile_off, nl);
    const uint64_t st_lines[4] = {scan_tiles(n_lines), 0, 0, 0};
    if ((rc = prepare_arena(ctx, st_lines, sizeof(MtxScalars) / 4, ar))) return rc;
    MtxScalars *d_ms = reinterpret_cast<MtxScalars *>(ar.counters);
    const unsigned grid_lines = grid_for(n_lines, MTX_THREADS, unsigned(ctx->sm_count) * 16u);
    LAUNCH(ctx, k_mtx_parse, grid_lines, MTX_THREADS, 0, d_text.as<char>(), len, nl, n_nl, symmetric, cnt, d_ms);
    MtxScalars hs;
    if ((rc = read_scalars(ctx, d_ms, hs))) return rc;
    // ---- slow lines: read on the host with the C library, in file order ----
    const uint64_t n_slow = hs.n_slow;
    osp_mtx::Piece slow;
    std::vector<uint64_t> slow_line_ids(n_slow), slow_off(n_slow + 1, 0);
    if (n_slow) {
        if ((rc = temp_alloc(ctx, d_slow, n_slow * sizeof(MtxSlowLine), "slow lines"))) return rc;
        LAUNCH(ctx, k_mtx_slow_list, grid_lines, MTX_THREADS, 0, cnt, nl, n_nl, len, d_slow.as<MtxSlowLine>(), d_ms);
        std::vector<MtxSlowLine> lines(n_slow);
        CU(ctx, cudaMemcpyAsync(lines.data(), d_slow.p, n_slow * sizeof(MtxSlowLine), cudaMemcpyDeviceToHost, ctx->stream));
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        std::sort(lines.begin(), lines.end(), [](const MtxSlowLine &a, const MtxSlowLine &b) { return a.line < b.line; });
        std::string text;
        for (uint64_t j = 0; j < n_slow; j++) {
            text.resize(size_t(lines[j].end - lines[j].begin));
            if (!src.read(body + lines[j].begin, text.size(), &text[0])) return fail(ctx, OSP_ERR_IO, "osp_readcoo_device: read error");
            if (osp_mtx::slow_line(text, symmetric, slow))
                return fail(ctx, OSP_ERR_INVALID, "osp_readcoo_device: line " + std::to_string(lines_before + lines[j].line + 1) +
                                                      " is neither an entry \"row col [value]\", a blank line nor a comment");
            slow_line_ids[j] = lines[j].line;
            slow_off[j + 1] = slow.rows.size();
        }
    }
    const uint64_t n_se = slow.rows.size(), total = hs.entries + n_se;
    if (total >= (1ull << 32)) return fail(ctx, OSP_ERR_UNSUPPORTED, "osp_readcoo_device: 2^32 or more entries (the device conversion takes fewer)");
    DevTemp d_se(ctx);
    if (n_slow) {
        std::vector<uint32_t> counts(n_slow);
        for (uint64_t j = 0; j < n_slow; j++) counts[j] = uint32_t(slow_off[j + 1] - slow_off[j]);
        const uint64_t o_off = align16(n_slow * 8), o_cnt = o_off + align16((n_slow + 1) * 8), o_rows = o_cnt + align16(n_slow * 4),
                       o_cols = o_rows + align16(n_se * 4), o_vals = o_cols + align16(n_se * 4);
        if ((rc = temp_alloc(ctx, d_se, o_vals + n_se * 4, "slow entries"))) return rc;
        CU(ctx, cudaMemcpyAsync(d_se.p, slow_line_ids.data(), n_slow * 8, cudaMemcpyHostToDevice, ctx->stream));
        CU(ctx, cudaMemcpyAsync(d_se.as<char>(o_off), slow_off.data(), (n_slow + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
        CU(ctx, cudaMemcpyAsync(d_se.as<char>(o_cnt), counts.data(), n_slow * 4, cudaMemcpyHostToDevice, ctx->stream));
        if (n_se) {
            CU(ctx, cudaMemcpyAsync(d_se.as<char>(o_rows), slow.rows.data(), n_se * 4, cudaMemcpyHostToDevice, ctx->stream));
            CU(ctx, cudaMemcpyAsync(d_se.as<char>(o_cols), slow.cols.data(), n_se * 4, cudaMemcpyHostToDevice, ctx->stream));
            CU(ctx, cudaMemcpyAsync(d_se.as<char>(o_vals), slow.vals.data(), n_se * 4, cudaMemcpyHostToDevice, ctx->stream));
        }
        LAUNCH(ctx, k_mtx_slow_counts, grid_for(n_slow, 256, unsigned(ctx->sm_count) * 16u), 256, 0, d_se.as<uint64_t>(),
               d_se.as<uint32_t>(o_cnt), n_slow, cnt);
        CU(ctx, cudaStreamSynchronize(ctx->stream));           // the host vectors above are released on return
    }
    // ---- entries: scan of the per-line counts (in place), then the scatter ----
    LAUNCH(ctx, (k_scan<U32In, U32Out>), unsigned(scan_tiles(n_lines)), SCAN_BLOCK, 0, U32In{cnt}, U32Out{cnt}, n_lines, ar.state[0],
           &ctx->d_sc->scan_ticket[0]);
    if (total) {
        cudaError_t e = cudaMallocAsync(reinterpret_cast<void **>(&c->d_rows), total * 4, ctx->stream);
        if (e == cudaSuccess) e = cudaMallocAsync(reinterpret_cast<void **>(&c->d_cols), total * 4, ctx->stream);
        if (e == cudaSuccess) e = cudaMallocAsync(reinterpret_cast<void **>(&c->d_vals), total * 4, ctx->stream);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(ctx, OSP_ERR_OOM, std::string("osp_readcoo_device: triplet allocation: ") + cudaGetErrorString(e));
        }
        LAUNCH(ctx, k_mtx_scatter, grid_lines, MTX_THREADS, 0, d_text.as<char>(), len, nl, n_nl, symmetric, cnt, c->d_rows, c->d_cols,
               c->d_vals, d_ms);
        if (n_se) {
            const uint64_t o_off = align16(n_slow * 8), o_cnt = o_off + align16((n_slow + 1) * 8), o_rows = o_cnt + align16(n_slow * 4),
                           o_cols = o_rows + align16(n_se * 4), o_vals = o_cols + align16(n_se * 4);
            LAUNCH(ctx, k_mtx_scatter_slow, grid_for(n_slow, 256, unsigned(ctx->sm_count) * 16u), 256, 0, d_se.as<uint64_t>(),
                   d_se.as<uint64_t>(o_off), n_slow, d_se.as<uint32_t>(o_rows), d_se.as<uint32_t>(o_cols), d_se.as<float>(o_vals), cnt,
                   c->d_rows, c->d_cols, c->d_vals);
        }
        if ((rc = read_scalars(ctx, d_ms, hs))) return rc;
        c->max_row = hs.max_row; c->max_col = hs.max_col;
        for (uint64_t k = 0; k < n_se; k++) {
            c->max_row = std::max(c->max_row, slow.rows[k]);
            c->max_col = std::max(c->max_col, slow.cols[k]);
        }
    }
    c->d_nnz = total;
    *out = c;
    guard.c = nullptr;
    return OSP_OK;
}

// No C++ exception crosses the C ABI: a host allocation that fails (slow lines, header text) is OSP_ERR_OOM.
int mtx_ingest(osp_ctx *ctx, const MtxSource &src, int symmetric, osp_coo **out) {
    try {
        return mtx_ingest_impl(ctx, src, symmetric, out);
    } catch (const std::bad_alloc &) {
        return fail(ctx, OSP_ERR_OOM, "osp_readcoo_device: host allocation failed");
    }
}

}  // namespace

// A device-resident osp_coo (osp_host.cpp hands these two over for it).
int osp_coo_device_copy(const osp_coo *c, uint32_t *rows, uint32_t *cols, float *vals) {
    osp_ctx *ctx = c->ctx;
    const uint64_t n = c->d_nnz;
    if (n && (!rows || !cols || !vals)) return fail(ctx, OSP_ERR_INVALID, "osp_coo_copy: NULL argument");
    if (!n) return OSP_OK;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemcpyAsync(rows, c->d_rows, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaMemcpyAsync(cols, c->d_cols, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaMemcpyAsync(vals, c->d_vals, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return OSP_OK;
}

void osp_coo_device_free(osp_coo *c) {
    osp_ctx *ctx = c->ctx;
    cudaSetDevice(ctx->device);
    for (void *p : {static_cast<void *>(c->d_rows), static_cast<void *>(c->d_cols), static_cast<void *>(c->d_vals)})
        if (p) cudaFreeAsync(p, ctx->stream);
    c->d_rows = c->d_cols = nullptr;
    c->d_vals = nullptr;
}

// ========================================================================================
// C ABI
// ========================================================================================
extern "C" {

const char *osp_version(void) { return "outerspace_b200 0.2 (sm_100a)"; }

int osp_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

const char *osp_last_error(const osp_ctx *ctx) { return ctx ? ctx->err.c_str() : g_last_error.c_str(); }

int osp_create(int device, osp_ctx **out) {
    if (!out) return fail(nullptr, OSP_ERR_INVALID, "osp_create: out is NULL");
    *out = nullptr;
    int n = osp_device_count();
    if (n <= 0) return fail(nullptr, OSP_ERR_NO_DEVICE, "no CUDA device visible: this engine has no CPU fallback");
    if (device < 0 || device >= n) return fail(nullptr, OSP_ERR_INVALID, "osp_create: device index out of range");
    osp_ctx *ctx = new osp_ctx();
    ctx->device = device;
    struct CtxGuard { osp_ctx *c; ~CtxGuard() { if (c) osp_destroy(c); } } ctx_guard{ctx};   // every early return below releases it
    CU(nullptr, cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(nullptr, cudaGetDeviceProperties(&prop, device));
    ctx->sm_count = prop.multiProcessorCount;
    ctx->total_mem = prop.totalGlobalMem;
    if (prop.l2CacheSize > 0) ctx->l2_bytes = size_t(prop.l2CacheSize);
    CU(nullptr, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    {   // the side stream runs ahead of the main one where both have work (the owner's merge beside the peers' multiply)
        int prio_lo = 0, prio_hi = 0;
        if (cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi) != cudaSuccess) { cudaGetLastError(); prio_hi = 0; }
        CU(nullptr, cudaStreamCreateWithPriority(&ctx->stream2, cudaStreamNonBlocking, prio_hi));
    }
    CU(nullptr, cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
    CU(nullptr, cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
    CU(nullptr, cudaEventCreateWithFlags(&ctx->ev_half[0], cudaEventDisableTiming));
    CU(nullptr, cudaEventCreateWithFlags(&ctx->ev_half[1], cudaEventDisableTiming));
    CU(nullptr, cudaMallocHost(reinterpret_cast<void **>(&ctx->h_sc), sizeof(DevScalars)));
    if (!std::getenv("OSP_NO_MAPPED_SYNC")) {
        CU(nullptr, cudaHostAlloc(reinterpret_cast<void **>(&ctx->h_slots), sizeof(ulonglong2) * PUBLISH_SLOTS, cudaHostAllocMapped));
        std::memset(ctx->h_slots, 0, sizeof(ulonglong2) * PUBLISH_SLOTS);
        void *dv = nullptr;
        if (cudaHostGetDevicePointer(&dv, ctx->h_slots, 0) == cudaSuccess) ctx->h_slots_dev = static_cast<ulonglong2 *>(dv);
        else cudaGetLastError();
    }
    CU(nullptr, cudaFuncSetAttribute(k_merge_long, cudaFuncAttributeMaxDynamicSharedMemorySize, int(LONG_SMEM)));
    CU(nullptr, cudaFuncSetAttribute(k_merge_dense, cudaFuncAttributeMaxDynamicSharedMemorySize, int(dense_smem(DENSE_MAX_COLS))));
    CU(nullptr, cudaFuncSetAttribute(k_fused_dense, cudaFuncAttributeMaxDynamicSharedMemorySize, int(fused_dense_smem(DENSE_MAX_COLS))));
    CU(nullptr, cudaFuncSetAttribute(k_fused_lanes<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(fused_lanes_smem(FL_MAX_COLS, 1))));
    CU(nullptr, cudaFuncSetAttribute(k_fused_lanes<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(fused_lanes_smem(FL_MAX_COLS, 1))));
    CU(nullptr, cudaFuncSetAttribute(k_bias_relu, cudaFuncAttributeMaxDynamicSharedMemorySize, int(DENSE_MAX_COLS * 4 + 256)));
    {
        auto k32 = k_merge_chain<uint32_t, false>;
        auto k64 = k_merge_chain<uint64_t, false>;
        auto kbm = k_merge_chain<uint32_t, true>;
        CU(nullptr, cudaFuncSetAttribute(k32, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sizeof(MergeChainSmem<false>))));
        CU(nullptr, cudaFuncSetAttribute(k64, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sizeof(MergeChainSmem<false>))));
        CU(nullptr, cudaFuncSetAttribute(kbm, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sizeof(MergeChainSmem<true>))));
        // persistent grids: as many CTAs as can be resident
        CU(nullptr, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->chain_occ[0], k32, MC_THREADS, sizeof(MergeChainSmem<false>)));
        CU(nullptr, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->chain_occ[1], k64, MC_THREADS, sizeof(MergeChainSmem<false>)));
        CU(nullptr, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->chain_occ[2], kbm, MC_THREADS, sizeof(MergeChainSmem<true>)));
        for (int &o : ctx->chain_occ) o = std::max(o, 1);
    }
    {   // fused band sweep of the long rows: opt-in (include/osp_b200.h, OSP_LONGROW_SWEEP); a device that cannot give
        // it its shared memory simply never takes that path
        auto kfill = k_long_fill<LR_THREADS, LR_BAND, LR_RUNS, LongRowsInBins>;
        ctx->sweep_ok = cudaFuncSetAttribute(kfill, cudaFuncAttributeMaxDynamicSharedMemorySize, int(LR_SMEM)) == cudaSuccess &&
                        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->sweep_occ, kfill, LR_THREADS, LR_SMEM) == cudaSuccess &&
                        ctx->sweep_occ >= 1;
        if (!ctx->sweep_ok) { cudaGetLastError(); ctx->sweep_occ = 1; }
        const char *env = std::getenv("OSP_LONGROW_SWEEP");
        ctx->sw.sweep = env && env[0] && env[0] != '0';
        const char *kw = std::getenv("OSP_KWAY");
        ctx->sw.kway = kw && kw[0] && kw[0] != '0';
        if (const char *fl = std::getenv("OSP_FUSED_LANES")) ctx->sw.fused_lanes_mode = fl[0] == '0' ? 0 : fl[0] == '2' ? 2 : 1;
        if (const char *fd = std::getenv("OSP_FL_DIRECT")) ctx->sw.fused_lanes_direct = fd[0] != '0';
        if (const char *bp = std::getenv("OSP_BPOS32_MIN_KB")) ctx->sw.bpos32_min = std::strtoull(bp, nullptr, 10) << 10;
        if (const char *m = std::getenv("OSP_LONGROW_SWEEP_MIN")) ctx->sw.sweep_min = std::strtoull(m, nullptr, 10);
    }
    {   // OSP_FUSED_SHORT: opt-in as well
        auto f32 = k_merge_chain_fused<uint32_t, false>;
        auto f64 = k_merge_chain_fused<uint64_t, false>;
        auto fbm = k_merge_chain_fused<uint32_t, true>;
        ctx->fused_short_ok =
            cudaFuncSetAttribute(f32, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sizeof(MergeChainSmem<false>))) == cudaSuccess &&
            cudaFuncSetAttribute(f64, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sizeof(MergeChainSmem<false>))) == cudaSuccess &&
            cudaFuncSetAttribute(fbm, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sizeof(MergeChainSmem<true>))) == cudaSuccess &&
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->chain_fused_occ[0], f32, MC_THREADS, sizeof(MergeChainSmem<false>)) == cudaSuccess &&
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->chain_fused_occ[1], f64, MC_THREADS, sizeof(MergeChainSmem<false>)) == cudaSuccess &&
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->chain_fused_occ[2], fbm, MC_THREADS, sizeof(MergeChainSmem<true>)) == cudaSuccess;
        if (!ctx->fused_short_ok) cudaGetLastError();
        for (int &o : ctx->chain_fused_occ) o = std::max(o, 1);
        const char *env = std::getenv("OSP_FUSED_SHORT");
        ctx->sw.fused_short = env && env[0] && env[0] != '0';
    }
    {   // k_chain2: the warp-specialised implementation of the same path
        auto c32 = k_chain2<uint32_t, false, C2SrcProduct>;
        auto c64 = k_chain2<uint64_t, false, C2SrcProduct>;
        auto cbm = k_chain2<uint32_t, true, C2SrcProduct>;
        ctx->chain2_ok =
            cudaFuncSetAttribute(c32, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sizeof(Chain2Smem<false>))) == cudaSuccess &&
            cudaFuncSetAttribute(c64, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sizeof(Chain2Smem<false>))) == cudaSuccess &&
            cudaFuncSetAttribute(cbm, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sizeof(Chain2Smem<true>))) == cudaSuccess &&
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->chain2_occ[0], c32, C2_THREADS, sizeof(Chain2Smem<false>)) == cudaSuccess &&
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->chain2_occ[1], c64, C2_THREADS, sizeof(Chain2Smem<false>)) == cudaSuccess &&
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->chain2_occ[2], cbm, C2_THREADS, sizeof(Chain2Smem<true>)) == cudaSuccess &&
            ctx->chain2_occ[0] >= 1 && ctx->chain2_occ[1] >= 1 && ctx->chain2_occ[2] >= 1;
        if (!ctx->chain2_ok) cudaGetLastError();
        for (int &o : ctx->chain2_occ) o = std::max(o, 1);
        const char *env = std::getenv("OSP_FUSED_SHORT_OLD");
        ctx->sw.chain2_old = env && env[0] && env[0] != '0';
    }
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        uint64_t thr = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    ctx->ws_limit = uint64_t(double(ctx->total_mem) * 0.35);
    if (const char *env = std::getenv("OSP_WORKSPACE_LIMIT_MB")) {
        uint64_t mb = std::strtoull(env, nullptr, 10);
        if (mb) ctx->ws_limit = mb << 20;
    }
    ctx_guard.c = nullptr;
    *out = ctx;
    return OSP_OK;
}

void osp_destroy(osp_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (DevBuf *b : {&ctx->arena, &ctx->op_a_pos, &ctx->op_a_data, &ctx->op_b_pos, &ctx->op_b_data, &ctx->conv_pos,
                      &ctx->conv_data, &ctx->conv_tmp, &ctx->conv_chk, &ctx->task_bs, &ctx->run_off, &ctx->row_bin, &ctx->tile_row,
                      &ctx->tile_start, &ctx->long_list, &ctx->xl_list, &ctx->uniq, &ctx->col_ptr, &ctx->tasks, &ctx->tile_state,
                      &ctx->xl_acc, &ctx->xl_bits, &ctx->bins, &ctx->swept, &ctx->lr_bands, &ctx->kw_scratch, &ctx->vbits,
                      &ctx->fl_meta, &ctx->fl_vals, &ctx->fl_colb, &ctx->fl_cnt, &ctx->fl_pos2, &ctx->bpos32})
        b->release();
    for (cudaEvent_t e : ctx->events) cudaEventDestroy(e);
    for (int i = 0; i < 2; i++) {
        if (ctx->mtx_stage[i]) cudaFreeHost(ctx->mtx_stage[i]);
        if (ctx->mtx_copied[i]) cudaEventDestroy(ctx->mtx_copied[i]);
    }
    if (ctx->h_sc) cudaFreeHost(ctx->h_sc);
    if (ctx->h_slots) cudaFreeHost(ctx->h_slots);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    for (cudaEvent_t e : ctx->ev_half) if (e) cudaEventDestroy(e);
    if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int osp_set_workspace_limit(osp_ctx *ctx, uint64_t bytes) {
    if (!ctx || bytes < 4096) return fail(ctx, OSP_ERR_INVALID, "osp_set_workspace_limit: bad argument");
    ctx->ws_limit = bytes;
    return OSP_OK;
}

int osp_set_result_limit(osp_ctx *ctx, uint64_t bytes) {
    if (!ctx) return fail(ctx, OSP_ERR_INVALID, "osp_set_result_limit: NULL context");
    ctx->result_limit = bytes;
    return OSP_OK;
}

void *osp_stream(osp_ctx *ctx) { return ctx ? static_cast<void *>(ctx->stream) : nullptr; }

int osp_spgemm(osp_ctx *ctx, const osp_spgemm_args *args, osp_result **out) {
    if (!ctx || !args || !out) return fail(ctx, OSP_ERR_INVALID, "osp_spgemm: NULL argument");
    *out = nullptr;
    if (!args->a_pos || !args->b_pos) return fail(ctx, OSP_ERR_INVALID, "osp_spgemm: NULL pos array");
    const bool a_is_csr = args->flags & OSP_A_IS_CSR;
    // k-dimension check: lmat.NRow() == rmat.NRow(), SimOuterSPACE.cpp:47
    if (!a_is_csr && args->a_slices != args->n_k)
        return fail(ctx, OSP_ERR_INVALID, "osp_spgemm: CSC(A) and CSR(B) must have the same number of slices");
    if (args->n_k >= (1ull << 32) || args->a_slices >= (1ull << 32) || args->rows_c >= (1ull << 32) ||
        args->cols_b >= (1ull << 32))
        return fail(ctx, OSP_ERR_INVALID, "osp_spgemm: dimensions must fit index_t (uint32)");
    int rc = begin_call(ctx, args->flags);
    if (rc) return rc;
    SpgemmCall c;
    c.args = args;
    c.validate = !(args->flags & OSP_NO_VALIDATE);
    c.n_k = args->n_k;
    rc = stage_operands(ctx, args, c.op);
    if (rc) return rc;
    cudaEvent_t ev_begin = next_event(ctx);
    c.m_a = args->a_slices;
    if (!a_is_csr) {
        rc = convert_a(ctx, c);
        if (rc) return rc;
    }
    c.m_plan = std::max<uint64_t>({c.m_a, args->rows_c, 1});
    c.cols_b = args->cols_b;
    c.paths = choose_paths(ctx, args, c.op.nnz_a, c.op.nnz_b, c.m_a);
    rc = launch_symbolic_and_plan(ctx, c);
    if (rc) return rc;
    cudaEvent_t ev_sym = next_event(ctx);
    // C.pos is allocated while the device is still busy with the symbolic pass and the plan
    PendingResult res(ctx);
    rc = alloc_result(ctx, res.r, c.m_plan + 1, 0);
    if (rc) return rc;
    rc = take_hand_over(ctx, c);
    if (rc) return rc;
    rc = launch_task_bitmap(ctx, c);
    if (rc) return rc;
    const Capacity cap = c_capacity(ctx, c);
    rc = alloc_result(ctx, res.r, 0, cap.c_cap);
    if (rc) return rc;
    c.job.c_pos = res->d_pos; c.job.c_data = res->d_data; c.job.c_cap = cap.c_cap;
    std::vector<Block> blocks;
    std::vector<uint64_t> h_row_bin;
    rc = cut_row_blocks(ctx, c, cap, blocks, h_row_bin);
    if (rc) return rc;
    std::vector<cudaEvent_t> ev_blocks;   // 3 per block: start, after multiply, after merge
    if (c.paths.fused) {
        ev_blocks.push_back(next_event(ctx));
        CU(ctx, ctx->tile_state.reserve((c.m_plan + 1) * 8));
        bool lanes = false;
        rc = fused_rows_lanes(ctx, c, res.r, ev_blocks, lanes);
        if (!rc && !lanes) rc = fused_rows_band(ctx, c, ev_blocks);
    } else {
        rc = run_blocks(ctx, c, cap, blocks, h_row_bin, ev_sym, ev_blocks);
    }
    if (rc) return rc;
    cudaEvent_t ev_end = next_event(ctx);
    rc = sync_scalars(ctx);
    if (rc) return rc;
    if (ctx->h_sc->err) return fail(ctx, OSP_ERR_CUDA, "osp_spgemm: internal capacity check failed on the device");
    const size_t n_blocks = blocks.size() - 1;
    const uint64_t nnz_a = c.op.nnz_a, nnz_b = c.op.nnz_b, n_k = c.n_k, P = c.P, nnz_c = ctx->h_sc->nnz_c[n_blocks & 1];
    res->rows = c.rows_c;
    res->nnz = nnz_c;
    osp_stats &stt = res->stats;
    stt.rows_c = c.rows_c; stt.cols_b = c.cols_b; stt.n_k = n_k;
    stt.nnz_a = nnz_a; stt.nnz_b = nnz_b; stt.nnz_c = nnz_c; stt.products = P;
    stt.algorithmic_bytes = 16 * P + 8 * nnz_c + 24 * nnz_a + 8 * nnz_b + 8 * (2 * c.rows_c + 3 * n_k + 5);
    stt.rows_medium = c.job.n_long; stt.rows_long = c.job.n_xl; stt.merge_tiles = c.job.n_tiles;
    stt.kernel_launches = ctx->launches;
    stt.row_chunks = n_blocks;
    stt.ms_h2d = c.op.ms_h2d;
    res->spans.push_back({&stt.ms_total, nullptr, ev_begin, ev_end});
    res->spans.push_back({&stt.ms_convert, nullptr, ev_begin, ev_sym});
    for (size_t b = 0; b < n_blocks; b++) {
        res->spans.push_back({&stt.ms_multiply, nullptr, ev_blocks[3 * b], ev_blocks[3 * b + 1]});
        res->spans.push_back({&stt.ms_merge, nullptr, ev_blocks[3 * b + 1], ev_blocks[3 * b + 2]});
    }
    return finish_result(ctx, res, out);
}

int osp_result_kernels(const osp_result *r, uint64_t *n, const char **names, float *ms) {
    if (!r || !n) return fail(nullptr, OSP_ERR_INVALID, "osp_result_kernels: NULL argument");
    resolve_times(const_cast<osp_result *>(r));
    if (names && ms)
        for (size_t i = 0; i < r->kernel_ms.size() && i < *n; i++) { names[i] = r->kernel_ms[i].first; ms[i] = r->kernel_ms[i].second; }
    *n = r->kernel_ms.size();
    return OSP_OK;
}

int osp_result_dims(const osp_result *r, uint64_t *rows, uint64_t *nnz) {
    if (!r) return fail(nullptr, OSP_ERR_INVALID, "osp_result_dims: NULL result");
    if (rows) *rows = r->rows;
    if (nnz) *nnz = r->nnz;
    return OSP_OK;
}

int osp_result_copy(osp_result *r, uint64_t *pos, void *data) {
    if (!r || !pos) return fail(nullptr, OSP_ERR_INVALID, "osp_result_copy: NULL argument");
    osp_ctx *ctx = r->ctx;
    if (r->nnz && !data) return fail(ctx, OSP_ERR_INVALID, "osp_result_copy: NULL data");
    CU(ctx, cudaSetDevice(ctx->device));
    cudaEvent_t e0 = next_event(ctx);
    CU(ctx, cudaMemcpyAsync(pos, r->d_pos, (r->rows + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (r->nnz) CU(ctx, cudaMemcpyAsync(data, r->d_data, r->nnz * 8, cudaMemcpyDeviceToHost, ctx->stream));
    cudaEvent_t e1 = next_event(ctx);
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    cudaEventElapsedTime(&r->stats.ms_d2h, e0, e1);
    return OSP_OK;
}

int osp_result_copy_rows(osp_result *r, uint64_t row_begin, uint64_t row_end, uint64_t *pos, void *data, uint64_t data_capacity) {
    if (!r || !pos) return fail(nullptr, OSP_ERR_INVALID, "osp_result_copy_rows: NULL argument");
    osp_ctx *ctx = r->ctx;
    if (row_begin > row_end || row_end > r->rows) return fail(ctx, OSP_ERR_INDEX, "osp_result_copy_rows: row range outside C");
    CU(ctx, cudaSetDevice(ctx->device));
    const uint64_t n = row_end - row_begin;
    CU(ctx, cudaMemcpyAsync(pos, r->d_pos + row_begin, (n + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    const uint64_t cnt = pos[n] - pos[0];
    if (!data) return OSP_OK;
    if (cnt > data_capacity) return fail(ctx, OSP_ERR_INVALID, "osp_result_copy_rows: data_capacity is smaller than the rows' non-zeros");
    if (cnt) {
        CU(ctx, cudaMemcpyAsync(data, r->d_data + pos[0], cnt * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return OSP_OK;
}

int osp_result_device(const osp_result *r, const uint64_t **d_pos, const void **d_data) {
    if (!r) return fail(nullptr, OSP_ERR_INVALID, "osp_result_device: NULL result");
    if (d_pos) *d_pos = r->d_pos;
    if (d_data) *d_data = r->d_data;
    return OSP_OK;
}

int osp_result_stats(const osp_result *r, osp_stats *stats) {
    if (!r || !stats) return fail(nullptr, OSP_ERR_INVALID, "osp_result_stats: NULL argument");
    resolve_times(const_cast<osp_result *>(r));
    *stats = r->stats;
    return OSP_OK;
}

void osp_result_free(osp_result *r) {
    if (!r) return;
    osp_ctx *ctx = r->ctx;
    cudaSetDevice(ctx->device);
    if (r->d_pos) cudaFreeAsync(r->d_pos, ctx->stream);
    if (r->d_data) cudaFreeAsync(r->d_data, ctx->stream);
    delete r;
}

// Sizes the reference's timing models read from TaskProvider (SimOuterSPACE.cpp:34-42,59-64), derived
// from the operand structure and the result's row pointer (host arithmetic on sizes only; no values).
int osp_task_sizes(osp_ctx *ctx, const osp_spgemm_args *args, const osp_result *r, uint64_t *n_multiply,
                   uint32_t *multiply_nnzc_nnzr, uint64_t *n_merge, uint32_t *merge_ways_out) {
    if (!ctx || !args || !r || !n_multiply || !n_merge) return fail(ctx, OSP_ERR_INVALID, "osp_task_sizes: NULL argument");
    const bool a_is_csr = args->flags & OSP_A_IS_CSR;
    const bool on_device = args->flags & OSP_DEVICE_POINTERS;
    const uint64_t n_k = args->n_k, a_slices = args->a_slices;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    std::vector<uint64_t> a_pos(a_slices + 1), b_pos(n_k + 1), c_pos(r->rows + 1);
    cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToHost : cudaMemcpyHostToHost;
    CU(ctx, cudaMemcpy(a_pos.data(), args->a_pos, (a_slices + 1) * 8, kind));
    CU(ctx, cudaMemcpy(b_pos.data(), args->b_pos, (n_k + 1) * 8, kind));
    CU(ctx, cudaMemcpy(c_pos.data(), r->d_pos, (r->rows + 1) * 8, cudaMemcpyDeviceToHost));
    const uint64_t nnz_a = a_pos[a_slices];
    std::vector<Elem> a_data(nnz_a);
    if (nnz_a) CU(ctx, cudaMemcpy(a_data.data(), args->a_data, nnz_a * 8, kind));
    std::vector<uint32_t> nnzc(n_k, 0), ways(r->rows, 0);
    if (a_is_csr) {
        for (uint64_t i = 0; i < a_slices; i++)
            for (uint64_t e = a_pos[i]; e < a_pos[i + 1]; e++) {
                uint32_t k = a_data[e].idx;
                if (k >= n_k) return fail(ctx, OSP_ERR_INDEX, "osp_task_sizes: index out of range");
                nnzc[k]++;
                if (b_pos[k + 1] > b_pos[k] && i < r->rows) ways[i]++;
            }
    } else {
        for (uint64_t k = 0; k < n_k; k++) {
            nnzc[k] = uint32_t(a_pos[k + 1] - a_pos[k]);
            if (b_pos[k + 1] > b_pos[k])
                for (uint64_t e = a_pos[k]; e < a_pos[k + 1]; e++)
                    if (a_data[e].idx < r->rows) ways[a_data[e].idx]++;
        }
    }
    uint64_t nm = 0;
    for (uint64_t k = 0; k < n_k; k++) {
        uint64_t nnzr = b_pos[k + 1] - b_pos[k];
        if (!nnzc[k] || !nnzr) continue;                       // skipped slices, SimOuterSPACE.cpp:82-83
        if (multiply_nnzc_nnzr) { multiply_nnzc_nnzr[2 * nm] = nnzc[k]; multiply_nnzc_nnzr[2 * nm + 1] = uint32_t(nnzr); }
        nm++;
    }
    *n_multiply = nm;
    *n_merge = r->rows;                                        // one MergeTask per row, empty rows included (:128)
    if (merge_ways_out)
        for (uint64_t i = 0; i < r->rows; i++) {
            merge_ways_out[2 * i] = ways[i];
            merge_ways_out[2 * i + 1] = uint32_t(c_pos[i + 1] - c_pos[i]);
        }
    return OSP_OK;
}

int osp_csr2csc(osp_ctx *ctx, uint64_t n_major, uint64_t n_minor, const uint64_t *pos, const void *data, uint32_t flags,
                uint64_t *pos_out, void *data_out) {
    if (!ctx || !pos || !pos_out) return fail(ctx, OSP_ERR_INVALID, "osp_csr2csc: NULL argument");
    if (n_major >= (1ull << 32) || n_minor >= (1ull << 32))
        return fail(ctx, OSP_ERR_INVALID, "osp_csr2csc: dimensions must fit index_t (uint32)");
    int rc = begin_call(ctx, 0);
    if (rc) return rc;
    if (flags & OSP_DEVICE_POINTERS) {
        uint64_t nnz = 0;
        CU(ctx, cudaMemcpyAsync(&nnz, pos + n_major, 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        return csr2csc_device(ctx, n_major, n_minor, pos, static_cast<const Elem *>(data), nnz, pos_out,
                              static_cast<Elem *>(data_out));
    }
    uint64_t nnz = pos[n_major];
    if (nnz && (!data || !data_out)) return fail(ctx, OSP_ERR_INVALID, "osp_csr2csc: NULL data");
    CU(ctx, ctx->op_a_pos.reserve((n_major + 1) * 8));
    CU(ctx, ctx->op_a_data.reserve(std::max<uint64_t>(nnz, 1) * 8));
    CU(ctx, ctx->conv_pos.reserve((n_minor + 1) * 8));
    CU(ctx, ctx->conv_data.reserve(std::max<uint64_t>(nnz, 1) * 8));
    CU(ctx, cudaMemcpyAsync(ctx->op_a_pos.p, pos, (n_major + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    if (nnz) CU(ctx, cudaMemcpyAsync(ctx->op_a_data.p, data, nnz * 8, cudaMemcpyHostToDevice, ctx->stream));
    rc = csr2csc_device(ctx, n_major, n_minor, ctx->op_a_pos.as<uint64_t>(), ctx->op_a_data.as<Elem>(), nnz,
                        ctx->conv_pos.as<uint64_t>(), ctx->conv_data.as<Elem>());
    if (rc) return rc;
    CU(ctx, cudaMemcpyAsync(pos_out, ctx->conv_pos.p, (n_minor + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (nnz) CU(ctx, cudaMemcpyAsync(data_out, ctx->conv_data.p, nnz * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return OSP_OK;
}

// relu(C + bias) kept sparse (SURVEY 8f rank 3): the step between two layers of the reference's MLP.
int osp_bias_relu(osp_ctx *ctx, const osp_result *c, uint64_t cols, const float *bias, uint32_t flags, osp_result **out) {
    if (!ctx || !c || !out) return fail(ctx, OSP_ERR_INVALID, "osp_bias_relu: NULL argument");
    *out = nullptr;
    if (cols == 0 || cols > DENSE_MAX_COLS) return fail(ctx, OSP_ERR_UNSUPPORTED, "osp_bias_relu: the row is densified in shared memory: 1 <= cols <= 16384");
    if (c->rows >= (1ull << 32)) return fail(ctx, OSP_ERR_INVALID, "osp_bias_relu: too many rows");
    int rc = begin_call(ctx, 0);
    if (rc) return rc;
    const uint64_t rows = c->rows;
    Arena ar;
    const uint64_t st0[4] = {0, 0, 0, 0};
    rc = prepare_arena(ctx, st0, 0, ar);
    if (rc) return rc;
    const float *d_bias = bias;
    if (bias && !(flags & OSP_DEVICE_POINTERS)) {
        CU(ctx, ctx->op_a_data.reserve(cols * 4));
        CU(ctx, cudaMemcpyAsync(ctx->op_a_data.p, bias, cols * 4, cudaMemcpyHostToDevice, ctx->stream));
        d_bias = ctx->op_a_data.as<float>();
    }
    PendingResult res(ctx);
    rc = alloc_result(ctx, res.r, rows + 1, std::max<uint64_t>(bias ? rows * cols : c->nnz, 1));
    if (rc) return rc;
    cudaEvent_t ev0 = next_event(ctx);
    if (rows == 0) {
        CU(ctx, cudaMemsetAsync(res->d_pos, 0, 8, ctx->stream));
    } else {
        CU(ctx, ctx->tile_state.reserve((rows + 1) * 8));
        CU(ctx, cudaMemsetAsync(ctx->tile_state.p, 0, (rows + 1) * 8, ctx->stream));
        const size_t sm = size_t((cols + 15) & ~15ull) * 4 + 64 * 4;
        int occ = 1;
        CU(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_bias_relu, BR_THREADS, sm));
        const unsigned grid = unsigned(std::min<uint64_t>(rows, uint64_t(ctx->sm_count) * std::max(occ, 1)));
        LAUNCH(ctx, k_bias_relu, grid, BR_THREADS, sm, c->d_pos, c->d_data, rows, uint32_t(cols), d_bias,
               ctx->tile_state.as<uint64_t>(), ctx->d_sc, res->d_pos, res->d_data);
    }
    res->spans.push_back({&res->stats.ms_total, nullptr, ev0, next_event(ctx)});
    rc = sync_scalars(ctx);
    if (rc) return rc;
    if (ctx->h_sc->err) return fail(ctx, OSP_ERR_INDEX, "osp_bias_relu: a column id of C is not below cols");
    res->rows = rows;
    res->nnz = rows ? ctx->h_sc->nnz_c[1] : 0;
    res->stats.rows_c = rows; res->stats.cols_b = cols; res->stats.nnz_c = res->nnz;
    res->stats.kernel_launches = ctx->launches;
    return finish_result(ctx, res, out);
}

// COO -> CSR / CSC on the device (SURVEY 8f rank 2): coo2csr<transpose> + dupcheck, SimSpGEMM.cpp:43-53,102-152.
int osp_coo2csr_device(osp_ctx *ctx, uint64_t nnz, const uint32_t *rows, const uint32_t *cols, const float *vals, uint64_t N,
                       uint64_t n_other, int transpose, uint32_t flags, uint64_t *pos, void *data) {
    if (!ctx || !pos || (nnz && (!rows || !cols || !vals || !data)))
        return fail(ctx, OSP_ERR_INVALID, "osp_coo2csr_device: NULL argument");
    if (N >= (1ull << 32) || n_other >= (1ull << 32) || nnz >= (1ull << 32))
        return fail(ctx, OSP_ERR_INVALID, "osp_coo2csr_device: dimensions must fit index_t (uint32)");
    int rc = begin_call(ctx, 0);
    if (rc) return rc;
    const uint32_t *major = transpose ? cols : rows, *minor = transpose ? rows : cols;
    if (flags & OSP_DEVICE_POINTERS) {
        if (!n_other) return fail(ctx, OSP_ERR_INVALID, "osp_coo2csr_device: the range of the other index is required with device pointers");
        CooSrc src{major, minor, vals};
        return csr2csc_device(ctx, n_other, N, nullptr, nullptr, nnz, pos, static_cast<Elem *>(data), &src);
    }
    if (!n_other)
        for (uint64_t i = 0; i < nnz; i++) n_other = std::max<uint64_t>(n_other, uint64_t(minor[i]) + 1);
    n_other = std::max<uint64_t>(n_other, 1);
    CU(ctx, ctx->op_a_pos.reserve(std::max<uint64_t>(nnz, 1) * 4));
    CU(ctx, ctx->op_b_pos.reserve(std::max<uint64_t>(nnz, 1) * 4));
    CU(ctx, ctx->op_a_data.reserve(std::max<uint64_t>(nnz, 1) * 4));
    CU(ctx, ctx->conv_pos.reserve((N + 1) * 8));
    CU(ctx, ctx->conv_data.reserve(std::max<uint64_t>(nnz, 1) * 8));
    if (nnz) {
        CU(ctx, cudaMemcpyAsync(ctx->op_a_pos.p, major, nnz * 4, cudaMemcpyHostToDevice, ctx->stream));
        CU(ctx, cudaMemcpyAsync(ctx->op_b_pos.p, minor, nnz * 4, cudaMemcpyHostToDevice, ctx->stream));
        CU(ctx, cudaMemcpyAsync(ctx->op_a_data.p, vals, nnz * 4, cudaMemcpyHostToDevice, ctx->stream));
    }
    CooSrc src{ctx->op_a_pos.as<uint32_t>(), ctx->op_b_pos.as<uint32_t>(), ctx->op_a_data.as<float>()};
    rc = csr2csc_device(ctx, n_other, N, nullptr, nullptr, nnz, ctx->conv_pos.as<uint64_t>(), ctx->conv_data.as<Elem>(), &src);
    if (rc) return rc;
    CU(ctx, cudaMemcpyAsync(pos, ctx->conv_pos.p, (N + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (nnz) CU(ctx, cudaMemcpyAsync(data, ctx->conv_data.p, nnz * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return OSP_OK;
}

// .mtx ingest on the device (SURVEY 8f rank 2): readcoo (SimSpGEMM.cpp:55-100) with the text parsed in HBM.
int osp_readcoo_device(osp_ctx *ctx, const char *path, int symmetric, osp_coo **out) {
    if (!ctx || !path || !out) return fail(ctx, OSP_ERR_INVALID, "osp_readcoo_device: NULL argument");
    *out = nullptr;
    int rc = begin_call(ctx, 0);
    if (rc) return rc;
    struct Fd { int fd; ~Fd() { if (fd >= 0) close(fd); } } f{open(path, O_RDONLY)};
    if (f.fd < 0) return fail(ctx, OSP_ERR_IO, std::string("osp_readcoo_device: cannot open ") + path);
    struct stat st;
    if (fstat(f.fd, &st) != 0) return fail(ctx, OSP_ERR_IO, std::string("osp_readcoo_device: cannot stat ") + path);
    MtxSource src;
    src.fd = f.fd;
    src.size = uint64_t(st.st_size);
    return mtx_ingest(ctx, src, symmetric, out);
}

int osp_readcoo_buffer_device(osp_ctx *ctx, const char *text, uint64_t len, int symmetric, osp_coo **out) {
    if (!ctx || (!text && len) || !out) return fail(ctx, OSP_ERR_INVALID, "osp_readcoo_buffer_device: NULL argument");
    *out = nullptr;
    int rc = begin_call(ctx, 0);
    if (rc) return rc;
    MtxSource src;
    src.mem = text;
    src.size = len;
    return mtx_ingest(ctx, src, symmetric, out);
}

int osp_coo_device(const osp_coo *c, const uint32_t **rows, const uint32_t **cols, const float **vals) {
    if (!c) return fail(nullptr, OSP_ERR_INVALID, "osp_coo_device: NULL argument");
    if (!c->ctx) return fail(nullptr, OSP_ERR_INVALID, "osp_coo_device: the triplets are on the host (osp_readcoo)");
    if (rows) *rows = c->d_rows;
    if (cols) *cols = c->d_cols;
    if (vals) *vals = c->d_vals;
    return OSP_OK;
}

// coo2csr<transpose> + dupcheck of device triplets into a device CSR (osp_coo2csr's errors and bytes).
int osp_coo2csr_result(osp_ctx *ctx, const osp_coo *c, uint64_t N, int transpose, osp_result **out) {
    if (!ctx || !c || !out) return fail(ctx, OSP_ERR_INVALID, "osp_coo2csr_result: NULL argument");
    *out = nullptr;
    if (c->ctx != ctx) return fail(ctx, OSP_ERR_INVALID, "osp_coo2csr_result: the triplets are not in this context's device memory");
    if (N >= (1ull << 32)) return fail(ctx, OSP_ERR_INVALID, "osp_coo2csr_result: dimensions must fit index_t (uint32)");
    int rc = begin_call(ctx, 0);
    if (rc) return rc;
    const uint64_t nnz = c->d_nnz;
    // the other index's range from the maxima recorded by the ingest
    const uint64_t n_other = nnz ? uint64_t(transpose ? c->max_row : c->max_col) + 1 : 1;
    PendingResult res(ctx);
    rc = alloc_result(ctx, res.r, N + 1, std::max<uint64_t>(nnz, 1));
    if (rc) return rc;
    cudaEvent_t ev0 = next_event(ctx);
    CooSrc src{transpose ? c->d_cols : c->d_rows, transpose ? c->d_rows : c->d_cols, c->d_vals};
    rc = csr2csc_device(ctx, n_other, N, nullptr, nullptr, nnz, res->d_pos, res->d_data, &src);
    if (rc) return rc;
    res->spans.push_back({&res->stats.ms_total, nullptr, ev0, next_event(ctx)});
    res->rows = N;
    res->nnz = nnz;
    res->stats.rows_c = N; res->stats.cols_b = n_other; res->stats.nnz_c = nnz;
    res->stats.kernel_launches = ctx->launches;
    return finish_result(ctx, res, out);
}

}  // extern "C"

#ifndef OSP_CUSIM            // the multi-GPU path needs peers and NCCL: not part of the emulated build
#include "osp_dist.inl"
#endif

// cusim.h -- a small CPU emulation of the CUDA execution model, for TESTS ONLY.
//
// It lets a kernel written in plain CUDA C++ (no inline PTX) run on the host so that its logic -- index arithmetic,
// barrier structure, warp collectives, arbitration loops -- can be checked against the oracle in the `-m "not gpu"`
// suite, where no GPU exists.  It is NOT a product path and nothing under outerspace_b200/ links it: the kernels are
// compiled by nvcc for sm_100a as always; a test translation unit defines OSP_CUSIM, includes this header instead of
// <cuda_runtime.h>, and calls cusim::launch().
//
// Model: the threads of a block are fibers scheduled round-robin on one OS thread, switching only inside the
// synchronising built-ins (__syncthreads*, warp collectives, __nanosleep).  That is a legal CUDA schedule, so a kernel
// that is correct under every schedule is correct here; the reverse does not hold (data races between barriers go
// unnoticed), which is why GPU parity tests stay the gate.
// Blocks: CUSIM_RESIDENT (default 1) blocks are resident at a time, each on its own OS thread, the next block of the
// grid starting when a resident one retires -- like CTAs on SMs.  With 1 the blocks of a launch run one after the
// other (a persistent kernel takes all its tickets in the first block); with more, blocks really run concurrently:
// tickets interleave, decoupled look-back chains wait on live predecessors, global atomics are real atomics.  Static
// __shared__ variables are thread-local statics (one copy per resident block).
#pragma once
#if !defined(__x86_64__)
#include <ucontext.h>
#endif

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <atomic>
#include <chrono>
#include <memory>
#include <thread>
#include <vector>

#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __noinline__
#define __shared__ static thread_local
#define __launch_bounds__(...)
#define __align__(n) __attribute__((aligned(n)))

struct dim3 {
    unsigned x, y, z;
    dim3(unsigned x_ = 1, unsigned y_ = 1, unsigned z_ = 1) : x(x_), y(y_), z(z_) {}
};
inline thread_local dim3 threadIdx, blockIdx;
inline dim3 blockDim, gridDim;

struct uint2 { unsigned x, y; };
struct alignas(16) uint4 { unsigned x, y, z, w; };
struct alignas(16) ulonglong2 { unsigned long long x, y; };
struct alignas(16) float4 { float x, y, z, w; };
inline uint2 make_uint2(unsigned x, unsigned y) { return uint2{x, y}; }
inline uint4 make_uint4(unsigned x, unsigned y, unsigned z, unsigned w) { return uint4{x, y, z, w}; }

namespace cusim {

// Context switch.  On x86-64 a dozen instructions (callee-saved registers + stack pointer): swapcontext() makes two
// signal-mask system calls per switch, and a barrier of a 512-thread block is 512 switches.
#if defined(__x86_64__)
extern "C" void cusim_swap(void **save_sp, void *load_sp);
asm(R"(
    .text
    .type cusim_swap,@function
cusim_swap:
    pushq %rbp
    pushq %rbx
    pushq %r12
    pushq %r13
    pushq %r14
    pushq %r15
    movq %rsp, (%rdi)
    movq %rsi, %rsp
    popq %r15
    popq %r14
    popq %r13
    popq %r12
    popq %rbx
    popq %rbp
    ret
    .size cusim_swap, .-cusim_swap
)");
struct Context {
    void *sp = nullptr;
    void prepare(char *stack, size_t bytes, void (*entry)()) {
        uintptr_t top = (reinterpret_cast<uintptr_t>(stack) + bytes) & ~uintptr_t(15);
        void **p = reinterpret_cast<void **>(top);
        *--p = nullptr;                                   // return address of `entry` (never used: entry does not return)
        *--p = reinterpret_cast<void *>(entry);           // popped by the first `ret`
        for (int i = 0; i < 6; i++) *--p = nullptr;       // rbp rbx r12 r13 r14 r15
        sp = p;
    }
};
inline void switch_context(Context &from, Context &to) { cusim_swap(&from.sp, to.sp); }
#else
struct Context {
    ucontext_t uc;
    void prepare(char *stack, size_t bytes, void (*entry)()) {
        getcontext(&uc);
        uc.uc_stack.ss_sp = stack; uc.uc_stack.ss_size = bytes; uc.uc_link = nullptr;
        makecontext(&uc, entry, 0);
    }
};
inline void switch_context(Context &from, Context &to) { swapcontext(&from.uc, &to.uc); }
#endif

struct Fiber {
    Context ctx;
    unsigned tid = 0;
    bool done = false;
};

struct Warp {
    unsigned arrived = 0, gen = 0;
    uint64_t slot[2][32];
};

struct Block {
    std::vector<Fiber> fibers;
    unsigned alive = 0, bar_count = 0, bar_gen = 0;
    int bar_or = 0, bar_and = 1, bar_cnt = 0;
    int res_or[2] = {0, 0}, res_and[2] = {0, 0}, res_cnt[2] = {0, 0};
    Warp warps[32];
    std::vector<unsigned char> dyn;
    std::function<void()> body;
};

inline thread_local Block *g_block = nullptr;
inline thread_local Fiber *g_fiber = nullptr;
inline thread_local Context g_sched;
inline thread_local unsigned long long g_progress = 0;
inline std::atomic<unsigned long long> g_switches{0};

inline void yield() {
    Fiber *me = g_fiber;
    g_switches.fetch_add(1, std::memory_order_relaxed);
    switch_context(me->ctx, g_sched);
    g_fiber = me;
    threadIdx.x = me->tid;
}

inline void release_barrier(Block &b) {
    const unsigned g = b.bar_gen & 1;
    b.res_or[g] = b.bar_or; b.res_and[g] = b.bar_and; b.res_cnt[g] = b.bar_cnt;
    b.bar_or = 0; b.bar_and = 1; b.bar_cnt = 0; b.bar_count = 0;
    b.bar_gen++;
    g_progress++;
}

// mode 0: plain, 1: or, 2: and, 3: count
inline int barrier(int pred, int mode) {
    Block &b = *g_block;
    const unsigned gen = b.bar_gen;
    b.bar_or |= pred != 0; b.bar_and &= pred != 0; b.bar_cnt += pred != 0;
    if (++b.bar_count == b.alive) release_barrier(b);
    else while (b.bar_gen == gen) yield();
    const unsigned g = gen & 1;
    return mode == 1 ? b.res_or[g] : mode == 2 ? b.res_and[g] : mode == 3 ? b.res_cnt[g] : 0;
}

inline unsigned live_lanes(unsigned warp) {
    Block &b = *g_block;
    unsigned m = 0;
    for (unsigned l = 0; l < 32; l++) {
        const unsigned t = warp * 32 + l;
        if (t < b.fibers.size() && !b.fibers[t].done) m |= 1u << l;
    }
    return m;
}

// Every lane named in `mask` deposits a word and gets the warp's 32 words back.
inline const uint64_t *exchange(unsigned mask, uint64_t v) {
    Block &b = *g_block;
    const unsigned tid = g_fiber->tid, w = tid >> 5, lane = tid & 31;
    Warp &wp = b.warps[w];
    const unsigned gen = wp.gen;
    wp.slot[gen & 1][lane] = v;
    wp.arrived |= 1u << lane;
    const unsigned need = mask & live_lanes(w);
    if ((wp.arrived & need) == need) { wp.arrived = 0; wp.gen++; g_progress++; }
    else while (wp.gen == gen) yield();
    return wp.slot[gen & 1];
}

template <class T> inline uint64_t to_word(T v) { static_assert(sizeof(T) <= 8, ""); uint64_t w = 0; std::memcpy(&w, &v, sizeof(T)); return w; }
template <class T> inline T from_word(uint64_t w) { T v; std::memcpy(&v, &w, sizeof(T)); return v; }

inline unsigned char *dyn_smem() { return g_block->dyn.data(); }

inline void trampoline() {
    Fiber *me = g_fiber;
    g_block->body();
    me->done = true;
    Block &b = *g_block;
    b.alive--;
    g_progress++;
    if (b.alive && b.bar_count == b.alive) release_barrier(b);       // the others were waiting for this thread only
    for (unsigned w = 0; w < 32; w++) {                               // likewise for a warp collective
        Warp &wp = b.warps[w];
        const unsigned need = live_lanes(w);
        if (wp.arrived && (wp.arrived & need) == need) { wp.arrived = 0; wp.gen++; }
    }
    switch_context(me->ctx, g_sched);
}

constexpr size_t STACK_BYTES = 256 << 10;
inline std::vector<std::unique_ptr<char[]>> &stack_pool() { static thread_local std::vector<std::unique_ptr<char[]>> p; return p; }
inline unsigned resident_blocks() {
    const char *e = std::getenv("CUSIM_RESIDENT");
    const unsigned n = e ? unsigned(std::strtoul(e, nullptr, 10)) : 1u;
    return n ? n : 1u;
}

// The order in which the runnable threads of a block get their turn in one scheduling pass.  Every order is a legal
// CUDA schedule; CUSIM_SCHEDULE picks it: unset / "forward" = ascending thread id, "reverse" = descending, "random:<seed>"
// = a fresh permutation of the block's threads every pass (who wins a racing store, an atomicCAS slot or a ticket
// then differs from pass to pass and from seed to seed).
inline void schedule_order(std::vector<unsigned> &order, unsigned n) {
    static thread_local int mode = -1;
    static thread_local uint64_t rng = 0x9E3779B97F4A7C15ull;
    if (mode < 0) {
        const char *e = std::getenv("CUSIM_SCHEDULE");
        mode = !e || !std::strcmp(e, "forward") ? 0 : !std::strcmp(e, "reverse") ? 1 : 2;
        if (mode == 2) { const char *c = std::strchr(e, ':'); rng ^= c ? std::strtoull(c + 1, nullptr, 10) * 0xD1342543DE82EF95ull : 0; }
    }
    for (unsigned i = 0; i < n; i++) order[i] = mode == 1 ? n - 1 - i : i;
    if (mode != 2) return;
    auto next = [&] { rng ^= rng << 13; rng ^= rng >> 7; rng ^= rng << 17; return rng; };
    for (unsigned i = n; i > 1; i--) std::swap(order[i - 1], order[next() % i]);
}

// One block: its threads as fibers on the calling OS thread, until all of them have returned.
template <class F> inline void run_block(unsigned bx, unsigned block, size_t dyn_bytes, F &body) {
    Block b;
    b.fibers.resize(block);
    b.alive = block;
    static const int fill = [] { const char *e = std::getenv("CUSIM_FILL"); return e ? int(std::strtol(e, nullptr, 0)) & 0xFF : 0xCD; }();
    b.dyn.assign(dyn_bytes + 16, (unsigned char)fill);             // shared memory starts as garbage too
    b.body = [&body] { body(); };
    g_block = &b;
    blockIdx = dim3(bx);
    auto &pool = stack_pool();                                    // stacks are reused across blocks and launches
    while (pool.size() < block) pool.emplace_back(new char[STACK_BYTES]);
    for (unsigned t = 0; t < block; t++) {
        Fiber &f = b.fibers[t];
        f.tid = t;
        f.ctx.prepare(pool[t].get(), STACK_BYTES, trampoline);
    }
    std::vector<unsigned> order(block);
    auto last_progress = std::chrono::steady_clock::now();
    unsigned idle_passes = 0;
    while (b.alive) {
        const unsigned long long before = g_progress;
        schedule_order(order, block);
        for (unsigned i = 0; i < block; i++) {
            const unsigned t = order[i];
            Fiber &f = b.fibers[t];
            if (f.done) continue;
            g_fiber = &f;
            threadIdx = dim3(t);
            switch_context(g_sched, f.ctx);
        }
        if (g_progress != before) { idle_passes = 0; continue; }
        // no thread of this block moved: alone on the device that is a deadlock; with other resident blocks it may be a
        // wait for one of them (look-back), so only a long silence counts
        if (idle_passes++ == 0) last_progress = std::chrono::steady_clock::now();
        const bool alone = resident_blocks() == 1;
        if ((alone && idle_passes > 1000) ||
            (!alone && (idle_passes & 1023) == 0 && std::chrono::steady_clock::now() - last_progress > std::chrono::seconds(60))) {
            std::fprintf(stderr, "cusim: deadlock in block %u (%u threads alive, %u at the barrier)\n", bx, b.alive, b.bar_count);
            std::abort();
        }
        if (!alone) std::this_thread::yield();
    }
    g_block = nullptr;
}

// Runs `body` (a call of the kernel function) once per thread of a grid x block launch, x dimension only.
template <class F> inline void launch(unsigned grid, unsigned block, size_t dyn_bytes, F &&body) {
    gridDim = dim3(grid); blockDim = dim3(block);
    const unsigned resident = std::min(resident_blocks(), grid);
    if (resident <= 1) {
        for (unsigned bx = 0; bx < grid; bx++) run_block(bx, block, dyn_bytes, body);
        return;
    }
    std::atomic<unsigned> next{0};
    std::vector<std::thread> sms;
    for (unsigned w = 0; w < resident; w++)
        sms.emplace_back([&] {
            for (unsigned bx = next.fetch_add(1); bx < grid; bx = next.fetch_add(1)) run_block(bx, block, dyn_bytes, body);
        });
    for (auto &t : sms) t.join();
}

}  // namespace cusim

// ---- synchronising built-ins -----------------------------------------------------------------------------------
inline void __syncthreads() { cusim::barrier(0, 0); }
inline int __syncthreads_or(int p) { return cusim::barrier(p, 1); }
inline int __syncthreads_and(int p) { return cusim::barrier(p, 2); }
inline int __syncthreads_count(int p) { return cusim::barrier(p, 3); }
inline void __syncwarp(unsigned mask = 0xffffffffu) { cusim::exchange(mask, 0); }
inline void __nanosleep(unsigned) { cusim::yield(); }
inline void __threadfence() { std::atomic_thread_fence(std::memory_order_seq_cst); }
inline void __threadfence_block() { std::atomic_thread_fence(std::memory_order_seq_cst); }

template <class T> inline T __shfl_sync(unsigned mask, T v, int src) {
    const uint64_t *s = cusim::exchange(mask, cusim::to_word(v));
    return cusim::from_word<T>(s[src & 31]);
}
template <class T> inline T __shfl_up_sync(unsigned mask, T v, unsigned d) {
    const unsigned lane = threadIdx.x & 31;
    const uint64_t *s = cusim::exchange(mask, cusim::to_word(v));
    return lane >= d ? cusim::from_word<T>(s[lane - d]) : v;
}
template <class T> inline T __shfl_down_sync(unsigned mask, T v, unsigned d) {
    const unsigned lane = threadIdx.x & 31;
    const uint64_t *s = cusim::exchange(mask, cusim::to_word(v));
    return lane + d < 32 ? cusim::from_word<T>(s[lane + d]) : v;
}
template <class T> inline T __shfl_xor_sync(unsigned mask, T v, int x) {
    const unsigned lane = threadIdx.x & 31;
    const uint64_t *s = cusim::exchange(mask, cusim::to_word(v));
    return cusim::from_word<T>(s[(lane ^ unsigned(x)) & 31]);
}
inline unsigned __ballot_sync(unsigned mask, int p) {
    const unsigned live = mask & cusim::live_lanes(threadIdx.x >> 5);
    const uint64_t *s = cusim::exchange(mask, p ? 1 : 0);
    unsigned r = 0;
    for (unsigned l = 0; l < 32; l++) if (((live >> l) & 1) && s[l]) r |= 1u << l;
    return r;
}
inline int __any_sync(unsigned mask, int p) { return __ballot_sync(mask, p) != 0; }
inline int __all_sync(unsigned mask, int p) { return __ballot_sync(mask, !p) == 0; }
template <class T> inline T __reduce_max_sync(unsigned mask, T v) {
    const unsigned live = mask & cusim::live_lanes(threadIdx.x >> 5);
    const uint64_t *s = cusim::exchange(mask, cusim::to_word(v));
    T r = v;
    for (unsigned l = 0; l < 32; l++) if ((live >> l) & 1) r = std::max(r, cusim::from_word<T>(s[l]));
    return r;
}
template <class T> inline T __reduce_min_sync(unsigned mask, T v) {
    const unsigned live = mask & cusim::live_lanes(threadIdx.x >> 5);
    const uint64_t *s = cusim::exchange(mask, cusim::to_word(v));
    T r = v;
    for (unsigned l = 0; l < 32; l++) if ((live >> l) & 1) r = std::min(r, cusim::from_word<T>(s[l]));
    return r;
}
template <class T> inline T __reduce_add_sync(unsigned mask, T v) {
    const unsigned live = mask & cusim::live_lanes(threadIdx.x >> 5);
    const uint64_t *s = cusim::exchange(mask, cusim::to_word(v));
    T r = 0;
    for (unsigned l = 0; l < 32; l++) if ((live >> l) & 1) r += cusim::from_word<T>(s[l]);
    return r;
}
template <class T> inline unsigned __match_any_sync(unsigned mask, T v) {
    const unsigned live = mask & cusim::live_lanes(threadIdx.x >> 5);
    const uint64_t mine = cusim::to_word(v);
    const uint64_t *s = cusim::exchange(mask, mine);
    unsigned r = 0;
    for (unsigned l = 0; l < 32; l++) if (((live >> l) & 1) && s[l] == mine) r |= 1u << l;
    return r;
}

// ---- arithmetic and memory built-ins ---------------------------------------------------------------------------
inline int __popc(unsigned v) { return __builtin_popcount(v); }
inline int __popcll(unsigned long long v) { return __builtin_popcountll(v); }
inline int __clz(int v) { return v ? __builtin_clz(unsigned(v)) : 32; }
inline int __ffs(int v) { return __builtin_ffs(v); }
inline float __uint_as_float(unsigned v) { float f; std::memcpy(&f, &v, 4); return f; }
inline unsigned __float_as_uint(float f) { unsigned v; std::memcpy(&v, &f, 4); return v; }
inline int __float_as_int(float f) { int v; std::memcpy(&v, &f, 4); return v; }
inline float __int_as_float(int v) { float f; std::memcpy(&f, &v, 4); return f; }
// A NaN result is the canonical 0x7FFFFFFF whatever the NaN operands carry, as measured on a B200 (tests/test_gpu_edges.py
// test_nan_payload_of_device_arithmetic); x86 would return the first operand's payload, or 0xFFC00000 for Inf - Inf.
// -DCUSIM_NAN_PAYLOADS keeps the x86 result: kernels must not depend on which NaN the hardware returns.
inline float cusim_nan_result(float r) {
#ifndef CUSIM_NAN_PAYLOADS
    if (r != r) return __uint_as_float(0x7FFFFFFFu);
#endif
    return r;
}
inline float __fadd_rn(float a, float b) { volatile float r = a + b; return cusim_nan_result(r); }
inline float __fmul_rn(float a, float b) { volatile float r = a * b; return cusim_nan_result(r); }
template <class T> inline T __ldcg(const T *p) { return *p; }
template <class T> inline T __ldg(const T *p) { return *p; }

// Atomics are real ones: with CUSIM_RESIDENT > 1 blocks run on different OS threads.
template <class T> inline T atomicAdd(T *p, T v) { return __atomic_fetch_add(p, v, __ATOMIC_RELAXED); }
template <class T> inline T atomicSub(T *p, T v) { return __atomic_fetch_sub(p, v, __ATOMIC_RELAXED); }
template <class T> inline T atomicOr(T *p, T v) { return __atomic_fetch_or(p, v, __ATOMIC_RELAXED); }
template <class T> inline T atomicAnd(T *p, T v) { return __atomic_fetch_and(p, v, __ATOMIC_RELAXED); }
template <class T> inline T atomicExch(T *p, T v) { return __atomic_exchange_n(p, v, __ATOMIC_RELAXED); }
template <class T> inline T atomicCAS(T *p, T cmp, T v) { __atomic_compare_exchange_n(p, &cmp, v, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED); return cmp; }
template <class T> inline T atomicMin(T *p, T v) {
    T o = __atomic_load_n(p, __ATOMIC_RELAXED);
    while (v < o && !__atomic_compare_exchange_n(p, &o, v, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
    return o;
}
template <class T> inline T atomicMax(T *p, T v) {
    T o = __atomic_load_n(p, __ATOMIC_RELAXED);
    while (v > o && !__atomic_compare_exchange_n(p, &o, v, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
    return o;
}

using std::max;
using std::min;

#include "cusim_runtime.h"

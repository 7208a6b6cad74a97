// cuda_emu.h -- TEST INFRASTRUCTURE: a functional emulator of the CUDA execution model for the host.
//
// Purpose: run the SOURCE TEXT of the tile-owner kernels (kindel_b200/csrc/pileup_tiled.cu, pileup_wide.cu, pileup_ws.cu)
// on the CPU, so that indexing, sentinels, flush conditions, warp collectives and the staging protocol of a
// kernel can be checked against the oracle without a GPU.  It models behaviour, not performance, and only the
// constructs those kernels use:
//
//   * one fibre (ucontext) per CUDA thread, blocks run one after another; fibres switch only at
//     __syncthreads / __syncwarp / warp collectives / mbarrier waits, round-robin in thread order;
//   * warp collectives (__shfl_xor_sync, __shfl_up_sync, __shfl_sync, __ballot_sync, __any_sync, __all_sync)
//     exchange values through a per-warp slot array between two warp barriers; full masks only;
//   * shared memory is one global array, filled with 0xCD before every block (nothing may rely on zeros);
//     "shared addresses" (smem_u32) are byte offsets into it;
//   * asynchronous copies are made LATE on purpose: a bulk copy (TMA) is performed when the scheduler has
//     gone once round all fibres after it was issued, and only then completes its mbarrier; a thread's
//     cp.async copies are performed at its own cp_async_wait_all.  A kernel that reads staged data before
//     waiting for it therefore sees garbage here, as it could on the device;
//   * a round in which no fibre makes progress is reported as a deadlock;
//   * the order in which fibres run within a round can be reversed or randomised (emu_set_schedule), which changes
//     how producers, consumers and pollers interleave.
//
// With g++ the CUDA headers turn __global__ / __device__ / __shared__ / __forceinline__ / __align__ into
// nothing or into GCC attributes, and give the vector types; everything else is defined below.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <ucontext.h>

#include <functional>
#include <vector>

#define __launch_bounds__(...)
#undef __shared__
#define __shared__ static  // blocks run one after another, so a static is shared by exactly one block's threads

uint3 threadIdx, blockIdx;
dim3 blockDim, gridDim;

namespace kdl {
__attribute__((aligned(128))) unsigned char smem_raw[232448];  // the kernels' `extern __shared__ smem_raw[]`
}

namespace emu {

constexpr int kStack = 256 * 1024;

struct Fibre {
    ucontext_t ctx;
    char* stack = nullptr;
    bool done = false;
    std::vector<std::function<void()>> async;  // this thread's pending cp.async copies
};

struct Deferred {
    std::function<void()> run;
    int age;
};

struct Machine {
    ucontext_t sched;
    std::vector<Fibre> fibres;
    int n = 0, cur = 0, live = 0;
    int warp_live[32];
    int block_arrived = 0;
    unsigned block_gen = 0;
    int warp_arrived[32];
    unsigned warp_gen[32];
    uint64_t slot[32][32];
    int named_arrived[16];
    unsigned named_gen[16];
    unsigned long long progress = 0;
    std::vector<Deferred> deferred;  // bulk copies in flight
    const std::function<void()>* body = nullptr;
    char error[256] = {0};
    std::vector<int> order;
    int schedule = 0;            // 0: threads in order each round, 1: reverse order, 2: a fresh random order per round
    uint64_t rng = 0x9E3779B97F4A7C15ull;
};

inline Machine& M() {
    static Machine m;
    return m;
}

inline void fail(const char* what) {
    Machine& m = M();
    if (!m.error[0]) snprintf(m.error, sizeof m.error, "%s (block %u, thread %d)", what, blockIdx.x, m.cur);
    // unwind is impossible from inside a fibre: mark every fibre done and go back to the scheduler
    for (auto& f : m.fibres) f.done = true;
    m.live = 0;
    swapcontext(&m.fibres[m.cur].ctx, &m.sched);
}

inline void yield() {
    Machine& m = M();
    swapcontext(&m.fibres[m.cur].ctx, &m.sched);
}

inline void block_barrier() {
    Machine& m = M();
    const unsigned gen = m.block_gen;
    if (++m.block_arrived >= m.live) {
        m.block_arrived = 0;
        ++m.block_gen;
        ++m.progress;
        return;
    }
    while (m.block_gen == gen) yield();
}

inline void warp_barrier() {
    Machine& m = M();
    const int w = m.cur >> 5;
    const unsigned gen = m.warp_gen[w];
    if (++m.warp_arrived[w] >= m.warp_live[w]) {
        m.warp_arrived[w] = 0;
        ++m.warp_gen[w];
        ++m.progress;
        return;
    }
    while (m.warp_gen[w] == gen) yield();
}

// bar.sync id, count: `count` threads of the block meet at named barrier `id`
inline void named_barrier(int id, int count) {
    Machine& m = M();
    if (id < 0 || id >= 16) fail("emulator: named barrier id out of range");
    const unsigned gen = m.named_gen[id];
    if (++m.named_arrived[id] >= count) {
        m.named_arrived[id] = 0;
        ++m.named_gen[id];
        ++m.progress;
        return;
    }
    while (m.named_gen[id] == gen) yield();
}

template <class T>
inline T exchange(unsigned mask, T v, int src_lane) {
    static_assert(sizeof(T) <= 8, "exchange: 64-bit values at most");
    Machine& m = M();
    if (mask != 0xffffffffu) fail("emulator: warp collectives with partial masks are not modelled");
    const int w = m.cur >> 5, lane = m.cur & 31;
    uint64_t raw = 0;
    memcpy(&raw, &v, sizeof(T));
    m.slot[w][lane] = raw;
    warp_barrier();
    raw = m.slot[w][src_lane & 31];
    warp_barrier();
    T out;
    memcpy(&out, &raw, sizeof(T));
    return out;
}

inline void on_exit_thread() {
    Machine& m = M();
    Fibre& f = m.fibres[m.cur];
    for (auto& c : f.async) c();
    f.async.clear();
    f.done = true;
    --m.live;
    --m.warp_live[m.cur >> 5];
    ++m.progress;
    // a barrier the remaining threads are waiting on may now be complete
    if (m.live > 0 && m.block_arrived >= m.live) {
        m.block_arrived = 0;
        ++m.block_gen;
    }
    const int w = m.cur >> 5;
    if (m.warp_live[w] > 0 && m.warp_arrived[w] >= m.warp_live[w]) {
        m.warp_arrived[w] = 0;
        ++m.warp_gen[w];
    }
}

inline void trampoline() {
    Machine& m = M();
    (*m.body)();
    on_exit_thread();
    swapcontext(&m.fibres[m.cur].ctx, &m.sched);
}

// run `body` as a grid of `grid` blocks of `block` threads; returns nullptr or an error text
inline const char* launch(unsigned grid, unsigned block, const std::function<void()>& body, unsigned block_y = 0,
                          unsigned grid_y = 1) {
    Machine& m = M();
    m.error[0] = 0;
    if (block > 1024 || block == 0 || grid == 0) return "emulator: bad launch configuration";
    if ((int)m.fibres.size() < (int)block) m.fibres.resize(block);
    for (unsigned t = 0; t < block; ++t)
        if (!m.fibres[t].stack) m.fibres[t].stack = (char*)malloc(kStack);
    gridDim = dim3(grid, grid_y, 1);
    blockDim = dim3(block, 1, 1);
    m.body = &body;
    for (unsigned b = 0; b < grid && !m.error[0]; ++b) {
        blockIdx.x = b; blockIdx.y = block_y; blockIdx.z = 0;
        memset(kdl::smem_raw, 0xCD, sizeof kdl::smem_raw);
        m.n = (int)block;
        m.live = m.n;
        m.block_arrived = 0;
        for (int k = 0; k < 16; ++k) m.named_arrived[k] = 0;
        m.deferred.clear();
        for (int w = 0; w < 32; ++w) {
            m.warp_live[w] = 0;
            m.warp_arrived[w] = 0;
        }
        for (int t = 0; t < m.n; ++t) {
            Fibre& f = m.fibres[t];
            f.done = false;
            f.async.clear();
            ++m.warp_live[t >> 5];
            getcontext(&f.ctx);
            f.ctx.uc_stack.ss_sp = f.stack;
            f.ctx.uc_stack.ss_size = kStack;
            f.ctx.uc_link = nullptr;
            makecontext(&f.ctx, (void (*)())trampoline, 0);
        }
        int idle_rounds = 0;
        while (m.live > 0) {
            const unsigned long long before = m.progress;
            // the order in which the fibres get their turn this round: different orders give different
            // interleavings of producers / consumers / pollers, i.e. a cheap search for protocol races
            m.order.resize((size_t)m.n);
            for (int t = 0; t < m.n; ++t) m.order[(size_t)t] = m.schedule == 1 ? m.n - 1 - t : t;
            if (m.schedule == 2) {
                for (int t = m.n - 1; t > 0; --t) {
                    m.rng = m.rng * 6364136223846793005ull + 1442695040888963407ull;
                    const int j = (int)((m.rng >> 33) % (uint64_t)(t + 1));
                    const int tmp = m.order[(size_t)t]; m.order[(size_t)t] = m.order[(size_t)j]; m.order[(size_t)j] = tmp;
                }
            }
            for (int k = 0; k < m.n && m.live > 0; ++k) {
                const int t = m.order[(size_t)k];
                if (m.fibres[t].done) continue;
                m.cur = t;
                threadIdx.x = (unsigned)t; threadIdx.y = threadIdx.z = 0;
                swapcontext(&m.sched, &m.fibres[t].ctx);
            }
            // bulk copies issued at least one full round ago land now
            for (size_t i = 0; i < m.deferred.size();) {
                if (--m.deferred[i].age < 0) {
                    m.deferred[i].run();
                    m.deferred.erase(m.deferred.begin() + i);
                    ++m.progress;
                } else {
                    ++i;
                }
            }
            if (m.progress == before) {
                if (++idle_rounds > 4) {
                    snprintf(m.error, sizeof m.error, "emulator: deadlock in block %u (%d threads alive)", b, m.live);
                    break;
                }
            } else {
                idle_rounds = 0;
            }
        }
    }
    return m.error[0] ? m.error : nullptr;
}

// the row blockIdx.y = block_y of a two-dimensional grid (grid x grid_y blocks)
inline const char* launch_y(unsigned grid, unsigned block_y, unsigned grid_y, unsigned block,
                            const std::function<void()>& body) {
    return launch(grid, block, body, block_y, grid_y);
}

}  // namespace emu

// ---- the CUDA built-ins the kernels use ---------------------------------------------------------------------
inline void __syncthreads() { emu::block_barrier(); }
inline void __syncwarp(unsigned mask = 0xffffffffu) {
    if (mask != 0xffffffffu) emu::fail("emulator: __syncwarp with a partial mask");
    emu::warp_barrier();
}
template <class T>
inline T __shfl_xor_sync(unsigned mask, T v, int lane_mask) {
    return emu::exchange(mask, v, (emu::M().cur & 31) ^ lane_mask);
}
template <class T>
inline T __shfl_up_sync(unsigned mask, T v, unsigned delta) {
    const int lane = emu::M().cur & 31;
    return emu::exchange(mask, v, lane >= (int)delta ? lane - (int)delta : lane);
}
template <class T>
inline T __shfl_down_sync(unsigned mask, T v, unsigned delta) {
    const int lane = emu::M().cur & 31;
    return emu::exchange(mask, v, lane + (int)delta < 32 ? lane + (int)delta : lane);
}
template <class T>
inline T __shfl_sync(unsigned mask, T v, int src) {
    return emu::exchange(mask, v, src);
}
inline unsigned __ballot_sync(unsigned mask, int pred) {
    emu::Machine& m = emu::M();
    if (mask != 0xffffffffu) emu::fail("emulator: __ballot_sync with a partial mask");
    const int w = m.cur >> 5, lane = m.cur & 31;
    m.slot[w][lane] = pred ? 1u : 0u;
    emu::warp_barrier();
    unsigned out = 0;
    for (int l = 0; l < 32; ++l)
        if (!m.fibres[(w << 5) + l].done && (w << 5) + l < m.n && m.slot[w][l]) out |= 1u << l;
    emu::warp_barrier();
    return out;
}
inline int __any_sync(unsigned mask, int pred) { return __ballot_sync(mask, pred) != 0u; }
inline int __all_sync(unsigned mask, int pred) { return __ballot_sync(mask, !pred) == 0u; }

template <class T>
inline T __ldg(const T* p) { return *p; }
inline int __ffs(unsigned v) { return __builtin_ffs((int)v); }
inline int __popc(unsigned v) { return __builtin_popcount(v); }
inline uint32_t __funnelshift_l(uint32_t lo, uint32_t hi, uint32_t shift) {
    return (uint32_t)(((((uint64_t)hi << 32) | lo) << (shift & 31)) >> 32);
}
inline int atomicOr(int* p, int v) { const int old = *p; *p = old | v; return old; }
inline unsigned atomicOr(unsigned* p, unsigned v) { const unsigned old = *p; *p = old | v; return old; }
inline unsigned long long atomicMin(unsigned long long* p, unsigned long long v) {
    const unsigned long long old = *p; if (v < old) *p = v; return old;
}
inline void __threadfence() {}
inline void __threadfence_system() {}
inline void __nanosleep(unsigned) { emu::yield(); }  // only ever called inside a polling loop
inline int atomicAdd(int* p, int v) { const int old = *p; *p = old + v; return old; }
inline unsigned atomicAdd(unsigned* p, unsigned v) { const unsigned old = *p; *p = old + v; return old; }
inline unsigned long long atomicAdd(unsigned long long* p, unsigned long long v) {
    const unsigned long long old = *p; *p = old + v; return old;
}

// ---- stand-ins for the PTX helpers of pileup_tiled.cu (same names, same contracts) ---------------------------
namespace kdl {

inline uint32_t smem_u32(const void* p) {
    const uintptr_t a = (uintptr_t)p, base = (uintptr_t)smem_raw;
    if (a < base || a >= base + sizeof smem_raw) emu::fail("emulator: smem_u32 of a pointer outside shared memory");
    return (uint32_t)(a - base);
}
inline uint32_t lds_u32(uint32_t addr) {  // ld.shared.u32
    if ((addr & 3u) || addr + 4u > sizeof smem_raw) emu::fail("emulator: ld.shared.u32 out of range or misaligned");
    uint32_t v;
    memcpy(&v, smem_raw + addr, 4);
    return v;
}

// mbarrier state in the 8 bytes of the barrier word: phase | pending arrivals | expected arrivals | tx bytes
struct MbarBits {
    uint32_t phase : 1, count : 15, pending : 16;
    int32_t tx;
};
static_assert(sizeof(MbarBits) == 8, "mbarrier emulation state must fit the 64-bit barrier word");
inline void mbar_check(MbarBits* b) {
    if (b->pending == 0 && b->tx == 0) {
        b->phase ^= 1u;
        b->pending = b->count;
        ++emu::M().progress;
    }
}
inline void mbar_init(uint64_t* bar, int count) {
    MbarBits b;
    b.phase = 0;
    b.count = (uint32_t)count;
    b.pending = (uint32_t)count;
    b.tx = 0;
    memcpy(bar, &b, 8);
}
inline void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {  // one arrival + `bytes` expected
    MbarBits* b = reinterpret_cast<MbarBits*>(bar);
    if (b->pending == 0) emu::fail("emulator: mbarrier arrival beyond its count");
    b->tx += (int32_t)bytes;
    b->pending -= 1;
    mbar_check(b);
}
inline void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    if ((bytes & 15u) || ((uintptr_t)dst & 15u) || ((uintptr_t)src & 15u))
        emu::fail("emulator: cp.async.bulk needs 16-byte aligned addresses and size");
    smem_u32(dst);
    if (bytes) smem_u32((const char*)dst + bytes - 1);
    emu::M().deferred.push_back({[=] {
                                     memcpy(dst, src, bytes);
                                     MbarBits* b = reinterpret_cast<MbarBits*>(bar);
                                     b->tx -= (int32_t)bytes;
                                     mbar_check(b);
                                 },
                                 1});
}
inline void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (reinterpret_cast<MbarBits*>(bar)->phase == (parity & 1u)) emu::yield();
}
inline void mbar_arrive(uint64_t* bar) {  // mbarrier.arrive: one arrival, no bytes
    MbarBits* b = reinterpret_cast<MbarBits*>(bar);
    if (b->pending == 0) emu::fail("emulator: mbarrier arrival beyond its count");
    b->pending -= 1;
    mbar_check(b);
}
inline void mbar_expect_tx_only(uint64_t* bar, uint32_t bytes) {  // mbarrier.expect_tx: bytes, no arrival
    reinterpret_cast<MbarBits*>(bar)->tx += (int32_t)bytes;
}
inline void producer_sync() { emu::named_barrier(1, 128); }  // bar.sync 1, 128
inline bool producer_sync_or(bool pred) {                    // bar.red.or.pred on the same barrier
    static unsigned tag[2] = {0u, 0u};  // generation of the barrier at which somebody last voted true, per parity
    const unsigned g = emu::M().named_gen[1];
    if (pred) tag[g & 1u] = g + 1u;
    emu::named_barrier(1, 128);
    return tag[g & 1u] == g + 1u;
}
template <int kRegs> inline void reg_dealloc() {}            // setmaxnreg: nothing to model
template <int kRegs> inline void reg_alloc() {}
// system-scope flag accesses of the exchange kernels (vote.cu): plain accesses here; a poll yields, so a flag
// that never arrives shows up as a deadlock
inline int ld_acquire_sys(const int32_t* p) { return *p; }
inline void st_release_sys(int32_t* p, int v) { *p = v; ++emu::M().progress; }
inline void cp_async4(void* dst, const void* src) {
    if (((uintptr_t)dst & 3u) || ((uintptr_t)src & 3u)) emu::fail("emulator: cp.async 4-byte alignment");
    smem_u32(dst);
    emu::M().fibres[emu::M().cur].async.push_back([=] { memcpy(dst, src, 4); });
}
inline void cp_async_wait_all() {
    auto& q = emu::M().fibres[emu::M().cur].async;
    for (auto& c : q) c();
    q.clear();
}

}  // namespace kdl

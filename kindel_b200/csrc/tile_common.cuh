// tile_common.cuh -- what the tile-owner pileup (pileup_tile.cu) is built from: K0 (the tile index), the PTX
// wrappers (mbarrier, 1-D bulk copy = TMA, cp.async, setmaxnreg, named barriers), the warp searches, the bit-sliced
// counters (Harley-Seal carry-save adders over one-hot nibbles) and the flush of a 64-slot window to the table.
//
// A BAM base is a one-hot nibble (A=1 C=2 G=4 T=8, N=15).  With 8 bases per 32-bit word, first base in the top
// nibble, the 8 bases a read puts on a lane's 8 slots are ONE funnel shift of two staged words, and the 32 bits of
// that word are 32 independent 1-bit inputs (8 slots x A,C,G,T) to vertical counters: 7 full adders (14 LOP3) per
// 8 reads instead of 8 x 150 read-modify-writes.  N (all four bits set) is not counted at all: per slot
// A+C+G+T (raw) = coverage + 3 N, and the coverage comes from a +1/-1 difference array (flush_window).
#pragma once
#include <stddef.h>

#include "kdl_common.cuh"

namespace kdl {

constexpr int F_WIN = 64;              // slots per warp window
constexpr int F_P = 8;                 // bit planes per stream: up to 255 reads between flushes
constexpr int F_FLUSH_BLOCKS = 31;     // 31 blocks x 8 reads = 248 <= 255
static_assert(F_FLUSH_BLOCKS % 2 == 1, "the counting loop folds exactly one pending carry at a mid-window flush");

// ---- K0: per tile, what K1 needs to start without dependent global loads: 8 x uint32
//   [0] lo, [1] hi   index range of the reads that can touch the tile: global start slot in
//                    [tile_lo - reach_right + 1, tile_hi + reach_left)
//   [2] wa, [3] wend word range of their blocks in seq4 (wa rounded down to a 16-byte boundary)
//   [4] c_lo, [5] c_hi contigs of read lo and of read hi - 1;  [6], [7] first slot of contig c_lo (64 bits)
// global slot of a read's first base = contig_slot[c] + ref_start; reads are sorted by it.
constexpr int F_IDX = 8;  // uint32 per tile in the index

// First read index whose global start slot is >= g, for TWO keys at once (a tile's lower and upper
// bound).  Warp-cooperative: the contig is found by every lane (few contigs), the read by a 32-ary
// search -- each round the 32 lanes probe 32 evenly spaced elements of the remaining range in ONE
// memory round trip (5 rounds for 10^7 reads, not 24); the two searches advance in lockstep so
// their round trips overlap.
struct Search {
    long long a, e, p;  // invariant: reads before a are < p, reads from e on are >= p (or e = end)
    bool live;
};

__device__ __forceinline__ Search search_begin(const kdl_batch& b, long long g) {
    Search s;
    s.live = false;
    s.a = s.e = 0;
    s.p = 0;
    if (b.n_contigs == 0) return s;
    int lo = 0, hi = b.n_contigs;  // first contig with slot + len + 1 > g
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (b.contig_slot[mid] + b.contig_len[mid] + 1 > g) hi = mid; else lo = mid + 1;
    }
    if (lo >= b.n_contigs) { s.a = s.e = b.n_reads; return s; }
    s.p = g - b.contig_slot[lo];  // position inside contig `lo` (may be < 0)
    s.a = b.contig_read_off[lo];
    s.e = b.contig_read_off[lo + 1];
    s.live = s.a < s.e;
    return s;
}

__device__ __forceinline__ void search_probe(const kdl_batch& b, const Search& s, int lane, long long& step, bool& ge) {
    step = (s.e - s.a + 31) >> 5;
    const long long idx = s.a + (long long)(lane + 1) * step - 1;  // last element of the lane's bucket
    ge = (s.live && idx < s.e) ? ((long long)b.ref_start[idx] >= s.p) : true;
}

__device__ __forceinline__ void search_narrow(Search& s, long long step, bool ge) {
    const unsigned m = __ballot_sync(0xffffffffu, ge);
    if (!s.live) return;
    if (m == 0u) { s.a = s.e; s.live = false; return; }  // even the very last element is < p
    const int k = __ffs(m) - 1;                          // first bucket whose last element is >= p
    const long long na = s.a + (long long)k * step;
    long long ne = s.a + (long long)(k + 1) * step - 1;  // that element is >= p: the answer is <= ne
    if (ne > s.e) ne = s.e;
    s.a = na;
    s.e = ne < na ? na : ne;
    if (step == 1) s.a = s.e;
    s.live = s.a < s.e;
}

__global__ void __launch_bounds__(256)
tile_index_kernel(kdl_batch b, long long tile_lo, long long n_tiles, uint32_t* __restrict__ index) {
    const int lane = threadIdx.x & 31;
    const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;  // one warp per tile
    if (w >= n_tiles) return;
    const long long t = tile_lo + w;
    const long long g0 = t * KDL_TILE;
    Search s1 = search_begin(b, g0 - b.reach_right + 1), s2 = search_begin(b, g0 + KDL_TILE + b.reach_left);
    while (s1.live || s2.live) {  // warp-uniform
        long long st1, st2;
        bool ge1, ge2;
        search_probe(b, s1, lane, st1, ge1);  // both probes are issued before either is consumed
        search_probe(b, s2, lane, st2, ge2);
        search_narrow(s1, st1, ge1);
        search_narrow(s2, st2, ge2);
    }
    const long long lo = s1.a, hi = s2.a;
    if (lane) return;
    uint32_t* e = index + F_IDX * t;
    e[0] = (uint32_t)lo;
    e[1] = (uint32_t)hi;
    e[2] = lo < b.n_reads ? (b.seq_off[lo] & ~3u) : 0u;
    e[3] = hi < b.n_reads ? b.seq_off[hi] : (uint32_t)b.seq4_words;
    const int c_lo = lo < hi ? find_contig(b.contig_read_off, b.n_contigs, lo) : 0;
    e[4] = (uint32_t)c_lo;
    e[5] = lo < hi ? (uint32_t)find_contig(b.contig_read_off, b.n_contigs, hi - 1) : 0u;
    const unsigned long long cs = lo < hi ? (unsigned long long)b.contig_slot[c_lo] : 0ull;
    e[6] = (uint32_t)cs;          // first slot of contig c_lo: K1 then needs no dependent load for it
    e[7] = (uint32_t)(cs >> 32);
}

// (KDL_HOST_EMU: tests/emu/ compiles this file for the host and supplies functional stand-ins for the PTX
// helpers below; the device build never defines it.)
#ifndef KDL_HOST_EMU
// ---- 1-D bulk copy global -> shared (TMA engine, SASS UBLKCP) completing on an mbarrier --------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// 4-byte asynchronous global -> shared copy (LDGSTS): no register staging, completes in background
__device__ __forceinline__ void cp_async4(void* dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// Plain polling: a nanosleep between polls or a suspend-time hint on try_wait measured the same to four digits, for
// producers and consumers alike (profiles/r02_ring_depth.txt).
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}
#endif  // KDL_HOST_EMU

#ifndef KDL_HOST_EMU
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// named barrier 1: the 128 producer threads only
__device__ __forceinline__ void producer_sync() { asm volatile("bar.sync 1, 128;" ::: "memory"); }
// the same barrier with an OR-reduction of a predicate over the 128 threads
__device__ __forceinline__ bool producer_sync_or(bool pred) {
    uint32_t r;
    asm volatile("{\n"
                 ".reg .pred p, q;\n"
                 "setp.ne.u32 p, %1, 0;\n"
                 "bar.red.or.pred q, 1, 128, p;\n"
                 "selp.u32 %0, 1, 0, q;\n"
                 "}\n"
                 : "=r"(r) : "r"((uint32_t)pred) : "memory");
    return r != 0;
}
template <int kRegs> __device__ __forceinline__ void reg_dealloc() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegs)); }
template <int kRegs> __device__ __forceinline__ void reg_alloc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegs)); }
#endif  // KDL_HOST_EMU

// first index i in [0, n) with g[i] >= key (n if none), for TWO keys at once (key_a <= key_e); g sorted,
// n <= 1024, whole warp calls.  Two 32-ary rounds: the lanes probe the last element of 32 buckets, then the
// elements of the first bucket whose last element is >= key.  One probe load serves both searches and the two
// dependent chains (load -> ballot -> load -> ballot) overlap.
__device__ __forceinline__ void lower_bound_warp2(const int* g, int n, int key_a, int key_e, int lane, int& ra, int& re) {
    const int step = (n + 31) >> 5;  // <= 32
    if (step == 0) { ra = re = 0; return; }
    const int i1 = (lane + 1) * step - 1;
    const int v1 = i1 < n ? g[i1] : 0x7fffffff;  // past the end: counts as >= key
    const unsigned ma = __ballot_sync(0xffffffffu, v1 >= key_a);
    const unsigned me = __ballot_sync(0xffffffffu, v1 >= key_e);
    const int ka = __ffs(ma) - 1, ke = __ffs(me) - 1;  // first bucket whose last element is >= key; -1: none
    const int ia = ka * step + lane, ie = ke * step + lane;
    const int va = (ka >= 0 && lane < step && ia < n) ? g[ia] : 0x7fffffff;
    const int ve = (ke >= 0 && lane < step && ie < n) ? g[ie] : 0x7fffffff;
    const unsigned m2a = __ballot_sync(0xffffffffu, va >= key_a);
    const unsigned m2e = __ballot_sync(0xffffffffu, ve >= key_e);
    const int qa = ka * step + __ffs(m2a) - 1, qe = ke * step + __ffs(m2e) - 1;
    ra = (ka < 0 || qa > n) ? n : qa;
    re = (ke < 0 || qe > n) ? n : qe;
}

// ---- bit-sliced counters ------------------------------------------------------------------------
__device__ __forceinline__ void csa(uint32_t& carry, uint32_t& sum, uint32_t a, uint32_t b, uint32_t c) {
    const uint32_t s = a ^ b ^ c;
    carry = (a & b) | (c & (a | b));
    sum = s;
}

struct Planes {
    uint32_t p[F_P];  // p[k] = bit k of 32 vertical counters
    __device__ __forceinline__ void clear() {
#pragma unroll
        for (int k = 0; k < F_P; ++k) p[k] = 0;
    }
    // Harley-Seal: 8 one-bit-per-counter inputs -> 7 full adders.  The carry out of the 4s plane (weight 8) is
    // handed back instead of being rippled up; the caller pairs two of them with one more full adder, so the
    // ripple runs once per 16 reads
    __device__ __forceinline__ uint32_t add8_carry(const uint32_t (&x)[8]) {
        uint32_t ta, tb, tc, td, fa, fb, e;
        csa(ta, p[0], p[0], x[0], x[1]);
        csa(tb, p[0], p[0], x[2], x[3]);
        csa(fa, p[1], p[1], ta, tb);
        csa(tc, p[0], p[0], x[4], x[5]);
        csa(td, p[0], p[0], x[6], x[7]);
        csa(fb, p[1], p[1], tc, td);
        csa(e, p[2], p[2], fa, fb);
        return e;
    }
    template <int K0>  // add one plane of weight 2^K0
    __device__ __forceinline__ void ripple(uint32_t e) {
#pragma unroll
        for (int k = K0; k < F_P; ++k) {
            const uint32_t t = p[k] & e;
            p[k] ^= e;
            e = t;
        }
    }
};

// sum of the same planes held by the 4 quarter-warps (lanes l, l^8, l^16, l^24): bit-sliced ripple
// adders over two butterfly stages; F_P planes in, F_P + 2 planes out, identical in all 4 lanes.
__device__ __forceinline__ void quarter_sum(const uint32_t (&in)[F_P], uint32_t (&out)[F_P + 2]) {
    uint32_t a[F_P + 2];
#pragma unroll
    for (int k = 0; k < F_P; ++k) a[k] = in[k];
    a[F_P] = 0;
    a[F_P + 1] = 0;
#pragma unroll
    for (int stage = 0; stage < 2; ++stage) {
        const int width = F_P + stage;  // planes that can be non-zero before this stage
        uint32_t carry = 0;
#pragma unroll
        for (int k = 0; k < F_P + 2; ++k) {
            if (k < width) {
                const uint32_t o = __shfl_xor_sync(0xffffffffu, a[k], 8 << stage);
                uint32_t c2, s;
                csa(c2, s, a[k], o, carry);
                a[k] = s;
                carry = c2;
            } else if (k == width) {
                a[k] = carry;
            }
        }
    }
#pragma unroll
    for (int k = 0; k < F_P + 2; ++k) out[k] = a[k];
}

// counters of bit `bit` (0..3) of every nibble: 8 integers, out[b] for the lane's slot b
// (slot b sits in nibble 7-b).  Planes: F_P + 2 <= 12 bits per counter.
__device__ __forceinline__ void extract8(const uint32_t (&pl)[F_P + 2], int bit, int (&out)[8]) {
    uint32_t v[3] = {0u, 0u, 0u};  // 4 planes per packed word: nibble j of v[g] = bits 4g..4g+3 of counter j
#pragma unroll
    for (int k = 0; k < F_P + 2; ++k) v[k >> 2] |= ((pl[k] >> bit) & 0x11111111u) << (k & 3);
#pragma unroll
    for (int b = 0; b < 8; ++b) {
        const int sh = 4 * (7 - b);
        out[b] = (int)(((v[0] >> sh) & 0xFu) | (((v[1] >> sh) & 0xFu) << 4) | (((v[2] >> sh) & 0xFu) << 8));
    }
}

// ---- flush: planes -> integers -> table ----------------------------------------------------------
// N is not counted: an N nibble (15) adds 1 to all four of A,C,G,T, so for every slot
//     A_raw + C_raw + G_raw + T_raw = cov + 3 N        (cov = staged reads / pieces covering the slot)
// and cov comes from a +1/-1 difference array over piece starts/ends (two shared-memory atomics per staged
// piece, one prefix sum per item).  The correction is applied by the FINAL flush of a window (kFinal); earlier
// flushes -- only needed when more than 248 reads per stream pile up on one window -- add raw counts and
// remember the raw total in `rawacc`.
// Quarter q owns column q (A,C,G,T); quarter 0 also writes column 4 (N).  Each lane holds 8 consecutive slots.
// kMode: F_STORE  = two 128-bit stores per column (first flush of a window whose columns hold stale data),
//        F_ADD    = 128-bit read-modify-writes (nobody else touches these slots during this kernel),
//        F_ATOMIC = one RED per non-zero value (several CTAs share the tile: depth split, see pileup_tile.cu).
enum { F_STORE = 0, F_ADD = 1, F_ATOMIC = 2 };

template <int kMode, bool kFinal>
__device__ __forceinline__ void flush_window(Planes& acc, int (&rawacc)[8], const int (&covacc)[8],
                                             int32_t* __restrict__ counts, long long n_slots, long long slot0,
                                             int lane) {
    const int q = lane >> 3;
    const long long s = slot0 + 8 * (lane & 7);
    int32_t* dcol = counts + (long long)q * n_slots + s;
    int4* dst = reinterpret_cast<int4*>(dcol);
    int4 v0 = make_int4(0, 0, 0, 0), v1 = v0;
    if (kMode == F_ADD) { v0 = dst[0]; v1 = dst[1]; }  // issued first: latency hides behind the transposition
    uint32_t m[F_P + 2];
    quarter_sum(acc.p, m);
    acc.clear();
    int cv[8], tot[8];
    extract8(m, q, cv);
#pragma unroll
    for (int k = 0; k < 8; ++k) {  // A+C+G+T raw of each slot: sum of the four quarters' columns
        int t = cv[k];
        t += __shfl_xor_sync(0xffffffffu, t, 8);
        t += __shfl_xor_sync(0xffffffffu, t, 16);
        tot[k] = t + rawacc[k];
    }
    int nn[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        if (kFinal) {
            nn[k] = (tot[k] - covacc[k]) / 3;  // exact by construction
            rawacc[k] = 0;
        } else {
            nn[k] = 0;
            rawacc[k] = tot[k];
        }
    }
    if (kMode == F_ATOMIC) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int d = cv[k] - nn[k];
            if (d) atomicAdd(dcol + k, d);
        }
        if (q == 0 && kFinal) {
            int32_t* ncol = counts + (long long)KDL_W_N * n_slots + s;
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (nn[k]) atomicAdd(ncol + k, nn[k]);
        }
        return;
    }
    v0.x += cv[0] - nn[0]; v0.y += cv[1] - nn[1]; v0.z += cv[2] - nn[2]; v0.w += cv[3] - nn[3];
    v1.x += cv[4] - nn[4]; v1.y += cv[5] - nn[5]; v1.z += cv[6] - nn[6]; v1.w += cv[7] - nn[7];
    dst[0] = v0;
    dst[1] = v1;
    if (q == 0 && (kFinal || kMode == F_STORE)) {
        int4* dn = reinterpret_cast<int4*>(counts + (long long)KDL_W_N * n_slots + s);
        int4 n0 = make_int4(0, 0, 0, 0), n1 = n0;
        if (kMode == F_ADD) { n0 = dn[0]; n1 = dn[1]; }
        n0.x += nn[0]; n0.y += nn[1]; n0.z += nn[2]; n0.w += nn[3];
        n1.x += nn[4]; n1.y += nn[5]; n1.z += nn[6]; n1.w += nn[7];
        dn[0] = n0;
        dn[1] = n1;
    }
}

// zero columns [col_lo, col_hi) of slots [slot_lo, slot_hi) (multiples of 4), 128-bit stores
__global__ void __launch_bounds__(256)
zero_cols_kernel(int32_t* __restrict__ counts, long long n_slots, int col_lo, int col_hi, long long slot_lo,
                 long long slot_hi) {
    const long long per_col = (slot_hi - slot_lo) >> 2;
    const long long total = per_col * (col_hi - col_lo);
    for (long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x; v < total;
         v += (long long)gridDim.x * blockDim.x) {
        const long long col = col_lo + v / per_col, off = v % per_col;
        reinterpret_cast<int4*>(counts + col * n_slots + slot_lo)[off] = make_int4(0, 0, 0, 0);
    }
}

}  // namespace kdl

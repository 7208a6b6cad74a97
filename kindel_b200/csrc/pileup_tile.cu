// pileup_tile.cu -- K1: the owner-computes pileup of coordinate-sorted reads, a warp-specialised pipeline.
//
// What it computes is the per-read loop of the reference, kindel/kindel.py:40-81, for every read that is not
// KDL_HARD: `weights[pos][base] += 1` for the bases of M/=/X ops (kindel.py:49-54) as a positional population
// count (tile_common.cuh), and -- for complex reads -- the insertion / deletion / clip updates (kindel.py:55-81).
//
//   * The slot space is cut into tiles of KDL_TILE = 512 slots.  Because the reads are coordinate-sorted, the
//     reads that can touch a tile are ONE index range and ONE byte range of seq4 (K0, tile_common.cuh); a tile
//     is owned by one CTA (or, for small references piled deep, by `split` CTAs that share it by read range and
//     flush with REDs), so the weight columns are written with plain 128-bit stores: no atomics, no memset.
//   * Two CTAs per SM, each 4 PRODUCER + 8 CONSUMER warps over a shared-memory ring (two stages), the register
//     file re-balanced with setmaxnreg.  An ITEM is (tile, up to kRmax reads).  Producers: wait for a free stage,
//     ONE 1-D bulk copy (TMA) of the item's bytes, per-read metadata, the coverage marks (+1 / -1 per window and the
//     carries between windows, TileStage::diff); each thread prefetches the metadata words of the reads it will
//     handle in the next item (cp.async), so the producers meet no barrier of their own in the simple path.
//     Consumers: each warp owns a 64-slot window, each quarter-warp walks a different read (one funnel shift of two
//     staged words per lane and read, 7 full adders per 8 reads), and flushes at the end of a tile.  Consumers never
//     touch global memory except for the table stores and never meet a CTA-wide barrier.
//   * Complex reads (indels, clips; include/kindel_b200.h) carry their CIGAR behind their bases in seq4, so it
//     arrives with the bulk copy.  A producer thread tracks the two cursors through it once per (read, tile): every
//     M/=/X segment that overlaps the tile becomes a PIECE (virtual start = slot of the read's base 0, clipped slot
//     range), which the consumers count with the same bit-sliced adders plus a nibble mask.  The sparse rest of
//     such a read -- insertion / deletion / clip updates, insertion events -- is K1e's (pileup_general.cu), once
//     per read.  Reads that could wrap a Python index or raise (KDL_HARD) are left to K1g.
//
// Preconditions (checked by the host side of the ABI): reads_sorted, classification as in include/kindel_b200.h.
#include "tile_common.cuh"

namespace kdl {

constexpr int W_CONSUMERS = 8;   // consumer warps (one 64-slot window each)
constexpr int W_PRODUCERS = 4;   // producer warps
// depth of the shared-memory ring.  Measured on B200 (cfg 4, all simple): 2 stages 0.216 ms, 3 stages 0.243 ms,
// 4 stages 0.262 ms for K0 + K1 -- see TileCfg and profiles/r02_ring_depth.txt
constexpr int W_STAGES = 2;
constexpr int W_THREADS = 32 * (W_CONSUMERS + W_PRODUCERS);
constexpr int W_PT = 32 * W_PRODUCERS;  // producer threads
// setmaxnreg per role: 128 * kProducer + 256 * kConsumer <= 384 * 80 (the launch bound's allocation)
template <bool kCx> struct TileRegs { static constexpr int kProducer = kCx ? 64 : 56, kConsumer = 88; };
static_assert(W_PT * TileRegs<true>::kProducer + 32 * W_CONSUMERS * TileRegs<true>::kConsumer <= W_THREADS * 80 &&
              W_PT * TileRegs<false>::kProducer + 32 * W_CONSUMERS * TileRegs<false>::kConsumer <= W_THREADS * 80,
              "register pool of the CTA");

// kCx = false: batches without tile-eligible complex reads (no piece list, larger stages)
template <bool kCx> struct TileCfg;
// An item is sized so that the whole ring fits half an SM's shared memory.  A tile of deep short-read data is
// several items, each a sub-range of the tile's (sorted) reads, and every item costs each consumer warp a wait, a
// search and a partly filled last block: FEW LARGE items beat a deeper ring of small ones (3 and 4 stages with
// proportionally smaller items were measured slower, profiles/r02_ring_depth.txt).
template <> struct TileCfg<false> {
    static constexpr int kRmax = 512;    // reads per item
    static constexpr int kCapW = 9728;   // words of seq4 per item (38 KB: ~510 reads of 150 bases)
    static constexpr int kPcap = 0;      // pieces of complex reads per item
};
template <> struct TileCfg<true> {
    static constexpr int kRmax = 384;
    static constexpr int kCapW = 7680;   // 30 KB
    static constexpr int kPcap = 672;
};

enum : int { ITEM_FIRST = 1, ITEM_LAST = 2, ITEM_EMPTY = 4, ITEM_END = 8 };

template <class C>
struct TileStage {
    uint32_t seq[C::kCapW];
    // per staged read (32 sentinels follow the last one); entry of read i at i + i/8 (one pad per 8: the four
    // quarter-warps' entries then sit 144 B = 4 banks apart):
    //   .x  4 * ceil(start / 8): byte offset, relative to the tile, of the first 8-slot group the read can serve
    //   .y  shared-memory address (u32) of the read's first word
    //   .z  bytes of packed bases (0 = not a simple read: adds nothing in the simple loop)
    //   .w  funnel-shift amount 4 * ((-start) & 7)
    int4 meta[C::kRmax + 40 + (C::kRmax + 40) / 8];
    // pieces of complex reads: .x/.y/.z as above with start = the slot of the read's base 0 (virtual start);
    // .w = shift | s0 << 8 | s1 << 20, [s0, s1) the piece's slots clipped to the tile.  px[kPcap] = a piece that
    // covers nothing (what idle lanes of a block read).
    int4 px[C::kPcap + 1];
    int gs[C::kRmax + 32];       // start slot relative to the tile (all reads: the array stays sorted)
    // coverage of the tile's slots by the item's reads / pieces, as a difference array PER WINDOW: +1 at a piece's
    // first slot, -1 behind its last (unless that is a window's first slot), and carry[w] = pieces that cover the
    // first slot of window w.  A consumer warp reads its own 64 + 1 entries and zeroes them again before it releases
    // the stage, so the producers never clean and nobody sums across windows.
    int diff[KDL_TILE + 32];
    int carry[W_CONSUMERS];
    long long tile_slot;
    int n_sub;
    int flags;
    int n_px;
    int pad0;
};

template <class C>
struct TileSmem {
    TileStage<C> st[W_STAGES];
    int raw[3][C::kRmax];          // producers: l_seq / ref_start / seq_off of the NEXT item's reads (cp.async)
    unsigned short queue[W_CONSUMERS][C::kPcap ? 64 : 4];  // consumers (kCx): indices of the pieces that overlap the warp's window
    int scan[W_PRODUCERS * 4 + 4];  // producers (kCx): per-group piece totals, cut counter
    uint64_t full[W_STAGES];       // producers -> consumers: 4 warp arrivals (metadata, pieces, coverage written)
    uint64_t landed[W_STAGES];     // the bulk copy's bytes (1 arrival + tx): consumers, and producers that explode
    uint64_t empty[W_STAGES];      // consumers -> producers: 8 warp arrivals
};
static_assert(sizeof(TileSmem<TileCfg<false>>) <= 113 * 1024 && sizeof(TileSmem<TileCfg<true>>) <= 113 * 1024,
              "K1 must fit two CTAs per SM");
static_assert(offsetof(TileStage<TileCfg<false>>, diff) % 16 == 0 && sizeof(TileStage<TileCfg<false>>) % 16 == 0 &&
              offsetof(TileStage<TileCfg<true>>, diff) % 16 == 0 && sizeof(TileStage<TileCfg<true>>) % 16 == 0 &&
              offsetof(TileStage<TileCfg<true>>, px) % 16 == 0 && offsetof(TileStage<TileCfg<true>>, meta) % 16 == 0,
              "128-bit shared accesses of the metadata and the pieces, 64-bit ones of the difference array");
static_assert(TileCfg<false>::kRmax % W_PT == 0 && TileCfg<true>::kRmax % W_PT == 0, "reads per producer thread");
static_assert(TileCfg<true>::kPcap >= KDL_TILE_MAXOPS && TileCfg<true>::kPcap < 1024, "one read's pieces fit; 10-bit piece slot");

// kFlush: F_STORE = the weight columns hold stale data (first flush of a window stores, untouched tiles are stored
// as zeros); F_ADD = add to what is there; F_ATOMIC = `split` CTAs share a tile, the table was zeroed, flush with REDs.
template <int kFlush, bool kCx>
__global__ void __launch_bounds__(W_THREADS, 2)
pileup_tile_kernel(kdl_batch b, int32_t* __restrict__ counts, long long n_slots,
                   const uint32_t* __restrict__ tile_index, long long tile_lo, long long n_tiles, int split,
                   int zero_rest) {
    KDL_DYNAMIC_SMEM(smem_raw);
    using C = TileCfg<kCx>;
    using Smem = TileSmem<C>;
    using Stage = TileStage<C>;
    constexpr int W_RMAX = C::kRmax, W_CAPW = C::kCapW, W_PCAP = C::kPcap;
    constexpr bool kFresh = kFlush == F_STORE;
    constexpr int kAdd = kFlush == F_ATOMIC ? F_ATOMIC : F_ADD;
    Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int maxlen = b.max_simple_len;
    const long long n_units = n_tiles * split;

    if (tid == 0) {
        for (int s = 0; s < W_STAGES; ++s) {
            mbar_init(&sm.full[s], W_PRODUCERS);
            mbar_init(&sm.landed[s], 1);
            mbar_init(&sm.empty[s], W_CONSUMERS);
        }
    }
    for (int s = 0; s < W_STAGES; ++s) {
        for (int k = tid; k < KDL_TILE + 32; k += W_THREADS) sm.st[s].diff[k] = 0;
        if (tid < W_CONSUMERS) sm.st[s].carry[tid] = 0;
        if (tid == 0) sm.st[s].px[W_PCAP] = make_int4(0x10000000, (int)smem_u32(sm.st[s].seq), 0, 0);
    }
    if (tid < W_PRODUCERS * 4 + 4) sm.scan[tid] = 0;
    __syncthreads();

    if (warp >= W_CONSUMERS) {
        // =========================== PRODUCERS ====================================================
        reg_dealloc<TileRegs<kCx>::kProducer>();
        const int pw = warp - W_CONSUMERS;          // 0..3
        const int ptid = tid - 32 * W_CONSUMERS;    // 0..127
        int ps = 0;           // the ring slot of the item being produced
        uint32_t pph = 0;     // parity of that slot's round (flips when ps wraps)
        bool wrapped = false;
        auto acquire_stage = [&]() -> Stage& {
            if (wrapped) mbar_wait(&sm.empty[ps], pph ^ 1u);  // consumers released its last use
            return sm.st[ps];
        };
        auto publish = [&]() {  // this warp's part of the item is written; on to the next ring slot
            __syncwarp();
            if (lane == 0) mbar_arrive(&sm.full[ps]);
            if (++ps == W_STAGES) { ps = 0; pph ^= 1u; wrapped = true; }
        };

        // The producers run a software pipeline of their own: while an item is prepared, the three metadata words
        // of the NEXT item's reads (the same unit's next chunk, or the next unit's first) stream into sm.raw with
        // cp.async -- each thread fetches exactly the elements it will consume, so they need no barrier -- and the
        // index entry of the next unit's tile is loaded a unit ahead.  The few seq_off lookups that size an item are
        // plain loads of lines the prefetch has just pulled into L1.
        constexpr int PER = W_RMAX / W_PT;  // reads per producer thread and item
        struct Unit { uint32_t lo, hi, wa, wend; uint2 ic; uint2 cs; };  // as K0 wrote it (read indices are < 2^31)
        auto load_unit = [&](long long w, Unit& u) {  // loads only: nothing here waits for them
            if (w >= n_units) { u.lo = u.hi = u.wa = u.wend = 0; u.ic = make_uint2(0, 0); u.cs = make_uint2(0, 0); return; }
            const long long t = tile_lo + (split == 1 ? w : w / split);
            const uint4 ix = __ldg(reinterpret_cast<const uint4*>(tile_index + F_IDX * t));
            const uint4 iy = __ldg(reinterpret_cast<const uint4*>(tile_index + F_IDX * t + 4));
            u.lo = ix.x; u.hi = ix.y; u.wa = ix.z; u.wend = ix.w;
            u.ic = make_uint2(iy.x, iy.y);
            u.cs = make_uint2(iy.z, iy.w);
        };
        auto part_of = [&](const Unit& u, long long w, uint32_t& plo, uint32_t& phi) {  // this unit's share of the tile's reads
            if (split == 1) { plo = u.lo; phi = u.hi; return; }
            const long long n = (long long)u.hi - u.lo;
            const int part = (int)(w % split);
            plo = u.lo + (uint32_t)(n * part / split);
            phi = u.lo + (uint32_t)(n * (part + 1) / split);
        };
        uint32_t pf_start = 0xFFFFFFFFu;  // sm.raw holds (once this thread's cp.async group lands) reads [pf_start, + pf_cnt)
        int pf_cnt = 0;
        auto prefetch_raw = [&](uint32_t start, uint32_t end) {
            const int cnt = end > start ? (int)(end - start < (uint32_t)W_RMAX ? end - start : (uint32_t)W_RMAX) : 0;
            pf_start = start;
            pf_cnt = cnt;
            for (int i = ptid; i < cnt; i += W_PT) {
                cp_async4(&sm.raw[0][i], b.l_seq + start + i);
                cp_async4(&sm.raw[1][i], b.ref_start + start + i);
                cp_async4(&sm.raw[2][i], b.seq_off + start + i);
            }
        };
        Unit u, nu;
        load_unit(blockIdx.x, u);
        {
            uint32_t plo, phi;
            part_of(u, blockIdx.x, plo, phi);
            prefetch_raw(plo, phi);
        }

        for (long long w = blockIdx.x; w < n_units; w += gridDim.x) {
            load_unit(w + gridDim.x, nu);  // consumed at the end of this iteration
            const long long tile_slot = (tile_lo + (split == 1 ? w : w / split)) * KDL_TILE;
            uint32_t plo, phi;
            part_of(u, w, plo, phi);
            if (plo >= phi) {
                if (kFresh) {  // consumers must store zeros: a header-only item
                    Stage& st = acquire_stage();
                    if (ptid == 0) {
                        st.tile_slot = tile_slot; st.n_sub = 0; st.n_px = 0; st.flags = ITEM_FIRST | ITEM_LAST | ITEM_EMPTY;
                        mbar_expect_tx(&sm.landed[ps], 0);
                    }
                    publish();
                }
                cp_async_wait_all();  // (a thread never has two prefetches in flight to the same words)
                uint32_t nplo, nphi;
                part_of(nu, w + gridDim.x, nplo, nphi);
                prefetch_raw(nplo, nphi);
                u = nu;
                continue;
            }
            const bool one_contig = u.ic.x == u.ic.y;
            const long long slot_base = one_contig ? (long long)(((unsigned long long)u.cs.y << 32) | u.cs.x) - tile_slot : 0;
            uint32_t c0 = plo;
            bool first = true;
            while (c0 < phi) {
                cp_async_wait_all();  // this thread's prefetched words have landed
                const bool have = pf_start == c0 && pf_cnt > 0;
                uint32_t c1 = phi - c0 > (uint32_t)W_RMAX ? c0 + W_RMAX : phi;
                const uint32_t wa = c0 == u.lo ? u.wa : (b.seq_off[c0] & ~3u);
                uint32_t wend = c1 == u.hi ? u.wend : ((long long)c1 < b.n_reads ? b.seq_off[c1] : (uint32_t)b.seq4_words);
                bool skip = false;
                while (wend - wa > (uint32_t)W_CAPW) {
                    if (c1 - c0 == 1) { skip = true; break; }  // one read too long to stage: never tile-eligible
                    const uint32_t n = c1 - c0;                // cut where the capacity ends
                    uint32_t n2 = (uint32_t)((unsigned long long)n * W_CAPW / (wend - wa));
                    n2 = n2 >= n ? n - 1 : (n2 < 1 ? 1 : n2);
                    c1 = c0 + n2;
                    wend = b.seq_off[c1];
                }
                int n_sub = skip ? 0 : (int)(c1 - c0);
                // this thread's reads of the item
                int l[PER], rs[PER];
                uint32_t so[PER];
                if (have) {
#pragma unroll
                    for (int k = 0; k < PER; ++k) {
                        const int i = ptid + k * W_PT;
                        const int ii = i < n_sub ? i : ptid;  // (its own elements only: nobody else's have to be visible)
                        l[k] = sm.raw[0][ii];
                        rs[k] = sm.raw[1][ii];
                        so[k] = (uint32_t)sm.raw[2][ii];
                    }
                } else {
#pragma unroll
                    for (int k = 0; k < PER; ++k) {
                        const int i = ptid + k * W_PT;
                        const long long r = (long long)c0 + (i < n_sub ? i : 0);
                        l[k] = b.l_seq[r];
                        rs[k] = b.ref_start[r];
                        so[k] = b.seq_off[r];
                    }
                }
                // ---- own elements are in registers: the next item's words start streaming in -- this unit's next
                // chunk, or the next unit's first.  (Should the piece list cut this item short below, the prefetch is
                // for the wrong reads and the next item loads directly.)
                if (c1 < phi) {
                    prefetch_raw(c1, phi);
                } else {
                    uint32_t nplo, nphi;
                    part_of(nu, w + gridDim.x, nplo, nphi);
                    prefetch_raw(nplo, nphi);
                }
                // ---- stage + bulk copy first: the bytes fly while the metadata is written.  (If the piece list
                // later cuts the item short the copy has fetched a little more than needed: harmless.)
                Stage& st = acquire_stage();
                const int stage_id = ps;
                const uint32_t stage_parity = pph;
                const uint32_t seq_base = smem_u32(st.seq);
                {
                    const long long n_words = skip ? 0 : (long long)(wend - wa);
                    const long long avail = b.seq4_words - (long long)wa;
                    const long long want = (n_words + 3) & ~3ll;
                    const long long bulk_words = want <= avail ? want : (avail & ~3ll);
                    const uint32_t tx = (uint32_t)(bulk_words * 4);
                    if (ptid == 0) {  // announce the bytes (one arrival), then let the TMA engine copy them
                        mbar_expect_tx(&sm.landed[stage_id], tx);
                        if (bulk_words) bulk_g2s(st.seq, b.seq4 + wa, tx, &sm.landed[stage_id]);
                    }
                    if (bulk_words < n_words && ptid < 4) {  // the (at most one) partial granule at the array's end, by hand
                        const long long wq = bulk_words + ptid;
                        st.seq[wq] = wq < avail ? b.seq4[wa + wq] : 0u;  // (visible to all after the barriers below)
                    }
                }
                // ---- complex reads: where each one's pieces go (exclusive prefix in read order of: M-op count in the
                // low 16 bits, 1 per tile-eligible complex read above), and a cut of the item if they do not fit
                int pre[PER];
                int n_px = 0, n_cx = 0;  // pieces / tile-eligible complex reads of the item
                if constexpr (kCx) {
                    int ub[PER];
                    bool mine = false;
#pragma unroll
                    for (int k = 0; k < PER; ++k) {
                        const int i = ptid + k * W_PT;
                        const uint32_t lw = (uint32_t)l[k];
                        ub[k] = (i < n_sub && (lw & (KDL_COMPLEX | KDL_HARD)) == KDL_COMPLEX)
                                    ? (int)((lw >> KDL_NM_SHIFT) & KDL_NM_MASK) | 0x10000 : 0;
                        pre[k] = 0;
                        mine |= ub[k] != 0;
                    }
                    if (producer_sync_or(mine)) {  // (items without complex reads pay one barrier, nothing else)
#pragma unroll
                        for (int k = 0; k < PER; ++k) {
                            int incl = ub[k];  // reads ptid + k * 128: group g = 4 k + pw holds 32 consecutive reads
#pragma unroll
                            for (int d = 1; d < 32; d <<= 1) {
                                const int o = __shfl_up_sync(0xffffffffu, incl, d);
                                if (lane >= d) incl += o;
                            }
                            pre[k] = incl - ub[k];
                            if (lane == 31) sm.scan[4 * k + pw] = incl;
                        }
                        producer_sync();
                        int run = 0;
#pragma unroll
                        for (int g = 0; g < 4 * PER; ++g) {
                            const int t = sm.scan[g];
#pragma unroll
                            for (int k = 0; k < PER; ++k)
                                if (g == 4 * k + pw) pre[k] += run;
                            run += t;
                        }
                        n_px = run & 0xFFFF;
                        n_cx = run >> 16;
                        if (n_px > W_PCAP) {  // rare: cut the item behind the last read whose pieces still fit
                            int fits = 0;
#pragma unroll
                            for (int k = 0; k < PER; ++k) {
                                const int i = ptid + k * W_PT;
                                fits += __popc(__ballot_sync(0xffffffffu, i < n_sub && (pre[k] & 0xFFFF) + (ub[k] & 0xFFFF) <= W_PCAP));
                            }
                            if (lane == 0) atomicAdd(&sm.scan[4 * W_PRODUCERS], fits);
                            producer_sync();
                            n_sub = sm.scan[4 * W_PRODUCERS];  // >= 1: one read has at most KDL_TILE_MAXOPS <= kPcap pieces
                            c1 = c0 + n_sub;
#pragma unroll
                            for (int k = 0; k < PER; ++k) {
                                const int i = ptid + k * W_PT;
                                if (i >= n_sub) ub[k] = 0;
                                if (i == n_sub - 1) sm.scan[4 * W_PRODUCERS + 1] = pre[k] + ub[k];
                            }
                            producer_sync();
                            n_px = sm.scan[4 * W_PRODUCERS + 1] & 0xFFFF;
                            n_cx = sm.scan[4 * W_PRODUCERS + 1] >> 16;
                            if (ptid == 0) sm.scan[4 * W_PRODUCERS] = 0;
                        }
                        // (the next item's first write to sm.scan[g] comes after at least one more producer barrier:
                        // no thread still reads the totals then)
                    }
                }
                const bool last = c1 >= phi;
#pragma unroll
                for (int k = 0; k < PER; ++k) {
                    const int i = ptid + k * W_PT;
                    if (i < n_sub) {
                        long long g;
                        if (one_contig) {
                            g = slot_base + rs[k];
                        } else {
                            const int c = find_contig(b.contig_read_off, b.n_contigs, (long long)c0 + i);
                            g = b.contig_slot[c] + rs[k] - tile_slot;
                        }
                        const int gs = (int)g;  // inside (-reach_right, 512 + reach_left) by construction of the index
                        const int raddr = (int)(seq_base + ((so[k] - wa) << 2));
                        const uint32_t lw = (uint32_t)l[k];
                        int4 en;
                        if (l[k] > 0) {  // simple read (bit 31 clear)
                            const int cs = gs < 0 ? 0 : gs, ce = gs + l[k] > KDL_TILE ? KDL_TILE : gs + l[k];
                            if (cs < ce) {
                                atomicAdd(st.diff + cs, 1);
                                if (ce & (F_WIN - 1)) atomicAdd(st.diff + ce, -1);
                                // (the 32 sorted reads of a warp carry into the same two or three windows; summing them
                                // with ballots first was measured slower than letting the atomics collide: 0.231 / 0.217 ms)
                                for (int w = (cs >> 6) + 1; w <= ((ce - 1) >> 6); ++w) atomicAdd(st.carry + w, 1);
                            }
                            en = make_int4(((gs + 7) >> 3) << 2, raddr, ((l[k] + 7) >> 3) << 2, ((-gs) & 7) << 2);
                        } else if (kCx && (lw & KDL_HARD) == 0) {
                            // tile-eligible complex read: .z = 0 keeps the entry inert in the simple loop; the rest is
                            // what the explode below needs -- start, block address, first piece slot, SEQ length,
                            // M-op count (.w: bit 31 = marker, 24..30 M ops, 10..23 length, 0..9 piece slot)
                            en = make_int4(gs, raddr, 0, (int)(0x80000000u | (((lw >> KDL_NM_SHIFT) & KDL_NM_MASK) << 24) |
                                                               ((lw & 0x3FFFu) << 10) | (uint32_t)(pre[k] & 0x3FF)));
                        } else {
                            en = make_int4(((gs + 7) >> 3) << 2, raddr, 0, 0);  // K1g's: adds nothing here
                        }
                        st.gs[i] = gs;
                        st.meta[i + (i >> 3)] = en;
                    }
                }
                if (ptid < 40) {  // sentinels behind the last read
                    const int i = n_sub + ptid;
                    if (ptid < 32) st.gs[i] = 0x10000000;
                    st.meta[i + (i >> 3)] = make_int4(0x10000000, (int)seq_base, 0, 0);
                }
                if (ptid == 0) {
                    st.tile_slot = tile_slot;
                    st.n_sub = n_sub;
                    st.n_px = n_px;
                    st.flags = (first ? ITEM_FIRST : 0) | (last ? ITEM_LAST : 0);
                }
                if constexpr (kCx) {
                    if (n_cx > 0) {
                        // ---- the M / = / X segments of the complex reads become pieces (their CIGARs came with the
                        // bulk copy).  One thread per read: it only tracks the two cursors through the ops -- the
                        // insertion / deletion / clip updates of these reads are K1e's (pileup_general.cu), once per
                        // read instead of once per tile it touches.
                        mbar_wait(&sm.landed[stage_id], stage_parity);
                        // carries of this thread's pieces into windows 0..3 / 4..7, one byte each (<= PER reads of
                        // <= KDL_TILE_MAXOPS pieces): a deep pileup puts every piece of the item across the same two or
                        // three window borders, so they are summed per thread, then per warp, before they touch st.carry
                        static_assert(PER * KDL_TILE_MAXOPS <= 255, "byte counters of the piece carries");
                        uint32_t clo = 0, chi = 0;
#pragma unroll 1
                        for (int i = ptid; i < n_sub; i += W_PT) {  // (its own entries: no barrier needed)
                            const int4 en = st.meta[i + (i >> 3)];
                            if (en.w >= 0) continue;
                            const int nbw = (((en.w >> 10) & 0x3FFF) + 7) >> 3;
                            const uint32_t* rw = st.seq + (((uint32_t)en.y - seq_base) >> 2);  // the read's block
                            const int n_ops = (int)rw[nbw];
                            const uint32_t* ops = rw + nbw + 2;
                            int pos = en.w & 0x3FF;
                            const int pend = pos + ((en.w >> 24) & 0x7F);
                            int r = en.x, q = 0;
                            for (int o = 0; o < n_ops; ++o) {
                                const uint32_t cg = ops[o];
                                const int len = (int)(cg >> 4);
                                const int op = (int)(cg & 0xF);
                                if (op == 0 || op == 7 || op == 8) {  // M = X (kindel.py:49-54)
                                    const int s0 = r < 0 ? 0 : r, s1 = r + len > KDL_TILE ? KDL_TILE : r + len;
                                    if (s0 < s1) {
                                        const int v = r - q;  // slot of the read's base 0
                                        atomicAdd(st.diff + s0, 1);
                                        if (s1 & (F_WIN - 1)) atomicAdd(st.diff + s1, -1);
                                        const uint32_t bits = ((2u << ((s1 - 1) >> 6)) - 1u) & ~((2u << (s0 >> 6)) - 1u);  // windows (w0, w1]
                                        clo += ((bits & 0xFu) * 0x00204081u) & 0x01010101u;  // bit k -> byte k
                                        chi += ((bits >> 4) * 0x00204081u) & 0x01010101u;
                                        st.px[pos++] = make_int4(((v + 7) >> 3) << 2, en.y, nbw << 2,
                                                                 (((-v) & 7) << 2) | (s0 << 8) | (s1 << 20));
                                    }
                                    r += len;
                                    q += len;
                                } else if (op == 1) {  // I
                                    q += len;
                                } else if (op == 2) {  // D
                                    r += len;
                                } else if (op == 4) {  // S: op #0 is a left clip (query only), any other advances both
                                    if (o) r += len;
                                    q += len;
                                }
                                // N, H, P: no-op (kindel.py:49-63 has no branch for them)
                            }
                            while (pos < pend) st.px[pos++] = make_int4(0x10000000, (int)seq_base, 0, 0);  // covers nothing
                        }
                        __syncwarp();
                        uint32_t cw[4] = {clo & 0x00FF00FFu, (clo >> 8) & 0x00FF00FFu, chi & 0x00FF00FFu, (chi >> 8) & 0x00FF00FFu};
#pragma unroll
                        for (int d = 16; d; d >>= 1) {
#pragma unroll
                            for (int k = 0; k < 4; ++k) cw[k] += __shfl_xor_sync(0xffffffffu, cw[k], d);  // 16-bit halves: <= 32 * 192
                        }
                        if (lane >= 1 && lane < W_CONSUMERS) {  // window `lane`: byte lane & 3 of clo (lane < 4) / chi
                            const uint32_t pair = cw[(lane & 1) + ((lane >> 2) << 1)];
                            const int v = (int)((lane & 2) ? pair >> 16 : pair & 0xFFFFu);
                            if (v) atomicAdd(st.carry + lane, v);
                        }
                    }
                }
                publish();
                first = false;
                c0 = c1;
            }
            u = nu;
        }
        {   // END item
            Stage& st = acquire_stage();
            if (ptid == 0) {
                st.tile_slot = 0; st.n_sub = 0; st.n_px = 0; st.flags = ITEM_END;
                mbar_expect_tx(&sm.landed[ps], 0);
            }
            publish();
        }
        return;
    }

    // =============================== CONSUMERS ===================================================
    reg_alloc<TileRegs<kCx>::kConsumer>();
    const int quarter = lane >> 3;
    const int wlo = warp * F_WIN;
    const int p8b = (wlo >> 1) + 4 * (lane & 7);  // 4 * (lane's first slot / 8): byte offset of its word
    Planes acc;
    acc.clear();
    int rawacc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) rawacc[k] = 0;
    int2 dacc = make_int2(0, 0);  // the tile's items' difference entries of slots wlo + 2 lane, + 1 (summed: the scan is linear)
    int cacc = 0;                 // ... and their carries into this window
    int blocks_since_flush = 0;
    uint32_t pend8 = 0;  // weight-8 carry of an odd block, waiting for its partner
    bool stored = false;
    long long tile_slot = 0;

    // one block = 8 words per lane (the quarter's 8 reads / pieces) into the counters; two blocks share one ripple
    auto add_block = [&](const uint32_t (&x)[8]) {
        const uint32_t e8 = acc.add8_carry(x);
        if (blocks_since_flush & 1) {  // second block of a pair: eights + eights -> sixteens, one ripple
            uint32_t c16;
            csa(c16, acc.p[3], acc.p[3], pend8, e8);
            acc.template ripple<4>(c16);
        } else {
            pend8 = e8;
        }
        if (++blocks_since_flush == F_FLUSH_BLOCKS) {
            acc.template ripple<3>(pend8);  // F_FLUSH_BLOCKS is odd: one carry is pending
            if (kFresh && !stored)
                flush_window<F_STORE, false>(acc, rawacc, rawacc, counts, n_slots, tile_slot + wlo, lane);
            else
                flush_window<kAdd, false>(acc, rawacc, rawacc, counts, n_slots, tile_slot + wlo, lane);  // (coverage unused)
            stored = true;
            blocks_since_flush = 0;
        }
    };
    // the two staged words of entry `mt` that cover the lane's 8 slots, funnel-shifted into place; words outside
    // the read are predicated off and read as zero
    auto extract = [&](const int4& mt) -> uint32_t {
        const uint32_t jb = (uint32_t)(p8b - mt.x);  // byte offset of the read's word
        const uint32_t addr = (uint32_t)mt.y + jb;
        uint32_t hw, lw;
#ifndef KDL_HOST_EMU
        asm("{\n"
            ".reg .pred p, q;\n"
            "setp.lt.u32 p, %2, %3;\n"
            "setp.lt.u32 q, %4, %3;\n"
            "mov.u32 %0, 0;\n"
            "mov.u32 %1, 0;\n"
            "@p ld.shared.u32 %0, [%5];\n"
            "@q ld.shared.u32 %1, [%5+4];\n"
            "}\n"
            : "=&r"(hw), "=&r"(lw)
            : "r"(jb), "r"((uint32_t)mt.z), "r"(jb + 4u), "r"(addr));
#else
        hw = jb < (uint32_t)mt.z ? lds_u32(addr) : 0u;
        lw = jb + 4u < (uint32_t)mt.z ? lds_u32(addr + 4u) : 0u;
#endif
        return __funnelshift_l(lw, hw, (uint32_t)mt.w);
    };

    int s = -1;
    uint32_t parity = 1;
    for (;;) {
        if (++s == W_STAGES) s = 0;
        if (s == 0) parity ^= 1u;
        mbar_wait(&sm.full[s], parity);
        mbar_wait(&sm.landed[s], parity);
        Stage& st = sm.st[s];
        const int flags = st.flags;
        const int n_sub = st.n_sub;
        if (flags & ITEM_END) break;
        if (flags & ITEM_FIRST) {
            tile_slot = st.tile_slot;
            stored = false;
            blocks_since_flush = 0;  // (already 0 after the previous tile's final flush)
        }
        if (n_sub > 0) {
            {   // this warp's difference entries of the item; zeroed again for the stage's next item
                int2* dp = reinterpret_cast<int2*>(st.diff + wlo) + lane;
                const int2 dd = *dp;
                cacc += st.carry[warp];
                dacc.x += dd.x;
                dacc.y += dd.y;
                __syncwarp();
                *dp = make_int2(0, 0);
                if (lane == 0) st.carry[warp] = 0;
            }
            // ---- simple reads: those with start in (wlo - maxlen, wlo + 64), two lower bounds over the sorted starts
            int a, e;
            lower_bound_warp2(st.gs, n_sub, wlo - maxlen + 1, wlo + F_WIN, lane, a, e);
            for (int base = a & ~7; base < e; base += 32) {
                // 8 reads per lane and block: quarter q takes the 8 CONSECUTIVE reads base + 8q .. + 7.  No bounds
                // logic: a read that does not reach the lane's 8 slots (the up to 7 reads before a, reads [e, ...)
                // right of the window, complex reads, the sentinels) fails both range tests and contributes zero.
                uint32_t x[8];
                int4 mt[8];
                const int i0 = base + 8 * quarter;
                const int4* mp = st.meta + i0 + (i0 >> 3);
#pragma unroll
                for (int k = 0; k < 8; ++k) mt[k] = mp[k];
#pragma unroll
                for (int k = 0; k < 8; ++k) x[k] = extract(mt[k]);
                add_block(x);
            }
            // ---- pieces of complex reads: unsorted, so the warp first collects the ones that overlap its window
            if constexpr (kCx) {
                const int n_px = st.n_px;
                if (n_px > 0) {
                    unsigned short* qu = sm.queue[warp];
                    int qn = 0, qh = 0;  // pending entries, ring head
                    const int p0 = wlo + 8 * (lane & 7);  // the lane's first slot
                    auto run_block = [&](int n_valid) {
                        uint32_t x[8];
#pragma unroll
                        for (int k = 0; k < 8; ++k) {
                            const int en = 8 * quarter + k;
                            const int idx = en < n_valid ? (int)qu[(qh + en) & 63] : W_PCAP;
                            const int4 pv = st.px[idx];
                            const int s0 = (pv.w >> 8) & 0xFFF, s1 = (pv.w >> 20) & 0xFFF;
                            int lead = s0 - p0, trail = p0 + 8 - s1;
                            lead = lead < 0 ? 0 : (lead > 8 ? 8 : lead);
                            trail = trail < 0 ? 0 : (trail > 8 ? 8 : trail);
                            uint32_t mask = lead >= 8 ? 0u : (0xFFFFFFFFu >> (4 * lead));
                            mask &= trail >= 8 ? 0u : (0xFFFFFFFFu << (4 * trail));
                            int4 mt = pv;
                            mt.w = pv.w & 31;
                            x[k] = extract(mt) & mask;
                        }
                        add_block(x);
                    };
                    for (int base = 0; base < n_px; base += 32) {
                        const int i = base + lane;
                        const int w3 = i < n_px ? st.px[i].w : 0;
                        const int s0 = (w3 >> 8) & 0xFFF, s1 = (w3 >> 20) & 0xFFF;
                        const bool hit = s0 < wlo + F_WIN && s1 > wlo;
                        const unsigned m = __ballot_sync(0xffffffffu, hit);
                        if (hit) qu[(qh + qn + __popc(m & ((1u << lane) - 1u))) & 63] = (unsigned short)i;
                        qn += __popc(m);
                        __syncwarp();
                        if (qn >= 32) {
                            run_block(32);
                            qh = (qh + 32) & 63;
                            qn -= 32;
                            __syncwarp();
                        }
                    }
                    if (qn > 0) {
                        run_block(qn);
                        __syncwarp();
                    }
                }
            }
        }
        // this warp is done reading the stage: hand it back before the (global-memory) flush
        __syncwarp();
        if (lane == 0) mbar_arrive(&sm.empty[s]);
        if (flags & ITEM_LAST) {
            if (blocks_since_flush & 1) acc.template ripple<3>(pend8);
            int covacc[8];  // coverage of the lane's 8 slots by the tile's reads / pieces: one scan of the summed entries
            {
                const int both = dacc.x + dacc.y;
                int run = both;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const int o = __shfl_up_sync(0xffffffffu, run, d);
                    if (lane >= d) run += o;
                }
                const int c0 = cacc + run - dacc.y, c1 = cacc + run;  // slots wlo + 2 lane, + 1
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int src = 4 * (lane & 7) + k;
                    covacc[2 * k] = __shfl_sync(0xffffffffu, c0, src);
                    covacc[2 * k + 1] = __shfl_sync(0xffffffffu, c1, src);
                }
                dacc = make_int2(0, 0);
                cacc = 0;
            }
            if (kFresh && !stored) flush_window<F_STORE, true>(acc, rawacc, covacc, counts, n_slots, tile_slot + wlo, lane);
            else flush_window<kAdd, true>(acc, rawacc, covacc, counts, n_slots, tile_slot + wlo, lane);
            if (kFresh && zero_rest) {
                // columns 5..18 of the window hold an earlier pileup's sparse counts: zero them here, under the
                // counting, instead of in a pass of their own (K1e / K1g add to them after this kernel)
                int32_t* z = counts + tile_slot + wlo + 8 * (lane & 7);
                for (int col = 5 + quarter; col < KDL_NCOL; col += 4) {
                    int4* zp = reinterpret_cast<int4*>(z + (long long)col * n_slots);
                    zp[0] = make_int4(0, 0, 0, 0);
                    zp[1] = make_int4(0, 0, 0, 0);
                }
            }
            blocks_since_flush = 0;
        }
    }
}

}  // namespace kdl

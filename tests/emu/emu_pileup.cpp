// emu_pileup.cpp -- TEST INFRASTRUCTURE: K0 + the tile-owner kernel K1 (and every other kernel) compiled for the host and run
// under tests/emu/cuda_emu.h.  The kernel sources are included as they are (KDL_HOST_EMU only swaps the inline
// PTX for functional stand-ins); nothing here is part of the product.
#define KDL_HOST_EMU 1
#include "cuda_emu.h"

#include <vector>

#include "../../kindel_b200/csrc/kdl_common.cuh"
#include "../../kindel_b200/csrc/pileup_tile.cu"
#include "../../kindel_b200/csrc/pileup_general.cu"
#include "../../kindel_b200/csrc/pileup_simple.cu"
#include "../../kindel_b200/csrc/vote.cu"
#include "../../kindel_b200/csrc/assemble.cu"

static char g_error[512];

extern "C" {

const char* emu_last_error() { return g_error; }

// 0: threads in order (default), 1: reverse order, 2: a fresh pseudo-random order every scheduler round
void emu_set_schedule(int mode, unsigned long long seed) {
    emu::M().schedule = mode;
    emu::M().rng = seed * 0x9E3779B97F4A7C15ull + 1;
}

// K0 + K1 as kdl_pileup_range launches them.  mode: 0 = F_STORE (weight columns hold garbage), 1 = F_ADD,
// 2 = F_ATOMIC (`split` CTAs share a tile; the table must be zero or hold counts to add to).  cx: 1 = the kCx
// instantiation (piece lists for tile-eligible complex reads), 0 = the lean one with K1e counting their bases too.  All pointers are HOST pointers; `counts` is
// int32 [KDL_NCOL][n_slots]; tile_index is scratch of 8 words per tile of the whole slot space.
// Returns 0, or 1 with emu_last_error() set.
int emu_pileup(const kdl_batch* batch, int32_t* counts, long long n_slots, uint32_t* tile_index, long long tile_lo,
               long long n_tiles, int mode, int cx, int split, int32_t* ins_events, int zero_rest, int grid) {
    g_error[0] = 0;
    if (n_tiles <= 0) return 0;
    const kdl_batch b = *batch;
    const unsigned idx_grid = (unsigned)((n_tiles * 32 + 255) / 256);
    const char* err = emu::launch(idx_grid, 256, [&] { kdl::tile_index_kernel(b, tile_lo, n_tiles, tile_index); });
    if (!err) {
        err = emu::launch((unsigned)grid, (unsigned)kdl::W_THREADS, [&] {
#define KDL_EMU_TILE(M, X) kdl::pileup_tile_kernel<M, X>(b, counts, n_slots, tile_index, tile_lo, n_tiles, split, zero_rest)
            if (mode == 0) { if (cx) KDL_EMU_TILE(kdl::F_STORE, true); else KDL_EMU_TILE(kdl::F_STORE, false); }
            else if (mode == 1) { if (cx) KDL_EMU_TILE(kdl::F_ADD, true); else KDL_EMU_TILE(kdl::F_ADD, false); }
            else { if (cx) KDL_EMU_TILE(kdl::F_ATOMIC, true); else KDL_EMU_TILE(kdl::F_ATOMIC, false); }
#undef KDL_EMU_TILE
        });
    }
    if (!err && b.n_complex > b.n_hard) {  // K1e: the sparse updates of the tile-eligible complex reads
        if (cx) err = emu::launch((unsigned)((b.n_complex + 255) / 256), 256,
                                  [&] { kdl::pileup_events_kernel<1>(b, counts, n_slots, ins_events, 0); });
        else err = emu::launch((unsigned)((b.n_complex + 31) / 32), 256,
                               [&] { kdl::pileup_events_kernel<8>(b, counts, n_slots, ins_events, 1); });
    }
    if (err) {
        snprintf(g_error, sizeof g_error, "%s", err);
        return 1;
    }
    return 0;
}

#define EMU_RUN(grid, block, ...)                                              \
    do {                                                                        \
        const char* e_ = emu::launch((unsigned)(grid), (unsigned)(block), [&] { __VA_ARGS__; }); \
        if (e_) { snprintf(g_error, sizeof g_error, "%s", e_); return 1; }      \
    } while (0)

// The other pileup kernels, as kdl_pileup_range launches them: K1s (atomic fallback, all simple reads of an
// unsorted batch) and K1g (complex reads).  grid is kept small on purpose so the grid-stride loops stride.
int emu_pileup_simple(const kdl_batch* batch, int32_t* counts, long long n_slots, int32_t* err_flag, int grid) {
    g_error[0] = 0;
    const kdl_batch b = *batch;
    EMU_RUN(grid, 256, kdl::pileup_simple_atomic_kernel(b, counts, n_slots, err_flag));
    return 0;
}
// K1g: all = 0 walks the KDL_HARD reads (batch.hard_idx), all = 1 every complex read (the unsorted fallback)
int emu_pileup_general(const kdl_batch* batch, int32_t* counts, long long n_slots, int32_t* ins_events,
                       int32_t* err_flag, int all, int grid) {
    g_error[0] = 0;
    const kdl_batch b = *batch;
    if (all) {
        if (b.n_complex > 0) EMU_RUN(grid, 256, kdl::pileup_general_kernel(b, nullptr, b.n_reads, counts, n_slots, ins_events, err_flag));
    } else if (b.n_hard > 0) {
        EMU_RUN(grid, 256, kdl::pileup_general_kernel(b, b.hard_idx, b.n_hard, counts, n_slots, ins_events, err_flag));
    }
    return 0;
}
int emu_diagnose(const kdl_batch* batch, kdl_diag* diag) {
    g_error[0] = 0;
    const kdl_batch b = *batch;
    EMU_RUN(1, 1, kdl::diagnose_init_kernel(diag));
    if (b.n_hard > 0) EMU_RUN((b.n_hard + 255) / 256, 256, kdl::diagnose_kernel(b, diag));
    EMU_RUN(1, 1, kdl::diagnose_final_kernel(diag));
    return 0;
}
int emu_vote(const int32_t* counts, long long n_slots, long long min_depth_ceil, uint8_t* calls) {
    g_error[0] = 0;
    kdl::Peers none;
    none.n = 0;
    EMU_RUN((n_slots / 4 + 255) / 256, 256,
            kdl::vote_kernel<false>(counts, none, n_slots, 0, n_slots, min_depth_ceil, calls, nullptr));
    return 0;
}
int emu_derive(const int32_t* counts, long long n_slots, int32_t* out) {
    g_error[0] = 0;
    EMU_RUN((n_slots + 255) / 256, 256, kdl::derive_kernel(counts, n_slots, out));
    return 0;
}
// K4 over slots [slot_lo, slot_hi), one thread per slot as kdl_cdr_flags launches it
int emu_cdr_flags(const int32_t* counts, long long n_slots, long long slot_lo, long long slot_hi, double decay,
                  uint8_t* flags, uint8_t* bases) {
    g_error[0] = 0;
    if (slot_hi <= slot_lo) return 0;
    EMU_RUN((slot_hi - slot_lo + 255) / 256, 256,
            kdl::cdr_flags_kernel(counts, n_slots, slot_lo, slot_hi, decay, flags, bases));
    return 0;
}
// K5: block sums, the one-CTA scan over them, the scatter -- the grids of kdl_assemble.  block_sums holds
// kdl_assemble_scratch_words(n_slots) words, offsets n_slots + 1.
int emu_assemble(const uint8_t* calls, long long n_slots, const int64_t* contig_slot, const int32_t* contig_len,
                 int n_contigs, const int64_t* ins_slot, const uint32_t* ins_off, const uint8_t* ins_bytes, long long n_ins,
                 uint32_t* block_sums, uint32_t* offsets, uint8_t* out) {
    g_error[0] = 0;
    kdl::AssembleArgs a;
    a.calls = calls; a.n_slots = n_slots; a.contig_slot = contig_slot; a.contig_len = contig_len; a.n_contigs = n_contigs;
    a.ins_slot = ins_slot; a.ins_off = ins_off; a.ins_bytes = ins_bytes; a.n_ins = n_ins;
    const long long n_blocks = (n_slots + 1 + kdl::A_BLOCK - 1) / kdl::A_BLOCK;
    EMU_RUN(n_blocks, kdl::A_THREADS, kdl::assemble_sums_kernel(a, block_sums));
    EMU_RUN(1, kdl::A_THREADS, kdl::assemble_scan_sums_kernel(block_sums, n_blocks));
    EMU_RUN(n_blocks, kdl::A_THREADS, kdl::assemble_scatter_kernel(a, block_sums, offsets, out));
    return 0;
}
// K2p: vote over the SUM of several tables, each non-zero only inside its footprint [lo, hi)
int emu_vote_peers(const int32_t* const* tables, const long long* lo, const long long* hi, int n, long long n_slots,
                   long long slot_lo, long long slot_hi, long long min_depth_ceil, uint8_t* calls, int32_t* reduced) {
    g_error[0] = 0;
    kdl::Peers peers;
    peers.n = n;
    for (int p = 0; p < n; ++p) {
        peers.tab[p] = tables[p];
        peers.lo[p] = lo ? lo[p] : 0;
        peers.hi[p] = hi ? hi[p] : n_slots;
    }
    const long long quads = (slot_hi - slot_lo + 3) / 4;
    EMU_RUN((quads + 255) / 256, 256,
            kdl::vote_kernel<true>(nullptr, peers, n_slots, slot_lo, slot_hi, min_depth_ceil, calls, reduced));
    return 0;
}
// One epoch of the fused exchange for ALL ranks on one machine: every rank's K2x (publish ready, wait for the
// peers' tables, reduce + vote its slice, publish done) and then every rank's K2g (pull the peers' call slices).
// A kernel runs to completion here, so rank r's K2x could never see a flag that a LATER kernel sets: like
// kdl_exchange_signal on the device, the ready flags are published first.
int emu_exchange_epoch(const kdl_exchange* xs, int n_ranks, long long n_slots, long long min_depth_ceil, int epoch,
                       int grid) {
    g_error[0] = 0;
    std::vector<kdl::Exchange> ex(n_ranks);
    for (int r = 0; r < n_ranks; ++r) {
        const kdl_exchange& x = xs[r];
        kdl::Exchange& e = ex[r];
        e.peers.n = x.n_ranks;
        e.rank = x.rank;
        e.counter = x.counter;
        for (int p = 0; p < x.n_ranks; ++p) {
            e.peers.tab[p] = x.tables[p];
            e.peers.lo[p] = x.foot_lo[p];
            e.peers.hi[p] = x.foot_hi[p] > n_slots ? n_slots : x.foot_hi[p];
            e.calls[p] = x.calls[p];
            e.ready[p] = x.ready[p];
            e.done[p] = x.done[p];
            e.slice_lo[p] = x.slice_lo[p];
            e.slice_hi[p] = x.slice_hi[p];
        }
        e.ready_local = x.ready[x.rank];
        e.done_local = x.done[x.rank];
    }
    for (int r = 0; r < n_ranks; ++r) EMU_RUN(1, 32, kdl::exchange_signal_kernel(ex[r], epoch));
    for (int r = 0; r < n_ranks; ++r) EMU_RUN(grid, 256, kdl::vote_exchange_kernel(ex[r], n_slots, min_depth_ceil, epoch));
    for (int r = 0; r < n_ranks; ++r) {
        for (int p = 0; p < n_ranks; ++p) {  // blockIdx.y = peer: the emulator's grid is one-dimensional
            const char* e_ = emu::launch_y((unsigned)grid, (unsigned)p, (unsigned)n_ranks, 256,
                                           [&] { kdl::exchange_gather_kernel(ex[r], epoch); });
            if (e_) { snprintf(g_error, sizeof g_error, "%s", e_); return 1; }
        }
    }
    return 0;
}

// ---- self-test of the emulator: a bulk copy must not be visible before its mbarrier completes -----------
namespace {
struct alignas(16) SelfSmem {
    uint32_t data[64];
    uint64_t bar;
};
int selftest(bool wait) {
    static uint32_t src[64] __attribute__((aligned(16)));
    static int mismatches;
    for (int i = 0; i < 64; ++i) src[i] = 0x1000u + (uint32_t)i;
    mismatches = 0;
    const char* err = emu::launch(1, 64, [&] {
        SelfSmem& sm = *reinterpret_cast<SelfSmem*>(kdl::smem_raw);
        const int tid = (int)threadIdx.x;
        if (tid == 0) kdl::mbar_init(&sm.bar, 1);
        __syncthreads();
        if (tid == 0) {
            kdl::mbar_expect_tx(&sm.bar, sizeof sm.data);
            kdl::bulk_g2s(sm.data, src, sizeof sm.data, &sm.bar);
        }
        if (wait) kdl::mbar_wait(&sm.bar, 0);
        if (sm.data[tid] != src[tid]) atomicAdd(&mismatches, 1);
        __syncthreads();
    });
    if (err) return -1;
    return mismatches ? 1 : 0;
}
}  // namespace

int emu_selftest_missing_wait() { return selftest(false); }
int emu_selftest_missing_wait_fixed() { return selftest(true); }

}  // extern "C"

// Fused bidirectional LSTM layer for sm_100a: input projection + recurrence in ONE kernel, no xg tensor in HBM.
//
// nn.LSTM semantics (PyanNet2.py:95,170; PyanNet.py:105,181): gates = W_ih x_t + b_ih + W_hh h_{t-1} + b_hh;
// i,f,o = sigmoid, g = tanh; c_t = f*c_{t-1} + i*g; h_t = o*tanh(c_t).
//
// The two-kernel layer (gemm_xg_pair_kernel -> xg in HBM -> lstm_tc_kernel) moved 8 KB of fp32 xg per frame and layer
// (107 of the 140 GB a 4096 x 8 s step moved) and had room for only ONE fp16 plane of W_hh in tensor memory.  Here a
// CLUSTER OF 4 CTAs owns up to 128 sequences of one direction and splits the HIDDEN UNITS: CTA r computes the four
// gates of units [32 r, 32 r + 32) = 128 gate rows = one MMA M tile.  Per CTA, tensor memory (512 columns) holds
//   * W_hh rows of its units as TWO fp16 planes (W_hi, W' -- the scaled split below): 128 columns,
//   * W_ih rows of its units as two planes (W_hi + W_lo or W_hi + W'):                <= 256 columns (D <= 256),
//   * the gate accumulators of up to 8 parts of 16 sequences:                           128 columns,
// so all weights of the layer stay resident for all T steps; the only HBM traffic is x_t in (fp16 planes) and h_t out
// (the layer output planes).
//
// Roles of a CTA (25 warps):
//   * TMA producer: x tiles of (step, pair of parts), multicast to the cluster (each CTA fetches a quarter of every tile);
//   * 2 input-product issuers (pairs of parts by parity):     acc(s, q)  = W_ih . x_s   (tcgen05.mma N = 32, A = weights in
//     TMEM), up to one step ahead of the recurrence;
//   * 2 recurrent-product issuers (parts by parity):          acc(s, q) += W_hh . h_{s-1}  as soon as the part's h tile is
//     complete -- the critical path.  Four issuing threads because tcgen05.mma issue blocks at the tensor pipe's pace and a
//     commit drains it: a single thread left the pipe idle during every barrier wait, and a thread spends ~2/3 of a part
//     slot in waits and commits;
//   * 16 pointwise warps: warp (pg, g) serves parts pg and pg + 4 alternately (while one part's h travels, the other is
//     computed) and owns TMEM lane quarter g.  Lane 32 g + l of the accumulator is gate l >> 3 of unit 8 g + (l & 7):
//     two 16x256b TMEM loads then give each lane all four gates of one unit for four sequences, with no (gate x sequence)
//     transposition through shared memory.  One warp of the group polls acc_ready and releases the other three through a
//     named barrier, and the staged h slice goes to the sender through another (F_BAR_ACC, F_BAR_SLICE): blocked warps
//     issue nothing, where polling ones took issue slots from the pointwise pass;
//   * 4 exchange-sender warps (h exchange over distributed shared memory): the pointwise warps write h_s (fp32) into the CTA's
//     own 2 KB staging slice of the part and end their pass there; a sender warp reads the slice, splits it into the two fp16
//     planes (operand layout) and stores them with 16-byte st.async stores into k-block `rank` of the part's operand tile in all
//     four CTAs (the destination mbarriers count the bytes), then the same chunks into the layer output planes.  The MMA K
//     index is free as long as A and B agree: K block r (64 slots = one 128-byte swizzled row) is [h1 of units 32r..32r+31 |
//     h2 of the same units], exactly what CTA r produces, so a CTA's contribution is ONE contiguous box.
//
// What bounds it (profiles/r02_lstm_fused.md): a step of a cluster with n parts in flight took ~1.6 us + 0.26 us (n - 1) in round 2
// (now ~1.1 us + 0.28 us (n - 1), see kStepUs in the launcher): a fixed
// chain latency (recurrent MMAs -> accumulator read -> cell arithmetic -> h exchange -> next MMAs, ~2 900 cycles) plus a per-part
// cost of ~475 cycles: a part needs 384 tensor-pipe cycles (16 recurrent MMAs x 8 + 16 input MMAs x 16), 6 KB out + 6 KB in over
// the SM-to-SM port (~17 B/clk: 360-720 cycles) and ~320 issue slots per SM sub-partition.  n = 8 is all the accumulator columns
// TMEM has left, so half of the step is unhidden latency.  Replacing 12 of the 16 acc_ready pollers and the 4 slice pollers by named
// barriers (~160 -> ~86 polls per step and CTA) cut the one-part step to 1.18 us and the layer by 3.4 %, but not the per-part slope
// (profiles/r03_lstm_fused_handoffs.md): the issue slots taken by polls are not what sets the per-part cost.  The pointwise pass
// is a dependent chain whose latency the step follows: taking the shared-memory transposition out of it (16x256b TMEM loads)
// cut the layer by 13 % (profiles/r04_lstm_fused_tmem_layout.md), while making the pass 32 columns wide on pairs of parts made it
// slower (profiles/r04_lstm_fused_pairs.md).  Moving the plane split and the layer-output store from the pass to the sender
// warps, which were idle most of the step, took ~95 of its ~225 instructions and cut the layer by another 9 %
// (profiles/r05_lstm_fused_sender_split.md).  Exchange mechanisms tried: cp.async.bulk by a sender thread (~3000 cycles per
// copy through the TMA unit), st.async from the pointwise warps (they stall on the port), and an exchange through the output
// planes in L2 (TMA store + multicast TMA load: two ~1-2 us TMA round trips on the per-step chain; that variant showed
// intermittent launch failures -- in hindsight probably the x_full race described at bar_x_full, which any delay of the x tiles
// exposes -- and is kept only as tools/experiments/lstm_fused_l2_exchange.cu.txt).
//
// Precision (DESIGN.md "Precision"): every product is split-precision with fp32 accumulation.  Activations travel as the
// scaled split x1 = fp16((1 - s) x), x2 = fp16(x - x1), s = 2^-6, weights as W_hi = fp16(W), W' = fp16(W_hi + W_lo / s):
// x1 . W_hi + x2 . W' = x . W to ~2^-18 with TWO fp16 MMAs.  The recurrent product uses the same split for h, so W_hh has
// the accuracy of two planes (the single-plane W_hh of lstm_tc.cu was the dominant error of the old path: 1.3e-3 on p at
// logit spread 2).  Layer 0 may take (hi, lo) planes and three MMAs (x_lo.W_hi + x_hi.W_lo + x_hi.W_hi).  The output
// planes are always the scaled split (they ARE the recurrent operand); a consumer that treats them as (hi, lo) in a
// three-term product (the head, or a terms = 3 layer) loses only the x2 . W_lo term, 2^-17 relative.
//
// Algorithmic work per (sequence, frame, direction): FLOPs 2 * 512 * (D + 128); HBM bytes 2 * 2 * D8 (x planes read,
// shared by both directions through L2) + 512 (y planes written).
#include "kernels.cuh"
#include "tc05.cuh"
#include <stdlib.h>
#include <algorithm>
#include <mutex>

namespace b200vad {

using namespace tc;

constexpr int FC = 4;                       // CTAs per cluster
constexpr int FU = kHidden / FC;            // hidden units per CTA (32)
constexpr int FPN = 16;                     // sequences per part (MMA N)
constexpr int FMAXP = 8;                    // parts per work item (128 sequences per cluster)
constexpr int F_PW_WARPS = 16;              // pointwise warps: warp w owns TMEM lane quarter w & 3 of parts (w >> 2) and (w >> 2) + 4
constexpr int F_W_PROD = F_PW_WARPS;        // TMA producer of the x tiles
constexpr int F_W_MMA = F_W_PROD + 1;       // 2 recurrent-product issuers (even / odd parts; the first also owns the TMEM allocation)
constexpr int F_W_MMAX = F_W_PROD + 3;      // 2 input-product issuers (even / odd parts)
constexpr int F_W_SEND = F_W_PROD + 5;      // 4 exchange senders (own staging slice -> k-block `rank` of all four CTAs' operand tiles):
                                            // sender k serves parts k and k + 4, like the pointwise warps (4 k .. 4 k + 3)
constexpr int F_THREADS = (F_W_PROD + 9) * 32;   // 25 warps = 800 threads
constexpr int F_BOX = FPN * 128;            // one h k-block of a part: 16 rows x 128 bytes = 2 KB
constexpr int F_XBOX = 2 * F_BOX;           // one x TMA box: the 32 rows of a PAIR of parts (the input products run on pairs, MMA N = 32)
constexpr int F_HTILE = FC * F_BOX;         // h operand tile of a part: 4 k-blocks (one per source CTA) = 8 KB
constexpr int F_STAGING = 2 * FMAXP * F_BOX; // own h slices [step parity][part][16 rows][128 B] (source of the exchange copies): 32 KB
constexpr int F_ACC_COL = 0;                // TMEM columns [0, 128): accumulators, part p at 16 p
constexpr int F_WHH_COL = FMAXP * FPN;      // [128, 256): W_hh, k-step j at 128 + 8 j
constexpr int F_WIH_COL = F_WHH_COL + 128;  // [256, 256 + 16 nk): W_ih plane a then plane b
constexpr int F_MAX_STAGES = 16;
constexpr int F_SMEM_FIXED = FMAXP * F_HTILE + F_STAGING;   // 96 KB
constexpr int F_SMEM_MAX = 232448;          // 227 KB per CTA

struct FusedParams {
    const __half* wih_hi;    // [2 * 512][ldw]  (gate-scaled, api.cu packing)
    const __half* wih_lo;
    const __half* whh_hi;    // [2][512][128]
    const __half* whh_lo;
    const float* bias;       // [2 * 512] b_ih + b_hh, gate-scaled
    __half* y_a;             // layer output planes [B][T][256]
    __half* y_b;
    int B, T;
    int nk;                  // k-steps of 16 of the input projection: ceil(D / 16)
    int kblocks;             // 64-wide k blocks per x plane (TMA boxes per plane)
    int ldw;                 // row pitch of wih planes (elements)
    int terms;               // 2: planes are the scaled (x1, x2) split, plane b of W_ih is W';  3: (hi, lo) planes, plane b is W_lo
    int items_per_dir;       // work items per direction; parts are spread evenly over them
    int stages;              // x ring depth
    int prefetch_steps;      // L2 prefetch distance of the x tiles, in time steps (0 = off)
    int flags;               // timing probes (wrong results): 2 no y store, 4 no cell math, 8 no recurrent MMAs, 16 no input MMAs, 32 wait-time table, 64 timeline
};

// wait-time probe (flags & 32, tools/fused_ablate.py): per (CTA, warp, wait tag) cycles spent in non-immediate waits, their count,
// and the mbarrier polls of the site (try_wait / test_wait instructions, immediate ones included); tag 0 = kernel cycles, steps run
constexpr int F_DBG_TAGS = 8, F_DBG_FIELDS = 3, F_DBG_WARPS = 25, F_DBG_MAX_CTAS = 148;
__device__ long long g_fused_dbg[F_DBG_MAX_CTAS * F_DBG_WARPS * F_DBG_TAGS * F_DBG_FIELDS];

// timeline probe (flags & 64): clock64 stamps of one part (part 0 of CTA 0's first item) over F_TRACE_STEPS steps, 16 per step:
// recurrent issuer 0 h_ready seen, 1 MMAs committed; pointwise warp 0: 2 acc_ready, 3 accumulator read, 4 / 5 exponentials,
// 10 cell arithmetic done, 12 pass done (fp32 h staged and handed over at the slice barrier); sender: 7 slice received, 8 exchange
// issued, 14 layer output stored; input issuer: 9 start, 13 x_full, 15 committed.  (Until the sender split the planes, 12 came
// after the plane split and the layer-output store of the pointwise warp, 8 was the sender's end and 14 was unused.)
constexpr int F_TRACE_S0 = 100, F_TRACE_STEPS = 8;
__device__ long long g_fused_trace[F_TRACE_STEPS * 16 + 128];   // + per-part stamps of the two MMA threads over two steps (flag 128)

// last words of a wait that timed out: written to page-locked HOST memory (readable after the context died), see lstm_fused_last_timeout
__device__ volatile int* g_fused_err_host = nullptr;

// h exchange variant: 0 = st.async (every 16-byte store credits the destination's h_ready barrier), 1 = plain remote
// shared-memory stores + ONE release arrive per destination CTA
#ifndef FUSED_EXCH_PLAIN
#define FUSED_EXCH_PLAIN 0
#endif
#define FUSED_WAIT(bar, parity, tag) mbar_wait_tag<false>(bar, parity, tag, wacc)
#define FUSED_WAIT_CLUSTER(bar, parity, tag) mbar_wait_tag<true>(bar, parity, tag, wacc)
template <bool CLUSTER_ACQUIRE>
__device__ __forceinline__ void mbar_wait_tag(uint32_t bar, uint32_t parity, int tag, long long* wacc) {
    if (!wacc && (CLUSTER_ACQUIRE ? mbar_try_wait_cluster(bar, parity) : mbar_try_wait(bar, parity))) return;
    if (wacc && !CLUSTER_ACQUIRE) {                                     // probe mode: count every wait that is not already satisfied
        wacc[F_DBG_FIELDS * tag + 2] += 1;
        if (mbar_test_wait(bar, parity)) return;
    }
    const long long t0 = wacc ? clock64() : 0;
    // suspended in hardware for up to 20 us per try (the default limit is ~80 cycles: see mbar_try_wait_hint); the time
    // bound (~2 s) is checked once per 64 tries
    unsigned tries = 0;
    long long tb = 0;
    while (!(CLUSTER_ACQUIRE ? mbar_try_wait_cluster(bar, parity) : mbar_try_wait_hint(bar, parity, 20000u))) {
        if ((++tries & 63u) != 0) continue;
        const long long now = clock64();
        if (tb == 0) tb = now;
        if (now - tb > 4000000000LL) {   // ~2 s
            volatile int* e = g_fused_err_host;
            if (e && e[0] == 0) {                              // (racy on purpose: any one record is enough)
                e[0] = 1; e[1] = (int)blockIdx.x; e[2] = (int)threadIdx.x; e[3] = tag; e[4] = (int)bar; e[5] = (int)parity; e[6] = (int)gridDim.x;
                __threadfence_system();
            }
            printf("b200vad lstm_fused: wait timed out (block %d thread %d tag %d bar 0x%x parity %u)\n", blockIdx.x, threadIdx.x, tag, bar,
                   parity);
            __trap();
        }
    }
    if (wacc) { wacc[F_DBG_FIELDS * tag] += clock64() - t0; wacc[F_DBG_FIELDS * tag + 1] += 1; wacc[F_DBG_FIELDS * tag + 2] += tries + 1; }
}

// Named barriers of the per-step chain (IDs 0 = __syncthreads and 9-15 are free).  A warp blocked in bar.sync issues nothing,
// where an mbarrier wait keeps polling (the suspend-time hint is capped by the hardware): polls were ~30 % of the kernel's
// issued instructions, on the same four schedulers that run the pointwise pass.
//   * F_BAR_ACC + pg (1-4), 128 threads: the 4 pointwise warps of part group pg, once per (step, part q in {pg, pg + 4} with
//     q < nparts), after the group's poller (warp 5 pg, lane quarter g == pg: one poller per SM sub-partition) has seen
//     acc_ready(q).  The poller's mbarrier wait keeps the bounded wait and its time-out record.
//   * F_BAR_SLICE + pg (5-8), 160 threads: the same 4 warps and sender warp pg, once per (step s < T, part q in {pg, pg + 4}
//     with q < nparts), when the part's fp32 h_s slice is staged.  The sender turns it into the fp16 planes, exchanges them
//     (s + 1 < T) and stores the layer output (every step, the last one included).  Replaces an mbarrier arrive + sender poll;
//     holding the pointwise warps until the sender arrives costs the chain nothing, because what they wait for next, acc_ready
//     of the group's other part, needs the sender's previous send (h of that part) to have landed anyway.
// Both sides of a barrier run the same (s, q) sequence from the same conditions (q < nparts per item, every s < T), and
// bar.sync blocks every participant until all have arrived: no participant can arrive at generation n + 1 before generation n
// completed, so generations cannot mix.  A participation mismatch would hang instead of trapping.
constexpr uint32_t F_BAR_ACC = 1, F_BAR_SLICE = 5;
__device__ __forceinline__ void fused_bar(uint32_t id, uint32_t threads, int tag, long long* wacc) {
    const long long t0 = wacc ? clock64() : 0;
    named_bar_sync(id, threads);
    // every passage, no polls.  The counts are exact; the times measured so far read implausibly low (0.2-0.6 % of the kernel for
    // warps that wait on the poller), so they are not used (profiles/r03_lstm_fused_handoffs.md)
    if (wacc) { wacc[F_DBG_FIELDS * tag] += clock64() - t0; wacc[F_DBG_FIELDS * tag + 1] += 1; }
}

// The MMA-issuing threads are serial resources (one tcgen05.mma of N = 16 occupies the tensor pipe for 8 cycles):
// descriptors are formed by ONE add on the low word of a per-slot base (the swizzled K-major tile layout makes the
// start-address field additive), the loops are fully unrolled (NK, TERMS are template parameters), and no divisions.
constexpr uint32_t F_DESC_HI = (uint32_t)(1024 >> 4) | (1u << 14) | (2u << 29);   // SBO 1024 B, descriptor version 1, SWIZZLE_128B
__device__ __forceinline__ uint64_t fdesc(uint32_t lo) {
    uint64_t d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo), "r"(F_DESC_HI));
    return d;
}
__device__ __forceinline__ uint32_t fdesc_lo(uint32_t smem_addr) { return (smem_addr & 0x3FFFFu) >> 4; }

// NK > 0: k-steps of the input projection known at compile time (5: 80 mel bins, 4: 60 SincNet channels, 16: 256 LSTM outputs);
// NK = 0: run-time p.nk / p.terms (any D <= 256; slower issue loop)
template <int NK, int TERMS, bool PROBE>
__global__ void __cluster_dims__(FC, 1, 1) __launch_bounds__(F_THREADS, 1)
lstm_fused_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, FusedParams p) {
    extern __shared__ unsigned char smem_dyn[];
    const uint32_t smem_base = (smem_u32(smem_dyn) + 1023u) & ~1023u;
    unsigned char* const smem_gen = smem_dyn + (smem_base - smem_u32(smem_dyn));
    const uint32_t h_off = 0;                                  // [part 8][k-block 4][16 rows][128 B]
    const uint32_t g_off = FMAXP * F_HTILE;                    // staging [step parity 2][part 8][16 rows][128 B]
    const uint32_t x_off = g_off + F_STAGING;                  // [stage][plane 2][k-block][16 rows][128 B]
    const int nk = NK > 0 ? NK : p.nk;
    const int terms = NK > 0 ? TERMS : p.terms;
    const uint32_t stage_bytes = 2u * p.kblocks * F_XBOX;     // one stage = the x tile of a pair of parts
    const uint32_t bar_base = smem_base + x_off + p.stages * stage_bytes;
    // x_full: ONE SET PER INPUT ISSUER (a slot of pair pp is consumed by issuer pp & 1).  With a single set and an odd ring depth
    // (3 stages at D = 256) successive phases of a stage's barrier are waited on by DIFFERENT threads; a thread that reaches its
    // slot before the other thread's (earlier) slot of the same stage has even landed then waits on a parity that aliases the
    // phase before last and passes at once -- stale tile, an extra commit on x_empty, and with it a corrupted ring (seen as an
    // `unspecified launch failure` whenever the x loads were slow: a second stream saturating HBM).  With its own set every
    // barrier is waited on by one thread, phase after phase.
    auto bar_x_full = [&](int me, int s) { return bar_base + (me ? 832 : 0) + 8 * s; };
    auto bar_x_empty = [&](int s) { return bar_base + 128 + 8 * s; };
    auto bar_acc_ready = [&](int q) { return bar_base + 256 + 8 * q; };
    auto bar_acc_free = [&](int q) { return bar_base + 320 + 8 * q; };
    auto bar_h_ready = [&](int q) { return bar_base + 384 + 8 * q; };
    auto bar_h_free = [&](int q) { return bar_base + 448 + 8 * q; };
    const uint32_t tmem_slot = bar_base + 512;
    auto bar_x_done = [&](int pp) { return bar_base + 592 + 8 * pp; };   // per pair of parts

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int cluster_id = blockIdx.x / FC, num_clusters = gridDim.x / FC;
    const int T = p.T;
    const int P = (p.B + FPN - 1) / FPN;                      // parts per direction
    const int ipd = p.items_per_dir;
    const int num_items = 2 * ipd;
    const int base_parts = P / ipd, rem_parts = P % ipd;

    if (threadIdx.x == 0) {
        for (int s = 0; s < F_MAX_STAGES; ++s) { mbar_init(bar_x_full(0, s), 1); mbar_init(bar_x_full(1, s), 1); mbar_init(bar_x_empty(s), FC); }
        for (int q = 0; q < FMAXP; ++q) {
            mbar_init(bar_acc_ready(q), 1);
            mbar_init(bar_acc_free(q), 4);
            mbar_init(bar_h_ready(q), FUSED_EXCH_PLAIN ? FC : 1);
            mbar_init(bar_h_free(q), FC);
            mbar_init(bar_x_done(q), 1);
        }
        mbar_fence_init();
    }
    if (warp == F_W_MMA) tmem_alloc<512>(tmem_slot);
    tc_fence_before();
    cluster_sync_all();                                       // every CTA's barriers exist before any remote arrive / multicast
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

    // wait-time probe: lane 0 of every warp accumulates straight into its row of the global table (probe mode only)
    long long* const wacc = (PROBE && (p.flags & 32) && lane == 0 && blockIdx.x < F_DBG_MAX_CTAS)
                                ? &g_fused_dbg[((size_t)blockIdx.x * F_DBG_WARPS + warp) * (F_DBG_FIELDS * F_DBG_TAGS)] : nullptr;
    if (wacc) {
        for (int i = 0; i < F_DBG_FIELDS * F_DBG_TAGS; ++i) wacc[i] = 0;
        wacc[0] = -clock64();
    }
    long long* const trace = (PROBE && (p.flags & 64) && blockIdx.x == 0 && lane == 0) ? g_fused_trace : nullptr;
    // persistent role state (phases carry over from item to item)
    int xst = 0;                                              // producer / input-product issuer: next x ring stage ...
    uint32_t xph = 0;                                         // ... and its phase
    uint32_t ph_a = 0, ph_b = 0;                              // per-part phase bits (meaning depends on the role)
    uint32_t xfph = 0;                                        // input-product issuer: phase bits of its own x_full set, per stage
    int loaded_dir = -1;

    for (int item = cluster_id; item < num_items; item += num_clusters) {
        const int dir = item / ipd, ii = item - dir * ipd;
        const int nparts = base_parts + (ii < rem_parts ? 1 : 0);
        const int part0 = ii * base_parts + min(ii, rem_parts);
        const int seq0 = part0 * FPN;
        if (nparts == 0) continue;                            // (uniform over the cluster)
        const bool tr_item = trace && item == cluster_id;
        if (wacc) wacc[1] += T;                               // steps this CTA runs (the per-step normaliser of the table)

        // ---------------- weights of this direction -> tensor memory (pointwise warps; only when the direction changes)
        if (warp < F_PW_WARPS && loaded_dir != dir) {
            const int wg = warp >> 2, g = warp & 3;
            const uint32_t lane_addr = tmem_base + ((uint32_t)(g * 32) << 16);
            // TMEM lane 32 g + l holds gate l >> 3 of unit 8 g + (l & 7) of this CTA: the row pattern of a 16x256b TMEM load, which
            // gives lane l rows l >> 2 and (l >> 2) + 8 of a 16-lane half, so that two loads bring it all four gates of unit l >> 2
            const int grow = dir * kGates + (lane >> 3) * kHidden + (int)rank * FU + 8 * g + (lane & 7);   // packed weight row of this TMEM lane
            // W_hh: k-step j holds plane (j >> 1) & 1 of units 32 (j >> 2) + 16 (j & 1) .. + 15  (K block j >> 2 = source CTA)
            for (int j = wg; j < 16; j += 4) {
                const int u0 = 32 * (j >> 2) + 16 * (j & 1), plane = (j >> 1) & 1;
                const uint4* hp = reinterpret_cast<const uint4*>(p.whh_hi + (size_t)grow * kHidden + u0);
                const uint4* lp = reinterpret_cast<const uint4*>(p.whh_lo + (size_t)grow * kHidden + u0);
                uint32_t r[8];
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const uint4 vh = __ldg(hp + i), vl = __ldg(lp + i);
                    const uint32_t hw[4] = {vh.x, vh.y, vh.z, vh.w}, lw[4] = {vl.x, vl.y, vl.z, vl.w};
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        if (plane == 0) {
                            r[4 * i + e] = hw[e];
                        } else {
                            const float2 fh = __half22float2(*reinterpret_cast<const __half2*>(&hw[e]));
                            const float2 fl = __half22float2(*reinterpret_cast<const __half2*>(&lw[e]));
                            const __half2 wp = __floats2half2_rn(fmaf(fl.x, 1.f / kPlaneScale, fh.x), fmaf(fl.y, 1.f / kPlaneScale, fh.y));
                            r[4 * i + e] = *reinterpret_cast<const uint32_t*>(&wp);
                        }
                    }
                }
                tmem_st8(lane_addr + F_WHH_COL + 8 * j, r);
            }
            // W_ih: plane a = W_hi, plane b = W_lo (terms 3) or W' (terms 2); k-step j of plane pl at F_WIH_COL + pl * 8 nk + 8 j
            for (int j = wg; j < 2 * nk; j += 4) {
                const int pl = j >= nk, kj = pl ? j - nk : j;
                const uint4* hp = reinterpret_cast<const uint4*>(p.wih_hi + (size_t)grow * p.ldw + 16 * kj);
                const uint4* lp = reinterpret_cast<const uint4*>(p.wih_lo + (size_t)grow * p.ldw + 16 * kj);
                uint32_t r[8];
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const uint4 vh = __ldg(hp + i), vl = __ldg(lp + i);
                    const uint32_t hw[4] = {vh.x, vh.y, vh.z, vh.w}, lw[4] = {vl.x, vl.y, vl.z, vl.w};
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        if (!pl) {
                            r[4 * i + e] = hw[e];
                        } else if (terms == 3) {
                            r[4 * i + e] = lw[e];
                        } else {
                            const float2 fh = __half22float2(*reinterpret_cast<const __half2*>(&hw[e]));
                            const float2 fl = __half22float2(*reinterpret_cast<const __half2*>(&lw[e]));
                            const __half2 wp = __floats2half2_rn(fmaf(fl.x, 1.f / kPlaneScale, fh.x), fmaf(fl.y, 1.f / kPlaneScale, fh.y));
                            r[4 * i + e] = *reinterpret_cast<const uint32_t*>(&wp);
                        }
                    }
                }
                tmem_st8(lane_addr + F_WIH_COL + 8 * j, r);
            }
            tmem_st_wait();
        }
        loaded_dir = dir;
        tc_fence_before();
        __syncthreads();
        tc_fence_after();

        if (warp == F_W_PROD) {
            // ===================== TMA producer: x tiles of (step, part) in issue order, multicast to the cluster =====================
            if (elect_one()) {
                const int nboxes = 2 * p.kblocks;
                const int pf = p.prefetch_steps;                                  // optional L2 prefetch distance (steps)
                const int npairs = (nparts + 1) >> 1;
                for (int s = 0; s < min(pf, T); ++s) {
                    const int t = dir == 0 ? s : T - 1 - s;
                    for (int pp = 0; pp < npairs; ++pp)
                        for (int bi = (int)rank; bi < nboxes; bi += FC) {
                            const int pl = bi >= p.kblocks, kb = pl ? bi - p.kblocks : bi;
                            tma_prefetch_l2_3d(pl ? &tm_b : &tm_a, kb * 64, t, seq0 + pp * 2 * FPN);
                        }
                }
                for (int s = 0; s < T; ++s) {
                    const int t = dir == 0 ? s : T - 1 - s;
                    const int sp = s + pf, tp = dir == 0 ? sp : T - 1 - sp;
                    for (int pp = 0; pp < npairs; ++pp) {
                        if (pf > 0 && sp < T)
                            for (int bi = (int)rank; bi < nboxes; bi += FC) {
                                const int pl = bi >= p.kblocks, kb = pl ? bi - p.kblocks : bi;
                                tma_prefetch_l2_3d(pl ? &tm_b : &tm_a, kb * 64, tp, seq0 + pp * 2 * FPN);
                            }
                        FUSED_WAIT(bar_x_empty(xst), xph ^ 1u, 1);                // all 4 CTAs' MMAs are done with this stage
                        if (PROBE && (p.flags & 256)) {                           // timing probe: no x loads (stale tiles)
                            mbar_arrive(bar_x_full(pp & 1, xst));
                            if (++xst == p.stages) { xst = 0; xph ^= 1u; }
                            continue;
                        }
                        mbar_expect_tx(bar_x_full(pp & 1, xst), stage_bytes);
                        const uint32_t dst = smem_base + x_off + xst * stage_bytes;
                        for (int bi = (int)rank; bi < nboxes; bi += FC) {
                            const int pl = bi >= p.kblocks, kb = pl ? bi - p.kblocks : bi;
                            tma_load_3d_mc(dst + bi * F_XBOX, pl ? &tm_b : &tm_a, kb * 64, t, seq0 + pp * 2 * FPN, bar_x_full(pp & 1, xst), (uint16_t)0xF);
                        }
                        if (++xst == p.stages) { xst = 0; xph ^= 1u; }
                    }
                }
            }
        } else if (warp == F_W_MMAX || warp == F_W_MMAX + 1) {
            // ===================== input-product issuers: acc(s, q) = W_ih . x_s, up to one step ahead of the recurrence =====================
            // (a thread spends ~2/3 of a part slot in barrier waits and commits, not in MMAs: parts are split by parity over two
            // issuers per product so that the tensor pipe always has the other thread's MMAs queued)
            if (elect_one()) {
                const int me = warp - F_W_MMAX;
                constexpr uint32_t idesc = idesc_f16(128, 2 * FPN);                 // a pair of parts per MMA: N = 32
                const uint32_t wa0 = tmem_base + F_WIH_COL, wb0 = wa0 + 8 * nk;
                const uint32_t plane_lo = (uint32_t)(p.kblocks * F_XBOX) >> 4;
                const int npairs = (nparts + 1) >> 1;
                // ph_b: acc_free phase bits (per part)
                for (int s = 0; s < T; ++s) {
                    for (int pp = 0; pp < npairs; ++pp) {
                        if ((pp & 1) != me) {                                      // the other issuer's slot of the x ring
                            if (++xst == p.stages) { xst = 0; xph ^= 1u; }
                            continue;
                        }
                        const bool trx = tr_item && pp == 0 && s >= F_TRACE_S0 && s < F_TRACE_S0 + F_TRACE_STEPS;
                        if (trx) trace[(s - F_TRACE_S0) * 16 + 9] = clock64();
                        long long* const t3 = (PROBE && (p.flags & 128) && tr_item && (s == F_TRACE_S0 || s == F_TRACE_S0 + 1))
                                                  ? g_fused_trace + F_TRACE_STEPS * 16 + 64 + (s - F_TRACE_S0) * 32 + pp * 8 : nullptr;
                        if (t3) t3[0] = clock64();
                        if (s > 0) {                                               // the pointwise warps have read acc(s - 1, .) of both parts
#pragma unroll
                            for (int h = 0; h < 2; ++h) {
                                const int q = 2 * pp + h;
                                if (q < nparts) {
                                    FUSED_WAIT(bar_acc_free(q), (ph_b >> q) & 1u, 2);
                                    ph_b ^= 1u << q;
                                }
                            }
                        }
                        if (t3) t3[1] = clock64();
                        FUSED_WAIT(bar_x_full(me, xst), (xfph >> xst) & 1u, 3);   // own barrier set: its phases are this thread's own uses of the stage
                        xfph ^= 1u << xst;
                        tc_fence_after();
                        if (t3) t3[2] = clock64();
                        if (trx) trace[(s - F_TRACE_S0) * 16 + 13] = clock64();
                        const uint32_t xa = fdesc_lo(smem_base + x_off + xst * stage_bytes), xb = xa + plane_lo;
                        const uint32_t d = tmem_base + F_ACC_COL + pp * 2 * FPN;
                        if (NK > 0) {
#pragma unroll
                            for (int j = 0; j < (NK > 0 ? NK : 1); ++j) {
                                if ((PROBE && (p.flags & 16)) && j > 0) break;
                                const uint32_t off = (uint32_t)((j >> 2) * (F_XBOX >> 4) + (j & 3) * 2);
                                if (TERMS == 3) {
                                    mma_f16_ts(d, wa0 + 8 * j, fdesc(xb + off), idesc, j != 0);   // x_lo . W_hi (small terms first)
                                    mma_f16_ts(d, wb0 + 8 * j, fdesc(xa + off), idesc, 1);        // x_hi . W_lo
                                } else {
                                    mma_f16_ts(d, wb0 + 8 * j, fdesc(xb + off), idesc, j != 0);   // x2 . W'
                                }
                                mma_f16_ts(d, wa0 + 8 * j, fdesc(xa + off), idesc, 1);            // x1 . W_hi
                            }
                        } else {
                            for (int j = 0; j < ((PROBE && (p.flags & 16)) ? 1 : nk); ++j) {
                                const uint32_t off = (uint32_t)((j >> 2) * (F_XBOX >> 4) + (j & 3) * 2);
                                if (terms == 3) {
                                    mma_f16_ts(d, wa0 + 8 * j, fdesc(xb + off), idesc, j != 0);
                                    mma_f16_ts(d, wb0 + 8 * j, fdesc(xa + off), idesc, 1);
                                } else {
                                    mma_f16_ts(d, wb0 + 8 * j, fdesc(xb + off), idesc, j != 0);
                                }
                                mma_f16_ts(d, wa0 + 8 * j, fdesc(xa + off), idesc, 1);
                            }
                        }
                        mma_commit_mc(bar_x_empty(xst), (uint16_t)0xF);
                        mma_commit(bar_x_done(pp));
                        if (++xst == p.stages) { xst = 0; xph ^= 1u; }
                        if (t3) t3[3] = clock64();
                        if (trx) trace[(s - F_TRACE_S0) * 16 + 15] = clock64();
                    }
                }
                // the accumulators of the last step must be read before the next item overwrites them
                for (int q = 0; q < nparts; ++q) {
                    if (((q >> 1) & 1) != me) continue;
                    FUSED_WAIT(bar_acc_free(q), (ph_b >> q) & 1u, 5);
                    ph_b ^= 1u << q;
                }
            }
        } else if (warp == F_W_MMA || warp == F_W_MMA + 1) {
            // ===================== recurrent-product issuers: acc(s, q) += W_hh . h_{s-1} =====================
            if (elect_one()) {
                const int me = warp - F_W_MMA;
                constexpr uint32_t idesc = idesc_f16(128, FPN);
                // ph_a: h_ready phase bits, ph_b: x_done phase bits
                // h_ready(q) = this thread's arming arrival + the 8 KB of h_s that the four CTAs' senders store into this CTA's
                // tile (st.async credits the bytes); armed before the step whose pointwise pass produces them
                if (T > 1 && !FUSED_EXCH_PLAIN)
                    for (int q = me; q < nparts; q += 2) mbar_expect_tx(bar_h_ready(q), (PROBE && (p.flags & 1)) ? F_HTILE / 2 : F_HTILE);
                for (int s = 0; s < T; ++s) {
                    for (int q = me; q < nparts; q += 2) {
                        const bool trh = tr_item && q == 0 && s >= F_TRACE_S0 && s < F_TRACE_S0 + F_TRACE_STEPS;
                        long long* const t2 = (PROBE && (p.flags & 128) && tr_item && (s == F_TRACE_S0 || s == F_TRACE_S0 + 1))
                                                  ? g_fused_trace + F_TRACE_STEPS * 16 + (s - F_TRACE_S0) * 32 + q * 4 : nullptr;
                        if (t2) t2[0] = clock64();
                        FUSED_WAIT(bar_x_done(q >> 1), (ph_b >> (q >> 1)) & 1u, 2);   // acc(s, q) holds the complete input product of its pair
                        ph_b ^= 1u << (q >> 1);
                        if (t2) t2[1] = clock64();
                        if (s > 0) {
#if FUSED_EXCH_PLAIN
                            FUSED_WAIT_CLUSTER(bar_h_ready(q), (ph_a >> q) & 1u, 4);   // four senders' release arrives (cluster scope)
#else
                            FUSED_WAIT(bar_h_ready(q), (ph_a >> q) & 1u, 4);       // h_{s-1} of this part: all four slices landed
#endif
                            ph_a ^= 1u << q;
                            if (!FUSED_EXCH_PLAIN && s < T - 1) mbar_expect_tx(bar_h_ready(q), (PROBE && (p.flags & 1)) ? F_HTILE / 2 : F_HTILE);   // arm for h_s
                            fence_proxy_async();                                   // st.async data -> tensor-core (async proxy) reads
                            tc_fence_after();
                            if (t2) t2[2] = clock64();
                            if (trh) trace[(s - F_TRACE_S0) * 16 + 0] = clock64();
                            const uint32_t hb = fdesc_lo(smem_base + h_off + q * F_HTILE);
                            const uint32_t d = tmem_base + F_ACC_COL + q * FPN;
                            if (!(PROBE && (p.flags & 8))) {
#pragma unroll
                                for (int jj = 0; jj < 16; ++jj)
                                    mma_f16_ts(d, tmem_base + F_WHH_COL + 8 * jj, fdesc(hb + (uint32_t)((jj >> 2) * (F_BOX >> 4) + (jj & 3) * 2)), idesc, 1);
                            }
                        }
                        mma_commit(bar_acc_ready(q));                              // (s = 0: h_{-1} = 0, the input product alone)
                        if (s < T - 1) mma_commit_mc(bar_h_free(q), (uint16_t)0xF);   // every CTA's copy of this part's h tile may be overwritten
                        if (t2) t2[3] = clock64();
                        if (trh) trace[(s - F_TRACE_S0) * 16 + 1] = clock64();
                    }
                }
            }
        } else if (warp >= F_W_SEND) {
            // ===================== exchange senders: own 2 KB slice of a part's h_s -> k-block `rank` of all four CTAs' operand tiles =====================
            // A whole warp per sender: the slice is copied with 16-byte st.async stores (SM-to-SM, a few hundred cycles; the
            // bytes are credited to the destination's h_ready barrier).  cp.async.bulk took ~3000 cycles per copy through the TMA
            // unit, and the same stores issued by the pointwise warps stalled them on the ~20 B/clk DSMEM port.
            uint32_t cta_delta[FC];                                            // [d]: address offset of CTA (rank + d) & 3 (static indices only)
#pragma unroll
            for (uint32_t d = 0; d < FC; ++d) cta_delta[d] = mapa_shared(smem_base, (rank + d) & (FC - 1)) - smem_base;
            // Lane l handles rows r(j) = (l >> 2) + 8 j (j = 0, 1), 8-unit chunk k = l & 3 of the fp32 slice: groups 2 k, 2 k + 1,
            // at the adjacent slots 2 (k ^ m) + {0, 1}, m = (r >> 1) & 3 = (l >> 3) & 3 (pointwise warps above).  The 16-byte loads
            // go by quarter warps; a quarter is two rows of the same m and all four k, so reading half (r & 1) of the chunk first
            // makes each load instruction cover 8 distinct slots of 16 bytes, i.e. all 32 banks.
            const int k = lane & 3, hs = (lane >> 2) & 1;
            const uint32_t src_lane = (uint32_t)((lane >> 2) * 128 + ((2 * (k ^ ((lane >> 3) & 3)) + hs) << 4));
            const float s1 = 1.f - kPlaneScale;
            // ph_b: h_free phase bits
            for (int s = 0; s < T; ++s) {
                const int t = dir == 0 ? s : T - 1 - s;
                const bool exchange = s + 1 < T;                                   // no h is exchanged after the last step, only y stored
                for (int q = warp - F_W_SEND; q < nparts; q += 4) {
                    const bool trl = tr_item && q == 0 && s >= F_TRACE_S0 && s < F_TRACE_S0 + F_TRACE_STEPS;
                    fused_bar(F_BAR_SLICE + (q & 3), 160, 1, wacc);               // the part's four pointwise warps have written h_s
                    if (trl) trace[(s - F_TRACE_S0) * 16 + 7] = clock64();
                    // h_s -> the scaled split (h1 . W_hi + h2 . W'), w1 / w2[j]: the 16-byte chunks (8 units) of row r(j); this
                    // needs no h_free and runs while the peers' recurrent MMAs may still read the operand tile
                    uint4 w1[2], w2[2];
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const uint32_t src = smem_base + g_off + ((s & 1) * FMAXP + q) * F_BOX + j * 1024 + src_lane;
                        float4 a, b;
                        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w) : "r"(src));
                        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "r"(src ^ 16u));
                        const float4 lo = hs ? b : a, hi = hs ? a : b;             // units 8 k .. 8 k + 3 and 8 k + 4 .. 8 k + 7
                        split_scaled_f16x2(lo.x, lo.y, s1, w1[j].x, w2[j].x);
                        split_scaled_f16x2(lo.z, lo.w, s1, w1[j].y, w2[j].y);
                        split_scaled_f16x2(hi.x, hi.y, s1, w1[j].z, w2[j].z);
                        split_scaled_f16x2(hi.z, hi.w, s1, w1[j].w, w2[j].w);
                    }
                    if (exchange) {
                        if (lane == 0) FUSED_WAIT(bar_h_free(q), (ph_b >> q) & 1u, 7);   // every CTA's recurrent MMAs of step s have read
                        ph_b ^= 1u << q;                                                  // the part's tile (it still holds h_{s-1})
                        __syncwarp();
                        // operand layout: row = sequence, chunk k (h1) / 4 + k (h2) of the 128-byte row at chunk ^ (row & 7)
                        const uint32_t bar = bar_h_ready(q);
#pragma unroll
                        for (int j = 0; j < 2; ++j) {
                            if (PROBE && (p.flags & 1) && j > 0) break;                   // timing probe: half the exchange bytes
                            const int row = (lane >> 2) + 8 * j;
                            const uint32_t dst_row = smem_base + h_off + q * F_HTILE + rank * F_BOX + row * 128;
#pragma unroll
                            for (int pl = 0; pl < 2; ++pl) {
                                const uint4 v = pl ? w2[j] : w1[j];
                                const uint32_t dst = dst_row + (((4 * pl + k) ^ (row & 7)) << 4);
                                // the three peers over DSMEM; the own copy is a plain shared-memory store (it does not take the SM-to-SM port)
#pragma unroll
                                for (uint32_t d = 1; d < FC; ++d) {
#if FUSED_EXCH_PLAIN
                                    asm volatile("st.shared::cluster.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(dst + cta_delta[d]),
                                                 "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
#else
                                    st_async_v4(dst + cta_delta[d], v, bar + cta_delta[d]);
#endif
                                }
                                asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
                            }
                        }
#if FUSED_EXCH_PLAIN
                        // every lane: its generic stores (local and remote) before the tensor cores' async-proxy reads, and before
                        // lane 0's release arrives at cluster scope
                        fence_proxy_async_all();
                        asm volatile("fence.acq_rel.cluster;" ::: "memory");
                        __syncwarp();
                        if (lane < FC) mbar_arrive_cluster(mapa_shared(bar, (uint32_t)lane));   // one arrive per destination CTA (own included)
#else
                        fence_proxy_async();                                       // own copy: generic stores before the tensor core's reads
                        __syncwarp();
                        if (lane == 0) mbar_complete_tx(bar, (PROBE && (p.flags & 1)) ? F_BOX / 2 : F_BOX);
#endif
                    }
                    if (trl) trace[(s - F_TRACE_S0) * 16 + 8] = clock64();
                    // layer output planes (B, T, 256): the same chunks, after the exchange so that the chain does not wait on them
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const int b = seq0 + q * FPN + (lane >> 2) + 8 * j;
                        if (b < p.B && !(PROBE && (p.flags & 2))) {
                            const size_t off = ((size_t)b * T + t) * (2 * kHidden) + dir * kHidden + (int)rank * FU + 8 * k;
                            *reinterpret_cast<uint4*>(p.y_a + off) = w1[j];
                            *reinterpret_cast<uint4*>(p.y_b + off) = w2[j];
                        }
                    }
                    if (trl) trace[(s - F_TRACE_S0) * 16 + 14] = clock64();
                }
            }
        } else if ((warp >> 2) < nparts) {
            // ===================== pointwise warps: warp (pg, g) = parts pg and pg + 4, units 8 g .. 8 g + 7 of this CTA =====================
            // Two 16x256b TMEM loads (lanes 32 g .. + 15 and 32 g + 16 .. + 31) hand lane l all four gates of unit 8 g + (l >> 2)
            // for the 4 sequences seq(i) = 2 (l & 3) + (i & 1) + 8 (i >> 1): the gate rows are laid out for exactly that (see the
            // weight loader), so no (gate x sequence) transposition through shared memory is needed.
            const int pg = warp >> 2, g = warp & 3;
            const int uu = lane >> 2, jj = lane & 3;
            const uint32_t lane_addr = tmem_base + ((uint32_t)(g * 32) << 16) + F_ACC_COL;
            float bias[4];                                                     // [gate] of unit 8 g + uu
#pragma unroll
            for (int k = 0; k < 4; ++k) bias[k] = __ldg(p.bias + dir * kGates + k * kHidden + (int)rank * FU + 8 * g + uu);
            const float L2E2 = 2.f * kLog2e;
            float cst[2][4];
#pragma unroll
            for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) cst[a][b] = 0.f;
            // staging slice of (step parity, part): fp32 h_s, [16 rows = sequences][8 groups of 4 units][4 B].  Group G = u >> 2 of
            // unit u sits at group slot G ^ (((row >> 1) & 3) << 1).  This lane's cells are unit u = 8 g + uu of rows 2 jj + {0, 1,
            // 8, 9}, all with (row >> 1) & 3 = jj: one column for all four, slot 2 (g ^ jj) + (uu >> 2), bank 4 slot + (uu & 3) --
            // over the warp's (jj, uu) 32 distinct banks per store.  A group stays 16 contiguous bytes for the sender's 16-byte loads.
            const int stg_col = ((((2 * g + (uu >> 2)) ^ (jj << 1)) << 2) + (uu & 3)) * 4 + 2 * jj * 128;
            // ph_a: acc_ready phase bits (bit pi; used by the group's poller only)
            const bool poller = g == pg;
            for (int s = 0; s < T; ++s) {
#pragma unroll
                for (int pi = 0; pi < 2; ++pi) {
                    const int q = pg + 4 * pi;
                    if (q >= nparts) break;
                    if (poller) FUSED_WAIT(bar_acc_ready(q), (ph_a >> pi) & 1u, 6);
                    ph_a ^= 1u << pi;
                    fused_bar(F_BAR_ACC + pg, 128, 5, wacc);                       // the poller saw acc_ready(q)
                    tc_fence_after();                                              // (commit -> mbarrier -> poller -> bar.sync -> tcgen05.ld)
                    const bool tr_on = tr_item && warp == 0 && pi == 0 && s >= F_TRACE_S0 && s < F_TRACE_S0 + F_TRACE_STEPS;
                    if (tr_on) trace[(s - F_TRACE_S0) * 16 + 2] = clock64();
                    float z[2][8];                                                 // [gates 2 h, 2 h + 1]: see tmem_ld_16x256b_x2
                    tmem_ld_16x256b_x2(lane_addr + q * FPN, z[0]);
                    tmem_ld_16x256b_x2(lane_addr + (16u << 16) + q * FPN, z[1]);
                    tmem_ld_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_acc_free(q));                   // the next step's input product may overwrite the accumulator
                    if (tr_on) trace[(s - F_TRACE_S0) * 16 + 3] = clock64();
                    float ev[4][4];                                                // [gate][cell i]: sequence seq(i)
#pragma unroll
                    for (int k = 0; k < 4; ++k)
#pragma unroll
                        for (int i = 0; i < 4; ++i)
                            ev[k][i] = fast_ex2(fminf(z[k >> 1][4 * (i >> 1) + 2 * (k & 1) + (i & 1)] + bias[k], 29.f));
                    if (tr_on) trace[(s - F_TRACE_S0) * 16 + 4] = clock64();
                    if (tr_on) trace[(s - F_TRACE_S0) * 16 + 5] = clock64();
                    float hv[4];
                    const f32x2 one = pack2(1.f, 1.f), mone = pack2(-1.f, -1.f), k2 = pack2(L2E2, L2E2);
#pragma unroll
                    for (int jp = 0; jp < 2; ++jp) {
                        if (PROBE && (p.flags & 4)) { hv[2 * jp] = ev[0][2 * jp] * 1e-3f; hv[2 * jp + 1] = ev[3][2 * jp + 1] * 1e-3f; continue; }
                        const f32x2 pei = pack2(ev[0][2 * jp], ev[0][2 * jp + 1]), pef = pack2(ev[1][2 * jp], ev[1][2 * jp + 1]);
                        const f32x2 peg = pack2(ev[2][2 * jp], ev[2][2 * jp + 1]), peo = pack2(ev[3][2 * jp], ev[3][2 * jp + 1]);
                        // c' = c / (1 + ef) + (eg - 1) / ((1 + ei)(eg + 1)) with one reciprocal (lstm_tc.cu)
                        const f32x2 di = add2(pei, one), df = add2(pef, one), dg = add2(peg, one);
                        const f32x2 dig = mul2(di, dg);
                        const f32x2 den = mul2(df, dig);
                        const f32x2 cn = mul2(fma2(pack2(cst[pi][2 * jp], cst[pi][2 * jp + 1]), dig, mul2(add2(peg, mone), df)), rcp2(den));
                        unpack2(cn, cst[pi][2 * jp], cst[pi][2 * jp + 1]);
                        const f32x2 ec = ex2_clamped2(mul2(cn, k2));
                        const f32x2 h2v = mul2(add2(ec, mone), rcp2(mul2(add2(peo, one), add2(ec, one))));
                        unpack2(h2v, hv[2 * jp], hv[2 * jp + 1]);
                    }
                    if (tr_on) trace[(s - F_TRACE_S0) * 16 + 10] = clock64();
                    // h_s -> the CTA's staging slice of (step parity, part); the sender splits it into the fp16 planes.  The slice of
                    // this parity was last read by the sender at step s - 2, before its exchange of step s - 1, which landed before
                    // any CTA could start step s.
                    unsigned char* const stg = smem_gen + g_off + ((s & 1) * FMAXP + q) * F_BOX + stg_col;
#pragma unroll
                    for (int c = 0; c < 4; ++c) *reinterpret_cast<float*>(stg + ((c & 1) + 8 * (c >> 1)) * 128) = hv[c];
                    fused_bar(F_BAR_SLICE + pg, 160, 4, wacc);                     // hand the slice to sender warp pg (it reads it with plain loads)
                    if (tr_on) trace[(s - F_TRACE_S0) * 16 + 12] = clock64();
                }
            }
        }
        // item boundary: every role of every CTA is done with this item's tiles and barriers
        tc_fence_before();
        cluster_sync_all();
        tc_fence_after();
    }
    // The last `stages` multicast commits onto x_empty are not consumed by any load: they must have LANDED in this CTA before it
    // exits (an arrive that finds its target CTA gone is a fault, and after the exit the shared memory may belong to another
    // kernel's CTA when a second stream keeps the SM busy).  The producer waits for them exactly as if it were to refill the ring.
    if (warp == F_W_PROD && elect_one()) {
        for (int k = 0; k < p.stages; ++k) {
            FUSED_WAIT(bar_x_empty(xst), xph ^ 1u, 1);
            if (++xst == p.stages) { xst = 0; xph ^= 1u; }
        }
    }
    if (wacc) wacc[0] += clock64();
    tc_fence_before();
    cluster_sync_all();                                       // no CTA exits while a peer may still signal or multicast into it
    if (warp == F_W_MMA) tmem_dealloc<512>(tmem_base);
}

// ---------------------------------------------------------------- launcher
static int g_fused_debug = -1, g_fused_lag = -1;
// timing probes (wrong results): 1 no h exchange, 2 no y store, 4 no cell math, 8 no recurrent MMAs, 16 no input MMAs
void lstm_fused_set_debug(int flags, int lag) { g_fused_debug = flags; if (lag >= 0) g_fused_lag = lag; }
int lstm_fused_read_debug(long long* host, int n) {
    if (n < 0) {                                             // the timeline table (flag 64)
        B200VAD_CUDA(cudaMemcpyFromSymbol(host, g_fused_trace, sizeof(long long) * std::min(-n, F_TRACE_STEPS * 16 + 128)));
        return B200VAD_OK;
    }
    const size_t bytes = sizeof(long long) * (size_t)std::min<long long>(n, (long long)F_DBG_MAX_CTAS * F_DBG_WARPS * F_DBG_TAGS * F_DBG_FIELDS);
    B200VAD_CUDA(cudaMemcpyFromSymbol(host, g_fused_dbg, bytes));
    return B200VAD_OK;
}
static int* g_fused_err_hostbuf = nullptr;
// {flag, block, thread, wait site, barrier address, parity, grid} of the first bounded wait that timed out (all zero: none)
int lstm_fused_last_timeout(int* out7) {
    for (int i = 0; i < 7; ++i) out7[i] = g_fused_err_hostbuf ? g_fused_err_hostbuf[i] : 0;
    return B200VAD_OK;
}
static int g_fused_clusters[64];
static std::once_flag g_fused_once[64];

typedef void (*FusedKern)(CUtensorMap, CUtensorMap, FusedParams);
static FusedKern fused_pick(int nk, int terms, int probe) {
    if (probe) {                                             // timing / ablation build of the bench shapes (tools/fused_ablate.py)
        if (nk == 16 && terms == 2) return lstm_fused_kernel<16, 2, true>;
        if (nk == 5 && terms == 3) return lstm_fused_kernel<5, 3, true>;
    }
    if (nk == 16) return terms == 2 ? lstm_fused_kernel<16, 2, false> : lstm_fused_kernel<16, 3, false>;
    if (nk == 5) return terms == 2 ? lstm_fused_kernel<5, 2, false> : lstm_fused_kernel<5, 3, false>;
    if (nk == 4) return terms == 2 ? lstm_fused_kernel<4, 2, false> : lstm_fused_kernel<4, 3, false>;
    return lstm_fused_kernel<0, 0, false>;
}

static int fused_smem_bytes(int kblocks, int* stages_out) {
    const int stage = 2 * kblocks * F_XBOX;
    int stages = (F_SMEM_MAX - 1024 - F_SMEM_FIXED - 1024) / stage;
    if (stages > F_MAX_STAGES) stages = F_MAX_STAGES;
    static int cap = -1;                                     // B200VAD_FUSED_STAGES: cap of the x ring depth (experiments)
    if (cap < 0) { const char* e = getenv("B200VAD_FUSED_STAGES"); cap = e ? atoi(e) : 0; }
    if (cap > 0 && stages > cap) stages = cap;
    *stages_out = stages;
    return 1024 + F_SMEM_FIXED + stages * stage + 1024;
}

// resident clusters of the kernel on this device (cudaOccupancyMaxActiveClusters); cached per device
static int fused_max_clusters() {
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 0;
    std::call_once(g_fused_once[dev], [&] {
        const void* fn = reinterpret_cast<const void*>(lstm_fused_kernel<16, 2, false>);
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(FC * 64);
        cfg.blockDim = dim3(F_THREADS);
        cfg.dynamicSmemBytes = F_SMEM_MAX - 1024;            // worst case
        cudaLaunchAttribute at;
        at.id = cudaLaunchAttributeClusterDimension;
        at.val.clusterDim.x = FC; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
        cfg.attrs = &at; cfg.numAttrs = 1;
        int n = 0;
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (set_max_dynamic_smem(fn, F_SMEM_MAX - 1024) != B200VAD_OK ||
            cudaOccupancyMaxActiveClusters(&n, fn, &cfg) != cudaSuccess || n <= 0) {
            cudaGetLastError();
            n = std::max(1, sms / FC - 4);
        }
        const char* e = getenv("B200VAD_FUSED_CLUSTERS");
        if (e && atoi(e) > 0) n = atoi(e);
        g_fused_clusters[dev] = n;
    });
    return g_fused_clusters[dev];
}

int lstm_fused_supported(int D) { return D >= 1 && D <= 256; }
int lstm_fused_clusters() { return fused_max_clusters(); }

// One bidirectional LSTM layer.  x_a / x_b: input planes (B, T, lda) fp16 (terms 2: scaled split; terms 3: hi / lo);
// weights as packed by api.cu (gate-scaled): wih planes [1024][ldw], whh planes [2][512][128], bias [1024];
// y_a / y_b: output planes (B, T, 256), scaled split if y_scaled else hi / lo.
int lstm_fused_launch(const __half* x_a, const __half* x_b, int64_t lda, int B, int T, int D, const __half* wih_hi,
                      const __half* wih_lo, int ldw, const __half* whh_hi, const __half* whh_lo, const float* bias, int terms,
                      __half* y_a, __half* y_b, int y_scaled, cudaStream_t st) {
    if (B <= 0 || T <= 0) return B200VAD_OK;
    if (!lstm_fused_supported(D) || (terms != 2 && terms != 3) || lda % 8 != 0 || ldw % 8 != 0 || ldw < (D + 15) / 16 * 16) {
        set_error("lstm_fused: unsupported shape (D=%d lda=%lld ldw=%d terms=%d)", D, (long long)lda, ldw, terms);
        return B200VAD_EINVAL;
    }
    FusedParams p;
    p.wih_hi = wih_hi; p.wih_lo = wih_lo; p.whh_hi = whh_hi; p.whh_lo = whh_lo; p.bias = bias; p.y_a = y_a; p.y_b = y_b;
    p.B = B; p.T = T; p.nk = (D + 15) / 16; p.kblocks = (D + 63) / 64; p.ldw = ldw; p.terms = terms;
    (void)y_scaled;                                          // the output planes are always the scaled split (see the header)
    int stages = 0;
    const int smem = fused_smem_bytes(p.kblocks, &stages);
    p.stages = stages;
    if (g_fused_debug < 0) { const char* e = getenv("B200VAD_FUSED_DEBUG"); g_fused_debug = e ? atoi(e) : 0; }
    if (g_fused_lag < 0) { const char* e = getenv("B200VAD_FUSED_LAG"); g_fused_lag = e ? atoi(e) : 2; }
    p.flags = g_fused_debug;
    static int pf_env = -1;
    if (pf_env < 0) { const char* e = getenv("B200VAD_FUSED_PREFETCH"); pf_env = e ? atoi(e) : 0; }
    p.prefetch_steps = pf_env;

    const int nc = fused_max_clusters();
    // work items: parts of 16 sequences, spread evenly over items_per_dir items per direction (<= 8 parts each); choose the
    // count that minimises waves x step time.  Measured step time (us) of a cluster with n parts in flight (B200 at 1 000 W,
    // `tools/lstm_modes_timing.py 256,...,2048 500 1`: one wave of n = B / 256 parts on each of 32 clusters; profiles/r05_*):
    // one part runs at the unloaded latency of the chain MMA -> pointwise -> exchange, eight parts overlap 2.8 chains' worth.
    // Small batches (streaming: 256 sequences) therefore spread over 32 clusters with one part each, large ones keep eight
    // parts per cluster.
    static const double kStepUs[FMAXP + 1] = {0.0, 1.11, 1.41, 1.53, 1.70, 2.15, 2.60, 2.73, 3.06};
    const int P = (B + FPN - 1) / FPN;
    int best_ipd = (P + FMAXP - 1) / FMAXP;
    double best_cost = 1e30;
    for (int ipd = (P + FMAXP - 1) / FMAXP; ipd <= P; ++ipd) {
        const int maxp = (P + ipd - 1) / ipd;
        const int waves = (2 * ipd + nc - 1) / nc;
        const double cost = waves * kStepUs[maxp];
        if (cost < best_cost - 1e-9) { best_cost = cost; best_ipd = ipd; }
        if (maxp == 1) break;
    }
    p.items_per_dir = best_ipd;
    const int grid = FC * std::min(nc, 2 * best_ipd);
    CUtensorMap tm_a, tm_b;
    int rc;
    if ((rc = make_tmap_3d(&tm_a, x_a, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, D, T, B, lda * 2, (uint64_t)T * lda * 2, 64, 1, 2 * FPN,
                           CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
    if ((rc = make_tmap_3d(&tm_b, x_b, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, D, T, B, lda * 2, (uint64_t)T * lda * 2, 64, 1, 2 * FPN,
                           CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
    const FusedKern kern = fused_pick(p.nk, terms, p.flags != 0);
    if ((rc = set_max_dynamic_smem(reinterpret_cast<const void*>(kern), smem))) return rc;
    if (!g_fused_err_hostbuf) {
        int* hb = nullptr;
        if (cudaHostAlloc(&hb, 64, cudaHostAllocMapped) == cudaSuccess) {
            for (int i = 0; i < 16; ++i) hb[i] = 0;
            int* dp = nullptr;
            if (cudaHostGetDevicePointer(&dp, hb, 0) == cudaSuccess &&
                cudaMemcpyToSymbol(g_fused_err_host, &dp, sizeof(dp)) == cudaSuccess) g_fused_err_hostbuf = hb;
        }
        cudaGetLastError();
    }
    prof_begin(0, st);
    kern<<<grid, F_THREADS, smem, st>>>(tm_a, tm_b, p);
    prof_end(0, st);
    B200VAD_LAUNCH_CHECK();
    return B200VAD_OK;
}

}  // namespace b200vad

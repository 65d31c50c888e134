// sm_100a primitives used by the tcgen05 kernels: mbarrier, TMA (cp.async.bulk.tensor), TMEM
// allocation, tcgen05.mma / commit / ld, and the shared-memory / instruction descriptors.
// Written against the PTX ISA for sm_100a; no CUTLASS dependency.
#pragma once
#include "common.cuh"
#include <cuda.h>

namespace b200vad {
namespace tc {

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// with a suspend-time hint (ns): the thread stays suspended in hardware until the phase completes or the hint elapses, instead
// of returning after the default (short) limit -- a waiting warp then issues a handful of instructions per wait instead of a
// nine-instruction poll every ~80 cycles (ncu: polls were ~45 % of all instructions the fused LSTM kernel executed)
__device__ __forceinline__ bool mbar_try_wait_hint(uint32_t bar, uint32_t parity, uint32_t ns) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity), "r"(ns)
        : "memory");
    return ok != 0;
}
// non-blocking probe of a phase (mbarrier.try_wait may suspend the thread for a system-dependent time)
__device__ __forceinline__ bool mbar_test_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// acquire at cluster scope: orders this thread's later accesses (including TMA issues) after writes that other CTAs of the
// cluster released before arriving on the barrier
__device__ __forceinline__ bool mbar_try_wait_cluster(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// generic-proxy writes (any state space) before, async-proxy accesses after
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
// Bounded wait: a protocol bug must abort the kernel instead of hanging the GPU box.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 8000000000LL) {   // ~4 s at 2 GHz
            printf("b200vad: mbarrier wait timed out (block %d thread %d bar 0x%x parity %u)\n", blockIdx.x, threadIdx.x, bar, parity);
            __trap();
        }
    }
}

__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t threads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}

// ------------------------------------------------------------------ TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, int c0, int c1, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(c0), "r"(c1), "r"(bar)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* m, int c0, int c1, int c2, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(c0), "r"(c1), "r"(c2), "r"(bar)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* m, int c0, int c1, int c2, int c3, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar)
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_l2_3d(const CUtensorMap* m, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global [%0, {%1, %2, %3}];"
                 ::"l"(reinterpret_cast<uint64_t>(m)), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, int c0, int c1, uint32_t src) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];"
                 ::"l"(reinterpret_cast<uint64_t>(m)), "r"(c0), "r"(c1), "r"(src)
                 : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, int c0, int c1, int c2, uint32_t src) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%1, %2, %3}], [%4];"
                 ::"l"(reinterpret_cast<uint64_t>(m)), "r"(c0), "r"(c1), "r"(c2), "r"(src)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_all() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ------------------------------------------------------------------ TMEM + tcgen05
template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t smem_result_addr) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_result_addr), "n"(COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc];  kind::f16 (fp16/bf16 operands, fp32 accumulate)
__device__ __forceinline__ void mma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// same with the A operand in TMEM (lane = row, two fp16 K-elements per 32-bit column)
__device__ __forceinline__ void mma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives (count 1) on the mbarrier once all previously issued tcgen05.mma of this thread completed
__device__ __forceinline__ void mma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// ------------------------------------------------------------------ CTA pairs (cta_group::2): two CTAs of a cluster on one TPC
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address -> shared::cluster address of the same offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
// Relaxed form for hand-overs whose payload is tensor memory already ordered by tcgen05.wait / tcgen05.fence ("I am done
// reading this accumulator"): a release at cluster scope adds a MEMBAR that waits for all of the thread's outstanding
// global stores (measured in the projection epilogue: the top stall reason).
__device__ __forceinline__ void mbar_arrive_cluster_relaxed(uint32_t cluster_bar) {
    asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
// TMA load issued by either CTA of a pair; the transaction bytes are credited to the mbarrier at the same offset in the
// pair's EVEN CTA (the MMA issuer): bit 24 of a shared::cluster address is the CTA's rank within the pair.
__device__ __forceinline__ void tma_load_3d_pair(uint32_t dst, const CUtensorMap* m, int c0, int c1, int c2, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(c0), "r"(c1), "r"(c2), "r"(bar & 0xFEFFFFFFu)
        : "memory");
}
// collective: the same warp index in both CTAs of the pair, the same shared-memory offset for the result
template <int COLS>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t smem_result_addr) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_result_addr), "n"(COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS) : "memory");
}
// D (M = 256: 128 rows in each CTA's TMEM) (+)= A (each CTA's own TMEM rows) * B (N split over the two CTAs' shared memory);
// issued by one thread of the even CTA on behalf of the pair
__device__ __forceinline__ void mma_f16_ts_pair(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives (count 1) on the mbarrier at this offset in BOTH CTAs once all previously issued MMAs of this thread completed
__device__ __forceinline__ void mma_commit_pair(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"((uint16_t)3) : "memory");
}

// same with an explicit cluster mask (clusters of two pairs: either the issuing pair's two CTAs or all four)
__device__ __forceinline__ void mma_commit_pair_mc(uint32_t bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"(mask) : "memory");
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, float (&v)[4]) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const float (&v)[4]) {
    const uint32_t* r = reinterpret_cast<const uint32_t*>(v);
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
                 ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
                 "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
                 : "memory");
}
// ------------------------------------------------------------------ clusters of more than two CTAs (lstm_fused.cu)
// TMA tile load delivered to the same shared-memory offset of every CTA in `mask`; each destination's mbarrier at that
// offset receives the bytes that landed in its own shared memory
__device__ __forceinline__ void tma_load_3d_mc(uint32_t dst, const CUtensorMap* m, int c0, int c1, int c2, uint32_t bar, uint16_t mask) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%2, %3, %4}], [%5], %6;"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(c0), "r"(c1), "r"(c2), "r"(bar), "h"(mask)
        : "memory");
}
// arrives (count 1) on the mbarrier at this offset in every CTA of `mask` once all previously issued MMAs of this thread completed
__device__ __forceinline__ void mma_commit_mc(uint32_t bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"(mask) : "memory");
}
// bulk copy own shared memory -> a peer CTA's shared memory (both shared::cluster addresses from mapa); the bytes are
// credited to the PEER's mbarrier (complete_tx) when they have landed
__device__ __forceinline__ void dsmem_bulk_copy(uint32_t dst_cluster, uint32_t src_cta, uint32_t bytes, uint32_t bar_cluster) {
    asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst_cluster), "r"(src_cta), "r"(bytes), "r"(bar_cluster) : "memory");
}
// 16-byte store into a peer CTA's shared memory (shared::cluster address from mapa); the bytes are credited to the PEER's
// mbarrier (complete_tx, release at cluster scope) when they have landed
__device__ __forceinline__ void st_async_v4(uint32_t dst_cluster, uint4 v, uint32_t bar_cluster) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];"
                 ::"r"(dst_cluster), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "r"(bar_cluster) : "memory");
}
// credits `bytes` to the transaction count of an mbarrier of this CTA (the counterpart of expect_tx for data written with plain stores)
__device__ __forceinline__ void mbar_complete_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.complete_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                   "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr)
                 : "memory");
}
// 16 lanes x 16 columns: lane l of the warp gets rows r = l >> 2 and r + 8 (of the 16 lanes at taddr), columns c = 2 (l & 3) + {0, 1}
// and c + 8: v = {(r, c), (r, c + 1), (r + 8, c), (r + 8, c + 1), (r, c + 8), (r, c + 9), (r + 8, c + 8), (r + 8, c + 9)}
__device__ __forceinline__ void tmem_ld_16x256b_x2(uint32_t taddr, float (&v)[8]) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------ descriptors
// K-major operand tile written by TMA with SWIZZLE_128B: rows of 128 bytes (64 fp16), 8-row swizzle
// atoms of 1024 bytes.  start address in 16-byte units; SBO = 1024 B between 8-row groups; LBO unused.
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);          // start address   [0,14)
    d |= (uint64_t)0 << 16;                                 // leading byte offset (ignored for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;                       // stride byte offset [32,46)
    d |= (uint64_t)1 << 46;                                 // descriptor version (sm_100)
    d |= (uint64_t)2 << 61;                                 // layout type: SWIZZLE_128B
    return d;
}
// kind::f16 instruction descriptor: fp16 A/B (K-major), fp32 accumulator, M x N tile
__host__ __device__ constexpr uint32_t idesc_f16(int M, int N) {
    return (1u << 4) | (0u << 7) | (0u << 10) | (0u << 15) | (0u << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

}  // namespace tc

// ------------------------------------------------------------------ host: tensor-map encoding
// cuTensorMapEncodeTiled is fetched through the runtime (no link-time dependency on libcuda).
int make_tmap_2d(CUtensorMap* out, const void* base, CUtensorMapDataType dtype, uint64_t inner, uint64_t outer,
                 uint64_t pitch_bytes, uint32_t box_inner, uint32_t box_outer, CUtensorMapSwizzle swizzle);
int make_tmap_3d(CUtensorMap* out, const void* base, CUtensorMapDataType dtype, uint64_t d0, uint64_t d1, uint64_t d2,
                 uint64_t pitch1_bytes, uint64_t pitch2_bytes, uint32_t b0, uint32_t b1, uint32_t b2, CUtensorMapSwizzle swizzle);
int make_tmap_4d(CUtensorMap* out, const void* base, CUtensorMapDataType dtype, const uint64_t dims[4], const uint64_t pitch_bytes[3],
                 const uint32_t box[4], CUtensorMapSwizzle swizzle);

}  // namespace b200vad

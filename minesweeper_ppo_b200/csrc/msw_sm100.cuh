// msw_sm100.cuh -- the one definition of each sm_100 asynchronous-copy and tensor-core instruction the kernels
// issue through inline PTX (mbarrier, TMA and bulk copies, cp.async, elect.sync, tcgen05), and the host-side
// tensor-map encoder the TMA copies read (defined in msw_capi.cu).
//
// Shared-memory operands are 32-bit shared-state-space addresses (smem_u32), as the PTX takes them; global
// operands and tensor maps are generic pointers.
#pragma once

#include <cuda.h>
#include <stdint.h>

namespace msw {

// ---------------------------------------------------------------------------
// Host: cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda at link time)
// ---------------------------------------------------------------------------
bool tensor_map_encoder_available();   // false when the driver does not provide cuTensorMapEncodeTiled

// Tiled map of a `rank`-D tensor at `base`: dims and box innermost first, `strides` = the rank - 1 outer byte
// strides.  Unit element strides, no interleave, 128-byte L2 promotion, and zeros for elements past the edges.
CUresult encode_tiled(CUtensorMap *map, CUtensorMapDataType dtype, cuuint32_t rank, const void *base,
                      const cuuint64_t *dims, const cuuint64_t *strides, const cuuint32_t *box,
                      CUtensorMapSwizzle swizzle);

// ---------------------------------------------------------------------------
// Shared memory and mbarriers
// ---------------------------------------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count));
}
// makes the initialised barriers visible to the async proxy (TMA, tcgen05.commit) and the other threads
__device__ __forceinline__ void mbar_fence_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity)
{
    unsigned done = 0;
    while (!done)
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
}

// ---------------------------------------------------------------------------
// TMA tensor copies and bulk copies.  Loads complete on an mbarrier (complete_tx); stores join the issuing
// thread's bulk group (bulk_commit / bulk_wait).
// ---------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(unsigned dst, const CUtensorMap *map, int c0, int c1, unsigned bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 :: "r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar) : "memory");
}
__device__ __forceinline__ void tma_load_4d(unsigned dst, const CUtensorMap *map, int c0, int c1, int c2, int c3, unsigned bar)
{
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
                 :: "r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar) : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap *map, int c0, int c1, unsigned src)
{
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];"
                 :: "l"(map), "r"(c0), "r"(c1), "r"(src) : "memory");
}
__device__ __forceinline__ void tma_prefetch(const CUtensorMap *map)
{
    asm volatile("prefetch.tensormap [%0];" :: "l"(map) : "memory");
}
// `bytes` contiguous bytes global -> shared (a multiple of 16, both ends 16-byte aligned)
__device__ __forceinline__ void bulk_load(unsigned dst, const void *src, unsigned bytes, unsigned bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void bulk_store(void *dst, unsigned src, unsigned bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" :: "l"(dst), "r"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// at most N bulk groups still pending (complete: the writes are done)
template <int N>
__device__ __forceinline__ void bulk_wait()
{
    asm volatile("cp.async.bulk.wait_group %0;" :: "n"(N) : "memory");
}
// at most N bulk groups still reading their shared-memory source (the source may be overwritten)
template <int N>
__device__ __forceinline__ void bulk_wait_read()
{
    asm volatile("cp.async.bulk.wait_group.read %0;" :: "n"(N) : "memory");
}
// generic-proxy writes to shared memory -> visible to a following TMA / bulk store
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---------------------------------------------------------------------------
// 16-byte cp.async (LDGSTS) and its groups
// ---------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(unsigned dst, const void *src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>   // at most N cp.async groups still pending
__device__ __forceinline__ void cp_async_wait()
{
    asm volatile("cp.async.wait_group %0;" :: "n"(N) : "memory");
}

// One lane of a converged warp.  ptxas knows that code guarded by elect.sync runs on exactly one thread, so the
// tcgen05 / TMA instructions inside take their uniform-register operands directly; guarded by `lane == 0` instead,
// every such instruction is wrapped in a divergence "waterfall" loop (ELECT / PLOP3 / BRA.U.ANY, ~10 dependent
// instructions per MMA).  Measured in round 2: the whole forward 4.04 -> 3.99 ms.
__device__ __forceinline__ bool elect_one()
{
    unsigned pred;
    asm volatile("{ .reg .pred p; elect.sync _|p, 0xffffffff; selp.u32 %0, 1, 0, p; }" : "=r"(pred));
    return pred != 0u;
}

// ---------------------------------------------------------------------------
// tcgen05: UMMA descriptors and MMAs, tensor-memory (TMEM) allocation and loads
// ---------------------------------------------------------------------------
// K-major operand descriptor (sm_100 version bit, LBO unused = 1, matrix base offset 0) for rows of ROW bytes:
// 8-row groups ROW * 8 bytes apart (SBO); ROW = 128 / 64 / 32 <-> layout type SWIZZLE_128B (2) / 64B (4) / 32B (6).
// `addr` is the shared-memory byte address.
template <unsigned ROW>
__device__ __forceinline__ uint64_t umma_desc(unsigned addr)
{
    constexpr uint64_t layout = ROW == 128 ? 2ull : ROW == 64 ? 4ull : 6ull;
    return (uint64_t)((addr >> 4) & 0x3FFFu) | (1ull << 16) | ((uint64_t)(ROW * 8u >> 4) << 32) | (1ull << 46) | (layout << 61);
}
// D[tmem] (+)= A[smem] . B[smem]^T (kind::f16), issued by one thread
__device__ __forceinline__ void umma_f16(unsigned d_tmem, uint64_t a, uint64_t b, unsigned idesc, unsigned accumulate)
{
    asm volatile("{ .reg .pred p; setp.ne.b32 p, %4, 0; tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p; }"
                 :: "r"(d_tmem), "l"(a), "l"(b), "r"(idesc), "r"(accumulate) : "memory");
}
// the same with a disable-output-lane mask: bit i of mask word w set = row 32w + i of D is not written
__device__ __forceinline__ void umma_f16_masked(unsigned d_tmem, uint64_t a, uint64_t b, unsigned idesc, unsigned accumulate,
                                                unsigned mask)
{
    asm volatile("{ .reg .pred p; setp.ne.b32 p, %4, 0; tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5}, p; }"
                 :: "r"(d_tmem), "l"(a), "l"(b), "r"(idesc), "r"(accumulate), "r"(mask) : "memory");
}
// arrive on `bar` once the MMAs this thread issued before have completed
__device__ __forceinline__ void umma_commit(unsigned bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar) : "memory");
}
// whole warp: allocate `cols` TMEM columns, their address written to shared memory at `dst`
__device__ __forceinline__ void tmem_alloc(unsigned dst, unsigned cols)
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(dst), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(unsigned tmem, unsigned cols)
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(cols) : "memory");
}
// order tcgen05 operations before / after a thread synchronisation (barrier, mbarrier wait)
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// the warp's 32 TMEM lanes x 16 / 32 consecutive 32-bit columns; valid after tmem_wait_ld
__device__ __forceinline__ void tmem_ld16(unsigned taddr, uint32_t (&v)[16])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld32(unsigned taddr, uint32_t (&v)[32])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
                 "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                   "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                   "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------------------
// Clusters and CTA pairs (tcgen05 cta_group::2): two CTAs of a 2-CTA cluster share each MMA.  The leader
// (rank 0) issues it; A rows 0..127 come from the leader's shared memory and rows 128..255 from the peer's at the
// same address, B's N rows are split in halves the same way, and D rows 0..127 / 128..255 land in the leader's /
// the peer's TMEM.  Barrier and shared-memory operands named `*_cluster` are shared::cluster addresses (mapa).
// ---------------------------------------------------------------------------
__device__ __forceinline__ unsigned cluster_ctarank()
{
    unsigned r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
// the shared::cluster address of this CTA's shared address `addr` in CTA `rank` of the cluster
__device__ __forceinline__ unsigned mapa_shared(unsigned addr, unsigned rank)
{
    unsigned r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
// all threads of all CTAs of the cluster (release / acquire)
__device__ __forceinline__ void cluster_sync()
{
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx_cluster(unsigned bar_cluster, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.release.cluster.shared::cluster.b64 _, [%0], %1;" :: "r"(bar_cluster), "r"(bytes) : "memory");
}
// releases this thread's earlier writes (st_shared_cluster included) to whoever waits on the barrier
__device__ __forceinline__ void mbar_arrive_cluster(unsigned bar_cluster)
{
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" :: "r"(bar_cluster) : "memory");
}
// mbar_wait with cluster-scope acquire: for barriers other CTAs of the cluster arrive on
__device__ __forceinline__ void mbar_wait_cluster(unsigned bar, unsigned parity)
{
    unsigned done = 0;
    while (!done)
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void st_shared_cluster_v4(unsigned addr_cluster, float4 v)
{
    asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" :: "r"(addr_cluster), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                 : "memory");
}
// TMA loads of a CTA pair: destination in this CTA's shared memory, completion on a barrier of either CTA
__device__ __forceinline__ void tma_load_2d_pair(unsigned dst, const CUtensorMap *map, int c0, int c1, unsigned bar_cluster)
{
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 :: "r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar_cluster) : "memory");
}
__device__ __forceinline__ void tma_load_4d_pair(unsigned dst, const CUtensorMap *map, int c0, int c1, int c2, int c3,
                                                 unsigned bar_cluster)
{
    asm volatile("cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
                 :: "r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar_cluster) : "memory");
}
// umma_f16_masked for the pair (M = 256): bit i of mask word w set = row 32w + i of the 256-row D is not written
__device__ __forceinline__ void umma_f16_masked_pair(unsigned d_tmem, uint64_t a, uint64_t b, unsigned idesc, unsigned accumulate,
                                                     unsigned mask)
{
    asm volatile("{ .reg .pred p; setp.ne.b32 p, %4, 0; tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, "
                 "{%5, %5, %5, %5, %5, %5, %5, %5}, p; }"
                 :: "r"(d_tmem), "l"(a), "l"(b), "r"(idesc), "r"(accumulate), "r"(mask) : "memory");
}
// arrive on the barrier at shared address `bar` in BOTH CTAs of the pair once the pair MMAs issued before complete
__device__ __forceinline__ void umma_commit_pair(unsigned bar)
{
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 :: "r"(bar), "h"((unsigned short)3) : "memory");
}
// tmem_alloc / tmem_dealloc for a pair: one warp of EACH CTA calls them, the columns are the same in both
__device__ __forceinline__ void tmem_alloc_pair(unsigned dst, unsigned cols)
{
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(dst), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(unsigned tmem, unsigned cols)
{
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(cols) : "memory");
}

}  // namespace msw

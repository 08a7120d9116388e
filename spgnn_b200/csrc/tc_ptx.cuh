// PTX wrappers shared by the TMA-fed tcgen05 kernels (gemm_tma.cu): mbarrier, TMA (cp.async.bulk.tensor), tcgen05
// alloc / mma / commit / ld, UMMA shared-memory and instruction descriptors.  sm_100a only.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace spgnn {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "LAB_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra LAB_DONE_%=;\n\t"
        "bra LAB_WAIT_%=;\n\t"
        "LAB_DONE_%=:\n\t"
        "}" ::"r"(bar), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// TMA tile loads global -> shared (this CTA), completion signalled on an mbarrier as transaction bytes
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}

// thread-block cluster helpers
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {          // every thread of every CTA of the cluster
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// one lane of a converged warp (the same lane every time): the issuing thread of the single-thread tcgen05 / TMA paths
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]; bf16 inputs, fp32 accumulate
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on an mbarrier once every previously issued UMMA of this thread has completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// UMMA shared-memory descriptor, SWIZZLE_128B (sm_100 "version 1" descriptor):
//   [0,14) start address >> 4 | [16,30) leading byte offset >> 4 | [32,46) stride byte offset >> 4 | [46,48) = 1 |
//   [61,64) layout type (2 = SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// instruction descriptor (kind::f16): c=f32 [4,6)=1, a=bf16 [7,10)=1, b=bf16 [10,13)=1, a_major bit 15, b_major bit 16
// (0 = K-major, 1 = MN-major), n>>3 at [17,23), m>>4 at [24,29); M = 128
__host__ __device__ __forceinline__ uint32_t make_idesc(int n, bool mn_major) {
    uint32_t d = (1u << 4) | (1u << 7) | (1u << 10);
    if (mn_major) d |= (1u << 15) | (1u << 16);
    d |= (uint32_t)(n >> 3) << 17;
    d |= (uint32_t)(128 >> 4) << 24;
    return d;
}

// ---- CTA pair (cta_group::2): two CTAs of a cluster on the two SMs of a TPC run ONE UMMA of M = 256; each CTA holds
// its 128 rows of A, HALF of the B tile (N / 2 rows) and its 128 lanes of the accumulator; the leader (rank 0) issues.
// address of the same shared-memory offset in CTA `rank` of the cluster (shared::cluster window)
__device__ __forceinline__ uint32_t mapa_u32(uint32_t saddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
// arrive on an mbarrier of any CTA of the cluster (cluster-window address)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
// TMA tile load into THIS CTA's shared memory, completion bytes signalled on an mbarrier that may live in the peer CTA
__device__ __forceinline__ void tma_load_3d_pair(uint32_t dst, const CUtensorMap* m, uint32_t cluster_bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(m)), "r"(cluster_bar), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
// both CTAs of the pair call these with the same warp and the same destination offset
__device__ __forceinline__ void tmem_alloc_pair(uint32_t dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on the mbarrier at this CTA-relative address in every CTA of cta_mask once the pair's UMMAs have completed
__device__ __forceinline__ void umma_commit_pair(uint32_t bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
                 "h"(cta_mask)
                 : "memory");
}
// instruction descriptor of the pair UMMA: M = 256 (128 per CTA), N = the whole tile width
__host__ __device__ __forceinline__ uint32_t make_idesc_pair(int n) {
    uint32_t d = (1u << 4) | (1u << 7) | (1u << 10);
    d |= (uint32_t)(n >> 3) << 17;
    d |= (uint32_t)(256 >> 4) << 24;
    return d;
}

// fp32 pair -> packed bf16 (hi) and packed bf16 of the remainders (lo); low half = first element.
// a = hi + lo + r with |r| <= 2^-17 |a| for normal a (the largest over all 2^23 mantissas of a binade is
// 2^-17.003: each rounding keeps 8 significant bits, the two together 16 and a sign).
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    hi = *reinterpret_cast<uint32_t*>(&h);
    const float ra = a - __uint_as_float(hi << 16);
    const float rb = b - __uint_as_float(hi & 0xFFFF0000u);
    __nv_bfloat162 l = __floats2bfloat162_rn(ra, rb);
    lo = *reinterpret_cast<uint32_t*>(&l);
}
// inverse: packed bf16 pair (hi) + packed pair (lo) -> two floats
__device__ __forceinline__ void join2(uint32_t hi, uint32_t lo, float& a, float& b) {
    a = __uint_as_float(hi << 16) + __uint_as_float(lo << 16);
    b = __uint_as_float(hi & 0xFFFF0000u) + __uint_as_float(lo & 0xFFFF0000u);
}

}  // namespace ptx
}  // namespace spgnn

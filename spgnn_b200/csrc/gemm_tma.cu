// TMA-fed tcgen05 GEMMs over "planes" operands (the production projection path).
//
// Planes: an fp32-valued matrix X[rows, cols] held as TWO bf16 matrices, X = hi + lo (|residual| <= 2^-17 |X|),
// both [rows, ld] row-major, lo = hi + plane_stride.  Same bytes as fp32, but directly consumable by the tensor
// cores: the product a*b is formed as a_hi*b_hi + a_hi*b_lo + a_lo*b_hi with fp32 accumulation in TMEM (three
// kind::f16 UMMAs per k-step, relative error ~3*2^-18 per product — inside the 1e-4 parity bar with margin, at 3/2 of
// the cost of ONE tf32 pass; a single tf32 pass would break that bar).
// The kernels that PRODUCE activations (aggregation epilogues, spgnn_split_planes) write planes, so no GEMM converts
// anything: operands go global -> shared by TMA (cp.async.bulk.tensor, SWIZZLE_128B) and shared -> tensor core by
// UMMA descriptors; no register staging, several stages (64-96 KB each) in flight per SM.
//
//   nt_planes_kernel : C[M,N] fp32 = [A1|A2][M,K] * B[N,K]^T (+bias)(act).  A: activation planes (K-major boxes
//                      64 x 128 x 2 planes), B: weight planes pre-split once per call.  Persistent over 128 x BN tiles,
//                      two TMEM accumulator buffers (epilogue of tile i overlaps the MMAs of tile i+1).
//                      Forward projection and dX = dY * W.
//   tn_planes_kernel : D[p, q] = sum over nodes m of P[m, p] * Q[m, q]  (weight gradient dW = dY^T X, reduction over
//                      the 1.2 M nodes, split across CTAs into partial sums reduced in fixed order).  Both operands
//                      are activation planes read MN-major: TMA boxes of 64 columns x 32 nodes x 2 planes land as
//                      [hi 4 KB][lo 4 KB] per 64-column block — exactly the SW128 MN-major UMMA layout, no transposition.
//                      A CTA owns up to 4 P blocks (two M=128 accumulators sharing the Q tile) x up to 4 Q blocks
//                      (N <= 256); blocks are enumerated across the concatenated sources ([X1 | X2]).
//
// Warp roles (192 threads): warps 0-3 epilogue (TMEM lanes 32w..32w+31), warp 4 TMEM alloc + single-thread UMMA
// issue, warp 5 single-thread TMA producer.
#include "common.cuh"
#include "tc_ptx.cuh"

namespace spgnn {
namespace tma {
using namespace ptx;

constexpr int BM = 128;
constexpr int BK = 64;                         // bf16 elements per k-block = one 128-byte swizzle row
constexpr int kThreads = 192;
constexpr int kEpiWarps = 4;
constexpr int kMaxStages = 6;
constexpr int kMaxBN = 256;
constexpr int kABytes = BM * 128 * 2;          // hi + lo planes of the A tile: 32 KB
constexpr int kStgLd = 36;                     // padded row of the per-warp 32x32 epilogue staging tile (floats)
constexpr int kStgBytes = kEpiWarps * 32 * kStgLd * 4;
constexpr int kSmemLimit = 232448;             // 227 KB opt-in limit per CTA
constexpr int kNtFixed = 1024 /*align*/ + 256 /*barriers*/ + kStgBytes;

// explicit shared-space accesses with 32-bit addresses: a float* carved out of the dynamic shared array compiles to
// generic LD.E / ST.E with 64-bit address arithmetic (ncu: the staging store was the top stall line of wide_kernel)
__device__ __forceinline__ float4 ld_shared4(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void st_shared4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

struct NtMaps { CUtensorMap a1, a2, b; };
struct NtArgs {
    const float* bias; int act; float slope;
    float* C; int64_t ldc;
    int64_t M; int N;
    int BN, nt_n; int64_t nt_m;
    int kb1, kb2;
    int stages, stage_bytes;
    // optional dropout mask on the OUTPUT (dX of a layer whose input went through feat_drop): 16 hash bits per
    // element, chunk index = row * mnch + col / 4 -- the convention of every plane producer (split_planes_kernel)
    uint32_t mthr; float mscale; uint64_t mseed; int64_t mnch, moff;
};
__device__ __forceinline__ float4 nt_mask4(const NtArgs& g, float4 x, int64_t row, int col) {
    const uint64_t h = chunk_hash(g.mseed, (uint64_t)row * (uint64_t)g.mnch + (uint64_t)(g.moff + (col >> 2)));
    x.x = ((uint32_t)(h) & 0xFFFFu) >= g.mthr ? x.x * g.mscale : 0.f;
    x.y = ((uint32_t)(h >> 16) & 0xFFFFu) >= g.mthr ? x.y * g.mscale : 0.f;
    x.z = ((uint32_t)(h >> 32) & 0xFFFFu) >= g.mthr ? x.z * g.mscale : 0.f;
    x.w = ((uint32_t)(h >> 48) & 0xFFFFu) >= g.mthr ? x.w * g.mscale : 0.f;
    return x;
}
struct NtShared {
    uint64_t full[kMaxStages];
    uint64_t empty[kMaxStages];
    uint64_t tmem_full[2];
    uint64_t tmem_empty[2];
    uint32_t tmem_base;
};

// Epilogue of one 128 x BN accumulator for one warp (TMEM lanes 32 * warp ..): TMEM -> registers -> padded smem staging
// tile -> global, so that every store instruction writes whole 128-byte row segments.
__device__ __forceinline__ void nt_epilogue_tile(const NtArgs& g, uint32_t stg, uint32_t taddr, int64_t m0, int n0,
                                                 int ncols, int warp, int lane, bool vec_ok, bool plain) {
    for (int c0 = 0; c0 < ncols; c0 += 32) {
        uint32_t v[32];
        tmem_ld16(taddr + c0, *reinterpret_cast<uint32_t(*)[16]>(&v[0]));
        tmem_ld16(taddr + c0 + 16, *reinterpret_cast<uint32_t(*)[16]>(&v[16]));
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 8; ++j)
            st_shared4(stg + (lane * kStgLd + 4 * j) * 4, v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        __syncwarp();
        const int cc = (lane & 7) * 4;
        const int col = n0 + c0 + cc;
        const int rsub = lane >> 3;                                   // row within each group of 4
        const int64_t row0 = m0 + warp * 32 + rsub;
        float* q = g.C + row0 * g.ldc + col;
        const int64_t qstep = 4 * g.ldc;
        const int nrow = (int)max((int64_t)0, min((int64_t)8, (g.M - row0 + 3) / 4));
        const uint32_t sp = stg + (rsub * kStgLd + cc) * 4;
        if (plain && vec_ok && c0 + 32 <= ncols) {
            if (g.mthr) {
#pragma unroll
                for (int itr = 0; itr < 8; ++itr)
                    if (itr < nrow)
                        st4(q + itr * qstep, nt_mask4(g, ld_shared4(sp + itr * (4 * kStgLd * 4)), row0 + 4 * itr, col));
            } else {
#pragma unroll
                for (int itr = 0; itr < 8; ++itr)
                    if (itr < nrow) st4(q + itr * qstep, ld_shared4(sp + itr * (4 * kStgLd * 4)));
            }
        } else {
            float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
            if (g.bias) {
                if (col + 0 < g.N) bv.x = __ldg(g.bias + col + 0);
                if (col + 1 < g.N) bv.y = __ldg(g.bias + col + 1);
                if (col + 2 < g.N) bv.z = __ldg(g.bias + col + 2);
                if (col + 3 < g.N) bv.w = __ldg(g.bias + col + 3);
            }
            const int nvalid = ncols - (c0 + cc);
            for (int itr = 0; itr < nrow; ++itr) {
                float4 x = ld_shared4(sp + itr * (4 * kStgLd * 4));
                x.x = act_fwd(x.x + bv.x, g.act, g.slope);
                x.y = act_fwd(x.y + bv.y, g.act, g.slope);
                x.z = act_fwd(x.z + bv.z, g.act, g.slope);
                x.w = act_fwd(x.w + bv.w, g.act, g.slope);
                if (g.mthr) x = nt_mask4(g, x, row0 + 4 * itr, col);
                float* qq = q + itr * qstep;
                if (vec_ok && nvalid >= 4) st4(qq, x);
                else {
                    if (nvalid > 0) qq[0] = x.x;
                    if (nvalid > 1) qq[1] = x.y;
                    if (nvalid > 2) qq[2] = x.z;
                    if (nvalid > 3) qq[3] = x.w;
                }
            }
        }
        __syncwarp();
    }
}

__global__ void __launch_bounds__(kThreads, 1) nt_planes_kernel(const __grid_constant__ NtMaps maps, const NtArgs g) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int stages_bytes = g.stages * g.stage_bytes;
    NtShared* sh = reinterpret_cast<NtShared*>(smem + stages_bytes);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem_base = smem_u32(smem);

    if (threadIdx.x == 0) {
        for (int s = 0; s < g.stages; ++s) {
            mbar_init(smem_u32(&sh->full[s]), 1);
            mbar_init(smem_u32(&sh->empty[s]), 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(smem_u32(&sh->tmem_full[b]), 1);
            mbar_init(smem_u32(&sh->tmem_empty[b]), kEpiWarps * 32);
        }
        fence_barrier_init();
    }
    if (warp == 5 && lane == 0) {
        prefetch_tmap(&maps.a1);
        if (g.kb2 > 0) prefetch_tmap(&maps.a2);
        prefetch_tmap(&maps.b);
    }
    if (warp == kEpiWarps) tmem_alloc(smem_u32(&sh->tmem_base), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = sh->tmem_base;

    const int64_t n_tiles = g.nt_m * g.nt_n;
    const int64_t tile0 = blockIdx.x, tile_step = gridDim.x;
    const int nkb = g.kb1 + g.kb2;

    if (warp < kEpiWarps) {
        // ===================================================== epilogue: TMEM -> registers -> smem staging -> global
        int it = 0;
        const uint32_t stg = smem_base + stages_bytes + 256 + warp * (32 * kStgLd * 4);
        const bool vec_ok = (g.ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(g.C) & 15) == 0);
        const bool plain = (g.act == SPGNN_ACT_NONE) && (g.bias == nullptr);
        for (int64_t tile = tile0; tile < n_tiles; tile += tile_step, ++it) {
            const int buf = it & 1;
            const uint32_t par = (it >> 1) & 1;
            const int64_t m0 = (tile / g.nt_n) * BM;
            const int n0 = (int)(tile % g.nt_n) * g.BN;
            const int ncols = min(g.BN, g.N - n0);
            mbar_wait(smem_u32(&sh->tmem_full[buf]), par);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(buf * kMaxBN);
            nt_epilogue_tile(g, stg, taddr, m0, n0, ncols, warp, lane, vec_ok, plain);
            tc_fence_before();
            mbar_arrive(smem_u32(&sh->tmem_empty[buf]));
        }
    } else if (warp == kEpiWarps) {
        // ===================================================== UMMA issuer: the whole warp walks the loop, one elected
        // lane issues (see nt_pair_kernel: `if (lane == 0)` around the loop costs an ELECT / R2UR waterfall per UMMA)
        {
            int it = 0;
            uint32_t kcount = 0;
            const uint32_t tbase = __shfl_sync(kFull, tmem_base, 0);
            for (int64_t tile = tile0; tile < n_tiles; tile += tile_step, ++it) {
                const int buf = it & 1;
                const uint32_t par = (it >> 1) & 1;
                const int n0 = (int)(tile % g.nt_n) * g.BN;
                const int ncols = min(g.BN, g.N - n0);
                const int n_mma = (ncols + 15) & ~15;
                const uint32_t idesc = make_idesc(n_mma, false);
                mbar_wait(smem_u32(&sh->tmem_empty[buf]), par ^ 1);     // epilogue drained this accumulator
                tc_fence_after();
                const uint32_t tmem_d = tbase + (uint32_t)(buf * kMaxBN);
                for (int kb = 0; kb < nkb; ++kb, ++kcount) {
                    const int s = kcount % g.stages;
                    const uint32_t sp = (kcount / g.stages) & 1;
                    mbar_wait(smem_u32(&sh->full[s]), sp);
                    tc_fence_after();
                    const uint32_t a_hi = smem_base + s * g.stage_bytes;
                    const uint32_t a_lo = a_hi + BM * 128;
                    const uint32_t b_hi = a_hi + kABytes;
                    const uint32_t b_lo = b_hi + g.BN * 128;
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < BK / 16; ++k) {
                            const uint32_t ko = k * 32;      // 16 bf16 = 32 bytes along the swizzled row
                            const uint64_t dah = make_desc(a_hi + ko, 16, 1024), dal = make_desc(a_lo + ko, 16, 1024);
                            const uint64_t dbh = make_desc(b_hi + ko, 16, 1024), dbl = make_desc(b_lo + ko, 16, 1024);
                            umma_bf16(tmem_d, dah, dbh, idesc, (kb | k) != 0);
                            umma_bf16(tmem_d, dah, dbl, idesc, 1);
                            umma_bf16(tmem_d, dal, dbh, idesc, 1);
                        }
                        umma_commit(smem_u32(&sh->empty[s]));          // frees the smem stage when these UMMAs retire
                    }
                    __syncwarp();
                }
                if (elect_one()) umma_commit(smem_u32(&sh->tmem_full[buf]));    // accumulator complete -> epilogue
                __syncwarp();
            }
        }
    } else if (lane == 0) {
        // ===================================================== TMA producer (one thread)
        uint32_t kcount = 0;
        const uint32_t tx = (uint32_t)g.stage_bytes;
        for (int64_t tile = tile0; tile < n_tiles; tile += tile_step) {
            const int m0 = (int)((tile / g.nt_n) * BM);
            const int n0 = (int)(tile % g.nt_n) * g.BN;
            for (int kb = 0; kb < nkb; ++kb, ++kcount) {
                const int s = kcount % g.stages;
                const uint32_t sp = (kcount / g.stages) & 1;
                mbar_wait(smem_u32(&sh->empty[s]), sp ^ 1);
                const uint32_t bar = smem_u32(&sh->full[s]);
                mbar_expect_tx(bar, tx);
                const uint32_t dst = smem_base + s * g.stage_bytes;
                if (kb < g.kb1) tma_load_3d(dst, &maps.a1, bar, kb * BK, m0, 0);
                else tma_load_3d(dst, &maps.a2, bar, (kb - g.kb1) * BK, m0, 0);
                tma_load_3d(dst + kABytes, &maps.b, bar, kb * BK, n0, 0);
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == kEpiWarps) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// ---------------------------------------------------------------------------------------------- NT, CTA pairs
// The same GEMM with tcgen05 cta_group::2: a cluster of two CTAs (the two SMs of a TPC) owns a 256 x BN tile.  Each
// CTA loads ITS 128 rows of A and HALF of the weight tile (BN / 2 rows), the leader issues one M = 256 UMMA per
// (k-step, pass) that reads both halves, and each CTA drains its own 128 accumulator lanes.  Per CTA and k-block that
// is 32 KB + BN * 128 B through the L2 -> SM path instead of 32 KB + BN * 256 B: the chip-wide L2 throughput
// (~6300 B/clk = 42.6 B/clk/SM) is what bounds the single-CTA kernel on the big projections (tensor pipe 62 - 73 %),
// and TMA multicast of the weight tile did not relieve it at cluster size 2 (measured neutral and removed,
// profiles/r01_gemm_check_cluster_vs_plain.txt).
// Barriers: full[s] of the LEADER collects the transaction bytes of both CTAs' loads (cp.async.bulk.tensor
// .cta_group::2 signals the peer's barrier); empty[s] / tmem_full[b] are arrived in both CTAs by multicast commits;
// tmem_empty[b] of the leader counts the epilogue threads of both CTAs (the peer arrives through the cluster window).
__global__ void __launch_bounds__(kThreads, 1) nt_pair_kernel(const __grid_constant__ NtMaps maps, const NtArgs g) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int stages_bytes = g.stages * g.stage_bytes;
    NtShared* sh = reinterpret_cast<NtShared*>(smem + stages_bytes);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;

    if (threadIdx.x == 0) {
        for (int s = 0; s < g.stages; ++s) {
            mbar_init(smem_u32(&sh->full[s]), 1);          // leader: its producer's arrive.expect_tx (bytes of both CTAs)
            mbar_init(smem_u32(&sh->empty[s]), 1);         // multicast commit of the leader's UMMA issuer
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(smem_u32(&sh->tmem_full[b]), 1);     // multicast commit
            mbar_init(smem_u32(&sh->tmem_empty[b]), 2 * kEpiWarps);        // leader: one arrival per epilogue warp of both CTAs
        }
        fence_barrier_init();
    }
    if (warp == 5 && lane == 0) {
        prefetch_tmap(&maps.a1);
        if (g.kb2 > 0) prefetch_tmap(&maps.a2);
        prefetch_tmap(&maps.b);
    }
    if (warp == kEpiWarps) tmem_alloc_pair(smem_u32(&sh->tmem_base), 512);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                      // both CTAs' barriers and TMEM exist before anything crosses the pair
    tc_fence_after();
    const uint32_t tmem_base = sh->tmem_base;

    const int64_t n_tiles = ((g.nt_m + 1) / 2) * g.nt_n;
    const int64_t tile0 = blockIdx.x / 2, tile_step = gridDim.x / 2;
    const int nkb = g.kb1 + g.kb2;
    const int half = g.BN / 2;               // weight rows held by each CTA

    if (warp < kEpiWarps) {
        // ===================================================== epilogue (both CTAs, own accumulator lanes)
        int it = 0;
        const uint32_t stg = smem_base + stages_bytes + 256 + warp * (32 * kStgLd * 4);
        const bool vec_ok = (g.ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(g.C) & 15) == 0);
        const bool plain = (g.act == SPGNN_ACT_NONE) && (g.bias == nullptr);
        for (int64_t tile = tile0; tile < n_tiles; tile += tile_step, ++it) {
            const int buf = it & 1;
            const uint32_t par = (it >> 1) & 1;
            const int64_t m0 = ((tile / g.nt_n) * 2 + rank) * BM;
            const int n0 = (int)(tile % g.nt_n) * g.BN;
            const int ncols = min(g.BN, g.N - n0);
            mbar_wait(smem_u32(&sh->tmem_full[buf]), par);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(buf * kMaxBN);
            nt_epilogue_tile(g, stg, taddr, m0, n0, ncols, warp, lane, vec_ok, plain);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&sh->tmem_empty[buf]), 0));
        }
    } else if (warp == kEpiWarps) {
        // ===================================================== UMMA issuer (leader CTA)
        // The WHOLE warp walks the loop and one elected lane issues: inside `if (lane == 0)` the operands of every
        // UMMA (descriptors, TMEM address, instruction descriptor) live in vector registers of a divergent thread and
        // ptxas wraps each tcgen05.mma in an ELECT / R2UR.BROADCAST / BRA.U.ANY waterfall (~16 instructions, ~110
        // cycles per UMMA for the single issuing thread -- more than an N = 128 UMMA takes to execute).
        if (leader) {
            int it = 0;
            uint32_t kcount = 0;
            const uint32_t idesc = make_idesc_pair(g.BN);
            const uint32_t tbase = __shfl_sync(kFull, tmem_base, 0);
            for (int64_t tile = tile0; tile < n_tiles; tile += tile_step, ++it) {
                const int buf = it & 1;
                const uint32_t par = (it >> 1) & 1;
                mbar_wait(smem_u32(&sh->tmem_empty[buf]), par ^ 1);     // both epilogues drained this accumulator
                tc_fence_after();
                const uint32_t tmem_d = tbase + (uint32_t)(buf * kMaxBN);
                for (int kb = 0; kb < nkb; ++kb, ++kcount) {
                    const int s = kcount % g.stages;
                    const uint32_t sp = (kcount / g.stages) & 1;
                    mbar_wait(smem_u32(&sh->full[s]), sp);
                    tc_fence_after();
                    const uint32_t a_hi = smem_base + s * g.stage_bytes;
                    const uint32_t a_lo = a_hi + BM * 128;
                    const uint32_t b_hi = a_hi + kABytes;
                    const uint32_t b_lo = b_hi + half * 128;
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < BK / 16; ++k) {
                            const uint32_t ko = k * 32;
                            const uint64_t dah = make_desc(a_hi + ko, 16, 1024), dal = make_desc(a_lo + ko, 16, 1024);
                            const uint64_t dbh = make_desc(b_hi + ko, 16, 1024), dbl = make_desc(b_lo + ko, 16, 1024);
                            umma_bf16_pair(tmem_d, dah, dbh, idesc, (kb | k) != 0);
                            umma_bf16_pair(tmem_d, dah, dbl, idesc, 1);
                            umma_bf16_pair(tmem_d, dal, dbh, idesc, 1);
                        }
                        umma_commit_pair(smem_u32(&sh->empty[s]), 3);       // the stage is free in both CTAs
                    }
                    __syncwarp();
                }
                if (elect_one()) umma_commit_pair(smem_u32(&sh->tmem_full[buf]), 3);   // accumulators complete
                __syncwarp();
            }
        }
    } else if (lane == 0) {
        // ===================================================== TMA producer (one thread per CTA)
        uint32_t kcount = 0;
        const uint32_t tx = 2u * (uint32_t)g.stage_bytes;               // both CTAs' loads land on the leader's barrier
        for (int64_t tile = tile0; tile < n_tiles; tile += tile_step) {
            const int m0 = (int)(((tile / g.nt_n) * 2 + rank) * BM);
            const int n0 = (int)(tile % g.nt_n) * g.BN + (int)rank * half;
            for (int kb = 0; kb < nkb; ++kb, ++kcount) {
                const int s = kcount % g.stages;
                const uint32_t sp = (kcount / g.stages) & 1;
                mbar_wait(smem_u32(&sh->empty[s]), sp ^ 1);
                const uint32_t bar = mapa_u32(smem_u32(&sh->full[s]), 0);
                if (leader) mbar_expect_tx(smem_u32(&sh->full[s]), tx);
                const uint32_t dst = smem_base + s * g.stage_bytes;
                if (kb < g.kb1) tma_load_3d_pair(dst, &maps.a1, bar, kb * BK, m0, 0);
                else tma_load_3d_pair(dst, &maps.a2, bar, (kb - g.kb1) * BK, m0, 0);
                tma_load_3d_pair(dst + kABytes, &maps.b, bar, kb * BK, n0, 0);
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                      // no CTA leaves (or frees TMEM) while its peer may still use the pair
    if (warp == kEpiWarps) {
        tc_fence_after();
        tmem_dealloc_pair(tmem_base, 512);
    }
}

// ---------------------------------------------------------------------------------------------- wide (output layer)
// out = 1/H sum_h act([Ax_h | x] * [W_fc,h | W_res,h]^T + b_h)   (spgnn_wide_linear, include/spgnn_b200.h)
// A = XA planes [M, (H+1)*kp] (block h = Ax_h, block H = x), B = weight planes [H*F, nparts*kp].  A tile is 128 rows x
// BN columns x H heads: H accumulators of BN TMEM columns each (x 2 buffers), the k-loop runs head after head; the
// epilogue walks the heads one at a time, so per thread only the running mean (mode 0) or the incoming gradient
// (mode 1) stays in registers.  Mode 0 can also write act'(pre_h) of every head (dact), which mode 2 reads back.
// Mode 2 (dpre from the gradient of a linear head on the output): A = the head's output-gradient planes [M, C],
// B = W_head^T planes [F, 64]; ONE accumulator (the head's dX, the same for every head h), and the epilogue forms
// dpre_h = (sum of the fp32 sources + acc) / H * dact_h -- the operation order of mode 1 with the head's dX as its
// last source, without recomputing the forward GEMM.
struct WideMaps { CUtensorMap a, b; };
struct WideArgs {
    int mode, H, F, act;
    const float* bias;
    float* out; int64_t ldo;
    __nv_bfloat16* outp; int64_t ldp, psp;
    float* dact; int64_t ldda;                 // mode 0: written when non-null; mode 2: read
    const float* g[3]; int64_t ldg[3]; int n_g;
    __nv_bfloat16* dpre; int64_t ldd, psd;
    float* dbias_ws;
    int64_t M; int BN, nt_n; int64_t nt_m;
    int hacc;                                  // accumulators per tile: H (modes 0 and 1) or 1 (mode 2)
    int kbp, nparts, kp;
    int stages, stage_bytes;
};
constexpr int kWideEpiWarps = 16;                      // four warps per TMEM lane quadrant, interleaved column chunks
constexpr int kWideThreads = (kWideEpiWarps + 2) * 32;
constexpr int kWideStgBytes = kWideEpiWarps * 32 * 16 * 4;   // one swizzled 32 x 16 fp32 tile per epilogue warp
constexpr int kWideFixed = 1024 /*align*/ + 256 /*barriers*/ + kWideStgBytes;

template <int ACT>
__device__ __forceinline__ float wide_act(float x, int act) {
    if (ACT == SPGNN_ACT_ELU) return x > 0.f ? x : exp_fast(x) - 1.f;     // FMUL + MUFU.EX2 + FADD on the x <= 0 side
    if (ACT == SPGNN_ACT_NONE) return x;
    return act_fwd(x, act, kGatLeakySlope);
}
template <int ACT>
__device__ __forceinline__ float wide_act_grad(float y, int act) {
    if (ACT == SPGNN_ACT_ELU) return y > 0.f ? 1.f : y + 1.f;
    if (ACT == SPGNN_ACT_NONE) return 1.f;
    return act_grad_from_out(y, act, kGatLeakySlope);
}
// act(x) and act'(x) from the pre-activation in one go (ELU: one exponential serves both)
template <int ACT>
__device__ __forceinline__ float wide_act_grad_pre(float x, int act) {
    if (ACT == SPGNN_ACT_ELU) return x > 0.f ? 1.f : exp_fast(x);
    if (ACT == SPGNN_ACT_NONE) return 1.f;
    return act_grad_from_out(act_fwd(x, act, kGatLeakySlope), act, kGatLeakySlope);
}
// run += act(x) and d = act'(x): the values of wide_act and wide_act_grad_pre, bit for bit
template <int ACT>
__device__ __forceinline__ void wide_act_and_grad(float x, int act, float& run, float& d) {
    if (ACT == SPGNN_ACT_ELU) {
        const float e = exp_fast(x);
        run += x > 0.f ? x : e - 1.f;
        d = x > 0.f ? 1.f : e;
    } else {
        run += wide_act<ACT>(x, act);
        d = wide_act_grad_pre<ACT>(x, act);
    }
}
__device__ __forceinline__ void st_planes4(__nv_bfloat16* q, int64_t ps, float4 d) {
    uint32_t h0, l0, h1, l1;
    split2(d.x, d.y, h0, l0);
    split2(d.z, d.w, h1, l1);
    *reinterpret_cast<uint2*>(q) = make_uint2(h0, h1);
    *reinterpret_cast<uint2*>(q + ps) = make_uint2(l0, l1);
}
// Epilogue of one 128 x BN x H tile for one warp: 16-column chunks; TMEM (lane = row) -> swizzled smem tile ->
// (row = lane/4 + 8i, 4 columns) per thread, so that global accesses are whole 32/64-byte row segments.  In mode 1
// the incoming gradient of the warp's four chunks is loaded BEFORE waiting for the accumulator, so its DRAM latency
// hides behind the MMAs of this tile.  The MMA work per output element is small here (K = 2 x 192), so the tile is
// only hidden behind the tensor pipe if the epilogue stays near ~1 issue slot per element: MODE and ACT are template
// parameters, the staging tile is addressed in the shared window, row pointers are hoisted out of the head loop.
// DACT (mode 0): also store act'(pre_h) of every head into dact [M, H*F].
template <int ACT, int MODE, bool DACT>
__device__ __forceinline__ void wide_epilogue_tile(const WideArgs& g, uint32_t stg, float* dbias_row, uint32_t taddr,
                                                   int64_t m0, int n0, int ncols, int warp, int lane,
                                                   uint32_t full_bar, uint32_t full_par) {
    const int quad = warp & 3, part = warp >> 2;
    const int r0 = lane >> 2, cq = lane & 3;
    const float inv_h = 1.f / (float)g.H;
    const int64_t row0 = m0 + quad * 32 + r0;
    const int nrow = (int)max((int64_t)0, min((int64_t)4, (g.M - row0 + 7) / 8));
    // staging addresses: this lane's TMEM row (write side) and the four rows it reads back
    const uint32_t st_w = stg + lane * 64;
    const int sw_w = (lane >> 1) & 3;
    uint32_t st_r[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = r0 + 8 * i;
        st_r[i] = stg + r * 64 + ((cq ^ ((r >> 1) & 3)) << 4);
    }
    const int colq = n0 + cq * 4;
    for (int cg = 0; cg < ncols; cg += 128) {
        float4 run[2][4];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int c0 = cg + q * 64 + part * 16;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                run[q][i] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (MODE == 1 && i < nrow && c0 < ncols)
                    run[q][i] = ldg4(g.g[0] + (row0 + 8 * i) * g.ldg[0] + colq + c0);
            }
        }
        if (MODE == 1) {
            for (int s = 1; s < g.n_g; ++s) {
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const int c0 = cg + q * 64 + part * 16;
                    float4 t[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        t[i] = (i < nrow && c0 < ncols) ? ldg4(g.g[s] + (row0 + 8 * i) * g.ldg[s] + colq + c0)
                                                        : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        run[q][i].x += t[i].x; run[q][i].y += t[i].y; run[q][i].z += t[i].z; run[q][i].w += t[i].w;
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < 2; ++q)
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    run[q][i].x *= inv_h; run[q][i].y *= inv_h; run[q][i].z *= inv_h; run[q][i].w *= inv_h;
                }
        }
        if (cg == 0) {
            mbar_wait(full_bar, full_par);
            tc_fence_after();
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int c0 = cg + q * 64 + part * 16;
            if (c0 >= ncols) break;
            const int col = colq + c0;
            __nv_bfloat16* dp = MODE == 1 ? g.dpre + row0 * g.ldd + col : nullptr;
            const int64_t dstep = 8 * g.ldd;
            float* da = DACT ? g.dact + row0 * g.ldda + col : nullptr;
            const int64_t astep = 8 * g.ldda;
            uint32_t v[16];
            tmem_ld16(taddr + c0, v);
            for (int h = 0; h < g.H; ++h) {
                const float4 bv = g.bias ? ldg4(g.bias + h * g.F + col) : make_float4(0.f, 0.f, 0.f, 0.f);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    st_shared4(st_w + ((j ^ sw_w) << 4), v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                __syncwarp();
                if (h + 1 < g.H) tmem_ld16(taddr + (h + 1) * g.BN + c0, v);      // next head: in flight during the math
                float4 bs = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    float4 x = ld_shared4(st_r[i]);
                    if (MODE == 0 && DACT) {
                        float4 a;
                        wide_act_and_grad<ACT>(x.x + bv.x, g.act, run[q][i].x, a.x);
                        wide_act_and_grad<ACT>(x.y + bv.y, g.act, run[q][i].y, a.y);
                        wide_act_and_grad<ACT>(x.z + bv.z, g.act, run[q][i].z, a.z);
                        wide_act_and_grad<ACT>(x.w + bv.w, g.act, run[q][i].w, a.w);
                        if (i < nrow) st4(da + i * astep + h * g.F, a);
                    } else if (MODE == 0) {
                        run[q][i].x += wide_act<ACT>(x.x + bv.x, g.act);
                        run[q][i].y += wide_act<ACT>(x.y + bv.y, g.act);
                        run[q][i].z += wide_act<ACT>(x.z + bv.z, g.act);
                        run[q][i].w += wide_act<ACT>(x.w + bv.w, g.act);
                    } else if (i < nrow) {
                        float4 d;
                        d.x = run[q][i].x * wide_act_grad_pre<ACT>(x.x + bv.x, g.act);
                        d.y = run[q][i].y * wide_act_grad_pre<ACT>(x.y + bv.y, g.act);
                        d.z = run[q][i].z * wide_act_grad_pre<ACT>(x.z + bv.z, g.act);
                        d.w = run[q][i].w * wide_act_grad_pre<ACT>(x.w + bv.w, g.act);
                        st_planes4(dp + i * dstep + h * g.F, g.psd, d);
                        bs.x += d.x; bs.y += d.y; bs.z += d.z; bs.w += d.w;
                    }
                }
                if (MODE == 1 && dbias_row) {
#pragma unroll
                    for (int o = 4; o < 32; o <<= 1) {
                        bs.x += __shfl_xor_sync(kFull, bs.x, o); bs.y += __shfl_xor_sync(kFull, bs.y, o);
                        bs.z += __shfl_xor_sync(kFull, bs.z, o); bs.w += __shfl_xor_sync(kFull, bs.w, o);
                    }
                    if (lane < 4) {                       // this CTA's partial row (L2 reductions, no return value)
                        float* p = dbias_row + h * g.F + col;
                        atomicAdd(p, bs.x); atomicAdd(p + 1, bs.y); atomicAdd(p + 2, bs.z); atomicAdd(p + 3, bs.w);
                    }
                }
                __syncwarp();
            }
            if (MODE == 0) {
                float* po = g.out ? g.out + row0 * g.ldo + col : nullptr;
                __nv_bfloat16* pp = g.outp ? g.outp + row0 * g.ldp + col : nullptr;
                const int64_t ostep = 8 * g.ldo, pstep = 8 * g.ldp;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    if (i < nrow) {
                        const float4 y = make_float4(run[q][i].x * inv_h, run[q][i].y * inv_h, run[q][i].z * inv_h,
                                                     run[q][i].w * inv_h);
                        if (po) st4(po + i * ostep, y);
                        if (pp) st_planes4(pp + i * pstep, g.psp, y);
                    }
                }
            }
        }
    }
}

// Mode 2 epilogue of one 128 x BN tile for one warp (same thread layout as wide_epilogue_tile).  The accumulator is
// the head's dX g (one per tile); run = (sources... + g) / H is formed once, then every head streams its dact in and
// its dpre planes out (the tile is bound by that traffic).
__device__ __forceinline__ void wide_dpre_tile(const WideArgs& g, uint32_t stg, float* dbias_row, uint32_t taddr,
                                               int64_t m0, int n0, int ncols, int warp, int lane, uint32_t full_bar,
                                               uint32_t full_par) {
    const int quad = warp & 3, part = warp >> 2;
    const int r0 = lane >> 2, cq = lane & 3;
    const float inv_h = 1.f / (float)g.H;
    const int64_t row0 = m0 + quad * 32 + r0;
    const int nrow = (int)max((int64_t)0, min((int64_t)4, (g.M - row0 + 7) / 8));
    const uint32_t st_w = stg + lane * 64;
    const int sw_w = (lane >> 1) & 3;
    uint32_t st_r[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = r0 + 8 * i;
        st_r[i] = stg + r * 64 + ((cq ^ ((r >> 1) & 3)) << 4);
    }
    const int colq = n0 + cq * 4;
    const int64_t dstep = 8 * g.ldd, astep = 8 * g.ldda;
    for (int cg = 0; cg < ncols; cg += 128) {
        float4 run[2][4];
        // the fp32 sources first (their loads overlap the MMAs), in the order mode 1 sums them
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int c0 = cg + q * 64 + part * 16;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                run[q][i] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (g.n_g > 0 && i < nrow && c0 < ncols)
                    run[q][i] = ldg4(g.g[0] + (row0 + 8 * i) * g.ldg[0] + colq + c0);
            }
        }
        for (int s = 1; s < g.n_g; ++s) {
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int c0 = cg + q * 64 + part * 16;
                float4 t[4];
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    t[i] = (i < nrow && c0 < ncols) ? ldg4(g.g[s] + (row0 + 8 * i) * g.ldg[s] + colq + c0)
                                                    : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    run[q][i].x += t[i].x; run[q][i].y += t[i].y; run[q][i].z += t[i].z; run[q][i].w += t[i].w;
                }
            }
        }
        if (cg == 0) {
            mbar_wait(full_bar, full_par);
            tc_fence_after();
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int c0 = cg + q * 64 + part * 16;
            if (c0 >= ncols) break;
            uint32_t v[16];
            tmem_ld16(taddr + c0, v);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 4; ++j)
                st_shared4(st_w + ((j ^ sw_w) << 4), v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float4 x = ld_shared4(st_r[i]);
                float4& r = run[q][i];
                if (g.n_g > 0) { r.x += x.x; r.y += x.y; r.z += x.z; r.w += x.w; }
                else r = x;
                r.x *= inv_h; r.y *= inv_h; r.z *= inv_h; r.w *= inv_h;
            }
            __syncwarp();
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int c0 = cg + q * 64 + part * 16;
            if (c0 >= ncols) break;
            const int col = colq + c0;
            const float* pa = g.dact + row0 * g.ldda + col;
            __nv_bfloat16* dp = g.dpre + row0 * g.ldd + col;
            for (int h = 0; h < g.H; ++h) {
                float4 a[4];
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    a[i] = i < nrow ? ldg4(pa + i * astep + h * g.F) : make_float4(0.f, 0.f, 0.f, 0.f);
                float4 bs = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    if (i < nrow) {
                        float4 d;
                        d.x = run[q][i].x * a[i].x;
                        d.y = run[q][i].y * a[i].y;
                        d.z = run[q][i].z * a[i].z;
                        d.w = run[q][i].w * a[i].w;
                        st_planes4(dp + i * dstep + h * g.F, g.psd, d);
                        bs.x += d.x; bs.y += d.y; bs.z += d.z; bs.w += d.w;
                    }
                }
                if (dbias_row) {
#pragma unroll
                    for (int o = 4; o < 32; o <<= 1) {
                        bs.x += __shfl_xor_sync(kFull, bs.x, o); bs.y += __shfl_xor_sync(kFull, bs.y, o);
                        bs.z += __shfl_xor_sync(kFull, bs.z, o); bs.w += __shfl_xor_sync(kFull, bs.w, o);
                    }
                    if (lane < 4) {
                        float* p = dbias_row + h * g.F + col;
                        atomicAdd(p, bs.x); atomicAdd(p + 1, bs.y); atomicAdd(p + 2, bs.z); atomicAdd(p + 3, bs.w);
                    }
                }
            }
        }
    }
}

template <int MODE, bool DACT>
__global__ void __launch_bounds__(kWideThreads, 1) wide_kernel(const __grid_constant__ WideMaps maps, const WideArgs g) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int stages_bytes = g.stages * g.stage_bytes;
    NtShared* sh = reinterpret_cast<NtShared*>(smem + stages_bytes);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem_base = smem_u32(smem);

    if (threadIdx.x == 0) {
        for (int s = 0; s < g.stages; ++s) {
            mbar_init(smem_u32(&sh->full[s]), 1);
            mbar_init(smem_u32(&sh->empty[s]), 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(smem_u32(&sh->tmem_full[b]), 1);
            mbar_init(smem_u32(&sh->tmem_empty[b]), kWideEpiWarps * 32);
        }
        fence_barrier_init();
    }
    if (warp == kWideEpiWarps + 1 && lane == 0) {
        prefetch_tmap(&maps.a);
        prefetch_tmap(&maps.b);
    }
    if (warp == kWideEpiWarps) tmem_alloc(smem_u32(&sh->tmem_base), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = sh->tmem_base;

    const int64_t n_tiles = g.nt_m * g.nt_n;
    const int nkb = g.nparts * g.kbp;                // k-blocks per head
    const int accw = g.H * g.BN;                     // TMEM columns per accumulator buffer

    if (warp < kWideEpiWarps) {
        // ===================================================== epilogue
        int it = 0;
        const uint32_t stg = smem_base + stages_bytes + 256 + warp * (32 * 16 * 4);
        float* dbias_row = g.dbias_ws ? g.dbias_ws + (int64_t)blockIdx.x * (g.H * g.F) : nullptr;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
            const int buf = it & 1;
            const uint32_t par = (it >> 1) & 1;
            const int64_t m0 = (tile / g.nt_n) * BM;
            const int n0 = (int)(tile % g.nt_n) * g.BN;
            const int ncols = min(g.BN, g.F - n0);
            const uint32_t taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(buf * accw);
            const uint32_t fb = smem_u32(&sh->tmem_full[buf]);
            if (MODE == 2) {
                wide_dpre_tile(g, stg, dbias_row, taddr, m0, n0, ncols, warp, lane, fb, par);
            } else if (g.act == SPGNN_ACT_ELU) {
                wide_epilogue_tile<SPGNN_ACT_ELU, MODE, DACT>(g, stg, dbias_row, taddr, m0, n0, ncols, warp, lane, fb, par);
            } else if (g.act == SPGNN_ACT_NONE) {
                wide_epilogue_tile<SPGNN_ACT_NONE, MODE, DACT>(g, stg, dbias_row, taddr, m0, n0, ncols, warp, lane, fb, par);
            } else {
                wide_epilogue_tile<-1, MODE, DACT>(g, stg, dbias_row, taddr, m0, n0, ncols, warp, lane, fb, par);
            }
            tc_fence_before();
            mbar_arrive(smem_u32(&sh->tmem_empty[buf]));
        }
    } else if (warp == kWideEpiWarps) {
        // ===================================================== UMMA issuer (whole warp in the loop, one lane issues)
        {
            int it = 0;
            uint32_t kcount = 0;
            const uint32_t tbase = __shfl_sync(kFull, tmem_base, 0);
            for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
                const int buf = it & 1;
                const uint32_t par = (it >> 1) & 1;
                const int n0 = (int)(tile % g.nt_n) * g.BN;
                const int ncols = min(g.BN, g.F - n0);
                const uint32_t idesc = make_idesc(ncols, false);
                mbar_wait(smem_u32(&sh->tmem_empty[buf]), par ^ 1);
                tc_fence_after();
                for (int h = 0; h < g.hacc; ++h) {
                    const uint32_t tmem_d = tbase + (uint32_t)(buf * accw + h * g.BN);
                    for (int kb = 0; kb < nkb; ++kb, ++kcount) {
                        const int s = kcount % g.stages;
                        const uint32_t sp = (kcount / g.stages) & 1;
                        mbar_wait(smem_u32(&sh->full[s]), sp);
                        tc_fence_after();
                        const uint32_t a_hi = smem_base + s * g.stage_bytes;
                        const uint32_t a_lo = a_hi + BM * 128;
                        const uint32_t b_hi = a_hi + kABytes;
                        const uint32_t b_lo = b_hi + g.BN * 128;
                        if (elect_one()) {
#pragma unroll
                            for (int k = 0; k < BK / 16; ++k) {
                                const uint32_t ko = k * 32;
                                const uint64_t dah = make_desc(a_hi + ko, 16, 1024), dal = make_desc(a_lo + ko, 16, 1024);
                                const uint64_t dbh = make_desc(b_hi + ko, 16, 1024), dbl = make_desc(b_lo + ko, 16, 1024);
                                umma_bf16(tmem_d, dah, dbh, idesc, (kb | k) != 0);
                                umma_bf16(tmem_d, dah, dbl, idesc, 1);
                                umma_bf16(tmem_d, dal, dbh, idesc, 1);
                            }
                            umma_commit(smem_u32(&sh->empty[s]));
                        }
                        __syncwarp();
                    }
                }
                if (elect_one()) umma_commit(smem_u32(&sh->tmem_full[buf]));
                __syncwarp();
            }
        }
    } else if (lane == 0) {
        // ===================================================== TMA producer
        uint32_t kcount = 0;
        const uint32_t tx = (uint32_t)g.stage_bytes;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const int m0 = (int)((tile / g.nt_n) * BM);
            const int n0 = (int)(tile % g.nt_n) * g.BN;
            for (int h = 0; h < g.hacc; ++h) {
                for (int kb = 0; kb < nkb; ++kb, ++kcount) {
                    const int s = kcount % g.stages;
                    const uint32_t sp = (kcount / g.stages) & 1;
                    mbar_wait(smem_u32(&sh->empty[s]), sp ^ 1);
                    const uint32_t bar = smem_u32(&sh->full[s]);
                    mbar_expect_tx(bar, tx);
                    const uint32_t dst = smem_base + s * g.stage_bytes;
                    const int part = kb / g.kbp, j = kb - part * g.kbp;
                    const int acol = (part == 0 ? h : g.H) * g.kp + j * BK;
                    tma_load_3d(dst, &maps.a, bar, acol, m0, 0);
                    tma_load_3d(dst + kABytes, &maps.b, bar, kb * BK, h * g.F + n0, 0);
                }
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == kWideEpiWarps) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

__global__ void wide_dbias_reduce_kernel(const float* __restrict__ part, int64_t nparts, int64_t HF, float* __restrict__ out) {
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < HF; c += (int64_t)gridDim.x * blockDim.x) {
        float s = 0.f;
        for (int64_t p = 0; p < nparts; ++p) s += part[p * HF + c];
        out[c] = s;
    }
}

// ---------------------------------------------------------------------------------------------- TN kernel (dW)
constexpr int T_BK = 32;                       // nodes per stage
constexpr int T_BLK = 2 * T_BK * 128;          // one 64-column block, hi + lo planes: 8 KB
constexpr int T_STAGE = 8 * T_BLK;             // up to 4 P blocks + 4 Q blocks: 64 KB
constexpr int T_STAGES = 3;
constexpr int T_SMEM = T_STAGES * T_STAGE + 1024 + 256;

struct TnMaps { CUtensorMap p[2], q[2]; };
struct TnArgs {
    int p_cols[2], q_cols[2];                  // columns of each source (0 = absent)
    int p_off[2], q_off[2];                    // first output index of each source
    float* out; int64_t ldo; int64_t split_stride; int transposed;   // transposed: out[q * ldo + p], else out[p * ldo + q]
    int64_t M; int64_t rows_per_split;
    int npb, nqb;                              // 64-column blocks over the concatenated sources
    int np_tiles, nq_tiles;
    int flush_kb;                              // k-blocks (of T_BK node rows) accumulated in TMEM between two drains
    int chunks_per_split;                      // slabs of the workspace per row range (one per drain)
};
struct TnShared {
    uint64_t full[T_STAGES];
    uint64_t empty[T_STAGES];
    uint64_t tmem_full;
    uint64_t tmem_empty;
    uint32_t tmem_base;
};
struct Blk { int src, col0, valid; };
__device__ __forceinline__ Blk blk_of(const int (&cols)[2], int b) {
    const int nb0 = (cols[0] + 63) >> 6;
    Blk r;
    r.src = b >= nb0;
    r.col0 = (r.src ? b - nb0 : b) << 6;
    r.valid = min(64, cols[r.src] - r.col0);
    return r;
}
__device__ __forceinline__ void tile_range(int nb, int tiles, int t, int& first, int& count) {
    const int base = nb / tiles, rem = nb % tiles;
    first = t * base + min(t, rem);
    count = base + (t < rem ? 1 : 0);
}

__global__ void __launch_bounds__(kThreads, 1) tn_planes_kernel(const __grid_constant__ TnMaps maps, const TnArgs g) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    TnShared* sh = reinterpret_cast<TnShared*>(smem + T_STAGES * T_STAGE);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem_base = smem_u32(smem);

    if (threadIdx.x == 0) {
        for (int s = 0; s < T_STAGES; ++s) {
            mbar_init(smem_u32(&sh->full[s]), 1);
            mbar_init(smem_u32(&sh->empty[s]), 1);
        }
        mbar_init(smem_u32(&sh->tmem_full), 1);
        mbar_init(smem_u32(&sh->tmem_empty), kEpiWarps);
        fence_barrier_init();
    }
    if (warp == 5 && lane == 0) {
        prefetch_tmap(&maps.p[0]);
        prefetch_tmap(&maps.q[0]);
        if (g.p_cols[1] > 0) prefetch_tmap(&maps.p[1]);
        if (g.q_cols[1] > 0) prefetch_tmap(&maps.q[1]);
    }
    if (warp == kEpiWarps) tmem_alloc(smem_u32(&sh->tmem_base), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = sh->tmem_base;

    const int tp = blockIdx.x / g.nq_tiles, tq = blockIdx.x % g.nq_tiles;
    int pb0, npb, qb0, nqb;
    tile_range(g.npb, g.np_tiles, tp, pb0, npb);
    tile_range(g.nqb, g.nq_tiles, tq, qb0, nqb);
    const int64_t mbeg = (int64_t)blockIdx.y * g.rows_per_split;
    const int64_t mend = min(g.M, mbeg + g.rows_per_split);
    const int nkb = mend > mbeg ? (int)((mend - mbeg + T_BK - 1) / T_BK) : 0;
    const int nacc = npb > 2 ? 2 : 1;
    const Blk qlast = blk_of(g.q_cols, qb0 + nqb - 1);
    const int n_mma = 64 * (nqb - 1) + ((qlast.valid + 15) & ~15);
    // The tensor core adds into its fp32 accumulator with truncation, not round-to-nearest: a chain of n UMMAs drifts
    // by ~n * 2^-24 of the running sum, always towards zero (measured: dW of 1.23 M rows over 9 row ranges, 25 k UMMAs
    // per accumulator, 4.8e-4 of the largest entry; scripts/fullsize_precision.py).  The accumulators are therefore
    // drained every flush_kb k-blocks (8192 node rows = 1536 UMMAs) into a slab of the workspace of their own (plain
    // coalesced stores, nothing is read back: a read-modify-write of one slab measured +6 ms per step) and
    // reduce_splits adds the slabs up in fp32 with round-to-nearest, in a fixed order.
    const int nchunks = (nkb + g.flush_kb - 1) / g.flush_kb;

    if (warp < kEpiWarps) {
        // ===================================================== epilogue: TMEM -> partial sums in the workspace
      for (int chunk = 0; chunk < g.chunks_per_split; ++chunk) {
        float* obase = g.out + ((int64_t)blockIdx.y * g.chunks_per_split + chunk) * g.split_stride;
        const bool live = chunk < nchunks;          // a short last row range leaves its trailing slabs zero
        if (live) {
            mbar_wait(smem_u32(&sh->tmem_full), chunk & 1);
            tc_fence_after();
        }
        for (int acc = 0; acc < nacc; ++acc) {
            const int pbi = acc * 2 + (warp >> 1);                 // P block of this warp's 32 lanes
            if (pbi >= npb) continue;
            const Blk pb = blk_of(g.p_cols, pb0 + pbi);
            const int pin = (warp & 1) * 32 + lane;                // column within the block
            const bool pok = pin < pb.valid;
            const int64_t pidx = g.p_off[pb.src] + pb.col0 + pin;
            const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(acc * 256);
            // 64 accumulator columns per round: four TMEM loads in flight behind ONE wait (a wait per 16 columns made
            // a drain of the 512 columns ~12 us, during which the tensor pipe idles)
            for (int c64 = 0; c64 < n_mma; c64 += 64) {
                uint32_t v[4][16];
                if (live) {
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        if (c64 + u * 16 < n_mma) tmem_ld16(taddr + c64 + u * 16, v[u]);
                    tmem_ld_wait();
                }
                const Blk qb = blk_of(g.q_cols, qb0 + (c64 >> 6));
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int qin = u * 16;
                    const int nv = min(16, qb.valid - qin);
                    if (c64 + qin < n_mma && pok && nv > 0) {
                        const int64_t qidx = g.q_off[qb.src] + qb.col0 + qin;
                        if (g.transposed) {
                            float* o = obase + qidx * g.ldo + pidx;
#pragma unroll
                            for (int j = 0; j < 16; ++j)
                                if (j < nv) o[(int64_t)j * g.ldo] = live ? __uint_as_float(v[u][j]) : 0.f;
                        } else {
                            float* o = obase + pidx * g.ldo + qidx;
#pragma unroll
                            for (int j = 0; j < 16; ++j)
                                if (j < nv) o[j] = live ? __uint_as_float(v[u][j]) : 0.f;
                        }
                    }
                }
            }
        }
        if (chunk + 1 < nchunks) {              // accumulators drained: the UMMA warp may overwrite them
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&sh->tmem_empty));
        }
      }
    } else if (warp == kEpiWarps) {
        // UMMA issuer: the whole warp walks the loop, one elected lane issues (see nt_pair_kernel)
        {
            const uint32_t idesc = make_idesc(n_mma, true);
            const uint32_t tbase = __shfl_sync(kFull, tmem_base, 0);
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % T_STAGES;
                const uint32_t sp = (kb / T_STAGES) & 1;
                const int kin = kb % g.flush_kb;            // position inside the accumulation chunk
                if (kb > 0 && kin == 0) {
                    if (elect_one()) umma_commit(smem_u32(&sh->tmem_full));
                    __syncwarp();
                    mbar_wait(smem_u32(&sh->tmem_empty), ((kb / g.flush_kb) - 1) & 1);
                    tc_fence_after();
                }
                mbar_wait(smem_u32(&sh->full[s]), sp);
                tc_fence_after();
                const uint32_t p_base = smem_base + s * T_STAGE;
                const uint32_t q_base = p_base + 4 * T_BLK;
                if (elect_one()) {
#pragma unroll
                    for (int k = 0; k < T_BK / 16; ++k) {
                        const uint32_t ko = k * 16 * 128;            // 16 node rows of 128 B
                        // MN-major SW128: 64-column blocks T_BLK apart (LBO), 8-row groups 1 KB apart (SBO)
                        const uint64_t dbh = make_desc(q_base + ko, T_BLK, 1024);
                        const uint64_t dbl = make_desc(q_base + T_BLK / 2 + ko, T_BLK, 1024);
                        for (int acc = 0; acc < nacc; ++acc) {
                            const uint32_t ao = p_base + acc * 2 * T_BLK + ko;
                            const uint64_t dah = make_desc(ao, T_BLK, 1024), dal = make_desc(ao + T_BLK / 2, T_BLK, 1024);
                            const uint32_t td = tbase + (uint32_t)(acc * 256);
                            umma_bf16(td, dah, dbh, idesc, (kin | k) != 0);
                            umma_bf16(td, dah, dbl, idesc, 1);
                            umma_bf16(td, dal, dbh, idesc, 1);
                        }
                    }
                    umma_commit(smem_u32(&sh->empty[s]));
                }
                __syncwarp();
            }
            if (nkb > 0 && elect_one()) umma_commit(smem_u32(&sh->tmem_full));
            __syncwarp();
        }
    } else if (lane == 0) {
        const uint32_t tx = (uint32_t)(npb + nqb) * T_BLK;
        for (int kb = 0; kb < nkb; ++kb) {
            const int s = kb % T_STAGES;
            const uint32_t sp = (kb / T_STAGES) & 1;
            mbar_wait(smem_u32(&sh->empty[s]), sp ^ 1);
            const uint32_t bar = smem_u32(&sh->full[s]);
            mbar_expect_tx(bar, tx);
            const uint32_t dst = smem_base + s * T_STAGE;
            const int m = (int)(mbeg + (int64_t)kb * T_BK);
            for (int i = 0; i < npb; ++i) {
                const Blk b = blk_of(g.p_cols, pb0 + i);
                tma_load_3d(dst + i * T_BLK, &maps.p[b.src], bar, b.col0, m, 0);
            }
            for (int i = 0; i < nqb; ++i) {
                const Blk b = blk_of(g.q_cols, qb0 + i);
                tma_load_3d(dst + (4 + i) * T_BLK, &maps.q[b.src], bar, b.col0, m, 0);
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == kEpiWarps) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// ---------------------------------------------------------------------------------------------- plane producers

// out planes [M, ldo] <- dropout([x1 | x2]) (scaled by 1/(1-p)); one thread per 4-column chunk of the concatenation.
// Mask: 16 hash bits per element, chunk index = row * nchunks + chunk (the convention of every plane producer).
__global__ void split_planes_kernel(const float* __restrict__ x1, int64_t ld1, int K1, const float* __restrict__ x2,
                                    int64_t ld2, int K2, uint32_t thr, float scale, uint64_t seed,
                                    int64_t cat_chunks, int64_t chunk_off, __nv_bfloat16* __restrict__ hi, int64_t ldo,
                                    int64_t ps, int64_t M) {
    const int K = K1 + K2;
    const int nch = (K + 3) >> 2;
    const int64_t total = M * nch;
    const bool v1 = (ld1 % 4 == 0) && ((reinterpret_cast<uintptr_t>(x1) & 15) == 0);
    const bool v2 = x2 && (ld2 % 4 == 0) && ((reinterpret_cast<uintptr_t>(x2) & 15) == 0) && (K1 % 4 == 0);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / nch;
        const int c = (int)(i - r * nch) * 4;
        float v[4];
        if (c + 3 < K1 && v1) {
            const float4 t = ldg4(x1 + r * ld1 + c);
            v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
        } else if (c >= K1 && c + 3 < K && v2) {
            const float4 t = ldg4(x2 + r * ld2 + (c - K1));
            v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int cc = c + j;
                v[j] = cc < K1 ? __ldg(x1 + r * ld1 + cc) : (cc < K ? __ldg(x2 + r * ld2 + (cc - K1)) : 0.f);
            }
        }
        if (thr) {
            const uint64_t h = chunk_hash(seed, (uint64_t)r * (uint64_t)cat_chunks + (uint64_t)(chunk_off + (c >> 2)));
#pragma unroll
            for (int j = 0; j < 4; ++j) v[j] = ((uint32_t)(h >> (16 * j)) & 0xFFFFu) >= thr ? v[j] * scale : 0.f;
        }
        uint32_t h0, l0, h1, l1;
        split2(v[0], v[1], h0, l0);
        split2(v[2], v[3], h1, l1);
        __nv_bfloat16* o = hi + r * ldo + c;
        *reinterpret_cast<uint2*>(o) = make_uint2(h0, h1);
        *reinterpret_cast<uint2*>(o + ps) = make_uint2(l0, l1);
    }
}

// weight planes.  transpose = 0: out[r, c] = W[r, map(c)], map: c < K1pad -> c (valid if c < K1), else
// K1 + (c - K1pad) (valid if < K1 + K2).  transpose = 1: out[r, c] = W[c, k_off + r] (c < Nvalid).
__global__ void split_weight_kernel(const float* __restrict__ W, int64_t ldw, int transpose, int64_t k_off, int R,
                                    int Cpad, int K1, int K1pad, int K2, int Nvalid, __nv_bfloat16* __restrict__ hi,
                                    __nv_bfloat16* __restrict__ lo, int64_t ldo) {
    const int64_t total = (int64_t)R * Cpad;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / Cpad), c = (int)(i - (int64_t)r * Cpad);
        float v = 0.f;
        if (!transpose) {
            if (c < K1pad) { if (c < K1) v = W[(int64_t)r * ldw + c]; }
            else if (c - K1pad < K2) v = W[(int64_t)r * ldw + K1 + (c - K1pad)];
        } else if (c < Nvalid) {
            v = W[(int64_t)c * ldw + k_off + r];
        }
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        hi[(int64_t)r * ldo + c] = h;
        lo[(int64_t)r * ldo + c] = __float2bfloat16_rn(v - __bfloat162float(h));
    }
}

// ---------------------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// planes [rows, cols] (ld elements between rows, ps elements between the hi and lo plane) -> 3-D map {cols, rows, 2}
static int make_planes_map(CUtensorMap* m, const void* hi, int64_t rows, int64_t cols, int64_t ld, int64_t ps,
                           int box_cols, int box_rows) {
    EncodeTiledFn fn = encode_fn();
    SPGNN_REQUIRE(fn, "cuTensorMapEncodeTiled is not available from the driver");
    SPGNN_REQUIRE(((uintptr_t)hi & 15) == 0 && (ld * 2) % 16 == 0 && (ps * 2) % 16 == 0 && rows > 0 && cols > 0,
                  "planes operand: base must be 16-byte aligned, ld (%lld) and plane stride (%lld) multiples of 8",
                  (long long)ld, (long long)ps);
    cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, 2};
    cuuint64_t strides[2] = {(cuuint64_t)ld * 2, (cuuint64_t)ps * 2};
    cuuint32_t box[3] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows, 2};
    cuuint32_t es[3] = {1, 1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(hi), dims, strides, box, es,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    SPGNN_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d) rows=%lld cols=%lld ld=%lld ps=%lld", (int)r,
                  (long long)rows, (long long)cols, (long long)ld, (long long)ps);
    return SPGNN_OK;
}

static inline int round_up(int64_t x, int m) { return (int)((x + m - 1) / m * m); }

// tile width: as few n-tiles as possible, equal widths, multiple of 16
static void pick_bn(int N, int* BN, int* nt) {
    const int n16 = round_up(N, 16);
    *nt = (n16 + kMaxBN - 1) / kMaxBN;
    *BN = round_up((n16 + *nt - 1) / *nt, 16);
}

static unsigned split_grid(int64_t total) {
    const int64_t want = ceil_div(total, 256), cap = (int64_t)sm_count() * 16;
    return (unsigned)(want < cap ? want : cap);
}

// Co-resident 2-CTA clusters of nt_pair_kernel on the CURRENT device (0: cluster launches unavailable).  Cached per
// device ordinal: the dynamic-shared-memory opt-in and the occupancy are per-device properties.
static int nt_pair_clusters() {
    struct Cache { int v[64]; Cache() { for (int& x : v) x = -1; } };
    static Cache cache;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 0;
    if (cache.v[dev] >= 0) return cache.v[dev];
    int n = 0;
    if (cudaFuncSetAttribute(nt_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit) == cudaSuccess) {
        cudaLaunchConfig_t cfg{};
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.gridDim = dim3((unsigned)(sm_count() / 2 * 2)); cfg.blockDim = dim3(kThreads);
        cfg.dynamicSmemBytes = kSmemLimit; cfg.attrs = at; cfg.numAttrs = 1;
        if (cudaOccupancyMaxActiveClusters(&n, nt_pair_kernel, &cfg) != cudaSuccess) n = 0;
    }
    (void)cudaGetLastError();
    cache.v[dev] = n;
    return n;
}

// C = [A1|A2] * Bplanes^T with Bplanes [N, ldb] already split (hi at Bhi, lo at Bhi + N*ldb)
static int launch_nt(const __nv_bfloat16* A1, int64_t lda1, int64_t ps1, int64_t K1, const __nv_bfloat16* A2,
                     int64_t lda2, int64_t ps2, int64_t K2, const __nv_bfloat16* Bhi, int64_t ldb, const float* bias,
                     int act, float slope, float* C, int64_t ldc, int64_t M, int64_t N, cudaStream_t st,
                     float mask_p = 0.f, uint64_t mask_seed = 0, int64_t mask_chunks = 0, int64_t mask_chunk_off = 0) {
    static DeviceOnce attr;
    if (attr.pending()) {
        SPGNN_CUDA_OK(cudaFuncSetAttribute(nt_planes_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
        attr.done();
    }
    NtMaps maps;
    NtArgs a{};
    pick_bn((int)N, &a.BN, &a.nt_n);
    // CTA pairs (cta_group::2), measured on 1.23 M rows (profiles/r02_nt_pair_vs_single.txt): gat0 / gat1 forward
    // -6..-12 % / -19..-25 %, dX of gat1 / the output layer (K = 4100 -> 192 columns) -17..-21 % / -28 %; output-bound
    // shapes (small K: pgnn0-2, K = 192 -> 4100 columns) lose 10 - 30 % to the coupling of the two epilogues and stay
    // on the single-CTA kernel
    const int pair_clusters = nt_pair_clusters();
    const int64_t Kt = K1 + K2;
    const bool pair = pair_clusters > 0 && Kt >= 256 && (N >= 320 || Kt >= 512) && N >= 64 &&
                      ceil_div(M, BM) >= 4 * (int64_t)pair_clusters;
    int rc = make_planes_map(&maps.a1, A1, M, K1, lda1, ps1, BK, BM);
    if (rc) return rc;
    if (A2 && K2 > 0) {
        rc = make_planes_map(&maps.a2, A2, M, K2, lda2, ps2, BK, BM);
        if (rc) return rc;
    } else {
        maps.a2 = maps.a1;
    }
    // each CTA of a pair loads half of the weight tile
    rc = make_planes_map(&maps.b, Bhi, N, ldb, ldb, N * ldb, BK, pair ? a.BN / 2 : a.BN);
    if (rc) return rc;
    a.bias = bias; a.act = act; a.slope = slope; a.C = C; a.ldc = ldc; a.M = M; a.N = (int)N;
    a.mthr = mask_p > 0.f ? (uint32_t)(mask_p * 65536.f + 0.5f) : 0u;
    a.mscale = mask_p > 0.f ? 1.f / (1.f - mask_p) : 1.f;
    a.mseed = mask_seed; a.mnch = mask_chunks > 0 ? mask_chunks : (N + 3) / 4; a.moff = mask_chunk_off;
    a.nt_m = ceil_div(M, BM);
    a.kb1 = (int)ceil_div(K1, BK);
    a.kb2 = (A2 && K2 > 0) ? (int)ceil_div(K2, BK) : 0;
    a.stage_bytes = kABytes + a.BN * (pair ? 128 : 256);
    a.stages = (kSmemLimit - kNtFixed) / a.stage_bytes;
    if (a.stages > kMaxStages) a.stages = kMaxStages;
    if (pair) {
        const int64_t items = ceil_div(a.nt_m, 2) * a.nt_n;
        cudaLaunchConfig_t cfg{};
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.gridDim = dim3((unsigned)(2 * (items < pair_clusters ? items : pair_clusters)));
        cfg.blockDim = dim3(kThreads);
        cfg.dynamicSmemBytes = kSmemLimit; cfg.stream = st; cfg.attrs = at; cfg.numAttrs = 1;
        SPGNN_CUDA_OK(cudaLaunchKernelEx(&cfg, nt_pair_kernel, maps, a));
        count_launch();
        return SPGNN_OK;
    }
    const int64_t tiles = a.nt_m * a.nt_n;
    const unsigned grid = (unsigned)(tiles < sm_count() ? tiles : sm_count());
    nt_planes_kernel<<<grid, kThreads, kSmemLimit, st>>>(maps, a);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

}  // namespace tma
}  // namespace spgnn

using namespace spgnn;
using namespace spgnn::tma;

namespace spgnn {
__global__ void reduce_splits_kernel(const float* __restrict__ ws, int64_t splits, int64_t split_stride, int64_t N,
                                     int64_t K, float* __restrict__ out, int64_t ldo) {
    const int64_t total = N * K;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        // fixed order: eight interleaved running sums (independent loads in flight), combined pairwise at the end
        float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        int64_t z = 0;
        for (; z + 8 <= splits; z += 8) {
#pragma unroll
            for (int u = 0; u < 8; ++u) s[u] += __ldg(ws + (z + u) * split_stride + i);
        }
        for (int u = 0; z < splits; ++z, ++u) s[u] += __ldg(ws + z * split_stride + i);
        out[(i / K) * ldo + (i % K)] = ((s[0] + s[1]) + (s[2] + s[3])) + ((s[4] + s[5]) + (s[6] + s[7]));
    }
}

void reduce_splits(const float* ws, int64_t splits, int64_t N, int64_t K, float* out, int64_t ldo, cudaStream_t st) {
    const int64_t total = N * K;
    const int64_t want = ceil_div(total, 256), cap = (int64_t)sm_count() * 8;
    reduce_splits_kernel<<<(unsigned)(want < cap ? want : cap), 256, 0, st>>>(ws, splits, N * K, N, K, out, ldo);
    count_launch();
}
}  // namespace spgnn

extern "C" int spgnn_split_planes(const float* x1, int64_t ld1, int64_t K1, const float* x2, int64_t ld2, int64_t K2,
                                  float p, uint64_t seed, int64_t concat_chunks, int64_t chunk_off, uint16_t* out_hi,
                                  int64_t ldo, int64_t plane_stride, int64_t M, void* stream) {
    SPGNN_REQUIRE(x1 && out_hi && M > 0 && K1 > 0 && K2 >= 0 && (K2 == 0 || x2), "split_planes: bad argument");
    SPGNN_REQUIRE(ldo % 4 == 0 && ldo >= ((K1 + K2 + 3) / 4) * 4 && plane_stride % 4 == 0 && ((uintptr_t)out_hi & 7) == 0,
                  "split_planes: output ld (%lld) must be a multiple of 4 covering the padded row", (long long)ldo);
    SPGNN_REQUIRE(p >= 0.f && p < 1.f, "split_planes: dropout p");
    const uint32_t thr = p > 0.f ? (uint32_t)(p * 65536.f + 0.5f) : 0u;
    const float scale = p > 0.f ? 1.f / (1.f - p) : 1.f;
    const int64_t total = M * ((K1 + K2 + 3) / 4);
    if (concat_chunks <= 0) { concat_chunks = (K1 + K2 + 3) / 4; chunk_off = 0; }
    split_planes_kernel<<<split_grid(total), 256, 0, as_stream(stream)>>>(
        x1, ld1, (int)K1, K2 > 0 ? x2 : nullptr, ld2, (int)K2, thr, scale, seed, concat_chunks, chunk_off,
        reinterpret_cast<__nv_bfloat16*>(out_hi), ldo, plane_stride, M);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

extern "C" int64_t spgnn_planes_linear_fwd_ws(int64_t N, int64_t K1, int64_t K2) {
    const int64_t kp = round_up(K1, BK) + (K2 > 0 ? round_up(K2, BK) : 0);
    return 2 * N * kp * (int64_t)sizeof(__nv_bfloat16) + 256;
}

extern "C" int spgnn_planes_linear_fwd(const uint16_t* A1, int64_t lda1, int64_t ps1, int64_t K1, const uint16_t* A2,
                                       int64_t lda2, int64_t ps2, int64_t K2, const float* W, int64_t ldw,
                                       const float* bias, int act, float slope, float* C, int64_t ldc, int64_t M,
                                       int64_t N, void* ws, int64_t ws_bytes, void* stream) {
    SPGNN_REQUIRE(A1 && W && C && ws && M > 0 && N > 0 && K1 > 0 && K2 >= 0, "planes_linear_fwd: bad argument");
    if (!A2) K2 = 0;
    SPGNN_REQUIRE(ldw >= K1 + K2 && ldc >= N, "planes_linear_fwd: leading dimension smaller than row length");
    SPGNN_REQUIRE(ws_bytes >= spgnn_planes_linear_fwd_ws(N, K1, K2), "planes_linear_fwd: workspace too small");
    SPGNN_REQUIRE(M < (1ll << 31) && N < (1 << 24), "planes_linear_fwd: shape too large");
    cudaStream_t st = as_stream(stream);
    const int k1p = round_up(K1, BK), k2p = K2 > 0 ? round_up(K2, BK) : 0;
    const int64_t ldb = k1p + k2p;
    __nv_bfloat16* hi = reinterpret_cast<__nv_bfloat16*>(((uintptr_t)ws + 127) & ~(uintptr_t)127);
    split_weight_kernel<<<split_grid(N * ldb), 256, 0, st>>>(W, ldw, 0, 0, (int)N, (int)ldb, (int)K1, k1p, (int)K2, 0,
                                                             hi, hi + N * ldb, ldb);
    SPGNN_LAUNCH_OK();
    return launch_nt(reinterpret_cast<const __nv_bfloat16*>(A1), lda1, ps1, K1,
                     reinterpret_cast<const __nv_bfloat16*>(A2), lda2, ps2, K2, hi, ldb, bias, act, slope, C, ldc, M, N,
                     st);
}

extern "C" int64_t spgnn_wide_linear_ws(int64_t H, int64_t F, int64_t kp, int has_res) {
    const int64_t b = 2 * H * F * (has_res ? 2 : 1) * kp * (int64_t)sizeof(__nv_bfloat16);
    return b + 256 + (int64_t)sm_count() * H * F * (int64_t)sizeof(float) + 256;
}

namespace {
// Tiling of the wide GEMM: 128 x BN tiles, BN = 256 / H columns per head (H accumulators fill the 512 TMEM columns
// of two buffers), as many pipeline stages as fit.
int wide_tiling(WideArgs& a) {
    a.BN = 256 / a.H;
    if (a.BN > a.F) a.BN = a.F;
    a.nt_n = (int)ceil_div(a.F, a.BN);
    a.nt_m = ceil_div(a.M, BM);
    a.stage_bytes = kABytes + a.BN * 256;
    a.stages = (kSmemLimit - kWideFixed) / a.stage_bytes;
    if (a.stages > kMaxStages) a.stages = kMaxStages;
    SPGNN_REQUIRE(a.stages >= 2, "wide_linear: not enough shared memory for two pipeline stages");
    return SPGNN_OK;
}

// Launches the kernel of a.mode with maps and tiling set up; dbias (modes 1 and 2, optional) goes through per-CTA
// partial rows at part_ws, reduced in fixed order.
int wide_launch(const WideMaps& maps, WideArgs& a, float* dbias, void* part_ws, cudaStream_t st) {
    static DeviceOnce attr;
    if (attr.pending()) {
        SPGNN_CUDA_OK(cudaFuncSetAttribute(wide_kernel<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
        SPGNN_CUDA_OK(cudaFuncSetAttribute(wide_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
        SPGNN_CUDA_OK(cudaFuncSetAttribute(wide_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
        SPGNN_CUDA_OK(cudaFuncSetAttribute(wide_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
        attr.done();
    }
    const int64_t HF = (int64_t)a.H * a.F;
    const int64_t tiles = a.nt_m * a.nt_n;
    const unsigned grid = (unsigned)(tiles < sm_count() ? tiles : sm_count());
    float* part = nullptr;
    if (a.mode != 0 && dbias) {
        part = reinterpret_cast<float*>(((uintptr_t)part_ws + 255) & ~(uintptr_t)255);
        a.dbias_ws = part;
        SPGNN_CUDA_OK(cudaMemsetAsync(part, 0, (size_t)grid * HF * sizeof(float), st));
    }
    if (a.mode == 0 && a.dact) wide_kernel<0, true><<<grid, kWideThreads, kSmemLimit, st>>>(maps, a);
    else if (a.mode == 0) wide_kernel<0, false><<<grid, kWideThreads, kSmemLimit, st>>>(maps, a);
    else if (a.mode == 1) wide_kernel<1, false><<<grid, kWideThreads, kSmemLimit, st>>>(maps, a);
    else wide_kernel<2, false><<<grid, kWideThreads, kSmemLimit, st>>>(maps, a);
    SPGNN_LAUNCH_OK();
    if (part) {
        wide_dbias_reduce_kernel<<<(unsigned)ceil_div(HF, 128), 128, 0, st>>>(part, grid, HF, dbias);
        SPGNN_LAUNCH_OK();
    }
    return SPGNN_OK;
}

int wide_linear(const uint16_t* XA, int64_t ldxa, int64_t psxa, int64_t kp, int64_t k_in, int64_t M, int H, int F,
                int has_res, const float* W, int64_t ldw, const float* bias, int act, int mode, float* out, int64_t ldo,
                uint16_t* out_planes, int64_t ldp, int64_t psp, float* dact, int64_t ldda, const float* g0,
                int64_t ldg0, const float* g1, int64_t ldg1, const float* g2, int64_t ldg2, uint16_t* dpre,
                int64_t ldd, int64_t psd, float* dbias, void* ws, int64_t ws_bytes, void* stream) {
    SPGNN_REQUIRE(XA && W && ws && M > 0 && k_in > 0, "wide_linear: bad argument");
    SPGNN_REQUIRE(H == 1 || H == 2 || H == 4, "wide_linear: H must be 1, 2 or 4 (got %d)", H);
    SPGNN_REQUIRE(F > 0 && F % 32 == 0 && (int64_t)H * F <= 8192, "wide_linear: F (%d) must be a multiple of 32, H*F <= 8192", F);
    SPGNN_REQUIRE(kp % BK == 0 && kp >= k_in && ldxa >= (H + 1) * kp && ldw >= k_in, "wide_linear: kp / ld mismatch");
    SPGNN_REQUIRE(mode == 0 || mode == 1, "wide_linear: mode must be 0 (forward) or 1 (gradient of the pre-activations)");
    SPGNN_REQUIRE(!bias || ((uintptr_t)bias & 15) == 0, "wide_linear: bias must be 16-byte aligned");
    SPGNN_REQUIRE(ws_bytes >= spgnn_wide_linear_ws(H, F, kp, has_res), "wide_linear: workspace too small");
    SPGNN_REQUIRE(M < (1ll << 31), "wide_linear: too many rows");
    WideMaps maps;
    WideArgs a{};
    a.mode = mode; a.H = H; a.F = F; a.act = act; a.bias = bias; a.M = M; a.hacc = H;
    if (mode == 0) {
        SPGNN_REQUIRE(out || out_planes, "wide_linear: no output");
        SPGNN_REQUIRE(!out || (ldo % 4 == 0 && ldo >= F && ((uintptr_t)out & 15) == 0), "wide_linear: out alignment");
        SPGNN_REQUIRE(!out_planes || (ldp % 4 == 0 && ldp >= F && psp % 4 == 0 && ((uintptr_t)out_planes & 7) == 0),
                      "wide_linear: out planes alignment");
        SPGNN_REQUIRE(!dact || (ldda % 4 == 0 && ldda >= (int64_t)H * F && ((uintptr_t)dact & 15) == 0),
                      "wide_linear: dact must be 16-byte aligned with ld %% 4 == 0 and ld >= H*F");
        a.out = out; a.ldo = ldo; a.outp = reinterpret_cast<__nv_bfloat16*>(out_planes); a.ldp = ldp; a.psp = psp;
        a.dact = dact; a.ldda = ldda;
    } else {
        SPGNN_REQUIRE(g0 && dpre, "wide_linear: mode 1 needs a gradient source and the dpre planes");
        SPGNN_REQUIRE(ldd % 4 == 0 && ldd >= (int64_t)H * F && psd % 4 == 0 && ((uintptr_t)dpre & 7) == 0,
                      "wide_linear: dpre planes alignment");
        const float* gs[3] = {g0, g1, g2};
        const int64_t lds[3] = {ldg0, ldg1, ldg2};
        for (int s = 0; s < 3; ++s) {
            if (!gs[s]) continue;
            SPGNN_REQUIRE(lds[s] % 4 == 0 && lds[s] >= F && ((uintptr_t)gs[s] & 15) == 0,
                          "wide_linear: gradient source %d must be 16-byte aligned with ld %% 4 == 0", s);
            a.g[a.n_g] = gs[s]; a.ldg[a.n_g] = lds[s]; ++a.n_g;
        }
        a.dpre = reinterpret_cast<__nv_bfloat16*>(dpre); a.ldd = ldd; a.psd = psd;
    }
    cudaStream_t st = as_stream(stream);
    const int nparts = has_res ? 2 : 1;
    const int64_t HF = (int64_t)H * F, ldb = nparts * kp;
    __nv_bfloat16* hi = reinterpret_cast<__nv_bfloat16*>(((uintptr_t)ws + 127) & ~(uintptr_t)127);
    for (int p = 0; p < nparts; ++p) {
        split_weight_kernel<<<split_grid(HF * kp), 256, 0, st>>>(W + (int64_t)p * HF * ldw, ldw, 0, 0, (int)HF, (int)kp,
                                                                 (int)k_in, (int)kp, 0, 0, hi + p * kp,
                                                                 hi + HF * ldb + p * kp, ldb);
        SPGNN_LAUNCH_OK();
    }
    int rc = wide_tiling(a);
    if (rc) return rc;
    a.kbp = (int)(kp / BK); a.nparts = nparts; a.kp = (int)kp;
    rc = make_planes_map(&maps.a, XA, M, (int64_t)(H + 1) * kp, ldxa, psxa, BK, BM);
    if (rc) return rc;
    rc = make_planes_map(&maps.b, hi, HF, ldb, ldb, HF * ldb, BK, a.BN);
    if (rc) return rc;
    // A CTA-pair variant was slower at the bench size and was removed (profiles/r02_wide_pair_probe.txt).
    return wide_launch(maps, a, dbias, hi + 2 * HF * ldb, st);
}
}  // namespace

extern "C" int spgnn_wide_linear(const uint16_t* XA, int64_t ldxa, int64_t psxa, int64_t kp, int64_t k_in, int64_t M,
                                 int H, int F, int has_res, const float* W, int64_t ldw, const float* bias, int act,
                                 int mode, float* out, int64_t ldo, uint16_t* out_planes, int64_t ldp, int64_t psp,
                                 const float* g0, int64_t ldg0, const float* g1, int64_t ldg1, const float* g2,
                                 int64_t ldg2, uint16_t* dpre, int64_t ldd, int64_t psd, float* dbias, void* ws,
                                 int64_t ws_bytes, void* stream) {
    return wide_linear(XA, ldxa, psxa, kp, k_in, M, H, F, has_res, W, ldw, bias, act, mode, out, ldo, out_planes, ldp,
                       psp, nullptr, 0, g0, ldg0, g1, ldg1, g2, ldg2, dpre, ldd, psd, dbias, ws, ws_bytes, stream);
}

extern "C" int spgnn_wide_linear_fwd_dact(const uint16_t* XA, int64_t ldxa, int64_t psxa, int64_t kp, int64_t k_in,
                                          int64_t M, int H, int F, int has_res, const float* W, int64_t ldw,
                                          const float* bias, int act, float* out, int64_t ldo, uint16_t* out_planes,
                                          int64_t ldp, int64_t psp, float* dact, int64_t ldda, void* ws,
                                          int64_t ws_bytes, void* stream) {
    SPGNN_REQUIRE(dact, "wide_linear_fwd_dact: no dact output");
    return wide_linear(XA, ldxa, psxa, kp, k_in, M, H, F, has_res, W, ldw, bias, act, 0, out, ldo, out_planes, ldp,
                       psp, dact, ldda, nullptr, 0, nullptr, 0, nullptr, 0, nullptr, 0, 0, nullptr, ws, ws_bytes,
                       stream);
}

extern "C" int64_t spgnn_wide_dpre_ws(int64_t H, int64_t F) {
    const int64_t b = 2 * F * BK * (int64_t)sizeof(__nv_bfloat16);
    return b + 256 + (int64_t)sm_count() * H * F * (int64_t)sizeof(float) + 256;
}

extern "C" int spgnn_wide_dpre(const uint16_t* GL, int64_t ldgl, int64_t psgl, int64_t C, int64_t M, int H, int F,
                               const float* Wh, int64_t ldwh, const float* dact, int64_t ldda, const float* g0,
                               int64_t ldg0, const float* g1, int64_t ldg1, uint16_t* dpre, int64_t ldd, int64_t psd,
                               float* dbias, void* ws, int64_t ws_bytes, void* stream) {
    SPGNN_REQUIRE(GL && Wh && dact && dpre && ws && M > 0, "wide_dpre: bad argument");
    SPGNN_REQUIRE(C > 0 && C <= BK && ldgl >= C && ldwh >= F, "wide_dpre: the head has 1..64 outputs (got %lld)",
                  (long long)C);
    SPGNN_REQUIRE(H == 1 || H == 2 || H == 4, "wide_dpre: H must be 1, 2 or 4 (got %d)", H);
    SPGNN_REQUIRE(F > 0 && F % 32 == 0 && (int64_t)H * F <= 8192, "wide_dpre: F (%d) must be a multiple of 32, H*F <= 8192", F);
    SPGNN_REQUIRE(ldda % 4 == 0 && ldda >= (int64_t)H * F && ((uintptr_t)dact & 15) == 0,
                  "wide_dpre: dact must be 16-byte aligned with ld %% 4 == 0 and ld >= H*F");
    SPGNN_REQUIRE(ldd % 4 == 0 && ldd >= (int64_t)H * F && psd % 4 == 0 && ((uintptr_t)dpre & 7) == 0,
                  "wide_dpre: dpre planes alignment");
    SPGNN_REQUIRE(ws_bytes >= spgnn_wide_dpre_ws(H, F), "wide_dpre: workspace too small");
    SPGNN_REQUIRE(M < (1ll << 31), "wide_dpre: too many rows");
    WideMaps maps;
    WideArgs a{};
    a.mode = 2; a.H = H; a.F = F; a.act = SPGNN_ACT_NONE; a.M = M; a.hacc = 1;
    a.dact = const_cast<float*>(dact); a.ldda = ldda;
    const float* gs[2] = {g0, g1};
    const int64_t lds[2] = {ldg0, ldg1};
    for (int s = 0; s < 2; ++s) {
        if (!gs[s]) continue;
        SPGNN_REQUIRE(lds[s] % 4 == 0 && lds[s] >= F && ((uintptr_t)gs[s] & 15) == 0,
                      "wide_dpre: gradient source %d must be 16-byte aligned with ld %% 4 == 0", s);
        a.g[a.n_g] = gs[s]; a.ldg[a.n_g] = lds[s]; ++a.n_g;
    }
    a.dpre = reinterpret_cast<__nv_bfloat16*>(dpre); a.ldd = ldd; a.psd = psd;
    cudaStream_t st = as_stream(stream);
    // B = W_head^T [F, C] split into planes with K padded to one 64-wide block, as spgnn_planes_linear_bwd_input does
    __nv_bfloat16* hi = reinterpret_cast<__nv_bfloat16*>(((uintptr_t)ws + 127) & ~(uintptr_t)127);
    split_weight_kernel<<<split_grid(F * BK), 256, 0, st>>>(Wh, ldwh, 1, 0, F, BK, 0, 0, 0, (int)C, hi, hi + F * BK, BK);
    SPGNN_LAUNCH_OK();
    int rc = wide_tiling(a);
    if (rc) return rc;
    a.kbp = 1; a.nparts = 1; a.kp = BK;
    rc = make_planes_map(&maps.a, GL, M, C, ldgl, psgl, BK, BM);
    if (rc) return rc;
    rc = make_planes_map(&maps.b, hi, F, BK, BK, F * BK, BK, a.BN);
    if (rc) return rc;
    return wide_launch(maps, a, dbias, hi + 2 * F * BK, st);
}

extern "C" int64_t spgnn_planes_linear_bwd_input_ws(int64_t N, int64_t K) {
    return 2 * K * (int64_t)round_up(N, BK) * 2 + 256;
}

// dA[M, K] = dC[M, N] * W[N, k_off : k_off + K]:  NT GEMM with B = (W^T)[K, N] pre-split
extern "C" int spgnn_planes_linear_bwd_input(const uint16_t* dC, int64_t lddc, int64_t ps, const float* W, int64_t ldw,
                                             int64_t k_off, float* dA, int64_t ldda, int64_t M, int64_t N, int64_t K,
                                             void* ws, int64_t ws_bytes, void* stream) {
    return spgnn_planes_linear_bwd_input_masked(dC, lddc, ps, W, ldw, k_off, dA, ldda, M, N, K, 0.f, 0, 0, ws, ws_bytes,
                                                stream);
}

// ... followed by the feat_drop mask of the layer whose (dropped) input dA is the gradient of: dA *= mask / (1 - p),
// mask chunk index = row * concat_chunks + (k_off + col) / 4 (dA column c is input column k_off + c)
extern "C" int spgnn_planes_linear_bwd_input_masked(const uint16_t* dC, int64_t lddc, int64_t ps, const float* W,
                                                    int64_t ldw, int64_t k_off, float* dA, int64_t ldda, int64_t M,
                                                    int64_t N, int64_t K, float drop_p, uint64_t seed,
                                                    int64_t concat_chunks, void* ws, int64_t ws_bytes, void* stream) {
    SPGNN_REQUIRE(dC && W && dA && ws && M > 0 && N > 0 && K > 0, "planes_linear_bwd_input: bad argument");
    SPGNN_REQUIRE(drop_p >= 0.f && drop_p < 1.f, "planes_linear_bwd_input: dropout p");
    SPGNN_REQUIRE(drop_p == 0.f || k_off % 4 == 0, "planes_linear_bwd_input: a masked output needs k_off %% 4 == 0");
    SPGNN_REQUIRE(ldw >= k_off + K && ldda >= K, "planes_linear_bwd_input: leading dimension too small");
    SPGNN_REQUIRE(ws_bytes >= spgnn_planes_linear_bwd_input_ws(N, K), "planes_linear_bwd_input: workspace too small");
    cudaStream_t st = as_stream(stream);
    const int np = round_up(N, BK);
    __nv_bfloat16* hi = reinterpret_cast<__nv_bfloat16*>(((uintptr_t)ws + 127) & ~(uintptr_t)127);
    split_weight_kernel<<<split_grid(K * np), 256, 0, st>>>(W, ldw, 1, k_off, (int)K, np, 0, 0, 0, (int)N, hi,
                                                            hi + K * np, np);
    SPGNN_LAUNCH_OK();
    return launch_nt(reinterpret_cast<const __nv_bfloat16*>(dC), lddc, ps, N, nullptr, 0, 0, 0, hi, np, nullptr, 0, 0.f,
                     dA, ldda, M, K, st, drop_p, seed, concat_chunks > 0 ? concat_chunks : (k_off + K + 3) / 4, k_off / 4);
}

namespace {
struct TnPlan {
    bool swap;                 // false: P = X (k), Q = dC (n) -> out[q][p];  true: P = dC, Q = X -> out[p][q]
    int npb, nqb, np_tiles, nq_tiles;
    int64_t splits, rows;
    double cost;               // modelled cycles of the launch (tile cost x stages per row range); < 0: not modelled
};
// 64-column blocks of up to two concatenated sources, with the valid columns of each block
int blocks_of(int64_t c0, int64_t c1, int* valid) {
    int n = 0;
    for (int64_t c : {c0, c1})
        for (int64_t o = 0; o < c; o += 64) valid[n++] = (int)(c - o < 64 ? c - o : 64);
    return n;
}
// Cycles one CTA spends per 32-node stage on a tile of pc P blocks x qc Q blocks: the tensor pipe needs
// 2 k-steps x 3 passes x nacc x n_mma / 2 cycles (tcgen05 floor: M = 128 costs N/2 cycles per k16, a half-filled second
// accumulator costs as much as a full one), the TMA fill needs (pc + qc) x 8 KB at the ~42.6 B/clk/SM share of the L2
// throughput cap (~6300 B/clk chip-wide).  Against profiles/r01_ncu_full_step_79ms_table.txt this reproduces the
// measured launches within a few percent (gat0 dW 7.7 ms, output-layer dW 2.1 ms with P = X vs 1.9 ms with P = dC).
double tn_tile_cost(const int* qvalid, int pc, int q0, int qc) {
    const int nacc = pc > 2 ? 2 : 1;
    const int n_mma = 64 * (qc - 1) + ((qvalid[q0 + qc - 1] + 15) & ~15);
    const double mma = 3.0 * nacc * n_mma, load = (pc + qc) * 8192.0 / 42.6;
    return (mma > load ? mma : load) + 60.0;
}
void tn_range(int nb, int tiles, int t, int& first, int& count) {
    const int base = nb / tiles, rem = nb % tiles;
    first = t * base + (t < rem ? t : rem);
    count = base + (t < rem ? 1 : 0);
}
// Orientation by the cost model (which operand is the M side: an accumulator takes 128 of its columns whether they
// are valid or not, the N side has a granularity of 16), tiles of up to 4 x 4 blocks, row ranges UNIFORM over the
// tile pairs: CTAs that share P or Q blocks then walk the same rows at the same time and meet in L2.  Measured
// (profiles/r01_gemm_check_cluster_vs_plain.txt): the orientation flip takes the output layer's dW from 5.5 to 4.4 ms;
// finer tilings that the model rates ~6 % better (6 x 6 x 4 for gat0) measure the same or worse, so they are not used.
TnPlan tn_plan(int64_t M, int64_t N, int64_t K1, int64_t K2) {
    int xv[1024], yv[1024];
    const bool small = K1 + K2 <= 64 * 500 && N <= 64 * 1000;
    const int xb = small ? blocks_of(K1, K2, xv) : (int)(ceil_div(K1, 64) + ceil_div(K2, 64));
    const int yb = small ? blocks_of(N, 0, yv) : (int)ceil_div(N, 64);
    const int sms = sm_count();
    const int64_t max_by_rows = ceil_div(M, 512);
    TnPlan best{};
    double best_t = -1.0;
    for (int sw = 0; small && sw < 2; ++sw) {
        const int npb = sw ? yb : xb, nqb = sw ? xb : yb;
        const int* qv = sw ? xv : yv;
        const int npt = (int)ceil_div(npb, 4), nqt = (int)ceil_div(nqb, 4);
        const int tiles = npt * nqt;
        if (tiles > sms) continue;
        double cmax = 0.0;
        for (int tp = 0; tp < npt; ++tp)
            for (int tq = 0; tq < nqt; ++tq) {
                int p0, pc, q0, qc;
                tn_range(npb, npt, tp, p0, pc);
                tn_range(nqb, nqt, tq, q0, qc);
                const double c = tn_tile_cost(qv, pc, q0, qc);
                cmax = c > cmax ? c : cmax;
            }
        int64_t want = sms / tiles;
        if (want > max_by_rows) want = max_by_rows;
        if (want < 1) want = 1;
        const int64_t rows = ceil_div(ceil_div(M, want), T_BK) * T_BK;
        const int64_t splits = ceil_div(M, rows);
        const double t = cmax * (double)(rows / T_BK);
        if (best_t < 0.0 || t < 0.97 * best_t) {          // P = X unless the flip is clearly better
            best_t = t;
            best.swap = sw != 0; best.npb = npb; best.nqb = nqb; best.np_tiles = npt; best.nq_tiles = nqt;
            best.splits = splits; best.rows = rows; best.cost = t;
        }
    }
    if (best_t >= 0.0) return best;
    // more tile pairs than SMs: one row range, CTAs queue on the hardware scheduler
    TnPlan t{};
    t.swap = false;
    t.npb = xb; t.nqb = yb;
    t.np_tiles = (int)ceil_div(t.npb, 4);
    t.nq_tiles = (int)ceil_div(t.nqb, 4);
    t.rows = ceil_div(M, T_BK) * T_BK;
    t.splits = 1;
    t.cost = -1.0;
    return t;
}
// Two concatenated sources whose block counts do not tile well TOGETHER are better served by two launches: gat0's
// X = [fvs 1024 | pos_enc 39] is 16 + 1 blocks, and 17 x 17 blocks make 25 tiles x 5 row ranges = 125 of 148 SMs with a
// half-empty accumulator on every 3-block tile, while 16 x 17 blocks make 20 tiles x 7 row ranges = 140 SMs of full
// tiles (model: 6.5 -> 4.6 + 0.7 ms).  Taken when the model rates the pair of launches at least 8 % cheaper.
bool tn_split_sources(int64_t M, int64_t N, int64_t K1, int64_t K2) {
    if (K2 <= 0) return false;
    static int enabled = -1;
    if (enabled < 0) {
        const char* e = getenv("SPGNN_TN_SPLIT_SOURCES");
        enabled = (e && atoi(e) == 0) ? 0 : 1;
    }
    if (!enabled) return false;
    const TnPlan both = tn_plan(M, N, K1, K2), a = tn_plan(M, N, K1, 0), b = tn_plan(M, N, K2, 0);
    if (both.cost < 0.0 || a.cost < 0.0 || b.cost < 0.0) return false;
    return a.cost + b.cost < 0.92 * both.cost;
}
}  // namespace

// node rows accumulated in TMEM between two drains of the accumulators (see tn_planes_kernel); SPGNN_TN_FLUSH_ROWS
// overrides it for experiments (0 = never drain: the round-1 behaviour)
static int tn_flush_kb() {
    static int cached = -1;
    if (cached < 0) {
        const char* e = getenv("SPGNN_TN_FLUSH_ROWS");
        long rows = e ? atol(e) : 8192;
        cached = rows <= 0 ? (1 << 30) : (int)((rows + T_BK - 1) / T_BK);
    }
    return cached;
}

static int64_t tn_chunks_per_split(const TnPlan& t) {
    const int64_t c = ceil_div(ceil_div(t.rows, T_BK), tn_flush_kb());
    return c < 1 ? 1 : c;
}

static int64_t tn_ws_one(int64_t M, int64_t N, int64_t K1, int64_t K2) {
    const TnPlan t = tn_plan(M, N, K1, K2);
    return t.splits * tn_chunks_per_split(t) * N * (K1 + K2) * (int64_t)sizeof(float) + 256;
}
extern "C" int64_t spgnn_planes_linear_bwd_weight_ws(int64_t M, int64_t N, int64_t K1, int64_t K2) {
    if (tn_split_sources(M, N, K1, K2)) {
        const int64_t a = tn_ws_one(M, N, K1, 0), b = tn_ws_one(M, N, K2, 0);
        return a > b ? a : b;
    }
    return tn_ws_one(M, N, K1, K2);
}

extern "C" int64_t spgnn_planes_linear_bwd_weight_plan(int64_t M, int64_t N, int64_t K1, int64_t K2, int32_t* out,
                                                       int64_t cap) {
    if (!out || cap < 8 || M <= 0 || N <= 0 || K1 <= 0 || K2 < 0) return 0;
    const bool split = tn_split_sources(M, N, K1, K2);      // then: the plan of the FIRST launch (X1 alone)
    const TnPlan t = tn_plan(M, N, K1, split ? 0 : K2);
    if (cap >= 9) out[8] = split ? 1 : 0;
    const int tiles = t.np_tiles * t.nq_tiles;
    const int64_t work = (int64_t)tiles * t.splits;
    const int32_t head[8] = {t.swap, t.np_tiles, t.nq_tiles, (int32_t)t.splits, (int32_t)work, (int32_t)t.rows, t.npb, t.nqb};
    int64_t n = 0;
    for (; n < 8 && n < cap; ++n) out[n] = head[n];
    return cap >= 9 ? 9 : n;
}

// dW[N, K1+K2] (lddw) = dC[M, N]^T * [X1 | X2][M, K1+K2], every operand in planes form
static int tn_launch(const uint16_t* dC, int64_t lddc, int64_t psc, const uint16_t* X1, int64_t ldx1, int64_t psx1,
                     int64_t K1, const uint16_t* X2, int64_t ldx2, int64_t psx2, int64_t K2, float* dW, int64_t lddw,
                     int64_t M, int64_t N, void* ws, void* stream);

extern "C" int spgnn_planes_linear_bwd_weight(const uint16_t* dC, int64_t lddc, int64_t psc, const uint16_t* X1,
                                              int64_t ldx1, int64_t psx1, int64_t K1, const uint16_t* X2, int64_t ldx2,
                                              int64_t psx2, int64_t K2, float* dW, int64_t lddw, int64_t M, int64_t N,
                                              void* ws, int64_t ws_bytes, void* stream) {
    SPGNN_REQUIRE(dC && X1 && dW && ws && M > 0 && N > 0 && K1 > 0 && K2 >= 0, "planes_linear_bwd_weight: bad argument");
    if (!X2) K2 = 0;
    SPGNN_REQUIRE(lddw >= K1 + K2, "planes_linear_bwd_weight: leading dimension too small");
    SPGNN_REQUIRE(ws_bytes >= spgnn_planes_linear_bwd_weight_ws(M, N, K1, K2), "planes_linear_bwd_weight: workspace too small");
    SPGNN_REQUIRE(M < (1ll << 31), "planes_linear_bwd_weight: too many rows");
    if (tn_split_sources(M, N, K1, K2)) {        // one launch per source (stream-ordered, the workspace is reused)
        int rc = tn_launch(dC, lddc, psc, X1, ldx1, psx1, K1, nullptr, 0, 0, 0, dW, lddw, M, N, ws, stream);
        if (rc) return rc;
        return tn_launch(dC, lddc, psc, X2, ldx2, psx2, K2, nullptr, 0, 0, 0, dW + K1, lddw, M, N, ws, stream);
    }
    return tn_launch(dC, lddc, psc, X1, ldx1, psx1, K1, X2, ldx2, psx2, K2, dW, lddw, M, N, ws, stream);
}

static int tn_launch(const uint16_t* dC, int64_t lddc, int64_t psc, const uint16_t* X1, int64_t ldx1, int64_t psx1,
                     int64_t K1, const uint16_t* X2, int64_t ldx2, int64_t psx2, int64_t K2, float* dW, int64_t lddw,
                     int64_t M, int64_t N, void* ws, void* stream) {
    static DeviceOnce attr;
    if (attr.pending()) {
        SPGNN_CUDA_OK(cudaFuncSetAttribute(tn_planes_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, T_SMEM));
        attr.done();
    }
    cudaStream_t st = as_stream(stream);
    const TnPlan t = tn_plan(M, N, K1, K2);
    const int64_t Kt = K1 + K2;
    TnMaps maps;
    TnArgs a{};
    CUtensorMap mx1, mx2, my;
    int rc = make_planes_map(&mx1, X1, M, K1, ldx1, psx1, 64, T_BK);
    if (rc) return rc;
    mx2 = mx1;
    if (K2 > 0) {
        rc = make_planes_map(&mx2, X2, M, K2, ldx2, psx2, 64, T_BK);
        if (rc) return rc;
    }
    rc = make_planes_map(&my, dC, M, N, lddc, psc, 64, T_BK);
    if (rc) return rc;
    if (!t.swap) {
        maps.p[0] = mx1; maps.p[1] = mx2; maps.q[0] = my; maps.q[1] = my;
        a.p_cols[0] = (int)K1; a.p_cols[1] = (int)K2; a.q_cols[0] = (int)N; a.q_cols[1] = 0;
        a.p_off[0] = 0; a.p_off[1] = (int)K1; a.q_off[0] = 0; a.q_off[1] = 0;
        a.transposed = 1;                       // out[n (q)][k (p)]
    } else {
        maps.p[0] = my; maps.p[1] = my; maps.q[0] = mx1; maps.q[1] = mx2;
        a.p_cols[0] = (int)N; a.p_cols[1] = 0; a.q_cols[0] = (int)K1; a.q_cols[1] = (int)K2;
        a.p_off[0] = 0; a.p_off[1] = 0; a.q_off[0] = 0; a.q_off[1] = (int)K1;
        a.transposed = 0;                       // out[n (p)][k (q)]
    }
    a.out = reinterpret_cast<float*>(((uintptr_t)ws + 127) & ~(uintptr_t)127);
    a.ldo = Kt; a.split_stride = N * Kt; a.M = M; a.rows_per_split = t.rows;
    a.npb = t.npb; a.nqb = t.nqb; a.np_tiles = t.np_tiles; a.nq_tiles = t.nq_tiles;
    a.flush_kb = tn_flush_kb();
    a.chunks_per_split = (int)tn_chunks_per_split(t);
    dim3 grid((unsigned)(t.np_tiles * t.nq_tiles), (unsigned)t.splits);
    tn_planes_kernel<<<grid, kThreads, T_SMEM, st>>>(maps, a);
    SPGNN_LAUNCH_OK();
    reduce_splits(a.out, t.splits * a.chunks_per_split, N, Kt, dW, lddw, st);
    return SPGNN_OK;
}

SPGNN_REGISTER_SALT(gemm_tma)

// tcgen05 tensor-core GEMMs for the dense projections (mode 1), fp32 in / fp32 out, fp32-grade accuracy.
//
// Arithmetic: every fp32 operand is split into two bf16 terms, a = a_hi + a_lo (|residual| <= 2^-17 |a|), and the
// product is formed as  a_hi*b_hi + a_hi*b_lo + a_lo*b_hi  with fp32 accumulation in TMEM ("bf16x3"): three
// kind::f16 UMMAs per k-step, relative error ~3*2^-18 per product — inside the 1e-4 parity bar with margin, at 3/2 of
// the cost of ONE tf32 pass (a single tf32 pass would break parity; 3xTF32 would cost twice this).
//
// Kernels (one CTA per SM, persistent over output tiles, 128 x BN x 64 tiles, BN a multiple of 16 up to 256):
//   tc_nt_kernel : C[M,N] = [A1|A2][M,K] * B[N,K]^T (+bias)(act).   A: fp32 activations, converted in-kernel by the
//                  producer warps into SW128 K-major tiles; B: weights pre-split to bf16 hi/lo once per call
//                  (a few MB) and streamed with cp.async.  Used for the forward projection and, with the
//                  transposed pre-split weight, for dX = dY * W.
//   tc_tn_kernel : dW[N,K] = dY[M,N]^T * X[M,K], reduction over the M nodes, split across CTAs into partial
//                  sums (fixed-order reduce afterwards).  Both operands are fp32 activations converted in-kernel
//                  into SW128 MN-major tiles (no transposition: the global row IS the smem k-row).
//
// Warp roles (416 threads): warps 0-3 epilogue (TMEM lanes 32w..32w+31), warp 4 TMEM alloc + single-thread UMMA
// issue, warps 5-12 producers in two groups that alternate k-blocks (group g owns smem stage g), so the global-load
// latency of one group hides behind the conversion work of the other and behind the MMAs.
// Accumulators are double-buffered in TMEM (2 x 256 columns): the epilogue of tile i overlaps the MMAs of tile i+1.
#include "common.cuh"
#include <cuda_bf16.h>

namespace spgnn {
namespace tc {

constexpr int BM = 128;            // UMMA M (cta_group::1)
constexpr int BK = 64;             // bf16 elements per k-block = one 128-byte swizzle row
constexpr int kStages = 2;
constexpr int kEpiWarps = 4, kProdWarps = 8;
constexpr int kThreads = 32 * (kEpiWarps + 1 + kProdWarps);   // 416
constexpr int kGroupThreads = 32 * kProdWarps / 2;             // 128 producer threads per stage group
constexpr int kMaxBN = 256;
constexpr uint32_t kTmemCols = 512;

constexpr int kATileBytes = BM * 128;          // 16 KB : 128 rows x 128 B (one of hi / lo)
constexpr int kBTileBytes = kMaxBN * 128;      // 32 KB
constexpr int kStageBytes = 2 * kATileBytes + 2 * kBTileBytes;   // 96 KB
constexpr int kStgLd = 36;                     // padded row of the per-warp 32x32 epilogue staging tile (floats)
constexpr int kStgBytes = kEpiWarps * 32 * kStgLd * 4;
constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align*/ + 256 /*barriers*/ + kStgBytes;

// ---------------------------------------------------------------------------------------------- PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}" ::"r"(bar), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

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

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void st_shared_v2(uint32_t addr, uint32_t a, uint32_t b) {
    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(a), "r"(b) : "memory");
}

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
// instruction descriptor: c=f32 [4,6)=1, a=bf16 [7,10)=1, b=bf16 [10,13)=1, a_major bit 15, b_major bit 16,
// n>>3 at [17,23), m>>4 at [24,29)
__host__ __device__ __forceinline__ uint32_t make_idesc(int n, bool mn_major) {
    uint32_t d = (1u << 4) | (1u << 7) | (1u << 10);
    if (mn_major) d |= (1u << 15) | (1u << 16);
    d |= (uint32_t)(n >> 3) << 17;
    d |= (uint32_t)(BM >> 4) << 24;
    return d;
}

// fp32 pair -> packed bf16 (hi) and packed bf16 of the remainders (lo); low half = first element
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    hi = *reinterpret_cast<uint32_t*>(&h);
    const float ra = a - __uint_as_float(hi << 16);
    const float rb = b - __uint_as_float(hi & 0xFFFF0000u);
    __nv_bfloat162 l = __floats2bfloat162_rn(ra, rb);
    lo = *reinterpret_cast<uint32_t*>(&l);
}

struct NtArgs {
    const float* A1; int64_t lda1; int K1;
    const float* A2; int64_t lda2; int K2;
    const __nv_bfloat16* Bhi; const __nv_bfloat16* Blo; int64_t ldb;   // [N, kb_total*64] pre-split, zero padded
    const float* bias; int act; float slope;
    float* C; int64_t ldc;
    int64_t M; int N;
    int BN; int nt_n; int64_t nt_m;       // tile width, tiles along n, tiles along m
    int kb1, kb2;                          // k-blocks of source 1 / source 2
};

struct Shared {
    uint64_t full[kStages];
    uint64_t empty[kStages];
    uint64_t tmem_full[2];
    uint64_t tmem_empty[2];
    uint32_t tmem_base;
};

// ---------------------------------------------------------------------------------------------- NT kernel
__global__ void __launch_bounds__(kThreads, 1) tc_nt_kernel(const NtArgs g) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    Shared* sh = reinterpret_cast<Shared*>(smem + kStages * kStageBytes);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem_base = smem_u32(smem);

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) {
            mbar_init(smem_u32(&sh->full[s]), kGroupThreads);
            mbar_init(smem_u32(&sh->empty[s]), 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(smem_u32(&sh->tmem_full[b]), 1);
            mbar_init(smem_u32(&sh->tmem_empty[b]), kEpiWarps * 32);
        }
        fence_barrier_init();
    }
    if (warp == kEpiWarps) tmem_alloc(smem_u32(&sh->tmem_base), kTmemCols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = sh->tmem_base;

    const int64_t n_tiles = g.nt_m * g.nt_n;
    const int nkb = g.kb1 + g.kb2;

    if (warp < kEpiWarps) {
        // ===================================================== epilogue: TMEM -> registers -> global
        int it = 0;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
            const int buf = it & 1;
            const uint32_t par = (it >> 1) & 1;
            const int64_t m0 = (tile / g.nt_n) * BM;
            const int n0 = (int)(tile % g.nt_n) * g.BN;
            const int ncols = min(g.BN, g.N - n0);
            mbar_wait(smem_u32(&sh->tmem_full[buf]), par);
            tc_fence_after();
            // TMEM lane = output row, so a raw store would scatter 16-byte pieces over 32 rows per instruction.
            // Stage 32x32 blocks through a per-warp smem tile and write 4 rows x 128 B per instruction instead.
            const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(buf * kMaxBN);
            float* stg = reinterpret_cast<float*>(smem + kStages * kStageBytes + 256) + warp * (32 * kStgLd);
            const bool vec_ok = (g.ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(g.C) & 15) == 0);
            const bool plain = (g.act == SPGNN_ACT_NONE) && (g.bias == nullptr);
            for (int c0 = 0; c0 < ncols; c0 += 32) {
                uint32_t v[32];
                tmem_ld16(taddr + c0, *reinterpret_cast<uint32_t(*)[16]>(&v[0]));
                tmem_ld16(taddr + c0 + 16, *reinterpret_cast<uint32_t(*)[16]>(&v[16]));
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    *reinterpret_cast<float4*>(stg + lane * kStgLd + 4 * j) =
                        make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                    __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
                __syncwarp();
                const int cc = (lane & 7) * 4;
                const int col = n0 + c0 + cc;
                const int rsub = lane >> 3;                                   // row within each group of 4
                const int64_t row0 = m0 + warp * 32 + rsub;
                float* q = g.C + row0 * g.ldc + col;
                const int64_t qstep = 4 * g.ldc;
                const int nrow = (int)min((int64_t)8, (g.M - row0 + 3) / 4);  // iterations with a valid row
                const float* sp = stg + rsub * kStgLd + cc;
                if (plain && vec_ok && c0 + 32 <= ncols) {
                    // interior block, no bias / activation: pure 128-bit copies
#pragma unroll
                    for (int itr = 0; itr < 8; ++itr)
                        if (itr < nrow) st4(q + itr * qstep, *reinterpret_cast<const float4*>(sp + itr * 4 * kStgLd));
                } else {
                    float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (g.bias) {
                        if (col + 0 < g.N) bv.x = __ldg(g.bias + col + 0);
                        if (col + 1 < g.N) bv.y = __ldg(g.bias + col + 1);
                        if (col + 2 < g.N) bv.z = __ldg(g.bias + col + 2);
                        if (col + 3 < g.N) bv.w = __ldg(g.bias + col + 3);
                    }
                    const int nvalid = ncols - (c0 + cc);                     // columns of this lane's float4 in range
                    for (int itr = 0; itr < nrow; ++itr) {
                        float4 x = *reinterpret_cast<const float4*>(sp + itr * 4 * kStgLd);
                        x.x = act_fwd(x.x + bv.x, g.act, g.slope);
                        x.y = act_fwd(x.y + bv.y, g.act, g.slope);
                        x.z = act_fwd(x.z + bv.z, g.act, g.slope);
                        x.w = act_fwd(x.w + bv.w, g.act, g.slope);
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
            tc_fence_before();
            mbar_arrive(smem_u32(&sh->tmem_empty[buf]));
        }
    } else if (warp == kEpiWarps) {
        // ===================================================== UMMA issuer (one elected thread)
        if (lane == 0) {
            int it = 0;
            uint32_t kcount = 0;
            for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
                const int buf = it & 1;
                const uint32_t par = (it >> 1) & 1;
                const int n0 = (int)(tile % g.nt_n) * g.BN;
                const int ncols = min(g.BN, g.N - n0);
                const int n_mma = (ncols + 15) & ~15;
                const uint32_t idesc = make_idesc(n_mma, false);
                mbar_wait(smem_u32(&sh->tmem_empty[buf]), par ^ 1);     // epilogue drained this accumulator
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + (uint32_t)(buf * kMaxBN);
                for (int kb = 0; kb < nkb; ++kb, ++kcount) {
                    const int s = kcount & 1;
                    const uint32_t sp = (kcount >> 1) & 1;
                    mbar_wait(smem_u32(&sh->full[s]), sp);
                    tc_fence_after();
                    const uint32_t a_hi = smem_base + s * kStageBytes;
                    const uint32_t a_lo = a_hi + kATileBytes;
                    const uint32_t b_hi = a_lo + kATileBytes;
                    const uint32_t b_lo = b_hi + kBTileBytes;
#pragma unroll
                    for (int k = 0; k < BK / 16; ++k) {
                        const uint32_t ko = k * 32;      // 16 bf16 = 32 bytes along the swizzled row
                        const uint64_t dah = make_desc(a_hi + ko, 16, 1024), dal = make_desc(a_lo + ko, 16, 1024);
                        const uint64_t dbh = make_desc(b_hi + ko, 16, 1024), dbl = make_desc(b_lo + ko, 16, 1024);
                        umma_bf16(tmem_d, dah, dbh, idesc, (kb | k) != 0);
                        umma_bf16(tmem_d, dah, dbl, idesc, 1);
                        umma_bf16(tmem_d, dal, dbh, idesc, 1);
                    }
                    umma_commit(smem_u32(&sh->empty[s]));      // frees the smem stage when these UMMAs retire
                }
                umma_commit(smem_u32(&sh->tmem_full[buf]));    // accumulator complete -> epilogue
            }
        }
    } else {
        // ===================================================== producers: group gidx owns stage gidx
        // The (tile, k-block) pairs of this CTA form one sequence; group g takes the elements with seq % 2 == g.
        // Global loads run one element AHEAD: as soon as a float4 of the current block is converted, the same
        // register is re-armed with the float4 of the group's next block, so ~16 loads per thread are always in
        // flight and their latency hides behind the conversion work and the barrier waits.
        const int pt = threadIdx.x - 32 * (kEpiWarps + 1);      // 0..255
        const int gidx = pt / kGroupThreads;                     // 0 / 1
        const int t = pt % kGroupThreads;                        // 0..127
        const int q = t & 15;                                    // float4 index within a 64-float row
        const int r0 = t >> 4;                                   // 0..7, rows r0 + 8*i
        const int64_t my_tiles = blockIdx.x < n_tiles ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
        const int64_t n_seq = my_tiles * nkb;

        // per-block load plan (computed once per k-block: the 64-bit div/mod must stay out of the 16-load loop)
        struct Plan { const float* p; int64_t step; int nrows; int kmode; };   // kmode: 0 none, 1..3 partial, 4 full float4
        auto make_plan = [&](int64_t seq) -> Plan {
            Plan pl{nullptr, 0, 0, 0};
            if (seq >= n_seq) return pl;
            const int64_t tile = blockIdx.x + (seq / nkb) * gridDim.x;
            const int kb = (int)(seq % nkb);
            const bool s2 = kb >= g.kb1;
            const float* Ap = s2 ? g.A2 : g.A1;
            const int64_t lda = s2 ? g.lda2 : g.lda1;
            const int Klim = s2 ? g.K2 : g.K1;
            const int k0 = (s2 ? kb - g.kb1 : kb) * BK + q * 4;
            const int64_t row = (tile / g.nt_n) * BM + r0;
            pl.p = Ap + row * lda + k0;
            pl.step = 8 * lda;
            const int64_t left = g.M - row;                       // rows row, row+8, ... < M
            pl.nrows = left <= 0 ? 0 : (int)min((int64_t)16, (left + 7) / 8);
            pl.kmode = k0 + 3 < Klim ? 4 : (k0 < Klim ? Klim - k0 : 0);
            return pl;
        };
        auto load_a = [&](const Plan& pl, int i) -> float4 {
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < pl.nrows && pl.kmode) {
                const float* p = pl.p + i * pl.step;
                if (pl.kmode == 4) v = ldg4(p);
                else {
                    v.x = __ldg(p);
                    if (pl.kmode > 1) v.y = __ldg(p + 1);
                    if (pl.kmode > 2) v.z = __ldg(p + 2);
                }
            }
            return v;
        };

        float4 av[16];
        {
            const Plan p0 = make_plan(gidx);
#pragma unroll
            for (int i = 0; i < 16; ++i) av[i] = load_a(p0, i);
        }
        for (int64_t seq = gidx; seq < n_seq; seq += 2) {
            const int64_t tile = blockIdx.x + (seq / nkb) * gridDim.x;
            const int kb = (int)(seq % nkb);
            const int n0 = (int)(tile % g.nt_n) * g.BN;
            const int ncols = min(g.BN, g.N - n0);
            const int brows = (ncols + 15) & ~15;
            const uint32_t sp = (uint32_t)(seq >> 1) & 1;
            const Plan nxt = make_plan(seq + 2);
            mbar_wait(smem_u32(&sh->empty[gidx]), sp ^ 1);
            const uint32_t a_hi = smem_base + gidx * kStageBytes;
            const uint32_t a_lo = a_hi + kATileBytes;
            const uint32_t b_hi = a_lo + kATileBytes;
            const uint32_t b_lo = b_hi + kBTileBytes;
            // ---- B: pre-split bf16 rows, 16-byte chunks straight into the swizzled layout (zero-fill past N)
            {
                const int64_t kcol = (int64_t)kb * BK;
                for (int idx = t; idx < brows * 8; idx += kGroupThreads) {
                    const int n = idx >> 3, c = idx & 7;
                    const uint32_t off = (uint32_t)n * 128 + (uint32_t)((c ^ (n & 7)) << 4);
                    const bool ok = n0 + n < g.N;
                    const int64_t go = (int64_t)(ok ? n0 + n : 0) * g.ldb + kcol + c * 8;
                    cp_async16(b_hi + off, g.Bhi + go, ok ? 16u : 0u);
                    cp_async16(b_lo + off, g.Blo + go, ok ? 16u : 0u);
                }
            }
            // ---- A: convert and store (8-byte stores; chunk index XOR (row & 7) = SWIZZLE_128B), then re-arm the load
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const int r = r0 + 8 * i;
                uint32_t h0, l0, h1, l1;
                split2(av[i].x, av[i].y, h0, l0);
                split2(av[i].z, av[i].w, h1, l1);
                const uint32_t off = (uint32_t)r * 128 + (uint32_t)(((q >> 1) ^ (r & 7)) << 4) + (uint32_t)(q & 1) * 8;
                st_shared_v2(a_hi + off, h0, h1);
                st_shared_v2(a_lo + off, l0, l1);
                av[i] = load_a(nxt, i);
            }
            cp_async_wait_all();
            fence_proxy_async();          // generic-proxy writes -> visible to the tensor core (async proxy)
            mbar_arrive(smem_u32(&sh->full[gidx]));
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == kEpiWarps) {
        tc_fence_after();
        tmem_dealloc(tmem_base, kTmemCols);
    }
}

// ---------------------------------------------------------------------------------------------- TN kernel (dW)
// dW partial [z][n, k] = sum over this split's node rows m of dY[m, n] * X[m, k]
struct TnArgs {
    const float* dY; int64_t lddy; int N;      // "A" operand: M dimension of the UMMA = n (rows of dW)
    const float* X; int64_t ldx; int K;        // "B" operand: N dimension of the UMMA = k (cols of dW)
    float* out; int64_t ldo; int64_t split_stride;
    int64_t M; int64_t rows_per_split;
    int nt_n, nt_k;                            // tiles along n (128) and k (128)
    uint32_t lbo, sbo;                         // MN-major SW128 descriptor strides (bytes)
};
constexpr int TN_BN = 128;                     // UMMA N for the weight gradient
constexpr int kTnTile = 64 * 128 * 2;          // 16 KB: 64 k-rows x 128 mn x bf16 (two 64-wide MN blocks of 8 KB)
constexpr int kTnStageBytes = 4 * kTnTile;     // A hi/lo + B hi/lo = 64 KB
constexpr int kTnStages = 3;
constexpr int kTnSmemBytes = kTnStages * kTnStageBytes + 1024 + 256;

struct SharedTn {
    uint64_t full[kTnStages];
    uint64_t empty[kTnStages];
    uint64_t tmem_full;
    uint32_t tmem_base;
};

__global__ void __launch_bounds__(kThreads, 1) tc_tn_kernel(const TnArgs g) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    SharedTn* sh = reinterpret_cast<SharedTn*>(smem + kTnStages * kTnStageBytes);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem_base = smem_u32(smem);
    constexpr int kProdThreads = 32 * kProdWarps;   // all 256 producer threads fill every stage

    if (threadIdx.x == 0) {
        for (int s = 0; s < kTnStages; ++s) {
            mbar_init(smem_u32(&sh->full[s]), kProdThreads);
            mbar_init(smem_u32(&sh->empty[s]), 1);
        }
        mbar_init(smem_u32(&sh->tmem_full), 1);
        fence_barrier_init();
    }
    if (warp == kEpiWarps) tmem_alloc(smem_u32(&sh->tmem_base), 128);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = sh->tmem_base;

    // one output tile per CTA: blockIdx.x = (tile_n * nt_k + tile_k), blockIdx.y = split
    const int tn = blockIdx.x / g.nt_k, tk = blockIdx.x % g.nt_k;
    const int n0 = tn * BM, k0 = tk * TN_BN;
    const int64_t mbeg = (int64_t)blockIdx.y * g.rows_per_split;
    const int64_t mend = min(g.M, mbeg + g.rows_per_split);
    const int nkb = (int)((mend - mbeg + BK - 1) / BK);

    if (warp < kEpiWarps) {
        mbar_wait(smem_u32(&sh->tmem_full), 0);
        tc_fence_after();
        const int row = n0 + warp * 32 + lane;
        float* orow = g.out + (int64_t)blockIdx.y * g.split_stride + (int64_t)row * g.ldo + k0;
        const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16);
        const int ncols = min(TN_BN, g.K - k0);
        for (int c0 = 0; c0 < ncols; c0 += 16) {
            uint32_t v[16];
            tmem_ld16(taddr + c0, v);
            tmem_ld_wait();
            if (row < g.N) {
                for (int j = 0; j < 16 && c0 + j < ncols; ++j) orow[c0 + j] = nkb > 0 ? __uint_as_float(v[j]) : 0.f;
            }
        }
    } else if (warp == kEpiWarps) {
        if (lane == 0) {
            const uint32_t idesc = make_idesc(TN_BN, true);
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % kTnStages;
                const uint32_t sp = (kb / kTnStages) & 1;
                mbar_wait(smem_u32(&sh->full[s]), sp);
                tc_fence_after();
                const uint32_t a_hi = smem_base + s * kTnStageBytes;
                const uint32_t a_lo = a_hi + kTnTile, b_hi = a_lo + kTnTile, b_lo = b_hi + kTnTile;
#pragma unroll
                for (int k = 0; k < BK / 16; ++k) {
                    const uint32_t ko = k * 16 * 128;     // 16 k-rows of 128 B
                    const uint64_t dah = make_desc(a_hi + ko, g.lbo, g.sbo), dal = make_desc(a_lo + ko, g.lbo, g.sbo);
                    const uint64_t dbh = make_desc(b_hi + ko, g.lbo, g.sbo), dbl = make_desc(b_lo + ko, g.lbo, g.sbo);
                    umma_bf16(tmem_base, dah, dbh, idesc, (kb | k) != 0);
                    umma_bf16(tmem_base, dah, dbl, idesc, 1);
                    umma_bf16(tmem_base, dal, dbh, idesc, 1);
                }
                umma_commit(smem_u32(&sh->empty[s]));
            }
            umma_commit(smem_u32(&sh->tmem_full));
        }
    } else {
        const int t = threadIdx.x - 32 * (kEpiWarps + 1);   // 0..255
        const int q = t & 31;                                // float4 index within a 128-float row segment
        const int r0 = t >> 5;                               // 0..7, k-rows r0 + 8*i
        const int n = n0 + q * 4, k = k0 + q * 4;
        // rolling prefetch (see tc_nt_kernel): registers are re-armed with the next k-block right after use
        auto load_ab = [&](int kb, int i, float4& va, float4& vb) {
            va = vb = make_float4(0.f, 0.f, 0.f, 0.f);
            const int64_t m = mbeg + (int64_t)kb * BK + r0 + 8 * i;
            if (kb < nkb && m < mend) {
                const float* pa = g.dY + m * g.lddy + n;
                const float* pb = g.X + m * g.ldx + k;
                if (n + 3 < g.N) va = ldg4(pa);
                else if (n < g.N) { va.x = __ldg(pa); if (n + 1 < g.N) va.y = __ldg(pa + 1); if (n + 2 < g.N) va.z = __ldg(pa + 2); }
                if (k + 3 < g.K) vb = ldg4(pb);
                else if (k < g.K) { vb.x = __ldg(pb); if (k + 1 < g.K) vb.y = __ldg(pb + 1); if (k + 2 < g.K) vb.z = __ldg(pb + 2); }
            }
        };
        float4 av[8], bv[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) load_ab(0, i, av[i], bv[i]);
        for (int kb = 0; kb < nkb; ++kb) {
            const int s = kb % kTnStages;
            const uint32_t sp = (kb / kTnStages) & 1;
            mbar_wait(smem_u32(&sh->empty[s]), sp ^ 1);
            const uint32_t a_hi = smem_base + s * kTnStageBytes;
            const uint32_t a_lo = a_hi + kTnTile, b_hi = a_lo + kTnTile, b_lo = b_hi + kTnTile;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int kk = r0 + 8 * i;
                // MN-major SW128: [mn block of 64][k-row][128 B], 16-byte chunk index XOR (k-row & 7)
                const int c = (q & 15) >> 1;
                const uint32_t off = (uint32_t)(q >> 4) * 8192 + (uint32_t)kk * 128 + (uint32_t)((c ^ (kk & 7)) << 4) +
                                     (uint32_t)(q & 1) * 8;
                uint32_t h0, l0, h1, l1;
                split2(av[i].x, av[i].y, h0, l0);
                split2(av[i].z, av[i].w, h1, l1);
                st_shared_v2(a_hi + off, h0, h1);
                st_shared_v2(a_lo + off, l0, l1);
                split2(bv[i].x, bv[i].y, h0, l0);
                split2(bv[i].z, bv[i].w, h1, l1);
                st_shared_v2(b_hi + off, h0, h1);
                st_shared_v2(b_lo + off, l0, l1);
                load_ab(kb + 1, i, av[i], bv[i]);
            }
            fence_proxy_async();
            mbar_arrive(smem_u32(&sh->full[s]));
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == kEpiWarps) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 128);
    }
}

// ---------------------------------------------------------------------------------------------- TN kernel v2 (dW)
// D[k, n] = sum over nodes m of X[m, k] * dY[m, n]  (= dW^T): a CTA owns 256 k-columns of X (two M=128 accumulators
// that SHARE the dY tile) x BN <= 256 dY-columns, so each fp32 operand element fetched from L2 feeds twice the
// math of a 128x128 tile (the v1 kernel was L2-bandwidth bound).  X may come from two sources ([X1 | X2], the
// un-materialised torch.cat).  BK = 32 nodes per stage, 3 stages, MN-major SW128 tiles, rolling register prefetch.
// TMEM lane = k, so the epilogue's per-column stores are 32 consecutive floats of a dW row: coalesced as is.
struct Tn2Args {
    const float* X1; int64_t ldx1; int K1;
    const float* X2; int64_t ldx2; int K2;
    const float* dY; int64_t lddy; int N;
    float* out; int64_t ldo; int64_t split_stride;      // partial sums [split][N][K1+K2]
    int64_t M; int64_t rows_per_split;
    int nk1, nk2, nt_n, BN;                             // 256-wide k tiles of source 1 / 2, n tiles, n tile width
};
constexpr int T2_BK = 32;
constexpr int T2_ABYTES = 4 * 4096;            // 256 mn x 32 rows x bf16 = 4 MN-blocks of 4 KB (one plane)
constexpr int T2_BBYTES = 4 * 4096;            // up to 256 mn
constexpr int T2_STAGE = 2 * T2_ABYTES + 2 * T2_BBYTES;   // 64 KB
constexpr int T2_STAGES = 3;
constexpr int T2_SMEM = T2_STAGES * T2_STAGE + 1024 + 256;

struct SharedTn2 {
    uint64_t full[T2_STAGES];
    uint64_t empty[T2_STAGES];
    uint64_t tmem_full;
    uint32_t tmem_base;
};

__global__ void __launch_bounds__(kThreads, 1) tc_tn2_kernel(const Tn2Args g) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    SharedTn2* sh = reinterpret_cast<SharedTn2*>(smem + T2_STAGES * T2_STAGE);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem_base = smem_u32(smem);
    constexpr int kProdThreads = 32 * kProdWarps;

    if (threadIdx.x == 0) {
        for (int s = 0; s < T2_STAGES; ++s) {
            mbar_init(smem_u32(&sh->full[s]), kProdThreads);
            mbar_init(smem_u32(&sh->empty[s]), 1);
        }
        mbar_init(smem_u32(&sh->tmem_full), 1);
        fence_barrier_init();
    }
    if (warp == kEpiWarps) tmem_alloc(smem_u32(&sh->tmem_base), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = sh->tmem_base;

    // work item: blockIdx.x = k-tile * nt_n + n-tile, blockIdx.y = split over the nodes
    const int tk = blockIdx.x / g.nt_n, tn = blockIdx.x % g.nt_n;
    const bool s2 = tk >= g.nk1;
    const float* X = s2 ? g.X2 : g.X1;
    const int64_t ldx = s2 ? g.ldx2 : g.ldx1;
    const int Kv = s2 ? g.K2 : g.K1;                         // valid columns of this source
    const int kbase = (s2 ? tk - g.nk1 : tk) * 256;          // first column within the source
    const int kout = (s2 ? g.K1 : 0) + kbase;                // first column in dW
    const int n0 = tn * g.BN;
    const int ncols = min(g.BN, g.N - n0);
    const int n_mma = (ncols + 15) & ~15;
    const int64_t mbeg = (int64_t)blockIdx.y * g.rows_per_split;
    const int64_t mend = min(g.M, mbeg + g.rows_per_split);
    const int nkb = (int)((mend - mbeg + T2_BK - 1) / T2_BK);
    const bool two_acc = kbase + 128 < Kv;                   // second accumulator has any valid column

    if (warp < kEpiWarps) {
        mbar_wait(smem_u32(&sh->tmem_full), 0);
        tc_fence_after();
        float* obase = g.out + (int64_t)blockIdx.y * g.split_stride;
        for (int acc = 0; acc < (two_acc ? 2 : 1); ++acc) {
            const int kk = kbase + acc * 128 + warp * 32 + lane;        // column within the source
            const bool kok = kk < Kv;
            const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(acc * 256);
            float* ocol = obase + (kout + acc * 128 + warp * 32 + lane);
            for (int c0 = 0; c0 < ncols; c0 += 16) {
                uint32_t v[16];
                tmem_ld16(taddr + c0, v);
                tmem_ld_wait();
                if (kok) {
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if (c0 + j < ncols) ocol[(int64_t)(n0 + c0 + j) * g.ldo] = __uint_as_float(v[j]);
                }
            }
        }
    } else if (warp == kEpiWarps) {
        if (lane == 0) {
            const uint32_t idesc = make_idesc(n_mma, true);
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % T2_STAGES;
                const uint32_t sp = (kb / T2_STAGES) & 1;
                mbar_wait(smem_u32(&sh->full[s]), sp);
                tc_fence_after();
                const uint32_t a_hi = smem_base + s * T2_STAGE;
                const uint32_t a_lo = a_hi + T2_ABYTES, b_hi = a_lo + T2_ABYTES, b_lo = b_hi + T2_BBYTES;
#pragma unroll
                for (int k = 0; k < T2_BK / 16; ++k) {
                    const uint32_t ko = k * 16 * 128;
                    const uint64_t dbh = make_desc(b_hi + ko, 4096, 1024), dbl = make_desc(b_lo + ko, 4096, 1024);
#pragma unroll
                    for (int acc = 0; acc < 2; ++acc) {
                        if (acc == 1 && !two_acc) break;
                        const uint32_t ao = acc * 8192 + ko;             // two 64-wide MN blocks per accumulator
                        const uint64_t dah = make_desc(a_hi + ao, 4096, 1024), dal = make_desc(a_lo + ao, 4096, 1024);
                        const uint32_t td = tmem_base + (uint32_t)(acc * 256);
                        umma_bf16(td, dah, dbh, idesc, (kb | k) != 0);
                        umma_bf16(td, dah, dbl, idesc, 1);
                        umma_bf16(td, dal, dbh, idesc, 1);
                    }
                }
                umma_commit(smem_u32(&sh->empty[s]));
            }
            umma_commit(smem_u32(&sh->tmem_full));
        }
    } else {
        const int t = threadIdx.x - 32 * (kEpiWarps + 1);   // 0..255
        // X tile: 32 rows x 64 float4; thread -> (q = t & 63, rows (t >> 6) + 4 i), 8 float4
        const int qa = t & 63, ra = t >> 6;
        const int ka = kbase + qa * 4;
        const uint32_t offa = (uint32_t)(qa >> 4) * 4096 + (uint32_t)(((qa & 15) >> 1) << 4) + (uint32_t)(qa & 1) * 8;
        // dY tile: 32 rows x (n_mma/4) float4, linear index t + 256 i; (row, q) fixed per thread -> computed once
        const int qpr = n_mma >> 2;
        constexpr int NB = 8;                                 // 32 * 64 / 256
        int brow[NB], bq[NB];
#pragma unroll
        for (int i = 0; i < NB; ++i) {
            const int idx = t + 256 * i;
            brow[i] = idx / qpr;
            bq[i] = idx - brow[i] * qpr;
            if (brow[i] >= T2_BK) brow[i] = -1;
        }
        auto load_x = [&](int kb, int i) -> float4 {
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            const int64_t m = mbeg + (int64_t)kb * T2_BK + ra + 4 * i;
            if (kb < nkb && m < mend && ka < Kv) {
                const float* p = X + m * ldx + ka;
                if (ka + 3 < Kv) v = ldg4(p);
                else { v.x = __ldg(p); if (ka + 1 < Kv) v.y = __ldg(p + 1); if (ka + 2 < Kv) v.z = __ldg(p + 2); }
            }
            return v;
        };
        auto load_y = [&](int kb, int i) -> float4 {
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (brow[i] < 0) return v;
            const int64_t m = mbeg + (int64_t)kb * T2_BK + brow[i];
            const int n = n0 + bq[i] * 4;
            if (kb < nkb && m < mend && n < g.N) {
                const float* p = g.dY + m * g.lddy + n;
                if (n + 3 < g.N) v = ldg4(p);
                else { v.x = __ldg(p); if (n + 1 < g.N) v.y = __ldg(p + 1); if (n + 2 < g.N) v.z = __ldg(p + 2); }
            }
            return v;
        };
        float4 xv[8], yv[NB];
#pragma unroll
        for (int i = 0; i < 8; ++i) xv[i] = load_x(0, i);
#pragma unroll
        for (int i = 0; i < NB; ++i) yv[i] = load_y(0, i);
        for (int kb = 0; kb < nkb; ++kb) {
            const int s = kb % T2_STAGES;
            const uint32_t sp = (kb / T2_STAGES) & 1;
            mbar_wait(smem_u32(&sh->empty[s]), sp ^ 1);
            const uint32_t a_hi = smem_base + s * T2_STAGE;
            const uint32_t a_lo = a_hi + T2_ABYTES, b_hi = a_lo + T2_ABYTES, b_lo = b_hi + T2_BBYTES;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int kk = ra + 4 * i;
                const uint32_t off = offa + (uint32_t)kk * 128;
                // chunk swizzle: XOR the 16-byte chunk index with (row & 7)
                const uint32_t sw = off ^ ((uint32_t)(kk & 7) << 4);
                uint32_t h0, l0, h1, l1;
                split2(xv[i].x, xv[i].y, h0, l0);
                split2(xv[i].z, xv[i].w, h1, l1);
                st_shared_v2(a_hi + sw, h0, h1);
                st_shared_v2(a_lo + sw, l0, l1);
                xv[i] = load_x(kb + 1, i);
            }
#pragma unroll
            for (int i = 0; i < NB; ++i) {
                if (brow[i] >= 0) {
                    const int kk = brow[i], q = bq[i];
                    const uint32_t off = (uint32_t)(q >> 4) * 4096 + (uint32_t)kk * 128 +
                                         (uint32_t)((((q & 15) >> 1) ^ (kk & 7)) << 4) + (uint32_t)(q & 1) * 8;
                    uint32_t h0, l0, h1, l1;
                    split2(yv[i].x, yv[i].y, h0, l0);
                    split2(yv[i].z, yv[i].w, h1, l1);
                    st_shared_v2(b_hi + off, h0, h1);
                    st_shared_v2(b_lo + off, l0, l1);
                    yv[i] = load_y(kb + 1, i);
                }
            }
            fence_proxy_async();
            mbar_arrive(smem_u32(&sh->full[s]));
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == kEpiWarps) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// ---------------------------------------------------------------------------------------------- weight pre-split
// out[r, c] (hi/lo bf16, ld = ldo): r < R rows, c < Cpad columns.
//   transpose = 0: out[r, c] = W[r, map(c)]  with map: c < K1pad -> c (valid if c < K1), else K1 + (c - K1pad) (valid if < K1+K2)
//   transpose = 1: out[r, c] = W[c, k_off + r]  (c < N valid)
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

static inline int round_up(int64_t x, int m) { return (int)((x + m - 1) / m * m); }

// choose the tile width: as few n-tiles as possible, equal widths, multiple of 16
static void pick_bn(int N, int* BN, int* nt) {
    const int n16 = round_up(N, 16);
    *nt = (n16 + kMaxBN - 1) / kMaxBN;
    *BN = round_up((n16 + *nt - 1) / *nt, 16);
}

static DeviceOnce g_attr_set_nt, g_attr_set_tn;

}  // namespace tc

using namespace tc;

int64_t tc_linear_ws_bytes(int64_t N, int64_t K1, int64_t K2) {
    const int64_t kp = round_up(K1, BK) + (K2 > 0 ? round_up(K2, BK) : 0);
    return 2 * N * kp * (int64_t)sizeof(__nv_bfloat16) + 256;
}

static int launch_nt(const NtArgs& a, cudaStream_t st) {
    if (g_attr_set_nt.pending()) {
        SPGNN_CUDA_OK(cudaFuncSetAttribute(tc_nt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
        g_attr_set_nt.done();
    }
    const int64_t tiles = a.nt_m * a.nt_n;
    const unsigned grid = (unsigned)(tiles < sm_count() ? tiles : sm_count());
    tc_nt_kernel<<<grid, kThreads, kSmemBytes, st>>>(a);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

int tc_linear_fwd(const float* A1, int64_t lda1, int64_t K1, const float* A2, int64_t lda2, int64_t K2, const float* W,
                  int64_t ldw, const float* bias, int act, float slope, float* C, int64_t ldc, int64_t M, int64_t N,
                  void* ws, cudaStream_t st) {
    const int k1p = round_up(K1, BK), k2p = A2 ? round_up(K2, BK) : 0;
    const int64_t ldb = k1p + k2p;
    __nv_bfloat16* hi = reinterpret_cast<__nv_bfloat16*>(((uintptr_t)ws + 127) & ~(uintptr_t)127);
    __nv_bfloat16* lo = hi + N * ldb;
    {
        const int64_t total = N * ldb;
        const unsigned blocks = (unsigned)(ceil_div(total, 256) < 4096 ? ceil_div(total, 256) : 4096);
        split_weight_kernel<<<blocks, 256, 0, st>>>(W, ldw, 0, 0, (int)N, (int)ldb, (int)K1, k1p, A2 ? (int)K2 : 0, 0, hi,
                                                    lo, ldb);
        SPGNN_LAUNCH_OK();
    }
    NtArgs a{};
    a.A1 = A1; a.lda1 = lda1; a.K1 = (int)K1; a.A2 = A2; a.lda2 = lda2; a.K2 = A2 ? (int)K2 : 0;
    a.Bhi = hi; a.Blo = lo; a.ldb = ldb; a.bias = bias; a.act = act; a.slope = slope;
    a.C = C; a.ldc = ldc; a.M = M; a.N = (int)N;
    pick_bn((int)N, &a.BN, &a.nt_n);
    a.nt_m = ceil_div(M, BM);
    a.kb1 = k1p / BK; a.kb2 = k2p / BK;
    return launch_nt(a, st);
}

int64_t tc_linear_bwd_input_ws_bytes(int64_t N, int64_t K) { return 2 * K * (int64_t)round_up(N, BK) * 2 + 256; }

// dA[M,K] = dC[M,N] * W[N, k_off:k_off+K]  ==  NT GEMM with B = (W^T)[K, N] pre-split
int tc_linear_bwd_input(const float* dC, int64_t lddc, const float* W, int64_t ldw, int64_t k_off, float* dA,
                        int64_t ldda, int64_t M, int64_t N, int64_t K, void* ws, cudaStream_t st) {
    const int np = round_up(N, BK);
    __nv_bfloat16* hi = reinterpret_cast<__nv_bfloat16*>(((uintptr_t)ws + 127) & ~(uintptr_t)127);
    __nv_bfloat16* lo = hi + K * np;
    {
        const int64_t total = K * np;
        const unsigned blocks = (unsigned)(ceil_div(total, 256) < 4096 ? ceil_div(total, 256) : 4096);
        split_weight_kernel<<<blocks, 256, 0, st>>>(W, ldw, 1, k_off, (int)K, np, 0, 0, 0, (int)N, hi, lo, np);
        SPGNN_LAUNCH_OK();
    }
    NtArgs a{};
    a.A1 = dC; a.lda1 = lddc; a.K1 = (int)N; a.A2 = nullptr; a.K2 = 0;
    a.Bhi = hi; a.Blo = lo; a.ldb = np; a.bias = nullptr; a.act = 0; a.slope = 0.f;
    a.C = dA; a.ldc = ldda; a.M = M; a.N = (int)K;
    pick_bn((int)K, &a.BN, &a.nt_n);
    a.nt_m = ceil_div(M, BM);
    a.kb1 = np / BK; a.kb2 = 0;
    return launch_nt(a, st);
}

static void tn_plan(int64_t M, int64_t N, int64_t K, int64_t* splits, int64_t* rows) {
    const int64_t tiles = ceil_div(N, BM) * ceil_div(K, TN_BN);
    int64_t want = ceil_div((int64_t)sm_count() * 2, tiles);
    const int64_t max_by_rows = ceil_div(M, 2048);
    if (want > max_by_rows) want = max_by_rows;
    if (want > 256) want = 256;
    if (want < 1) want = 1;
    *rows = ceil_div(ceil_div(M, want), BK) * BK;
    *splits = ceil_div(M, *rows);
}

int64_t tc_linear_bwd_weight_ws_bytes(int64_t M, int64_t N, int64_t K) {
    int64_t splits, rows;
    tn_plan(M, N, K, &splits, &rows);
    return splits * N * K * (int64_t)sizeof(float);
}

void reduce_splits(const float* ws, int64_t splits, int64_t N, int64_t K, float* out, int64_t ldo, cudaStream_t st);

int tc_linear_bwd_weight(const float* dC, int64_t lddc, const float* A, int64_t lda, float* dW, int64_t lddw,
                         int64_t k_off, int64_t M, int64_t N, int64_t K, void* ws, cudaStream_t st) {
    if (g_attr_set_tn.pending()) {
        SPGNN_CUDA_OK(cudaFuncSetAttribute(tc_tn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTnSmemBytes));
        g_attr_set_tn.done();
    }
    int64_t splits, rows;
    tn_plan(M, N, K, &splits, &rows);
    TnArgs a{};
    a.dY = dC; a.lddy = lddc; a.N = (int)N; a.X = A; a.ldx = lda; a.K = (int)K;
    a.out = (float*)ws; a.ldo = K; a.split_stride = N * K; a.M = M; a.rows_per_split = rows;
    a.nt_n = (int)ceil_div(N, BM); a.nt_k = (int)ceil_div(K, TN_BN);
    a.lbo = 8192; a.sbo = 1024;      // 64-wide MN blocks are 8 KB apart, 8-row k groups 1 KB apart (validated on B200)
    dim3 grid((unsigned)(a.nt_n * a.nt_k), (unsigned)splits);
    tc_tn_kernel<<<grid, kThreads, kTnSmemBytes, st>>>(a);
    SPGNN_LAUNCH_OK();
    reduce_splits((const float*)ws, splits, N, K, dW + k_off, lddw, st);
    return SPGNN_OK;
}


static DeviceOnce g_attr_set_tn2;

static void tn2_plan(int64_t M, int64_t N, int64_t K1, int64_t K2, int* BN, int* nt_n, int* nk1, int* nk2,
                     int64_t* splits, int64_t* rows) {
    tc::pick_bn((int)N, BN, nt_n);
    *nk1 = (int)ceil_div(K1, 256);
    *nk2 = K2 > 0 ? (int)ceil_div(K2, 256) : 0;
    const int64_t tiles = (int64_t)(*nk1 + *nk2) * *nt_n;
    int64_t want = ceil_div((int64_t)sm_count() * 4, tiles);
    const int64_t max_by_rows = ceil_div(M, 1024);
    if (want > max_by_rows) want = max_by_rows;
    if (want > 512) want = 512;
    if (want < 1) want = 1;
    *rows = ceil_div(ceil_div(M, want), tc::T2_BK) * tc::T2_BK;
    *splits = ceil_div(M, *rows);
}

int64_t tc_linear_bwd_weight2_ws_bytes(int64_t M, int64_t N, int64_t K1, int64_t K2) {
    int BN, nt_n, nk1, nk2;
    int64_t splits, rows;
    tn2_plan(M, N, K1, K2, &BN, &nt_n, &nk1, &nk2, &splits, &rows);
    return splits * N * (K1 + K2) * (int64_t)sizeof(float);
}

// dW[N, K1+K2] = dC[M,N]^T * [X1 | X2][M, K1+K2]
int tc_linear_bwd_weight2(const float* dC, int64_t lddc, const float* X1, int64_t ldx1, int64_t K1, const float* X2,
                          int64_t ldx2, int64_t K2, float* dW, int64_t lddw, int64_t M, int64_t N, void* ws,
                          cudaStream_t st) {
    if (g_attr_set_tn2.pending()) {
        SPGNN_CUDA_OK(cudaFuncSetAttribute(tc::tc_tn2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::T2_SMEM));
        g_attr_set_tn2.done();
    }
    tc::Tn2Args a{};
    int64_t splits, rows;
    tn2_plan(M, N, K1, X2 ? K2 : 0, &a.BN, &a.nt_n, &a.nk1, &a.nk2, &splits, &rows);
    a.X1 = X1; a.ldx1 = ldx1; a.K1 = (int)K1; a.X2 = X2; a.ldx2 = ldx2; a.K2 = X2 ? (int)K2 : 0;
    a.dY = dC; a.lddy = lddc; a.N = (int)N;
    const int64_t Kt = K1 + (X2 ? K2 : 0);
    a.out = (float*)ws; a.ldo = Kt; a.split_stride = N * Kt; a.M = M; a.rows_per_split = rows;
    dim3 grid((unsigned)((a.nk1 + a.nk2) * a.nt_n), (unsigned)splits);
    tc::tc_tn2_kernel<<<grid, tc::kThreads, tc::T2_SMEM, st>>>(a);
    SPGNN_LAUNCH_OK();
    reduce_splits((const float*)ws, splits, N, Kt, dW, lddw, st);
    return SPGNN_OK;
}

}  // namespace spgnn

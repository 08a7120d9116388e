// Elementwise half of a projection's backward in ONE pass (spgnn_act_bwd_planes, include/spgnn_b200.h):
//   d = mask(g) * act'(y)   ->   split-bf16 planes of d (the operand of the dX / dW GEMMs)  +  column sums of d (bias gradient)
// instead of act_bwd (read g, y; write d), split_planes (read d; write planes) and colsum (read d): 12 bytes per
// element instead of 28.  HBM-bound; one warp per row segment of 128 columns, float4 per lane.
// spgnn_colsum is the column sum alone, for the bias gradients of the paths that do not go through that pass.
#include "common.cuh"
#include "tc_ptx.cuh"

namespace spgnn {
namespace {

constexpr int kFbThreads = 256;
constexpr int64_t kFbMaxBands = 1184;     // 8 x 148 row bands at most (workspace bound)

template <bool SUM>
__global__ void __launch_bounds__(kFbThreads) act_bwd_planes_kernel(const float* __restrict__ g, int64_t ldg,
                                                                    const float* __restrict__ y, int64_t ldy, int act,
                                                                    float slope, uint32_t thr, float scale,
                                                                    uint64_t seed, __nv_bfloat16* __restrict__ hi,
                                                                    int64_t ldo, int64_t ps, int64_t M, int N,
                                                                    int64_t rows_per_band, float* __restrict__ part) {
    __shared__ float4 red[kFbThreads / 32][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int c = (blockIdx.x * 32 + lane) * 4;                 // first column of this lane's chunk
    const bool in_row = c < N;
    const int64_t r0 = (int64_t)blockIdx.y * rows_per_band;
    const int64_t r1 = r0 + rows_per_band < M ? r0 + rows_per_band : M;
    float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
    if (in_row) {
        const bool m1 = c + 1 < N, m2 = c + 2 < N, m3 = c + 3 < N;       // ragged last chunk: padding columns -> 0
        const int nch = (N + 3) >> 2;
        for (int64_t r = r0 + w; r < r1; r += kFbThreads / 32) {
            float4 d = ldg4(g + r * ldg + c);
            if (thr) {           // g is the gradient of a tensor that was dropped on its way into the consumer
                const uint64_t h = chunk_hash(seed, (uint64_t)r * (uint64_t)nch + (uint64_t)(c >> 2));
                d.x = ((uint32_t)(h) & 0xFFFFu) >= thr ? d.x * scale : 0.f;
                d.y = ((uint32_t)(h >> 16) & 0xFFFFu) >= thr ? d.y * scale : 0.f;
                d.z = ((uint32_t)(h >> 32) & 0xFFFFu) >= thr ? d.z * scale : 0.f;
                d.w = ((uint32_t)(h >> 48) & 0xFFFFu) >= thr ? d.w * scale : 0.f;
            }
            if (y) {
                const float4 yv = ldg4(y + r * ldy + c);
                d.x *= act_grad_from_out(yv.x, act, slope); d.y *= act_grad_from_out(yv.y, act, slope);
                d.z *= act_grad_from_out(yv.z, act, slope); d.w *= act_grad_from_out(yv.w, act, slope);
            }
            if (!m1) d.y = 0.f;
            if (!m2) d.z = 0.f;
            if (!m3) d.w = 0.f;
            uint32_t h0, l0, h1, l1;
            ptx::split2(d.x, d.y, h0, l0);
            ptx::split2(d.z, d.w, h1, l1);
            __nv_bfloat16* o = hi + r * ldo + c;
            *reinterpret_cast<uint2*>(o) = make_uint2(h0, h1);
            *reinterpret_cast<uint2*>(o + ps) = make_uint2(l0, l1);
            if (SUM) { sum.x += d.x; sum.y += d.y; sum.z += d.z; sum.w += d.w; }
        }
    }
    if (SUM) {
        red[w][lane] = sum;
        __syncthreads();
        if (w == 0 && in_row) {
            float4 t = red[0][lane];
#pragma unroll
            for (int q = 1; q < kFbThreads / 32; ++q) {
                const float4 u = red[q][lane];
                t.x += u.x; t.y += u.y; t.z += u.z; t.w += u.w;
            }
            float* p = part + (int64_t)blockIdx.y * N + c;
            p[0] = t.x;
            if (c + 1 < N) p[1] = t.y;
            if (c + 2 < N) p[2] = t.z;
            if (c + 3 < N) p[3] = t.w;
        }
    }
}

__global__ void sum_bands_kernel(const float* __restrict__ part, int64_t bands, int N, float* __restrict__ out) {
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < N; c += gridDim.x * blockDim.x) {
        float s = 0.f;
        for (int64_t b = 0; b < bands; ++b) s += part[b * N + c];
        out[c] = s;
    }
}

}  // namespace

// column sums: partial per block over a row band, then a fixed-order final reduce
__global__ void colsum_partial_kernel(const float* __restrict__ X, int64_t ldx, int64_t M, int64_t N,
                                      int64_t rows_per_block, float* __restrict__ part) {
    const int64_t r0 = (int64_t)blockIdx.y * rows_per_block;
    const int64_t r1 = r0 + rows_per_block < M ? r0 + rows_per_block : M;
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < N; c += (int64_t)gridDim.x * blockDim.x) {
        float s = 0.f;
        for (int64_t r = r0; r < r1; ++r) s += __ldg(X + r * ldx + c);
        part[(int64_t)blockIdx.y * N + c] = s;
    }
}
// one warp per column: lane l adds the partial rows l, l + 32, ... then a butterfly (a fixed order, hence reproducible);
// one thread per column walked 592 dependent loads: 50 us for the 22 columns of the head's bias gradient
__global__ void colsum_final_kernel(const float* __restrict__ part, int64_t nparts, int64_t N, float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t c = warp; c < N; c += nwarps) {
        float s = 0.f;
        for (int64_t p = lane; p < nparts; p += 32) s += part[p * N + c];
        s = warp_sum(s);
        if (lane == 0) out[c] = s;
    }
}

constexpr int64_t kColsumParts = 592;   // 4 x 148 row bands

}  // namespace spgnn

using namespace spgnn;

extern "C" int64_t spgnn_colsum_ws(int64_t N) { return kColsumParts * N * (int64_t)sizeof(float); }

extern "C" int spgnn_colsum(const float* X, int64_t ldx, int64_t M, int64_t N, float* out, void* ws, void* stream) {
    SPGNN_REQUIRE(X && out && ws && M > 0 && N > 0, "colsum: bad argument");
    cudaStream_t st = as_stream(stream);
    int64_t parts = M < kColsumParts ? M : kColsumParts;
    int64_t rpb = ceil_div(M, parts);
    parts = ceil_div(M, rpb);
    dim3 grid((unsigned)ceil_div(N, 128), (unsigned)parts);
    colsum_partial_kernel<<<grid, 128, 0, st>>>(X, ldx, M, N, rpb, (float*)ws);
    SPGNN_LAUNCH_OK();
    const int64_t fblocks = ceil_div(N * 32, 128), fcap = (int64_t)sm_count() * 8;
    colsum_final_kernel<<<(unsigned)(fblocks < fcap ? fblocks : fcap), 128, 0, st>>>((const float*)ws, parts, N, out);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

extern "C" int64_t spgnn_act_bwd_planes_ws(int64_t N) { return kFbMaxBands * N * (int64_t)sizeof(float) + 16; }

extern "C" int spgnn_act_bwd_planes(const float* g, int64_t ldg, const float* y, int64_t ldy, int act, float slope,
                                    float drop_p, uint64_t drop_seed, uint16_t* out_hi, int64_t ldo,
                                    int64_t plane_stride, int64_t M, int64_t N, float* colsum_out, void* ws,
                                    void* stream) {
    SPGNN_REQUIRE(g && out_hi && M > 0 && N > 0 && N < (1 << 24), "act_bwd_planes: bad argument");
    const int64_t n4 = (N + 3) / 4 * 4;
    SPGNN_REQUIRE(ldg % 4 == 0 && ldg >= n4 && ((uintptr_t)g & 15) == 0,
                  "act_bwd_planes: g rows must be 16-byte aligned and padded to a multiple of 4 columns (ld %lld)", (long long)ldg);
    SPGNN_REQUIRE(!y || (ldy % 4 == 0 && ldy >= n4 && ((uintptr_t)y & 15) == 0),
                  "act_bwd_planes: y rows must be 16-byte aligned and padded to a multiple of 4 columns (ld %lld)", (long long)ldy);
    SPGNN_REQUIRE(ldo % 4 == 0 && ldo >= n4 && plane_stride % 4 == 0 && ((uintptr_t)out_hi & 7) == 0,
                  "act_bwd_planes: output ld (%lld) must be a multiple of 4 covering the padded row", (long long)ldo);
    SPGNN_REQUIRE(!colsum_out || ws, "act_bwd_planes: column sums need the workspace");
    SPGNN_REQUIRE(drop_p >= 0.f && drop_p < 1.f, "act_bwd_planes: dropout p");
    const uint32_t thr = drop_p > 0.f ? (uint32_t)(drop_p * 65536.f + 0.5f) : 0u;
    const float scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
    if (act == SPGNN_ACT_NONE) y = nullptr;
    cudaStream_t st = as_stream(stream);
    const int64_t ncg = ceil_div(n4 / 4, 32);
    int64_t bands = ceil_div(kFbMaxBands, ncg);
    const int64_t max_bands = ceil_div(M, kFbThreads / 32);
    if (bands > max_bands) bands = max_bands;
    const int64_t rpb = ceil_div(M, bands);
    bands = ceil_div(M, rpb);
    dim3 grid((unsigned)ncg, (unsigned)bands);
    __nv_bfloat16* hi = reinterpret_cast<__nv_bfloat16*>(out_hi);
    if (colsum_out) {
        act_bwd_planes_kernel<true><<<grid, kFbThreads, 0, st>>>(g, ldg, y, ldy, act, slope, thr, scale, drop_seed, hi,
                                                                 ldo, plane_stride, M, (int)N, rpb, (float*)ws);
        SPGNN_LAUNCH_OK();
        sum_bands_kernel<<<(unsigned)ceil_div(N, 128), 128, 0, st>>>((const float*)ws, bands, (int)N, colsum_out);
        SPGNN_LAUNCH_OK();
    } else {
        act_bwd_planes_kernel<false><<<grid, kFbThreads, 0, st>>>(g, ldg, y, ldy, act, slope, thr, scale, drop_seed, hi,
                                                                  ldo, plane_stride, M, (int)N, rpb, nullptr);
        SPGNN_LAUNCH_OK();
    }
    return SPGNN_OK;
}

SPGNN_REGISTER_SALT(fused_bwd)

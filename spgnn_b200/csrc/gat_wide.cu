// Aggregate-first evaluation of the head-averaged GAT output layer (spgnn_gat_aggx_fwd / _bwd; the GEMM half is
// spgnn_wide_linear in gemm_tma.cu).  See include/spgnn_b200.h for the contract.
//
// Aggregation is linear, so for the output layer GATConv(k_in -> H x F) with H*F >> k_in the edge softmax and the
// neighbour aggregation run on the NARROW input rows:  Ax_h[v] = sum_u a[u->v,h] x[u]  (k_in columns instead of
// H*F), and the projection to H x F happens afterwards in one tcgen05 GEMM whose epilogue applies bias, activation
// and the head mean.  These kernels are the narrow half:
//   aggx_fwd      edge softmax (from the el/er projection) + Ax_h for every head + a copy of x, all as planes
//   aggx_bwd_dst  <d(Ax_h)[v], x[u]> per edge, softmax + LeakyReLU backward, d(er)
//   aggx_bwd_src  d(el), dX[u] = sum_h sum_{u->v} a * d(Ax_h)[v] + residual path + logit path, d_eler planes
//
// Same structure as gat_layer.cu: a CTA owns 128 consecutive nodes; phase A is thread-parallel over (node, head)
// and stages neighbour ids and weights of the <= 4 edges in shared memory; phase B is warp-per-node over 128-bit
// column chunks.  HBM roofline: rows are k_in (192) wide, so all three kernels together move ~6 KB per node —
// 5 % of what the projection-first layer kernels moved for the same layer.
#include <stdlib.h>
#include "layer_util.cuh"

namespace spgnn {
namespace wide {
using namespace layer;

constexpr int kNPC = 128;
constexpr int kThreads = 256;
constexpr int kMaxH = 4;

struct WArgs {
    const int32_t *in_ptr, *in_src, *out_ptr, *out_dst, *out_slot;
    int64_t N; int H, has_res;
    const __nv_bfloat16* X1; int64_t ldx1, psx1;
    const __nv_bfloat16* X2; int64_t ldx2, psx2;
    int K1, K2r;                 // K2r = K2 rounded up to 4 (plane producers write whole 4-column chunks)
    int k4;                      // k_in rounded up to 4
    const float* eler; int64_t ld_eler;
    float neg_slope, drop_p; uint64_t seed;
    float* att;
    __nv_bfloat16* XA; int64_t ldxa, psxa; int kp;
    const float* dXA; int64_t ld_dxa, head_stride;
    const float* w_eler; int64_t ld_w;
    float* ds;
    float* d_eler; int64_t ld_de;
    __nv_bfloat16* dep; int64_t ld_dep, ps_dep;
    float* dX; int64_t ld_dx;
};

__device__ __forceinline__ float keep_scale(const WArgs& a, int64_t slot, int h) {
    if (a.drop_p <= 0.f) return 1.f;
    return u01(a.seed, (uint64_t)slot * (uint64_t)a.H + (uint64_t)h) >= a.drop_p ? 1.f / (1.f - a.drop_p) : 0.f;
}
// 4 columns of the concatenated input row u (zeros in the padding up to kp)
__device__ __forceinline__ float4 load_x(const WArgs& a, int64_t u, int c) {
    if (c < a.K1) return load_planes4(a.X1 + u * a.ldx1 + c, a.psx1);
    const int c2 = c - a.K1;
    if (c2 < a.K2r) return load_planes4(a.X2 + u * a.ldx2 + c2, a.psx2);
    return zero4();
}
__device__ __forceinline__ float4 load_xa(const WArgs& a, int64_t u, int c) {      // the copy of x inside XA
    return load_planes4(a.XA + u * a.ldxa + (int64_t)a.H * a.kp + c, a.psxa);
}

struct Stage {
    int* deg;        // [kNPC]
    int* beg;        // [kNPC]
    int* nb;         // [kNPC][4]
    float* w;        // [kNPC][H][4] attention weight after dropout scaling (0 beyond the degree)
    float* at;       // [kNPC][H][4] softmax weight before dropout        (bwd-dst)
    float* lk;       // [kNPC][H][4] LeakyReLU slope factor of the logit   (bwd-dst)
    float* dd;       // [kNPC][H][4] <d(Ax_h)[v], x_j>                      (bwd-dst); del | der [kNPC][2H] (bwd-src)
    float* we;       // [2H][k4] logit projection weights                   (bwd-src)
};
__device__ __forceinline__ Stage carve(uint8_t* smem, int H) {
    Stage s;
    s.deg = reinterpret_cast<int*>(smem);
    s.beg = s.deg + kNPC;
    s.nb = s.beg + kNPC;
    s.w = reinterpret_cast<float*>(s.nb + 4 * kNPC);
    s.at = s.w + kNPC * H * 4;
    s.lk = s.at + kNPC * H * 4;
    s.dd = s.lk + kNPC * H * 4;
    s.we = s.dd + kNPC * H * 4;
    return s;
}
static size_t stage_bytes(int H, int k4) {
    return (size_t)kNPC * 6 * 4 + (size_t)kNPC * H * 4 * 4 * 4 + (size_t)2 * H * k4 * 4 + 16;
}
// the forward only stages deg | beg | nb | w (at / lk / dd / we belong to the backward): independent of k_in
static size_t stage_bytes_fwd(int H) { return (size_t)kNPC * 6 * 4 + (size_t)kNPC * H * 4 * 4 + 16; }


// Phase B of the three kernels runs LPN lanes per node (32: one warp per node; 16: two nodes per warp).  The output
// layer's input is 192 columns = 48 four-column chunks: with 32 lanes the second pass of the chunk loop leaves half the
// warp idle, with 16 lanes every pass is full.
template <int LPN>
__device__ __forceinline__ float group_sum(float v, unsigned mask) {
#pragma unroll
    for (int o = LPN / 2; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o);
    return v;
}
template <int LPN>
__device__ __forceinline__ unsigned group_mask(int lane) {
    return LPN == 32 ? 0xFFFFFFFFu : (0xFFFFu << (lane & 16));
}

// ------------------------------------------------------------------------------------------------ forward
template <int H, int LPN>
__global__ void __launch_bounds__(kThreads) aggx_fwd_kernel(const WArgs a) {
    extern __shared__ __align__(16) uint8_t smem[];
    const Stage st = carve(smem, H);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t nchunks = (a.N + kNPC - 1) / kNPC;
    const int nch = a.kp >> 2;
    for (int64_t chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
        const int64_t base = chunk * kNPC;
        // ---------------- phase A: edge softmax, one thread per (node, head)
        for (int it = threadIdx.x; it < kNPC * H; it += kThreads) {
            const int n = it / H, h = it - n * H;
            const int64_t v = base + n;
            if (v >= a.N) continue;
            const int beg = __ldg(a.in_ptr + v), deg = __ldg(a.in_ptr + v + 1) - beg;
            const float er = __ldg(a.eler + v * a.ld_eler + H + h);
            if (h == 0) { st.deg[n] = deg; st.beg[n] = beg; }
            if (deg <= 4) {
                int u[4];
                float e[4], m = -INFINITY;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    u[j] = deg > 0 ? __ldg(a.in_src + beg + min(j, deg - 1)) : (int)v;
                    e[j] = leaky(__ldg(a.eler + (int64_t)u[j] * a.ld_eler + h) + er, a.neg_slope);
                    if (j < deg) m = fmaxf(m, e[j]);
                }
                float p[4], sum = 0.f;
#pragma unroll
                for (int j = 0; j < 4; ++j) { p[j] = j < deg ? __expf(e[j] - m) : 0.f; sum += p[j]; }
                const float inv = deg > 0 ? 1.f / sum : 0.f;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float at = p[j] * inv;
                    if (j < deg) a.att[(int64_t)(beg + j) * H + h] = at;
                    st.w[(n * H + h) * 4 + j] = j < deg ? at * keep_scale(a, beg + j, h) : 0.f;
                    if (h == 0) st.nb[n * 4 + j] = u[j];
                }
            } else {
                float m = -INFINITY;
                for (int s = beg; s < beg + deg; ++s)
                    m = fmaxf(m, leaky(__ldg(a.eler + (int64_t)__ldg(a.in_src + s) * a.ld_eler + h) + er, a.neg_slope));
                float sum = 0.f;
                for (int s = beg; s < beg + deg; ++s)
                    sum += __expf(leaky(__ldg(a.eler + (int64_t)__ldg(a.in_src + s) * a.ld_eler + h) + er, a.neg_slope) - m);
                const float inv = 1.f / sum;
                for (int s = beg; s < beg + deg; ++s)
                    a.att[(int64_t)s * H + h] =
                        __expf(leaky(__ldg(a.eler + (int64_t)__ldg(a.in_src + s) * a.ld_eler + h) + er, a.neg_slope) - m) * inv;
            }
        }
        __syncthreads();
        // ---------------- phase B: Ax_h for every head + the copy of x, one warp per node
        for (int n = warp * (32 / LPN) + lane / LPN; n < kNPC; n += kThreads / LPN) {
            const int64_t v = base + n;
            if (v >= a.N) continue;
            const int gl = lane & (LPN - 1);
            const int deg = st.deg[n];
            __nv_bfloat16* orow = a.XA + v * a.ldxa;
            if (deg <= 4) {
                const int4 nb = *reinterpret_cast<const int4*>(st.nb + n * 4);
                float4 w[H];
#pragma unroll
                for (int h = 0; h < H; ++h) w[h] = *reinterpret_cast<const float4*>(st.w + (n * H + h) * 4);
                for (int ch = gl; ch < nch; ch += LPN) {
                    const int c = ch * 4;
                    const float4 x0 = load_x(a, nb.x, c), x1 = load_x(a, nb.y, c), x2 = load_x(a, nb.z, c),
                                 x3 = load_x(a, nb.w, c);
                    const float4 xv = load_x(a, v, c);
#pragma unroll
                    for (int h = 0; h < H; ++h) {
                        float4 acc = scale4(w[h].x, x0);
                        acc = fma4(w[h].y, x1, acc); acc = fma4(w[h].z, x2, acc); acc = fma4(w[h].w, x3, acc);
                        store_planes4(orow + h * a.kp + c, a.psxa, acc);
                    }
                    store_planes4(orow + H * a.kp + c, a.psxa, xv);
                }
            } else {
                const int beg = st.beg[n];
                for (int ch = gl; ch < nch; ch += LPN) {
                    const int c = ch * 4;
#pragma unroll
                    for (int h = 0; h < H; ++h) {
                        float4 acc = zero4();
                        for (int s = beg; s < beg + deg; ++s)
                            acc = fma4(a.att[(int64_t)s * H + h] * keep_scale(a, s, h), load_x(a, __ldg(a.in_src + s), c), acc);
                        store_planes4(orow + h * a.kp + c, a.psxa, acc);
                    }
                    store_planes4(orow + H * a.kp + c, a.psxa, load_x(a, v, c));
                }
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------ backward, dst side
template <int H, int LPN>
__global__ void __launch_bounds__(kThreads) aggx_bwd_dst_kernel(const WArgs a) {
    extern __shared__ __align__(16) uint8_t smem[];
    const Stage st = carve(smem, H);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t nchunks = (a.N + kNPC - 1) / kNPC;
    const int nch = a.k4 >> 2;
    for (int64_t chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
        const int64_t base = chunk * kNPC;
        for (int it = threadIdx.x; it < kNPC * H; it += kThreads) {
            const int n = it / H, h = it - n * H;
            const int64_t v = base + n;
            if (v >= a.N) continue;
            const int beg = __ldg(a.in_ptr + v), deg = __ldg(a.in_ptr + v + 1) - beg;
            if (h == 0) { st.deg[n] = deg; st.beg[n] = beg; }
            if (deg <= 4) {
                const float er = __ldg(a.eler + v * a.ld_eler + H + h);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int u = deg > 0 ? __ldg(a.in_src + beg + min(j, deg - 1)) : (int)v;
                    const float raw = __ldg(a.eler + (int64_t)u * a.ld_eler + h) + er;
                    const float at = j < deg ? __ldg(a.att + (int64_t)(beg + j) * H + h) : 0.f;
                    const int o = (n * H + h) * 4 + j;
                    st.at[o] = at;
                    st.w[o] = j < deg ? at * keep_scale(a, beg + j, h) : 0.f;
                    st.lk[o] = raw > 0.f ? 1.f : a.neg_slope;
                    if (h == 0) st.nb[n * 4 + j] = u;
                }
            }
        }
        __syncthreads();
        // ---------------- phase B: <d(Ax_h)[v], x[u_j]> for the (<= 4) in-edges of v
        for (int n = warp * (32 / LPN) + lane / LPN; n < kNPC; n += kThreads / LPN) {
            const int64_t v = base + n;
            if (v >= a.N) continue;
            const int gl = lane & (LPN - 1);
            const unsigned gm = group_mask<LPN>(lane);
            const int deg = st.deg[n];
            if (deg <= 4) {
                const int4 nb = *reinterpret_cast<const int4*>(st.nb + n * 4);
                float d[H][4];
#pragma unroll
                for (int h = 0; h < H; ++h) d[h][0] = d[h][1] = d[h][2] = d[h][3] = 0.f;
                for (int ch = gl; ch < nch; ch += LPN) {
                    const int c = ch * 4;
                    const float4 x0 = load_xa(a, nb.x, c), x1 = load_xa(a, nb.y, c), x2 = load_xa(a, nb.z, c),
                                 x3 = load_xa(a, nb.w, c);
#pragma unroll
                    for (int h = 0; h < H; ++h) {
                        const float4 g = ldg4(a.dXA + h * a.head_stride + v * a.ld_dxa + c);
                        d[h][0] += dot4(g, x0); d[h][1] += dot4(g, x1); d[h][2] += dot4(g, x2); d[h][3] += dot4(g, x3);
                    }
                }
#pragma unroll
                for (int h = 0; h < H; ++h) {
                    const float d0 = group_sum<LPN>(d[h][0], gm), d1 = group_sum<LPN>(d[h][1], gm),
                                d2 = group_sum<LPN>(d[h][2], gm), d3 = group_sum<LPN>(d[h][3], gm);
                    if (gl == 0) *reinterpret_cast<float4*>(st.dd + (n * H + h) * 4) = make_float4(d0, d1, d2, d3);
                }
            } else {
                const int beg = st.beg[n];
                for (int h = 0; h < H; ++h)
                    for (int s = beg; s < beg + deg; ++s) {
                        const int u = __ldg(a.in_src + s);
                        float dsum = 0.f;
                        for (int ch = gl; ch < nch; ch += LPN)
                            dsum += dot4(ldg4(a.dXA + h * a.head_stride + v * a.ld_dxa + ch * 4), load_xa(a, u, ch * 4));
                        dsum = group_sum<LPN>(dsum, gm);
                        if (gl == 0) a.ds[(int64_t)s * H + h] = dsum * keep_scale(a, s, h);
                    }
            }
        }
        __syncthreads();
        // ---------------- phase C: softmax + LeakyReLU backward, one thread per (node, head)
        for (int it = threadIdx.x; it < kNPC * H; it += kThreads) {
            const int n = it / H, h = it - n * H;
            const int64_t v = base + n;
            if (v >= a.N) continue;
            const int deg = st.deg[n], beg = st.beg[n];
            float der = 0.f;
            if (deg <= 4) {
                const int o = (n * H + h) * 4;
                float da[4], wsum = 0.f;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float at = st.at[o + j];
                    da[j] = at > 0.f ? st.dd[o + j] * (st.w[o + j] / at) : 0.f;
                    wsum += at * da[j];
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (j < deg) {
                        const float dsv = st.at[o + j] * (da[j] - wsum) * st.lk[o + j];
                        a.ds[(int64_t)(beg + j) * H + h] = dsv;
                        der += dsv;
                    }
                }
            } else {
                const float er = __ldg(a.eler + v * a.ld_eler + H + h);
                float wsum = 0.f;
                for (int s = beg; s < beg + deg; ++s) wsum += __ldg(a.att + (int64_t)s * H + h) * a.ds[(int64_t)s * H + h];
                for (int s = beg; s < beg + deg; ++s) {
                    const float raw = __ldg(a.eler + (int64_t)__ldg(a.in_src + s) * a.ld_eler + h) + er;
                    const float dsv = __ldg(a.att + (int64_t)s * H + h) * (a.ds[(int64_t)s * H + h] - wsum) *
                                      (raw > 0.f ? 1.f : a.neg_slope);
                    a.ds[(int64_t)s * H + h] = dsv;
                    der += dsv;
                }
            }
            a.d_eler[v * a.ld_de + H + h] = der;
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------ backward, src side
template <int H, int LPN>
__global__ void __launch_bounds__(kThreads) aggx_bwd_src_kernel(const WArgs a) {
    extern __shared__ __align__(16) uint8_t smem[];
    const Stage st = carve(smem, H);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t nchunks = (a.N + kNPC - 1) / kNPC;
    const int nch = a.k4 >> 2;
    for (int i = threadIdx.x; i < 2 * H * a.k4; i += kThreads) {
        const int r = i / a.k4, c = i - r * a.k4;
        st.we[i] = __ldg(a.w_eler + (int64_t)r * a.ld_w + c);     // packed-weight rows are padded to k4 with zeros
    }
    __syncthreads();
    for (int64_t chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
        const int64_t base = chunk * kNPC;
        for (int it = threadIdx.x; it < kNPC * H; it += kThreads) {
            const int n = it / H, h = it - n * H;
            const int64_t u = base + n;
            if (u >= a.N) continue;
            const int beg = __ldg(a.out_ptr + u), deg = __ldg(a.out_ptr + u + 1) - beg;
            if (h == 0) { st.deg[n] = deg; st.beg[n] = beg; }
            float del = 0.f;
            if (deg <= 4) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int q = beg + min(j, max(deg - 1, 0));
                    const int s = deg > 0 ? __ldg(a.out_slot + q) : 0;
                    const int v = deg > 0 ? __ldg(a.out_dst + q) : (int)u;
                    const bool on = j < deg;
                    st.w[(n * H + h) * 4 + j] = on ? __ldg(a.att + (int64_t)s * H + h) * keep_scale(a, s, h) : 0.f;
                    if (on) del += a.ds[(int64_t)s * H + h];
                    if (h == 0) st.nb[n * 4 + j] = v;
                }
            } else {
                for (int q = beg; q < beg + deg; ++q) del += a.ds[(int64_t)__ldg(a.out_slot + q) * H + h];
            }
            const float der = a.d_eler[u * a.ld_de + H + h];
            a.d_eler[u * a.ld_de + h] = del;
            st.dd[n * 2 * H + h] = del;
            st.dd[n * 2 * H + H + h] = der;
            store_planes1(a.dep + u * a.ld_dep + h, a.ps_dep, del);
            store_planes1(a.dep + u * a.ld_dep + H + h, a.ps_dep, der);
        }
        __syncthreads();
        for (int n = warp * (32 / LPN) + lane / LPN; n < kNPC; n += kThreads / LPN) {
            const int64_t u = base + n;
            if (u >= a.N) continue;
            const int gl = lane & (LPN - 1);
            const int deg = st.deg[n];
            float del[H], der[H];
#pragma unroll
            for (int h = 0; h < H; ++h) { del[h] = st.dd[n * 2 * H + h]; der[h] = st.dd[n * 2 * H + H + h]; }
            float* orow = a.dX + u * a.ld_dx;
            if (deg <= 4) {
                const int4 nb = *reinterpret_cast<const int4*>(st.nb + n * 4);
                float4 w[H];
#pragma unroll
                for (int h = 0; h < H; ++h) w[h] = *reinterpret_cast<const float4*>(st.w + (n * H + h) * 4);
                for (int ch = gl; ch < nch; ch += LPN) {
                    const int c = ch * 4;
                    float4 acc = zero4();
#pragma unroll
                    for (int h = 0; h < H; ++h) {
                        const float* gh = a.dXA + h * a.head_stride + c;
                        acc = fma4(w[h].x, ldg4(gh + (int64_t)nb.x * a.ld_dxa), acc);
                        acc = fma4(w[h].y, ldg4(gh + (int64_t)nb.y * a.ld_dxa), acc);
                        acc = fma4(w[h].z, ldg4(gh + (int64_t)nb.z * a.ld_dxa), acc);
                        acc = fma4(w[h].w, ldg4(gh + (int64_t)nb.w * a.ld_dxa), acc);
                        if (a.has_res) acc = add4(acc, ldg4(gh + u * a.ld_dxa + a.k4));
                        acc = fma4(del[h], *reinterpret_cast<const float4*>(st.we + h * a.k4 + c), acc);
                        acc = fma4(der[h], *reinterpret_cast<const float4*>(st.we + (H + h) * a.k4 + c), acc);
                    }
                    st4(orow + c, acc);
                }
            } else {
                const int beg = st.beg[n];
                for (int ch = gl; ch < nch; ch += LPN) {
                    const int c = ch * 4;
                    float4 acc = zero4();
#pragma unroll
                    for (int h = 0; h < H; ++h) {
                        const float* gh = a.dXA + h * a.head_stride + c;
                        for (int q = beg; q < beg + deg; ++q) {
                            const int s = __ldg(a.out_slot + q);
                            acc = fma4(__ldg(a.att + (int64_t)s * H + h) * keep_scale(a, s, h),
                                       ldg4(gh + (int64_t)__ldg(a.out_dst + q) * a.ld_dxa), acc);
                        }
                        if (a.has_res) acc = add4(acc, ldg4(gh + u * a.ld_dxa + a.k4));
                        acc = fma4(del[h], *reinterpret_cast<const float4*>(st.we + h * a.k4 + c), acc);
                        acc = fma4(der[h], *reinterpret_cast<const float4*>(st.we + (H + h) * a.k4 + c), acc);
                    }
                    st4(orow + c, acc);
                }
            }
        }
        __syncthreads();
    }
}

static unsigned wide_grid(int64_t N) {
    const int64_t chunks = ceil_div(N, kNPC), cap = (int64_t)sm_count() * 8;
    return (unsigned)(chunks < cap ? chunks : cap);
}

static int fill(WArgs& a, const spgnn_gat_wide* L, bool bwd) {
    SPGNN_REQUIRE(L, "gat_aggx: null descriptor");
    SPGNN_REQUIRE(L->in_ptr && L->in_src && L->X1 && L->eler && L->att && L->XA && L->N > 0, "gat_aggx: null pointer");
    SPGNN_REQUIRE(L->H == 1 || L->H == 2 || L->H == 4, "gat_aggx: H must be 1, 2 or 4 (got %d)", (int)L->H);
    SPGNN_REQUIRE(L->K1 > 0 && L->K1 % 64 == 0 && L->K2 >= 0 && (L->K2 == 0 || L->X2),
                  "gat_aggx: K1 (%d) must be a positive multiple of 64", (int)L->K1);
    const int k_in = L->K1 + L->K2;
    SPGNN_REQUIRE(L->kp % 64 == 0 && L->kp >= k_in && L->ldxa >= (int64_t)(L->H + 1) * L->kp && L->ldxa % 4 == 0 &&
                      L->psxa % 4 == 0 && ((uintptr_t)L->XA & 7) == 0,
                  "gat_aggx: XA must hold (H+1)*kp columns, kp %% 64 == 0");
    SPGNN_REQUIRE(L->ldx1 % 4 == 0 && L->psx1 % 4 == 0 && ((uintptr_t)L->X1 & 7) == 0 &&
                      (L->K2 == 0 || (L->ldx2 % 4 == 0 && L->psx2 % 4 == 0 && ((uintptr_t)L->X2 & 7) == 0 &&
                                      L->ldx2 >= (L->K2 + 3) / 4 * 4)),
                  "gat_aggx: input planes must have ld and plane stride multiples of 4");
    SPGNN_REQUIRE(L->attn_drop_p >= 0.f && L->attn_drop_p < 1.f, "gat_aggx: attention dropout p");
    a.in_ptr = L->in_ptr; a.in_src = L->in_src; a.out_ptr = L->out_ptr; a.out_dst = L->out_dst; a.out_slot = L->out_slot;
    a.N = L->N; a.H = L->H; a.has_res = L->has_res;
    a.X1 = reinterpret_cast<const __nv_bfloat16*>(L->X1); a.ldx1 = L->ldx1; a.psx1 = L->psx1;
    a.X2 = reinterpret_cast<const __nv_bfloat16*>(L->X2); a.ldx2 = L->ldx2; a.psx2 = L->psx2;
    a.K1 = L->K1; a.K2r = (L->K2 + 3) / 4 * 4; a.k4 = (k_in + 3) / 4 * 4;
    a.eler = L->eler; a.ld_eler = L->ld_eler; a.neg_slope = L->negative_slope; a.drop_p = L->attn_drop_p;
    a.seed = L->attn_seed; a.att = L->att;
    a.XA = reinterpret_cast<__nv_bfloat16*>(L->XA); a.ldxa = L->ldxa; a.psxa = L->psxa; a.kp = (int)L->kp;
    if (bwd) {
        SPGNN_REQUIRE(L->out_ptr && L->out_dst && L->out_slot && L->dXA && L->w_eler && L->ds_ws && L->d_eler &&
                          L->d_eler_planes && L->dX,
                      "gat_aggx_bwd: null pointer");
        SPGNN_REQUIRE(L->ld_dxa % 4 == 0 && L->head_stride % 4 == 0 && ((uintptr_t)L->dXA & 15) == 0 &&
                          L->ld_dxa >= (L->has_res ? 2 : 1) * a.k4,
                      "gat_aggx_bwd: dXA must be 16-byte aligned with ld %% 4 == 0 and (1+has_res)*k4 columns");
        SPGNN_REQUIRE(L->ld_dx % 4 == 0 && L->ld_dx >= a.k4 && ((uintptr_t)L->dX & 15) == 0, "gat_aggx_bwd: dX alignment");
        SPGNN_REQUIRE(L->ld_w >= a.k4, "gat_aggx_bwd: w_eler rows must be padded to k4 = %d columns", a.k4);
        SPGNN_REQUIRE(L->ld_de >= 2 * L->H && L->ld_dep >= 2 * L->H, "gat_aggx_bwd: d_eler needs 2H columns");
        a.dXA = L->dXA; a.ld_dxa = L->ld_dxa; a.head_stride = L->head_stride;
        a.w_eler = L->w_eler; a.ld_w = L->ld_w; a.ds = L->ds_ws; a.d_eler = L->d_eler; a.ld_de = L->ld_de;
        a.dep = reinterpret_cast<__nv_bfloat16*>(L->d_eler_planes); a.ld_dep = L->ld_dep; a.ps_dep = L->ps_dep;
        a.dX = L->dX; a.ld_dx = L->ld_dx;
    }
    return SPGNN_OK;
}

}  // namespace wide
}  // namespace spgnn

using namespace spgnn;
using namespace spgnn::wide;

extern "C" int64_t spgnn_gat_wide_sizeof(void) { return (int64_t)sizeof(spgnn_gat_wide); }

// NCH = four-column chunks per row: 16 lanes per node when that fills every pass of the chunk loop and 32 would not
// (profiles/r02_aggx_lanes_per_node.txt)
#define WIDE_DISPATCH_H(KERNEL, HH, NCH, ...)                                                   \
    do {                                                                                        \
        if ((NCH) % 32 != 0 && (NCH) % 16 == 0)                                                 \
            KERNEL<HH, 16><<<grid, kThreads, smem, st>>>(__VA_ARGS__);                          \
        else KERNEL<HH, 32><<<grid, kThreads, smem, st>>>(__VA_ARGS__);                         \
    } while (0)
#define WIDE_DISPATCH(KERNEL, NCH, ...)                                     \
    do {                                                                    \
        if (a.H == 1) WIDE_DISPATCH_H(KERNEL, 1, NCH, __VA_ARGS__);         \
        else if (a.H == 2) WIDE_DISPATCH_H(KERNEL, 2, NCH, __VA_ARGS__);    \
        else WIDE_DISPATCH_H(KERNEL, 4, NCH, __VA_ARGS__);                  \
        SPGNN_LAUNCH_OK();                                                  \
    } while (0)

extern "C" int spgnn_gat_aggx_fwd(const spgnn_gat_wide* L, void* stream) {
    WArgs a{};
    int rc = fill(a, L, false);
    if (rc) return rc;
    cudaStream_t st = as_stream(stream);
    const unsigned grid = wide_grid(a.N);
    const size_t smem = stage_bytes_fwd(a.H);
    WIDE_DISPATCH(aggx_fwd_kernel, a.kp >> 2, a);
    return SPGNN_OK;
}

// the most dynamic shared memory one block can opt into on sm_100
constexpr size_t kBwdSmemMax = 227 * 1024;
#define WIDE_INSTANCES(KERNEL)                                                                                 \
    (const void*)KERNEL<1, 16>, (const void*)KERNEL<1, 32>, (const void*)KERNEL<2, 16>, (const void*)KERNEL<2, 32>, \
        (const void*)KERNEL<4, 16>, (const void*)KERNEL<4, 32>
static cudaError_t set_bwd_smem() {
    const void* fns[] = {WIDE_INSTANCES(aggx_bwd_dst_kernel), WIDE_INSTANCES(aggx_bwd_src_kernel)};
    for (const void* f : fns) {
        const cudaError_t e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBwdSmemMax);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

extern "C" int spgnn_gat_aggx_bwd(const spgnn_gat_wide* L, void* stream) {
    WArgs a{};
    int rc = fill(a, L, true);
    if (rc) return rc;
    cudaStream_t st = as_stream(stream);
    const unsigned grid = wide_grid(a.N);
    const size_t smem = stage_bytes(a.H, a.k4);
    // The logit-weight stage grows with k_in: past 48 KB (H = 4 above k_in = 415) the kernels opt into more dynamic
    // shared memory, so every layer StackPlan marks wide (H*F <= 8192, k_in <= H*F / 4: at most 101 KB) trains.
    SPGNN_REQUIRE(smem <= kBwdSmemMax, "gat_aggx_bwd: k_in too large for the logit-weight stage (%zu bytes)", smem);
    static DeviceOnce attr;
    if (smem > 48 * 1024 && attr.pending()) {
        SPGNN_CUDA_OK(set_bwd_smem());
        attr.done();
    }
    WIDE_DISPATCH(aggx_bwd_dst_kernel, a.k4 >> 2, a);
    WIDE_DISPATCH(aggx_bwd_src_kernel, a.k4 >> 2, a);
    return SPGNN_OK;
}

SPGNN_REGISTER_SALT(gat_wide)

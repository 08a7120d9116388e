// Non-attention aggregations and the elementwise glue between projections:
//   spmm            weighted neighbour sum with degree norms  (GraphConv 'both', GINConv 'mean', SAGEConv 'mean'/'gcn')
//   sage_maxpool    elementwise neighbour max with arg-slot    (SAGEConv 'pool')
//   bias_act / act_bwd / concat_dropout(+bwd)
// One warp per node, lanes over 128-bit column chunks (scalar lanes when the width is not a multiple of 4).
// All HBM-bound: ~one read of x (neighbour rows hit L1/L2 inside a tree) and one write of out.
#include "common.cuh"

namespace spgnn {

constexpr int kThreads = 256;

static inline unsigned node_grid(int64_t N) {
    int64_t want = ceil_div(N, kThreads / 32);
    int64_t cap = (int64_t)sm_count() * 32;
    return (unsigned)(want < cap ? want : cap);
}
static inline unsigned elem_grid(int64_t n) {
    int64_t want = ceil_div(n, kThreads);
    int64_t cap = (int64_t)sm_count() * 16;
    if (want < 1) want = 1;
    return (unsigned)(want < cap ? want : cap);
}

template <int VEC>
struct Vec;
template <>
struct Vec<4> {
    using T = float4;
    static __device__ __forceinline__ T zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
    static __device__ __forceinline__ T ld(const float* p) { return ldg4(p); }
    static __device__ __forceinline__ void st(float* p, T v) { st4(p, v); }
    static __device__ __forceinline__ T fma(float s, T x, T a) {
        return make_float4(fmaf(s, x.x, a.x), fmaf(s, x.y, a.y), fmaf(s, x.z, a.z), fmaf(s, x.w, a.w));
    }
    template <typename Fn>
    static __device__ __forceinline__ T map(T v, Fn f) { return make_float4(f(v.x), f(v.y), f(v.z), f(v.w)); }
};
template <>
struct Vec<1> {
    using T = float;
    static __device__ __forceinline__ T zero() { return 0.f; }
    static __device__ __forceinline__ T ld(const float* p) { return __ldg(p); }
    static __device__ __forceinline__ void st(float* p, T v) { *p = v; }
    static __device__ __forceinline__ T fma(float s, T x, T a) { return fmaf(s, x, a); }
    template <typename Fn>
    static __device__ __forceinline__ T map(T v, Fn f) { return f(v); }
};

template <int VEC>
__global__ void __launch_bounds__(kThreads) spmm_kernel(const float* __restrict__ x, int64_t ldx,
                                                        const int32_t* __restrict__ ptr,
                                                        const int32_t* __restrict__ nbr,
                                                        const float* __restrict__ pre, const float* __restrict__ post,
                                                        const float* __restrict__ self_eps, int self_in,
                                                        int64_t n_self, const float* __restrict__ add, int64_t ld_add,
                                                        const float* __restrict__ bias, int act, float slope,
                                                        float* __restrict__ out, int64_t ldo, int64_t N, int F) {
    using V = Vec<VEC>;
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const float self_coef = self_eps ? 1.f + __ldg(self_eps) : 0.f;
    for (int64_t v = warp0; v < N; v += nwarps) {
        const int beg = __ldg(ptr + v), end = __ldg(ptr + v + 1);
        const float pv = post ? __ldg(post + v) : 1.f;
        const bool has_self = v < n_self;
        const float self_w = (self_in && has_self) ? (pre ? __ldg(pre + v) : 1.f) : 0.f;
        for (int col = lane * VEC; col < F; col += 32 * VEC) {
            typename V::T acc = V::zero();
            for (int s = beg; s < end; ++s) {
                const int u = __ldg(nbr + s);
                const float w = pre ? __ldg(pre + u) : 1.f;
                acc = V::fma(w, V::ld(x + (int64_t)u * ldx + col), acc);
            }
            // self term inside the norm, post-scale, self term outside it, addend, bias, activation
            if (self_w != 0.f) acc = V::fma(self_w, V::ld(x + v * ldx + col), acc);
            typename V::T r = V::fma(pv, acc, V::zero());
            if (self_eps && has_self) r = V::fma(self_coef, V::ld(x + v * ldx + col), r);
            if (add) r = V::fma(1.f, V::ld(add + v * ld_add + col), r);
            if (bias) r = V::fma(1.f, V::ld(bias + col), r);
            r = V::map(r, [&](float t) { return act_fwd(t, act, slope); });
            V::st(out + v * ldo + col, r);
        }
    }
}

__global__ void degree_norms_kernel(const int32_t* __restrict__ ptr, int64_t N, float* __restrict__ nsqrt,
                                    float* __restrict__ ninv) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
        float d = (float)(ptr[i + 1] - ptr[i]);
        d = fmaxf(d, 1.f);
        if (nsqrt) nsqrt[i] = powf(d, -0.5f);
        if (ninv) ninv[i] = 1.f / d;
    }
}

__global__ void inv_degree_kernel(const int32_t* __restrict__ ptr, int64_t N, float add, float* __restrict__ out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = 1.f / fmaxf((float)(ptr[i + 1] - ptr[i]) + add, 1.f);
}

template <int VEC>
__global__ void __launch_bounds__(kThreads) maxpool_fwd_kernel(const float* __restrict__ m, int64_t ldm,
                                                               const int32_t* __restrict__ in_ptr,
                                                               const int32_t* __restrict__ in_src,
                                                               float* __restrict__ out, int64_t ldo,
                                                               int32_t* __restrict__ arg, int64_t N, int F) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t v = warp0; v < N; v += nwarps) {
        const int beg = __ldg(in_ptr + v), end = __ldg(in_ptr + v + 1);
        for (int col = lane * VEC; col < F; col += 32 * VEC) {
            float best[VEC];
            int bs[VEC];
#pragma unroll
            for (int i = 0; i < VEC; ++i) { best[i] = -INFINITY; bs[i] = -1; }
            for (int s = beg; s < end; ++s) {
                const float* q = m + (int64_t)__ldg(in_src + s) * ldm + col;
                float val[VEC];
                if (VEC == 4) { float4 t = ldg4(q); val[0] = t.x; val[1] = t.y; val[2] = t.z; val[3] = t.w; }
                else val[0] = __ldg(q);
#pragma unroll
                for (int i = 0; i < VEC; ++i)
                    if (val[i] > best[i]) { best[i] = val[i]; bs[i] = s; }   // strict > keeps the first max
            }
#pragma unroll
            for (int i = 0; i < VEC; ++i) {
                out[v * ldo + col + i] = bs[i] >= 0 ? best[i] : 0.f;        // DGL zero-fills empty neighbourhoods
                arg[v * (int64_t)F + col + i] = bs[i];
            }
        }
    }
}

template <int VEC>
__global__ void __launch_bounds__(kThreads) maxpool_bwd_kernel(const float* __restrict__ g, int64_t ldg,
                                                               const int32_t* __restrict__ arg,
                                                               const int32_t* __restrict__ out_ptr,
                                                               const int32_t* __restrict__ out_dst,
                                                               const int32_t* __restrict__ out_slot,
                                                               float* __restrict__ dm, int64_t lddm, int64_t N, int F) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t u = warp0; u < N; u += nwarps) {
        const int beg = __ldg(out_ptr + u), end = __ldg(out_ptr + u + 1);
        for (int col = lane * VEC; col < F; col += 32 * VEC) {
            float acc[VEC];
#pragma unroll
            for (int i = 0; i < VEC; ++i) acc[i] = 0.f;
            for (int q = beg; q < end; ++q) {
                const int v = __ldg(out_dst + q);
                const int slot = __ldg(out_slot + q);
                if (VEC == 4) {
                    const int4 a4 = __ldg(reinterpret_cast<const int4*>(arg + (int64_t)v * F + col));
                    const float4 g4 = ldg4(g + (int64_t)v * ldg + col);
                    if (a4.x == slot) acc[0] += g4.x;
                    if (a4.y == slot) acc[1] += g4.y;
                    if (a4.z == slot) acc[2] += g4.z;
                    if (a4.w == slot) acc[3] += g4.w;
                } else {
                    if (__ldg(arg + (int64_t)v * F + col) == slot) acc[0] += __ldg(g + (int64_t)v * ldg + col);
                }
            }
            if (VEC == 4) st4(dm + u * lddm + col, make_float4(acc[0], acc[1], acc[2], acc[3]));
            else dm[u * lddm + col] = acc[0];
        }
    }
}

// Elementwise glue.  VEC = 4: rows are whole float4 chunks (N % 4 == 0, every ld % 4 == 0, bases 16-byte aligned).
template <int VEC>
__global__ void bias_act_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ bias, int act,
                                float slope, float* __restrict__ y, int64_t ldy, int64_t M, int64_t N) {
    const int64_t nc = N / VEC, total = M * nc;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / nc, c = (i - r * nc) * VEC;
        if (VEC == 4) {
            float4 v = ldg4(x + r * ldx + c);
            if (bias) {
                const float4 b = ldg4(bias + c);
                v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
            }
            st4(y + r * ldy + c, make_float4(act_fwd(v.x, act, slope), act_fwd(v.y, act, slope),
                                             act_fwd(v.z, act, slope), act_fwd(v.w, act, slope)));
        } else {
            float v = x[r * ldx + c];
            if (bias) v += __ldg(bias + c);
            y[r * ldy + c] = act_fwd(v, act, slope);
        }
    }
}

template <int VEC>
__global__ void act_bwd_kernel(const float* __restrict__ g, int64_t ldg, const float* __restrict__ y, int64_t ldy,
                               int act, float slope, float* __restrict__ dx, int64_t lddx, int64_t M, int64_t N) {
    const int64_t nc = N / VEC, total = M * nc;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / nc, c = (i - r * nc) * VEC;
        if (VEC == 4) {
            const float4 gv = ldg4(g + r * ldg + c), yv = ldg4(y + r * ldy + c);
            st4(dx + r * lddx + c, make_float4(gv.x * act_grad_from_out(yv.x, act, slope),
                                               gv.y * act_grad_from_out(yv.y, act, slope),
                                               gv.z * act_grad_from_out(yv.z, act, slope),
                                               gv.w * act_grad_from_out(yv.w, act, slope)));
        } else {
            dx[r * lddx + c] = g[r * ldg + c] * act_grad_from_out(y[r * ldy + c], act, slope);
        }
    }
}

// mask index = row * (K1+K2) + col  — the same element index forward and backward
template <int VEC>
__global__ void concat_dropout_kernel(const float* __restrict__ x1, int64_t ld1, int64_t K1,
                                      const float* __restrict__ x2, int64_t ld2, int64_t K2, float p, uint64_t seed,
                                      float* __restrict__ out, int64_t ldo, int64_t M) {
    const int64_t K = K1 + K2, nc = K / VEC, total = M * nc;
    const float sc = p > 0.f ? 1.f / (1.f - p) : 1.f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / nc, c = (i - r * nc) * VEC;
        if (VEC == 4) {
            float4 v = c < K1 ? ldg4(x1 + r * ld1 + c) : ldg4(x2 + r * ld2 + (c - K1));
            if (p > 0.f) {
                const uint64_t e = (uint64_t)(r * K + c);
                v.x = u01(seed, e) >= p ? v.x * sc : 0.f;
                v.y = u01(seed, e + 1) >= p ? v.y * sc : 0.f;
                v.z = u01(seed, e + 2) >= p ? v.z * sc : 0.f;
                v.w = u01(seed, e + 3) >= p ? v.w * sc : 0.f;
            }
            st4(out + r * ldo + c, v);
        } else {
            float v = c < K1 ? __ldg(x1 + r * ld1 + c) : __ldg(x2 + r * ld2 + (c - K1));
            if (p > 0.f) v = u01(seed, (uint64_t)(r * K + c)) >= p ? v * sc : 0.f;
            out[r * ldo + c] = v;
        }
    }
}

template <int VEC>
__global__ void concat_dropout_bwd_kernel(const float* __restrict__ g, int64_t ldg, int64_t K1, int64_t K2, float p,
                                          uint64_t seed, float* __restrict__ d1, int64_t ldd1,
                                          float* __restrict__ d2, int64_t ldd2, int64_t M) {
    const int64_t K = K1 + K2, nc = K / VEC, total = M * nc;
    const float sc = p > 0.f ? 1.f / (1.f - p) : 1.f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / nc, c = (i - r * nc) * VEC;
        if (VEC == 4) {
            float4 v = ldg4(g + r * ldg + c);
            if (p > 0.f) {
                const uint64_t e = (uint64_t)(r * K + c);
                v.x = u01(seed, e) >= p ? v.x * sc : 0.f;
                v.y = u01(seed, e + 1) >= p ? v.y * sc : 0.f;
                v.z = u01(seed, e + 2) >= p ? v.z * sc : 0.f;
                v.w = u01(seed, e + 3) >= p ? v.w * sc : 0.f;
            }
            if (c < K1) { if (d1) st4(d1 + r * ldd1 + c, v); }
            else if (d2) st4(d2 + r * ldd2 + (c - K1), v);
        } else {
            float v = g[r * ldg + c];
            if (p > 0.f) v = u01(seed, (uint64_t)(r * K + c)) >= p ? v * sc : 0.f;
            if (c < K1) { if (d1) d1[r * ldd1 + c] = v; }
            else if (d2) d2[r * ldd2 + (c - K1)] = v;
        }
    }
}

static inline bool vec_ok(const void* p, int64_t ld, int64_t F) { return ((uintptr_t)p & 15) == 0 && ld % 4 == 0 && F % 4 == 0; }

}  // namespace spgnn

using namespace spgnn;

extern "C" int spgnn_spmm(const float* x, int64_t ldx, const int32_t* ptr, const int32_t* nbr, const float* pre,
                          const float* post, const float* self_eps_ptr, int self_in, int64_t n_self, const float* add,
                          int64_t ld_add, const float* bias, int act, float slope, float* out, int64_t ldo, int64_t N,
                          int64_t F, void* stream) {
    SPGNN_REQUIRE(x && ptr && nbr && out && N > 0 && F > 0 && ldx >= F && ldo >= F && n_self >= 0 && n_self <= N &&
                  (!add || ld_add >= F), "spmm: bad argument");
    cudaStream_t st = as_stream(stream);
    if (vec_ok(x, ldx, F) && vec_ok(out, ldo, F) && (!bias || ((uintptr_t)bias & 15) == 0) &&
        (!add || vec_ok(add, ld_add, F)))
        spmm_kernel<4><<<node_grid(N), kThreads, 0, st>>>(x, ldx, ptr, nbr, pre, post, self_eps_ptr, self_in, n_self,
                                                          add, ld_add, bias, act, slope, out, ldo, N, (int)F);
    else
        spmm_kernel<1><<<node_grid(N), kThreads, 0, st>>>(x, ldx, ptr, nbr, pre, post, self_eps_ptr, self_in, n_self,
                                                          add, ld_add, bias, act, slope, out, ldo, N, (int)F);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

extern "C" int spgnn_degree_norms(const int32_t* ptr, int64_t N, float* norm_sqrt, float* norm_inv, void* stream) {
    SPGNN_REQUIRE(ptr && N > 0, "degree_norms: bad argument");
    degree_norms_kernel<<<elem_grid(N), kThreads, 0, as_stream(stream)>>>(ptr, N, norm_sqrt, norm_inv);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

extern "C" int spgnn_inv_degree(const int32_t* ptr, int64_t N, float add, float* out, void* stream) {
    SPGNN_REQUIRE(ptr && out && N > 0, "inv_degree: bad argument");
    inv_degree_kernel<<<elem_grid(N), kThreads, 0, as_stream(stream)>>>(ptr, N, add, out);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

extern "C" int spgnn_sage_maxpool_fwd(const float* m, int64_t ldm, const int32_t* in_ptr, const int32_t* in_src,
                                      float* out, int64_t ldo, int32_t* arg, int64_t N, int64_t F, void* stream) {
    SPGNN_REQUIRE(m && in_ptr && in_src && out && arg && N > 0 && F > 0, "sage_maxpool_fwd: bad argument");
    cudaStream_t st = as_stream(stream);
    if (vec_ok(m, ldm, F))
        maxpool_fwd_kernel<4><<<node_grid(N), kThreads, 0, st>>>(m, ldm, in_ptr, in_src, out, ldo, arg, N, (int)F);
    else
        maxpool_fwd_kernel<1><<<node_grid(N), kThreads, 0, st>>>(m, ldm, in_ptr, in_src, out, ldo, arg, N, (int)F);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

extern "C" int spgnn_sage_maxpool_bwd(const float* g, int64_t ldg, const int32_t* arg, const int32_t* out_ptr,
                                      const int32_t* out_dst, const int32_t* out_slot, float* dm, int64_t lddm,
                                      int64_t N, int64_t F, void* stream) {
    SPGNN_REQUIRE(g && arg && out_ptr && out_dst && out_slot && dm && N > 0 && F > 0, "sage_maxpool_bwd: bad argument");
    cudaStream_t st = as_stream(stream);
    if (vec_ok(g, ldg, F) && vec_ok(dm, lddm, F) && ((uintptr_t)arg & 15) == 0)
        maxpool_bwd_kernel<4><<<node_grid(N), kThreads, 0, st>>>(g, ldg, arg, out_ptr, out_dst, out_slot, dm, lddm, N, (int)F);
    else
        maxpool_bwd_kernel<1><<<node_grid(N), kThreads, 0, st>>>(g, ldg, arg, out_ptr, out_dst, out_slot, dm, lddm, N, (int)F);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

extern "C" int spgnn_bias_act(const float* x, int64_t ldx, const float* bias, int act, float slope, float* y,
                              int64_t ldy, int64_t M, int64_t N, void* stream) {
    SPGNN_REQUIRE(x && y && M > 0 && N > 0, "bias_act: bad argument");
    cudaStream_t st = as_stream(stream);
    if (vec_ok(x, ldx, N) && vec_ok(y, ldy, N) && (!bias || ((uintptr_t)bias & 15) == 0))
        bias_act_kernel<4><<<elem_grid(M * N / 4), kThreads, 0, st>>>(x, ldx, bias, act, slope, y, ldy, M, N);
    else
        bias_act_kernel<1><<<elem_grid(M * N), kThreads, 0, st>>>(x, ldx, bias, act, slope, y, ldy, M, N);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

extern "C" int spgnn_act_bwd(const float* g, int64_t ldg, const float* y, int64_t ldy, int act, float slope,
                             float* dx, int64_t lddx, int64_t M, int64_t N, void* stream) {
    SPGNN_REQUIRE(g && y && dx && M > 0 && N > 0, "act_bwd: bad argument");
    cudaStream_t st = as_stream(stream);
    if (vec_ok(g, ldg, N) && vec_ok(y, ldy, N) && vec_ok(dx, lddx, N))
        act_bwd_kernel<4><<<elem_grid(M * N / 4), kThreads, 0, st>>>(g, ldg, y, ldy, act, slope, dx, lddx, M, N);
    else
        act_bwd_kernel<1><<<elem_grid(M * N), kThreads, 0, st>>>(g, ldg, y, ldy, act, slope, dx, lddx, M, N);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

extern "C" int spgnn_concat_dropout(const float* x1, int64_t ld1, int64_t K1, const float* x2, int64_t ld2,
                                    int64_t K2, float p, uint64_t seed, float* out, int64_t ldo, int64_t M,
                                    void* stream) {
    SPGNN_REQUIRE(x1 && out && M > 0 && K1 > 0 && (K2 == 0 || x2) && p >= 0.f && p < 1.f, "concat_dropout: bad argument");
    cudaStream_t st = as_stream(stream);
    if (vec_ok(x1, ld1, K1) && (K2 == 0 || vec_ok(x2, ld2, K2)) && vec_ok(out, ldo, K1 + K2))
        concat_dropout_kernel<4><<<elem_grid(M * (K1 + K2) / 4), kThreads, 0, st>>>(x1, ld1, K1, x2, ld2, K2, p, seed, out, ldo, M);
    else
        concat_dropout_kernel<1><<<elem_grid(M * (K1 + K2)), kThreads, 0, st>>>(x1, ld1, K1, x2, ld2, K2, p, seed, out, ldo, M);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

extern "C" int spgnn_concat_dropout_bwd(const float* g, int64_t ldg, int64_t K1, int64_t K2, float p, uint64_t seed,
                                        float* d1, int64_t ldd1, float* d2, int64_t ldd2, int64_t M, void* stream) {
    SPGNN_REQUIRE(g && M > 0 && K1 > 0 && p >= 0.f && p < 1.f, "concat_dropout_bwd: bad argument");
    cudaStream_t st = as_stream(stream);
    if (vec_ok(g, ldg, K1 + K2) && K1 % 4 == 0 && (!d1 || vec_ok(d1, ldd1, K1)) && (!d2 || K2 == 0 || vec_ok(d2, ldd2, K2)))
        concat_dropout_bwd_kernel<4><<<elem_grid(M * (K1 + K2) / 4), kThreads, 0, st>>>(g, ldg, K1, K2, p, seed, d1, ldd1, d2, ldd2, M);
    else
        concat_dropout_bwd_kernel<1><<<elem_grid(M * (K1 + K2)), kThreads, 0, st>>>(g, ldg, K1, K2, p, seed, d1, ldd1, d2, ldd2, M);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

SPGNN_REGISTER_SALT(aggs)

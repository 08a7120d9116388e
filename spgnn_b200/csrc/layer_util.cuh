// Device helpers shared by the GAT layer kernels (gat_layer.cu, gat_wide.cu): float4 arithmetic, the feat_drop mask
// convention of the planes pipeline, and split-bf16 plane loads / stores.
#pragma once
#include "common.cuh"
#include "tc_ptx.cuh"

namespace spgnn {
namespace layer {
using ptx::join2;
using ptx::split2;

__device__ __forceinline__ float4 fma4(float s, float4 x, float4 acc) {
    acc.x = fmaf(s, x.x, acc.x); acc.y = fmaf(s, x.y, acc.y);
    acc.z = fmaf(s, x.z, acc.z); acc.w = fmaf(s, x.w, acc.w);
    return acc;
}
__device__ __forceinline__ float4 add4(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ float4 mul4(float4 a, float4 b) { return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w); }
__device__ __forceinline__ float4 scale4(float s, float4 a) { return make_float4(s * a.x, s * a.y, s * a.z, s * a.w); }
__device__ __forceinline__ float dot4(float4 a, float4 b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }
__device__ __forceinline__ float4 zero4() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ float4 act4(float4 p, int act) {
    return make_float4(act_fast(p.x, act), act_fast(p.y, act), act_fast(p.z, act), act_fast(p.w, act));
}
__device__ __forceinline__ float4 actgrad4(float4 y, int act) {
    return make_float4(act_grad_from_out(y.x, act, kGatLeakySlope), act_grad_from_out(y.y, act, kGatLeakySlope),
                       act_grad_from_out(y.z, act, kGatLeakySlope), act_grad_from_out(y.w, act, kGatLeakySlope));
}
__device__ __forceinline__ float leaky(float x, float slope) { return x > 0.f ? x : slope * x; }

// feat_drop of a consumer on a 4-column chunk (16 hash bits per element; same convention as spgnn_split_planes)
__device__ __forceinline__ float4 drop4(float4 v, uint32_t thr, float scale, uint64_t seed, uint64_t chunk_idx) {
    if (!thr) return v;
    const uint64_t h = chunk_hash(seed, chunk_idx);
    v.x = ((uint32_t)(h) & 0xFFFFu) >= thr ? v.x * scale : 0.f;
    v.y = ((uint32_t)(h >> 16) & 0xFFFFu) >= thr ? v.y * scale : 0.f;
    v.z = ((uint32_t)(h >> 32) & 0xFFFFu) >= thr ? v.z * scale : 0.f;
    v.w = ((uint32_t)(h >> 48) & 0xFFFFu) >= thr ? v.w * scale : 0.f;
    return v;
}
__device__ __forceinline__ void store_planes4(__nv_bfloat16* hi, int64_t ps, float4 v) {
    uint32_t h0, l0, h1, l1;
    split2(v.x, v.y, h0, l0);
    split2(v.z, v.w, h1, l1);
    *reinterpret_cast<uint2*>(hi) = make_uint2(h0, h1);
    *reinterpret_cast<uint2*>(hi + ps) = make_uint2(l0, l1);
}
__device__ __forceinline__ float4 load_planes4(const __nv_bfloat16* hi, int64_t ps) {
    const uint2 h = *reinterpret_cast<const uint2*>(hi);
    const uint2 l = *reinterpret_cast<const uint2*>(hi + ps);
    float4 v;
    join2(h.x, l.x, v.x, v.y);
    join2(h.y, l.y, v.z, v.w);
    return v;
}
__device__ __forceinline__ void store_planes1(__nv_bfloat16* hi, int64_t ps, float x) {
    const __nv_bfloat16 h = __float2bfloat16_rn(x);
    hi[0] = h;
    hi[ps] = __float2bfloat16_rn(x - __bfloat162float(h));
}

struct Sink {
    __nv_bfloat16* hi; int64_t ld, ps; int64_t nch, ch_off; uint32_t thr; float scale; uint64_t seed;
};
struct GSrc {
    const float* g; int64_t ld; int64_t nch, ch_off; uint32_t thr; float scale; uint64_t seed;
};
struct Args {
    const int32_t *in_ptr, *in_src, *out_ptr, *out_dst, *out_slot;
    int64_t N; int H, F;
    const float* Y; int64_t ldy, res_off, el_off, er_off; int res_mode, act; float neg_slope; int mean_heads;
    const float* bias; float drop_p; uint64_t seed;
    float* att;
    float* out; int64_t ldo; int n_sinks; Sink sinks[2];
    int n_g; GSrc gs[3];
    __nv_bfloat16* dY; int64_t dld, dps;
    float* g_ws; float* ds; float* dbias_ws;
};

__device__ __forceinline__ float keep_scale(const Args& a, int64_t slot, int h) {
    if (a.drop_p <= 0.f) return 1.f;
    return u01(a.seed, (uint64_t)slot * (uint64_t)a.H + (uint64_t)h) >= a.drop_p ? 1.f / (1.f - a.drop_p) : 0.f;
}

__device__ __forceinline__ void emit(const Args& a, int64_t v, int c, float4 y) {
    if (a.out) st4(a.out + v * a.ldo + c, y);
    for (int s = 0; s < a.n_sinks; ++s) {
        const Sink& k = a.sinks[s];
        const float4 d = drop4(y, k.thr, k.scale, k.seed, (uint64_t)v * (uint64_t)k.nch + (uint64_t)(k.ch_off + (c >> 2)));
        store_planes4(k.hi + v * k.ld + c, k.ps, d);
    }
}

__device__ __forceinline__ float4 load_g(const Args& a, int64_t v, int c) {
    float4 g = zero4();
    for (int s = 0; s < a.n_g; ++s) {
        const GSrc& k = a.gs[s];
        const float4 t = ldg4(k.g + v * k.ld + c);
        g = add4(g, drop4(t, k.thr, k.scale, k.seed, (uint64_t)v * (uint64_t)k.nch + (uint64_t)(k.ch_off + (c >> 2))));
    }
    return g;
}
static inline uint32_t thr_of(float p) { return p > 0.f ? (uint32_t)(p * 65536.f + 0.5f) : 0u; }

static inline int fill_common(Args& a, const spgnn_gat_layer* L) {
    SPGNN_REQUIRE(L, "gat_layer: null descriptor");
    SPGNN_REQUIRE(L->in_ptr && L->in_src && L->Y && L->att && L->N > 0 && L->H > 0 && L->H <= 8 && L->F > 0,
                  "gat_layer: bad argument (N=%lld H=%d F=%d)", (long long)L->N, (int)L->H, (int)L->F);
    SPGNN_REQUIRE(L->F % 4 == 0 && L->ldy % 4 == 0 && ((uintptr_t)L->Y & 15) == 0 && L->res_off % 4 == 0,
                  "gat_layer: F (%d), ldy (%lld) and res_off must be multiples of 4 and Y 16-byte aligned", (int)L->F,
                  (long long)L->ldy);
    SPGNN_REQUIRE(L->res_mode == 0 || L->res_mode == 1, "gat_layer: res_mode must be 0 (none) or 1 (linear, in Y)");
    SPGNN_REQUIRE(!L->bias || ((uintptr_t)L->bias & 15) == 0, "gat_layer: bias must be 16-byte aligned");
    SPGNN_REQUIRE(L->attn_drop_p >= 0.f && L->attn_drop_p < 1.f, "gat_layer: attention dropout p");
    a.in_ptr = L->in_ptr; a.in_src = L->in_src; a.out_ptr = L->out_ptr; a.out_dst = L->out_dst; a.out_slot = L->out_slot;
    a.N = L->N; a.H = L->H; a.F = L->F;
    a.Y = L->Y; a.ldy = L->ldy; a.res_off = L->res_off; a.el_off = L->el_off; a.er_off = L->er_off;
    a.res_mode = L->res_mode; a.act = L->act; a.neg_slope = L->negative_slope; a.mean_heads = L->mean_heads;
    a.bias = L->bias; a.drop_p = L->attn_drop_p; a.seed = L->attn_seed; a.att = L->att;
    return SPGNN_OK;
}

}  // namespace layer
}  // namespace spgnn

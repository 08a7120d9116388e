// SAGEConv 'lstm' reducer: the per-destination LSTM over in-edge messages, run as row prefixes of destinations
// sorted by in-degree (include/spgnn_b200.h, "SAGEConv lstm reducer").  The recurrent products H_{t-1} W_hh^T and
// their gradients are the planes GEMMs (gemm_tma.cu); the kernels here are the HBM-bound parts around them:
//   order_count / order_scatter   stable counting sort of the destinations by descending in-degree
//   cell_fwd / cell_bwd           one LSTM step over n_t rows: gather P, gates, c, h (and their gradients)
//   dp                            dP[u] = sum of the gate gradients of u's out-edges (out-CSR gather, no atomics)
// Threads own 4 hidden units of one row: the four gates of those units are four float4 column chunks (i, f, g, o).
#include "common.cuh"
#include "layer_util.cuh"

namespace spgnn {
namespace {

constexpr int kThreads = 256;
constexpr int kSortChunk = 256;
constexpr int64_t kMaxSortKeys = 12288;

using layer::load_planes4;
using layer::store_planes4;

static inline unsigned grid_for(int64_t items) {
    int64_t want = ceil_div(items, kThreads);
    int64_t cap = (int64_t)sm_count() * 16;
    if (want < 1) want = 1;
    return (unsigned)(want < cap ? want : cap);
}

__device__ __forceinline__ float sigm(float x) { return 1.f / (1.f + __expf(-x)); }

// fp32 values kept as their two 16-bit halves in the two planes of a planes buffer: the gate-gradient planes later
// written over them occupy exactly the same bytes, element by element.
__device__ __forceinline__ void store_halves4(__nv_bfloat16* hi, int64_t ps, float4 v) {
    const uint32_t a = __float_as_uint(v.x), b = __float_as_uint(v.y), c = __float_as_uint(v.z),
                   d = __float_as_uint(v.w);
    *reinterpret_cast<uint2*>(hi) = make_uint2((a >> 16) | (b & 0xFFFF0000u), (c >> 16) | (d & 0xFFFF0000u));
    *reinterpret_cast<uint2*>(hi + ps) = make_uint2((a & 0xFFFFu) | (b << 16), (c & 0xFFFFu) | (d << 16));
}
__device__ __forceinline__ float4 load_halves4(const __nv_bfloat16* hi, int64_t ps) {
    const uint2 h = *reinterpret_cast<const uint2*>(hi);
    const uint2 l = *reinterpret_cast<const uint2*>(hi + ps);
    return make_float4(__uint_as_float((h.x << 16) | (l.x & 0xFFFFu)), __uint_as_float((h.x & 0xFFFF0000u) | (l.x >> 16)),
                       __uint_as_float((h.y << 16) | (l.y & 0xFFFFu)), __uint_as_float((h.y & 0xFFFF0000u) | (l.y >> 16)));
}

__device__ __forceinline__ int sort_key(const int32_t* in_ptr, int64_t v, int64_t N, int64_t max_deg) {
    return v < N ? (int)(max_deg - (__ldg(in_ptr + v + 1) - __ldg(in_ptr + v))) : (int)(max_deg + 1);
}

__global__ void __launch_bounds__(kSortChunk) order_count_kernel(const int32_t* __restrict__ in_ptr, int64_t N,
                                                                 int64_t max_deg, int64_t* __restrict__ counts) {
    extern __shared__ int hist[];
    const int nb = (int)max_deg + 1;
    for (int i = threadIdx.x; i < nb; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    const int64_t v = (int64_t)blockIdx.x * kSortChunk + threadIdx.x;
    if (v < N) atomicAdd(&hist[sort_key(in_ptr, v, N, max_deg)], 1);
    __syncthreads();
    for (int i = threadIdx.x; i < nb; i += blockDim.x) counts[(int64_t)i * gridDim.x + blockIdx.x] = hist[i];
}

// Stable within a chunk: the warps take their turn in order, and inside a warp lanes with equal keys rank by lane.
__global__ void __launch_bounds__(kSortChunk) order_scatter_kernel(const int32_t* __restrict__ in_ptr, int64_t N,
                                                                   int64_t max_deg, const int64_t* __restrict__ offs,
                                                                   int32_t* __restrict__ perm,
                                                                   int32_t* __restrict__ rank) {
    extern __shared__ int hist[];
    const int nb = (int)max_deg + 2;
    for (int i = threadIdx.x; i < nb; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    const int64_t v = (int64_t)blockIdx.x * kSortChunk + threadIdx.x;
    const int key = sort_key(in_ptr, v, N, max_deg);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned peers = __match_any_sync(0xFFFFFFFFu, key);
    const int below = __popc(peers & ((1u << lane) - 1u));
    for (int w = 0; w < kSortChunk / 32; ++w) {
        if (warp == w) {
            if (v < N) {
                const int64_t pos = offs[(int64_t)key * gridDim.x + blockIdx.x] + hist[key] + below;
                perm[pos] = (int32_t)v;
                rank[v] = (int32_t)pos;
            }
            __syncwarp();
            if (below == 0) hist[key] += __popc(peers);
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(kThreads) cell_fwd_kernel(int t, int64_t n_t, int64_t n_next,
                                                            const int32_t* __restrict__ perm,
                                                            const int32_t* __restrict__ in_ptr,
                                                            const int32_t* __restrict__ in_src,
                                                            const float* __restrict__ P, int64_t ldp,
                                                            const float* __restrict__ R, int64_t ldr,
                                                            __nv_bfloat16* __restrict__ gates, int64_t ldg, int64_t psg,
                                                            const float* __restrict__ c_prev, float* __restrict__ c_cur,
                                                            __nv_bfloat16* __restrict__ h_next, int64_t ldh, int64_t psh,
                                                            float* __restrict__ out, int64_t ldo, int D) {
    const int nc = D / 4;
    const int64_t total = n_t * nc;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / nc;
        const int c = (int)(i - r * nc) * 4;
        const int v = __ldg(perm + r);
        const int u = __ldg(in_src + __ldg(in_ptr + v) + t);
        const float* p = P + (int64_t)u * ldp + c;
        float4 gi = ldg4(p), gf = ldg4(p + D), gg = ldg4(p + 2 * D), go = ldg4(p + 3 * D);
        if (R) {
            const float* q = R + r * ldr + c;
            gi = layer::add4(gi, ldg4(q)); gf = layer::add4(gf, ldg4(q + D));
            gg = layer::add4(gg, ldg4(q + 2 * D)); go = layer::add4(go, ldg4(q + 3 * D));
        }
        gi = make_float4(sigm(gi.x), sigm(gi.y), sigm(gi.z), sigm(gi.w));
        gf = make_float4(sigm(gf.x), sigm(gf.y), sigm(gf.z), sigm(gf.w));
        gg = make_float4(tanhf(gg.x), tanhf(gg.y), tanhf(gg.z), tanhf(gg.w));
        go = make_float4(sigm(go.x), sigm(go.y), sigm(go.z), sigm(go.w));
        const float4 cp = c_prev ? ldg4(c_prev + r * D + c) : layer::zero4();
        const float4 cn = make_float4(fmaf(gf.x, cp.x, gi.x * gg.x), fmaf(gf.y, cp.y, gi.y * gg.y),
                                      fmaf(gf.z, cp.z, gi.z * gg.z), fmaf(gf.w, cp.w, gi.w * gg.w));
        const float4 h = make_float4(go.x * tanhf(cn.x), go.y * tanhf(cn.y), go.z * tanhf(cn.z), go.w * tanhf(cn.w));
        __nv_bfloat16* gr = gates + r * ldg + c;
        store_halves4(gr, psg, gi);
        store_halves4(gr + D, psg, gf);
        store_halves4(gr + 2 * D, psg, gg);
        store_halves4(gr + 3 * D, psg, go);
        st4(c_cur + r * D + c, cn);
        if (r < n_next) store_planes4(h_next + r * ldh + c, psh, h);
        else st4(out + (int64_t)v * ldo + c, h);
    }
}

__global__ void __launch_bounds__(kThreads) cell_bwd_kernel(int t, int64_t n_t, int64_t n_next,
                                                            const int32_t* __restrict__ perm,
                                                            const float* __restrict__ g_out, int64_t ldgo,
                                                            const float* __restrict__ dh_rec, int64_t ldr,
                                                            float* __restrict__ dcc,
                                                            __nv_bfloat16* __restrict__ gates, int64_t ldg, int64_t psg,
                                                            const float* __restrict__ c_prev,
                                                            const float* __restrict__ c_cur, int D) {
    const int nc = D / 4;
    const int64_t total = n_t * nc;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / nc;
        const int c = (int)(i - r * nc) * 4;
        const bool cont = r < n_next;
        const float4 dh = cont ? ldg4(dh_rec + r * ldr + c) : ldg4(g_out + (int64_t)__ldg(perm + r) * ldgo + c);
        __nv_bfloat16* gr = gates + r * ldg + c;
        const float4 gi = load_halves4(gr, psg), gf = load_halves4(gr + D, psg);
        const float4 gg = load_halves4(gr + 2 * D, psg), go = load_halves4(gr + 3 * D, psg);
        const float4 cn = ldg4(c_cur + r * D + c);
        const float4 cp = t > 0 ? ldg4(c_prev + r * D + c) : layer::zero4();
        const float4 dcn = cont ? *reinterpret_cast<const float4*>(dcc + r * D + c) : layer::zero4();
        float dci[4], dgi[4], dgf[4], dgg[4], dgo[4];
        const float vi[4] = {gi.x, gi.y, gi.z, gi.w}, vf[4] = {gf.x, gf.y, gf.z, gf.w};
        const float vg[4] = {gg.x, gg.y, gg.z, gg.w}, vo[4] = {go.x, go.y, go.z, go.w};
        const float vc[4] = {cn.x, cn.y, cn.z, cn.w}, vp[4] = {cp.x, cp.y, cp.z, cp.w};
        const float vdh[4] = {dh.x, dh.y, dh.z, dh.w}, vdc[4] = {dcn.x, dcn.y, dcn.z, dcn.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float tc = tanhf(vc[k]);
            const float dc = fmaf(vdh[k] * vo[k], 1.f - tc * tc, vdc[k]);
            dci[k] = dc * vf[k];
            dgi[k] = dc * vg[k] * vi[k] * (1.f - vi[k]);
            dgf[k] = dc * vp[k] * vf[k] * (1.f - vf[k]);
            dgg[k] = dc * vi[k] * (1.f - vg[k] * vg[k]);
            dgo[k] = vdh[k] * tc * vo[k] * (1.f - vo[k]);
        }
        if (t > 0) *reinterpret_cast<float4*>(dcc + r * D + c) = make_float4(dci[0], dci[1], dci[2], dci[3]);
        store_planes4(gr, psg, make_float4(dgi[0], dgi[1], dgi[2], dgi[3]));
        store_planes4(gr + D, psg, make_float4(dgf[0], dgf[1], dgf[2], dgf[3]));
        store_planes4(gr + 2 * D, psg, make_float4(dgg[0], dgg[1], dgg[2], dgg[3]));
        store_planes4(gr + 3 * D, psg, make_float4(dgo[0], dgo[1], dgo[2], dgo[3]));
    }
}

// One warp per source node, lanes over 4-column chunks of the 4D gate columns.
__global__ void __launch_bounds__(kThreads) dp_kernel(const __nv_bfloat16* __restrict__ dG, int64_t ldg, int64_t psg,
                                                      const int64_t* __restrict__ off,
                                                      const int32_t* __restrict__ rank,
                                                      const int32_t* __restrict__ in_ptr,
                                                      const int32_t* __restrict__ out_ptr,
                                                      const int32_t* __restrict__ out_dst,
                                                      const int32_t* __restrict__ out_slot, float* __restrict__ dP,
                                                      int64_t lddp, int64_t n_src, int G) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t u = warp0; u < n_src; u += nwarps) {
        const int beg = __ldg(out_ptr + u), end = __ldg(out_ptr + u + 1);
        for (int col = lane * 4; col < G; col += 128) {
            float4 acc = layer::zero4();
            for (int q = beg; q < end; ++q) {
                const int v = __ldg(out_dst + q);
                const int t = __ldg(out_slot + q) - __ldg(in_ptr + v);
                const int64_t row = __ldg(off + t) + __ldg(rank + v);
                acc = layer::add4(acc, load_planes4(dG + row * ldg + col, psg));
            }
            st4(dP + u * lddp + col, acc);
        }
    }
}

}  // namespace
}  // namespace spgnn

using namespace spgnn;

static inline bool al16(const void* p) { return ((uintptr_t)p & 15) == 0; }

extern "C" int spgnn_lstm_order_count(const int32_t* in_ptr, int64_t N, int64_t max_deg, int64_t* counts,
                                      void* stream) {
    SPGNN_REQUIRE(in_ptr && counts && N > 0 && max_deg >= 0, "lstm_order_count: bad argument");
    SPGNN_REQUIRE(max_deg < kMaxSortKeys, "lstm_order_count: in-degree above the sort's key range");
    const unsigned chunks = (unsigned)ceil_div(N, kSortChunk);
    order_count_kernel<<<chunks, kSortChunk, (size_t)(max_deg + 1) * sizeof(int), as_stream(stream)>>>(
        in_ptr, N, max_deg, counts);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

extern "C" int spgnn_lstm_order_scatter(const int32_t* in_ptr, int64_t N, int64_t max_deg, const int64_t* offs,
                                        int32_t* perm, int32_t* rank, void* stream) {
    SPGNN_REQUIRE(in_ptr && offs && perm && rank && N > 0 && max_deg >= 0, "lstm_order_scatter: bad argument");
    SPGNN_REQUIRE(max_deg < kMaxSortKeys, "lstm_order_scatter: in-degree above the sort's key range");
    // max_deg + 2 keys (the padding lanes of the last chunk take key max_deg + 1): at max_deg = kMaxSortKeys - 1 that
    // is 4 bytes over the 48 KB a launch gets without opting in
    static DeviceOnce attr;
    if (attr.pending()) {
        SPGNN_CUDA_OK(cudaFuncSetAttribute(order_scatter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)((kMaxSortKeys + 1) * sizeof(int))));
        attr.done();
    }
    const unsigned chunks = (unsigned)ceil_div(N, kSortChunk);
    order_scatter_kernel<<<chunks, kSortChunk, (size_t)(max_deg + 2) * sizeof(int), as_stream(stream)>>>(
        in_ptr, N, max_deg, offs, perm, rank);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

extern "C" int spgnn_lstm_cell_fwd(int64_t t, int64_t n_t, int64_t n_next, const int32_t* perm, const int32_t* in_ptr,
                                   const int32_t* in_src, const float* P, int64_t ldp, const float* R, int64_t ldr,
                                   uint16_t* gates, int64_t ldg, int64_t psg, const float* c_prev, float* c_cur,
                                   uint16_t* h_next, int64_t ldh, int64_t psh, float* out, int64_t ldo, int64_t D,
                                   void* stream) {
    SPGNN_REQUIRE(perm && in_ptr && in_src && P && gates && c_cur && out && n_t > 0 && D > 0 && D % 4 == 0 &&
                  t >= 0 && n_next >= 0 && n_next <= n_t && (t == 0 || (R && c_prev)) && (n_next == 0 || h_next),
                  "lstm_cell_fwd: bad argument");
    SPGNN_REQUIRE(al16(P) && ldp % 4 == 0 && (!R || (al16(R) && ldr % 4 == 0)) && ldg % 8 == 0 && psg % 8 == 0 &&
                  al16(gates) && (!h_next || (ldh % 8 == 0 && psh % 8 == 0 && al16(h_next))) && al16(out) &&
                  ldo % 4 == 0 && al16(c_cur) && (!c_prev || al16(c_prev)), "lstm_cell_fwd: operands not 16-byte aligned");
    cell_fwd_kernel<<<grid_for(n_t * (D / 4)), kThreads, 0, as_stream(stream)>>>(
        (int)t, n_t, n_next, perm, in_ptr, in_src, P, ldp, R, ldr, reinterpret_cast<__nv_bfloat16*>(gates), ldg, psg,
        c_prev, c_cur, reinterpret_cast<__nv_bfloat16*>(h_next), ldh, psh, out, ldo, (int)D);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

extern "C" int spgnn_lstm_cell_bwd(int64_t t, int64_t n_t, int64_t n_next, const int32_t* perm, const float* g_out,
                                   int64_t ldgo, const float* dh_rec, int64_t ldr, float* dc, uint16_t* gates,
                                   int64_t ldg, int64_t psg, const float* c_prev, const float* c_cur, int64_t D,
                                   void* stream) {
    SPGNN_REQUIRE(perm && g_out && gates && c_cur && n_t > 0 && D > 0 && D % 4 == 0 && t >= 0 && n_next >= 0 &&
                  n_next <= n_t && (t == 0 || (c_prev && dc)) && (n_next == 0 || (dh_rec && dc)),
                  "lstm_cell_bwd: bad argument");
    SPGNN_REQUIRE(al16(g_out) && ldgo % 4 == 0 && (!dh_rec || (al16(dh_rec) && ldr % 4 == 0)) && (!dc || al16(dc)) &&
                  al16(gates) && ldg % 8 == 0 && psg % 8 == 0 && al16(c_cur) && (!c_prev || al16(c_prev)),
                  "lstm_cell_bwd: operands not 16-byte aligned");
    cell_bwd_kernel<<<grid_for(n_t * (D / 4)), kThreads, 0, as_stream(stream)>>>(
        (int)t, n_t, n_next, perm, g_out, ldgo, dh_rec, ldr, dc, reinterpret_cast<__nv_bfloat16*>(gates), ldg, psg,
        c_prev, c_cur, (int)D);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

extern "C" int spgnn_lstm_dp(const uint16_t* dgates, int64_t ldg, int64_t psg, const int64_t* off, const int32_t* rank,
                             const int32_t* in_ptr, const int32_t* out_ptr, const int32_t* out_dst,
                             const int32_t* out_slot, float* dP, int64_t lddp, int64_t n_src, int64_t D, void* stream) {
    SPGNN_REQUIRE(dgates && off && rank && in_ptr && out_ptr && out_dst && out_slot && dP && n_src > 0 && D > 0 &&
                  D % 4 == 0 && al16(dgates) && ldg % 8 == 0 && psg % 8 == 0 && al16(dP) && lddp % 4 == 0 &&
                  lddp >= 4 * D, "lstm_dp: bad argument");
    int64_t want = ceil_div(n_src, kThreads / 32), cap = (int64_t)sm_count() * 32;
    dp_kernel<<<(unsigned)(want < cap ? want : cap), kThreads, 0, as_stream(stream)>>>(
        reinterpret_cast<const __nv_bfloat16*>(dgates), ldg, psg, off, rank, in_ptr, out_ptr, out_dst, out_slot, dP,
        lddp, n_src, (int)(4 * D));
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

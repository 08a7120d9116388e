// Fused GAT edge-softmax + neighbour aggregation + residual + bias + activation (+ head mean), forward and
// backward.  One warp per node; lanes own 128-bit column chunks, so every global access of a row is a run of
// coalesced float4s.  Airway trees have in-degree <= 4 (incl. the self loop) and the nodes of a tree are stored
// contiguously, so neighbour rows are re-read from L1/L2 and DRAM traffic stays ~one pass over Y and out.
//
// HBM roofline: algorithmic bytes per node fwd = 4*(HF_z + HF_res + 2H + W_out) (+ indices), see DESIGN.md.
#include "common.cuh"

namespace spgnn {

constexpr int kAggThreads = 256;
constexpr int kMaxCh = 8;   // float4 chunks per lane per head in backward: F <= 32*4*8 = 1024

struct GatArgs {
    const float* Y; int64_t ldy; int64_t res_off, el_off, er_off;
    int res_mode; const float* xres; int64_t ldxres; int xres_cols;
    const float* bias; int act; float neg_slope; int mean_heads;
    float drop_p; uint64_t seed;
    const int32_t* in_ptr; const int32_t* in_src;
    const int32_t* out_ptr; const int32_t* out_dst; const int32_t* out_slot;
    int64_t N; int H; int F;
    // forward
    float* out; int64_t ldo; float* att;
    // backward
    const float* g_out; int64_t ldg; const float* out_saved; const float* att_in;
    float* dY; float* G; int64_t ldG; float* dxres; float* ds;
    int skip_fast;   // general kernels: leave nodes with 1..4 in/out-edges to the fast kernels
};

__device__ __forceinline__ float keep_scale(const GatArgs& a, int64_t slot, int h) {
    if (a.drop_p <= 0.f) return 1.f;
    return u01(a.seed, (uint64_t)slot * (uint64_t)a.H + (uint64_t)h) >= a.drop_p ? 1.f / (1.f - a.drop_p) : 0.f;
}

__device__ __forceinline__ float leaky(float x, float slope) { return x > 0.f ? x : slope * x; }

__device__ __forceinline__ float edge_logit(const GatArgs& a, int u, float er, int h) {
    return leaky(__ldg(a.Y + (int64_t)u * a.ldy + a.el_off + h) + er, a.neg_slope);
}

// softmax over the in-edges of v for head h (DGL edge_softmax: max-subtracted); writes att[slot*H+h]
__device__ __forceinline__ void edge_softmax_warp(const GatArgs& a, int64_t v, int h, int beg, int end, int lane) {
    const float er = __ldg(a.Y + v * a.ldy + a.er_off + h);
    float m = -INFINITY;
    for (int s = beg + lane; s < end; s += 32) m = fmaxf(m, edge_logit(a, __ldg(a.in_src + s), er, h));
    m = warp_max(m);
    float sum = 0.f;
    for (int s = beg + lane; s < end; s += 32) sum += expf(edge_logit(a, __ldg(a.in_src + s), er, h) - m);
    sum = warp_sum(sum);
    const float inv = 1.f / sum;
    for (int s = beg + lane; s < end; s += 32)
        a.att[(int64_t)s * a.H + h] = expf(edge_logit(a, __ldg(a.in_src + s), er, h) - m) * inv;
}

__device__ __forceinline__ float4 fma4(float s, float4 x, float4 acc) {
    acc.x = fmaf(s, x.x, acc.x); acc.y = fmaf(s, x.y, acc.y);
    acc.z = fmaf(s, x.z, acc.z); acc.w = fmaf(s, x.w, acc.w);
    return acc;
}
__device__ __forceinline__ float4 add4(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ float4 mul4(float4 a, float4 b) { return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w); }
__device__ __forceinline__ float4 scale4(float s, float4 a) { return make_float4(s * a.x, s * a.y, s * a.z, s * a.w); }
__device__ __forceinline__ float dot4(float4 a, float4 b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }
__device__ __forceinline__ float4 act4(float4 p, int act) {
    return make_float4(act_fast(p.x, act), act_fast(p.y, act), act_fast(p.z, act), act_fast(p.w, act));
}
__device__ __forceinline__ float4 actgrad4(float4 y, int act) {
    return make_float4(act_grad_from_out(y.x, act, kGatLeakySlope), act_grad_from_out(y.y, act, kGatLeakySlope),
                       act_grad_from_out(y.z, act, kGatLeakySlope), act_grad_from_out(y.w, act, kGatLeakySlope));
}

// pre-activation chunk for (v, h, col): sum_j a_drop_j * z[u_j] + residual + bias.   att: plain (coherent) loads —
// in forward the values were written by this same warp just before (ordered by __syncwarp).
__device__ __forceinline__ float4 pre_chunk(const GatArgs& a, const float* att, int64_t v, int h, int col, int beg,
                                            int end) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    const int hc = h * a.F + col;
    for (int s = beg; s < end; ++s) {
        const int u = __ldg(a.in_src + s);
        const float w = att[(int64_t)s * a.H + h] * keep_scale(a, s, h);
        acc = fma4(w, ldg4(a.Y + (int64_t)u * a.ldy + hc), acc);
    }
    if (a.res_mode == 1) acc = add4(acc, ldg4(a.Y + v * a.ldy + a.res_off + hc));
    else if (a.res_mode == 2) acc = add4(acc, ldg4(a.xres + v * a.ldxres + (hc % a.xres_cols)));
    if (a.bias) acc = add4(acc, ldg4(a.bias + hc));
    return acc;
}

// Fast-path helper: attention weights (after dropout scaling) and source ids of up to 4 in-edges, warp-uniform.
struct Edge4 {
    int u[4];
    float w[4];
};
__device__ __forceinline__ Edge4 load_edges4(const GatArgs& a, const float* att, int beg, int deg, int h) {
    Edge4 e;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const bool on = j < deg;
        e.u[j] = on ? __ldg(a.in_src + beg + j) : 0;
        e.w[j] = on ? att[(int64_t)(beg + j) * a.H + h] * keep_scale(a, beg + j, h) : 0.f;
    }
    return e;
}
// sum_j w_j * z[u_j, h, col..col+3] with the (<= 4) row loads issued back to back
__device__ __forceinline__ float4 gather4(const GatArgs& a, const Edge4& e, int deg, int hc) {
    float4 z[4];
#pragma unroll
    for (int j = 0; j < 4; ++j)
        z[j] = j < deg ? ldg4(a.Y + (int64_t)e.u[j] * a.ldy + hc) : make_float4(0.f, 0.f, 0.f, 0.f);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int j = 0; j < 4; ++j) acc = fma4(e.w[j], z[j], acc);
    return acc;
}
__device__ __forceinline__ float4 add_res_bias(const GatArgs& a, float4 acc, int64_t v, int hc) {
    if (a.res_mode == 1) acc = add4(acc, ldg4(a.Y + v * a.ldy + a.res_off + hc));
    else if (a.res_mode == 2) acc = add4(acc, ldg4(a.xres + v * a.ldxres + (hc % a.xres_cols)));
    if (a.bias) acc = add4(acc, ldg4(a.bias + hc));
    return acc;
}

// ------------------------------------------------------------------------------------------------------------
// Fast path: in-degree <= 4 and H <= 2 (every airway-tree node: <= 3 neighbours + the self loop).
// Lanes 0..7 own one (edge j = lane & 3, head h = lane >> 2) pair for the softmax; everything is then broadcast
// with shuffles, neighbour rows are addressed through 4 precomputed row pointers (edges beyond the degree alias the
// last real edge with weight 0, so the row loads need no predication) and issued back to back.
// ------------------------------------------------------------------------------------------------------------
template <int H>
struct Nbr4 {
    const float* row[4];     // Y rows of the (<= 4) sources
    float w[H][4];           // attention weights after dropout scaling, 0 beyond the degree
    float att[H][4];         // softmax weights before dropout
    int u[4];
};

// forward: computes the edge softmax from el/er, optionally writes att[]
template <int H, bool kWriteAtt>
__device__ __forceinline__ Nbr4<H> softmax4(const GatArgs& a, int64_t v, int beg, int deg, int lane, float* att_out) {
    const int j = lane & 3, h = min((lane >> 2) & 1, H - 1);
    const int s = beg + min(j, deg - 1);
    const int u = __ldg(a.in_src + s);
    const float raw = __ldg(a.Y + (int64_t)u * a.ldy + a.el_off + h) + __ldg(a.Y + v * a.ldy + a.er_off + h);
    const float e = leaky(raw, a.neg_slope);
    const bool valid = j < deg;
    float m = valid ? e : -INFINITY;
    m = fmaxf(m, __shfl_xor_sync(kFull, m, 1));
    m = fmaxf(m, __shfl_xor_sync(kFull, m, 2));
    const float p = valid ? __expf(e - m) : 0.f;
    float sum = p + __shfl_xor_sync(kFull, p, 1);
    sum += __shfl_xor_sync(kFull, sum, 2);
    const float att = p / sum;
    if (kWriteAtt && valid && lane < 4 * H) att_out[(int64_t)s * H + h] = att;
    const float w = att * keep_scale(a, s, h);
    Nbr4<H> n;
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
        n.u[jj] = __shfl_sync(kFull, u, jj);
        n.row[jj] = a.Y + (int64_t)n.u[jj] * a.ldy;
#pragma unroll
        for (int hh = 0; hh < H; ++hh) {
            n.w[hh][jj] = __shfl_sync(kFull, w, jj + 4 * hh);
            n.att[hh][jj] = __shfl_sync(kFull, att, jj + 4 * hh);
        }
    }
    return n;
}

template <int H>
__device__ __forceinline__ float4 gather_rows(const Nbr4<H>& n, int h, int hc, float4 (&z)[4]) {
#pragma unroll
    for (int j = 0; j < 4; ++j) z[j] = ldg4(n.row[j] + hc);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int j = 0; j < 4; ++j) acc = fma4(n.w[h][j], z[j], acc);
    return acc;
}

template <int H>
__device__ __forceinline__ void fwd_node_fast(const GatArgs& a, int64_t v, int beg, int deg, int lane) {
    const Nbr4<H> n = softmax4<H, true>(a, v, beg, deg, lane, a.att);
    const float inv_h = 1.f / (float)H;
    float* orow = a.out + v * a.ldo;
    for (int col = lane * 4; col < a.F; col += 128) {
        float4 y[H];
#pragma unroll
        for (int h = 0; h < H; ++h) {
            float4 z[4];
            y[h] = act4(add_res_bias(a, gather_rows<H>(n, h, h * a.F + col, z), v, h * a.F + col), a.act);
        }
        if (a.mean_heads) {
            float4 m = y[0];
#pragma unroll
            for (int h = 1; h < H; ++h) m = add4(m, y[h]);
            st4(orow + col, scale4(inv_h, m));
        } else {
#pragma unroll
            for (int h = 0; h < H; ++h) st4(orow + h * a.F + col, y[h]);
        }
    }
}

// backward, destination side: one pass over the chunks computes g (and stores it), and the 4 x H dot products
// <g, z[u_j]> from the SAME z registers that the (mean-mode) recomputation of the pre-activation used.
template <int H>
__device__ __forceinline__ void bwd_dst_node_fast(const GatArgs& a, int64_t v, int beg, int deg, int lane) {
    const Nbr4<H> n = softmax4<H, false>(a, v, beg, deg, lane, nullptr);   // recomputed: same values as forward
    const float inv_h = 1.f / (float)H;
    float d[H][4];
#pragma unroll
    for (int h = 0; h < H; ++h)
#pragma unroll
        for (int j = 0; j < 4; ++j) d[h][j] = 0.f;
    for (int col = lane * 4; col < a.F; col += 128) {
        float4 idsum = make_float4(0.f, 0.f, 0.f, 0.f);
        float4 gom;
        if (a.mean_heads) gom = scale4(inv_h, ldg4(a.g_out + v * a.ldg + col));
#pragma unroll
        for (int h = 0; h < H; ++h) {
            const int hc = h * a.F + col;
            float4 z[4];
            float4 go, y;
            if (a.mean_heads) {
                y = act4(add_res_bias(a, gather_rows<H>(n, h, hc, z), v, hc), a.act);
                go = gom;
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) z[j] = ldg4(n.row[j] + hc);
                go = ldg4(a.g_out + v * a.ldg + hc);
                y = ldg4(a.out_saved + v * a.ldo + hc);
            }
            const float4 gq = mul4(go, actgrad4(y, a.act));
            st4(a.G + v * a.ldG + hc, gq);
            if (a.res_mode == 2) {
                if (a.xres_cols == a.F) idsum = add4(idsum, gq);
                else st4(a.dxres + v * a.ldxres + hc, gq);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) d[h][j] += dot4(gq, z[j]);
        }
        if (a.res_mode == 2 && a.xres_cols == a.F) st4(a.dxres + v * a.ldxres + col, idsum);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
        for (int h = 0; h < H; ++h)
#pragma unroll
            for (int j = 0; j < 4; ++j) d[h][j] += __shfl_xor_sync(kFull, d[h][j], o);
    // softmax + LeakyReLU backward, redundantly on every lane (<= 4 edges x H heads)
#pragma unroll
    for (int h = 0; h < H; ++h) {
        const float er = __ldg(a.Y + v * a.ldy + a.er_off + h);
        float da[4], wsum = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            // d(a_drop)/d(a) = keep/(1-p) = w/att (0 when dropped or beyond the degree)
            const float ks = n.att[h][j] > 0.f ? n.w[h][j] / n.att[h][j] : 0.f;
            da[j] = j < deg ? d[h][j] * ks : 0.f;
            wsum += n.att[h][j] * da[j];
        }
        float der = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j < deg) {
                const float raw = __ldg(n.row[j] + a.el_off + h) + er;
                const float dsv = n.att[h][j] * (da[j] - wsum) * (raw > 0.f ? 1.f : a.neg_slope);
                if (lane == j) a.ds[(int64_t)(beg + j) * H + h] = dsv;
                der += dsv;
            }
        }
        if (lane == 0) a.dY[v * a.ldy + a.er_off + h] = der;
    }
}

// backward, source side: dz[u,h,:] = sum over out-edges (u->v) of a_drop * g[v,h,:];  del[u,h] = sum of ds
template <int H>
__device__ __forceinline__ void bwd_src_node_fast(const GatArgs& a, int64_t u, int beg, int deg, int lane) {
    const int j = lane & 3, h = min((lane >> 2) & 1, H - 1);
    const int qidx = beg + min(j, deg - 1);
    const int s = __ldg(a.out_slot + qidx);
    const int v = __ldg(a.out_dst + qidx);
    const bool valid = j < deg;
    const float w = valid ? __ldg(a.att_in + (int64_t)s * H + h) * keep_scale(a, s, h) : 0.f;
    float dsv = valid ? __ldg(a.ds + (int64_t)s * H + h) : 0.f;
    dsv += __shfl_xor_sync(kFull, dsv, 1);
    dsv += __shfl_xor_sync(kFull, dsv, 2);
    if (j == 0 && lane < 4 * H) a.dY[u * a.ldy + a.el_off + h] = dsv;
    const float* grow[4];
    float wj[H][4];
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
        grow[jj] = a.G + (int64_t)__shfl_sync(kFull, v, jj) * a.ldG;
#pragma unroll
        for (int hh = 0; hh < H; ++hh) wj[hh][jj] = __shfl_sync(kFull, w, jj + 4 * hh);
    }
    float* drow = a.dY + u * a.ldy;
    for (int col = lane * 4; col < a.F; col += 128) {
#pragma unroll
        for (int hh = 0; hh < H; ++hh) {
            const int hc = hh * a.F + col;
            float4 gv[4];
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) gv[jj] = ldg4(grow[jj] + hc);
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) acc = fma4(wj[hh][jj], gv[jj], acc);
            st4(drow + hc, acc);
        }
    }
}

__global__ void __launch_bounds__(kAggThreads) gat_agg_fwd_kernel(const GatArgs a) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const float inv_h = 1.f / (float)a.H;
    for (int64_t v = warp0; v < a.N; v += nwarps) {
        const int beg = __ldg(a.in_ptr + v), end = __ldg(a.in_ptr + v + 1);
        const int deg = end - beg;
        if (a.skip_fast && deg >= 1 && deg <= 4) continue;
        for (int h = 0; h < a.H; ++h) edge_softmax_warp(a, v, h, beg, end, lane);
        __syncwarp();
        if (false) {
            // airway trees: in-degree <= 4 (3 neighbours + self loop)
            const Edge4 e0 = load_edges4(a, a.att, beg, deg, 0);
            const Edge4 e1 = a.H > 1 ? load_edges4(a, a.att, beg, deg, 1) : e0;
            for (int col = lane * 4; col < a.F; col += 128) {
                float4 y0 = act4(add_res_bias(a, gather4(a, e0, deg, col), v, col), a.act);
                if (a.H > 1) {
                    float4 y1 = act4(add_res_bias(a, gather4(a, e1, deg, a.F + col), v, a.F + col), a.act);
                    if (a.mean_heads) st4(a.out + v * a.ldo + col, scale4(inv_h, add4(y0, y1)));
                    else { st4(a.out + v * a.ldo + col, y0); st4(a.out + v * a.ldo + a.F + col, y1); }
                } else {
                    st4(a.out + v * a.ldo + col, y0);      // one head: its mean is itself
                }
            }
            continue;
        }
        for (int col = lane * 4; col < a.F; col += 128) {
            float4 mean = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int h = 0; h < a.H; ++h) {
                const float4 y = act4(pre_chunk(a, a.att, v, h, col, beg, end), a.act);
                if (a.mean_heads) mean = add4(mean, y);
                else st4(a.out + v * a.ldo + h * a.F + col, y);
            }
            if (a.mean_heads) st4(a.out + v * a.ldo + col, scale4(inv_h, mean));
        }
    }
}

// Backward phase 1, one warp per DESTINATION node v:
//   g[v,h,:]  = g_out * act'(y)                      -> G (== the dres columns of dY when the residual is linear)
//   dot_j     = <g[v,h,:], z[u_j,h,:]>                -> d(a_drop_j)
//   ds_j      = a_j (da_j - sum_k a_k da_k) * leaky'(el[u_j]+er[v])   -> ds[slot*H+h];   der[v,h] = sum_j ds_j
template <int NCH>
__global__ void __launch_bounds__(kAggThreads) gat_agg_bwd_dst_kernel(const GatArgs a) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const float inv_h = 1.f / (float)a.H;
    for (int64_t v = warp0; v < a.N; v += nwarps) {
        const int beg = __ldg(a.in_ptr + v), end = __ldg(a.in_ptr + v + 1);
        const int deg = end - beg;
        if (a.skip_fast && deg >= 1 && deg <= 4) continue;
        const bool fast = false;
        float4 idsum[NCH];   // identity-residual gradient (summed over heads when xres_cols == F)
#pragma unroll
        for (int c = 0; c < NCH; ++c) idsum[c] = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int h = 0; h < a.H; ++h) {
            Edge4 e;
            if (fast) e = load_edges4(a, a.att_in, beg, deg, h);
            float4 gq[NCH];
#pragma unroll
            for (int c = 0; c < NCH; ++c) {
                gq[c] = make_float4(0.f, 0.f, 0.f, 0.f);
                const int col = (c * 32 + lane) * 4;
                if (col < a.F) {
                    float4 go, y;
                    if (a.mean_heads) {
                        go = scale4(inv_h, ldg4(a.g_out + v * a.ldg + col));
                        const float4 pre = fast ? add_res_bias(a, gather4(a, e, deg, h * a.F + col), v, h * a.F + col)
                                                : pre_chunk(a, a.att_in, v, h, col, beg, end);
                        y = act4(pre, a.act);
                    } else {
                        go = ldg4(a.g_out + v * a.ldg + h * a.F + col);
                        y = ldg4(a.out_saved + v * a.ldo + h * a.F + col);
                    }
                    gq[c] = mul4(go, actgrad4(y, a.act));
                    st4(a.G + v * a.ldG + h * a.F + col, gq[c]);
                    if (a.res_mode == 2) {
                        if (a.xres_cols == a.F) idsum[c] = add4(idsum[c], gq[c]);
                        else st4(a.dxres + v * a.ldxres + h * a.F + col, gq[c]);
                    }
                }
            }
            const float er = __ldg(a.Y + v * a.ldy + a.er_off + h);
            if (fast) {
                // d(a_drop_j) = <g, z[u_j]> for the (<= 4) in-edges: row loads issued together, reductions interleaved
                float d[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int c = 0; c < NCH; ++c) {
                    const int col = (c * 32 + lane) * 4;
                    if (col < a.F) {
                        float4 z[4];
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            z[j] = j < deg ? ldg4(a.Y + (int64_t)e.u[j] * a.ldy + h * a.F + col)
                                           : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                        for (int j = 0; j < 4; ++j) d[j] += dot4(gq[c], z[j]);
                    }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) d[j] += __shfl_xor_sync(kFull, d[j], o);
                }
                // softmax backward, every lane redundantly (4 edges)
                float att_j[4], da[4], wsum = 0.f;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    att_j[j] = j < deg ? __ldg(a.att_in + (int64_t)(beg + j) * a.H + h) : 0.f;
                    da[j] = j < deg ? d[j] * keep_scale(a, beg + j, h) : 0.f;
                    wsum += att_j[j] * da[j];
                }
                float der = 0.f;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (j < deg) {
                        const float raw = __ldg(a.Y + (int64_t)e.u[j] * a.ldy + a.el_off + h) + er;
                        const float dsv = att_j[j] * (da[j] - wsum) * (raw > 0.f ? 1.f : a.neg_slope);
                        if (lane == j) a.ds[(int64_t)(beg + j) * a.H + h] = dsv;
                        der += dsv;
                    }
                }
                if (lane == 0) a.dY[v * a.ldy + a.er_off + h] = der;
            } else {
                // general degree: d(a_drop_j) staged in ds[]
                for (int s = beg; s < end; ++s) {
                    const int u = __ldg(a.in_src + s);
                    float d = 0.f;
#pragma unroll
                    for (int c = 0; c < NCH; ++c) {
                        const int col = (c * 32 + lane) * 4;
                        if (col < a.F) d += dot4(gq[c], ldg4(a.Y + (int64_t)u * a.ldy + h * a.F + col));
                    }
                    d = warp_sum(d);
                    if (lane == 0) a.ds[(int64_t)s * a.H + h] = d * keep_scale(a, s, h);
                }
                __syncwarp();
                float wsum = 0.f;
                for (int s = beg + lane; s < end; s += 32)
                    wsum += __ldg(a.att_in + (int64_t)s * a.H + h) * a.ds[(int64_t)s * a.H + h];
                wsum = warp_sum(wsum);
                float der = 0.f;
                for (int s = beg + lane; s < end; s += 32) {
                    const int u = __ldg(a.in_src + s);
                    const float raw = __ldg(a.Y + (int64_t)u * a.ldy + a.el_off + h) + er;
                    const float de = __ldg(a.att_in + (int64_t)s * a.H + h) * (a.ds[(int64_t)s * a.H + h] - wsum);
                    const float dsv = de * (raw > 0.f ? 1.f : a.neg_slope);
                    a.ds[(int64_t)s * a.H + h] = dsv;
                    der += dsv;
                }
                der = warp_sum(der);
                if (lane == 0) a.dY[v * a.ldy + a.er_off + h] = der;
                __syncwarp();
            }
        }
        if (a.res_mode == 2 && a.xres_cols == a.F) {
#pragma unroll
            for (int c = 0; c < NCH; ++c) {
                const int col = (c * 32 + lane) * 4;
                if (col < a.F) st4(a.dxres + v * a.ldxres + col, idsum[c]);
            }
        }
    }
}

// Backward phase 2, one warp per SOURCE node u:
//   del[u,h] = sum over out-edges of ds;   dz[u,h,:] = sum over out-edges (u->v) of a_drop * g[v,h,:]
__global__ void __launch_bounds__(kAggThreads) gat_agg_bwd_src_kernel(const GatArgs a) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t u = warp0; u < a.N; u += nwarps) {
        const int beg = __ldg(a.out_ptr + u), end = __ldg(a.out_ptr + u + 1);
        if (a.skip_fast && end - beg >= 1 && end - beg <= 4) continue;
        for (int h = 0; h < a.H; ++h) {
            float del = 0.f;
            for (int q = beg + lane; q < end; q += 32) del += __ldg(a.ds + (int64_t)__ldg(a.out_slot + q) * a.H + h);
            del = warp_sum(del);
            if (lane == 0) a.dY[u * a.ldy + a.el_off + h] = del;
            for (int col = lane * 4; col < a.F; col += 128) {
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                for (int q = beg; q < end; ++q) {
                    const int s = __ldg(a.out_slot + q);
                    const int v = __ldg(a.out_dst + q);
                    const float w = __ldg(a.att_in + (int64_t)s * a.H + h) * keep_scale(a, s, h);
                    acc = fma4(w, ldg4(a.G + (int64_t)v * a.ldG + h * a.F + col), acc);
                }
                st4(a.dY + u * a.ldy + h * a.F + col, acc);
            }
        }
    }
}

// which = 0 forward, 1 backward-destination, 2 backward-source
template <int H, int WHICH>
__global__ void __launch_bounds__(kAggThreads) gat_fast_kernel(const GatArgs a) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int32_t* ptr = WHICH == 2 ? a.out_ptr : a.in_ptr;
    for (int64_t v = warp0; v < a.N; v += nwarps) {
        const int beg = __ldg(ptr + v), deg = __ldg(ptr + v + 1) - beg;
        if (deg < 1 || deg > 4) continue;            // left to the general kernel
        if (WHICH == 0) fwd_node_fast<H>(a, v, beg, deg, lane);
        else if (WHICH == 1) bwd_dst_node_fast<H>(a, v, beg, deg, lane);
        else bwd_src_node_fast<H>(a, v, beg, deg, lane);
    }
}

template <int WHICH>
static int launch_fast(const GatArgs& a, cudaStream_t st, unsigned grid) {
    if (a.H == 1) gat_fast_kernel<1, WHICH><<<grid, kAggThreads, 0, st>>>(a);
    else gat_fast_kernel<2, WHICH><<<grid, kAggThreads, 0, st>>>(a);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

static inline unsigned agg_grid(int64_t N) {
    int64_t want = ceil_div(N, kAggThreads / 32);
    int64_t cap = (int64_t)sm_count() * 32;
    return (unsigned)(want < cap ? want : cap);
}

static int check_common(const float* Y, int64_t ldy, int64_t N, int64_t H, int64_t F, int res_mode, const float* xres,
                        int64_t ldxres, int64_t xres_cols, const float* bias) {
    SPGNN_REQUIRE(Y && N > 0 && H > 0 && F > 0, "gat_agg: bad argument");
    SPGNN_REQUIRE(F % 4 == 0 && ldy % 4 == 0 && ((uintptr_t)Y & 15) == 0,
                  "gat_agg: F (%lld) and ldy (%lld) must be multiples of 4 and Y 16-byte aligned", (long long)F,
                  (long long)ldy);
    SPGNN_REQUIRE(!bias || ((uintptr_t)bias & 15) == 0, "gat_agg: bias must be 16-byte aligned");
    if (res_mode == 2) {
        SPGNN_REQUIRE(xres && ldxres % 4 == 0 && ((uintptr_t)xres & 15) == 0 &&
                          (xres_cols == F || xres_cols == H * F),
                      "gat_agg: identity residual needs xres with F or H*F columns (got %lld), ld multiple of 4",
                      (long long)xres_cols);
    }
    SPGNN_REQUIRE(res_mode >= 0 && res_mode <= 2, "gat_agg: res_mode");
    return SPGNN_OK;
}

}  // namespace spgnn

using namespace spgnn;

extern "C" int spgnn_gat_agg_fwd(const float* Y, int64_t ldy, int64_t res_off, int64_t el_off, int64_t er_off,
                                 int res_mode, const float* xres, int64_t ldxres, int64_t xres_cols,
                                 const float* bias, int act, float negative_slope, int mean_heads, float attn_drop_p,
                                 uint64_t seed, const int32_t* in_ptr, const int32_t* in_src, int64_t N, int64_t H,
                                 int64_t F, float* out, int64_t ldo, float* att, void* stream) {
    int rc = check_common(Y, ldy, N, H, F, res_mode, xres, ldxres, xres_cols, bias);
    if (rc) return rc;
    SPGNN_REQUIRE(in_ptr && in_src && out && att, "gat_agg_fwd: null pointer");
    SPGNN_REQUIRE(ldo % 4 == 0 && ((uintptr_t)out & 15) == 0 && (res_mode != 1 || res_off % 4 == 0),
                  "gat_agg_fwd: out/res alignment");
    SPGNN_REQUIRE(attn_drop_p >= 0.f && attn_drop_p < 1.f, "gat_agg_fwd: dropout p");
    GatArgs a{};
    a.Y = Y; a.ldy = ldy; a.res_off = res_off; a.el_off = el_off; a.er_off = er_off;
    a.res_mode = res_mode; a.xres = xres; a.ldxres = ldxres; a.xres_cols = (int)xres_cols;
    a.bias = bias; a.act = act; a.neg_slope = negative_slope; a.mean_heads = mean_heads;
    a.drop_p = attn_drop_p; a.seed = seed; a.in_ptr = in_ptr; a.in_src = in_src;
    a.N = N; a.H = (int)H; a.F = (int)F; a.out = out; a.ldo = ldo; a.att = att;
    a.skip_fast = H <= 2;
    if (a.skip_fast) {
        rc = launch_fast<0>(a, as_stream(stream), agg_grid(N));
        if (rc) return rc;
    }
    gat_agg_fwd_kernel<<<agg_grid(N), kAggThreads, 0, as_stream(stream)>>>(a);   // nodes with other degrees (none in a tree)
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

extern "C" int spgnn_gat_agg_bwd(const float* g_out, int64_t ldg, const float* out, int64_t ldo, const float* Y,
                                 int64_t ldy, int64_t res_off, int64_t el_off, int64_t er_off, int res_mode,
                                 const float* xres, int64_t ldxres, int64_t xres_cols, const float* bias, int act,
                                 float negative_slope, int mean_heads, float attn_drop_p, uint64_t seed,
                                 const float* att, const int32_t* in_ptr, const int32_t* in_src,
                                 const int32_t* out_ptr, const int32_t* out_dst, const int32_t* out_slot, int64_t N,
                                 int64_t H, int64_t F, float* dY, float* dxres, float* g_ws, float* ds_ws,
                                 void* stream) {
    int rc = check_common(Y, ldy, N, H, F, res_mode, xres, ldxres, xres_cols, bias);
    if (rc) return rc;
    SPGNN_REQUIRE(g_out && att && in_ptr && in_src && out_ptr && out_dst && out_slot && dY && ds_ws,
                  "gat_agg_bwd: null pointer");
    SPGNN_REQUIRE(mean_heads || out, "gat_agg_bwd: saved output required unless mean_heads");
    SPGNN_REQUIRE(res_mode == 1 || g_ws, "gat_agg_bwd: g_ws [N,H*F] required when the residual is not linear");
    SPGNN_REQUIRE(res_mode != 2 || dxres, "gat_agg_bwd: dxres required for identity residual");
    SPGNN_REQUIRE(F <= 128 * kMaxCh, "gat_agg_bwd: F=%lld exceeds %d", (long long)F, 128 * kMaxCh);
    SPGNN_REQUIRE(ldg % 4 == 0 && ((uintptr_t)g_out & 15) == 0 && ((uintptr_t)dY & 15) == 0 &&
                      (mean_heads || (ldo % 4 == 0 && ((uintptr_t)out & 15) == 0)),
                  "gat_agg_bwd: alignment");
    GatArgs a{};
    a.Y = Y; a.ldy = ldy; a.res_off = res_off; a.el_off = el_off; a.er_off = er_off;
    a.res_mode = res_mode; a.xres = xres; a.ldxres = ldxres; a.xres_cols = (int)xres_cols;
    a.bias = bias; a.act = act; a.neg_slope = negative_slope; a.mean_heads = mean_heads;
    a.drop_p = attn_drop_p; a.seed = seed; a.in_ptr = in_ptr; a.in_src = in_src;
    a.out_ptr = out_ptr; a.out_dst = out_dst; a.out_slot = out_slot;
    a.N = N; a.H = (int)H; a.F = (int)F; a.ldo = ldo;
    a.g_out = g_out; a.ldg = ldg; a.out_saved = out; a.att_in = att;
    a.dY = dY; a.dxres = dxres; a.ds = ds_ws;
    if (res_mode == 1) { a.G = dY + res_off; a.ldG = ldy; } else { a.G = g_ws; a.ldG = H * F; }
    cudaStream_t st = as_stream(stream);
    a.skip_fast = H <= 2;
    if (a.skip_fast) {
        rc = launch_fast<1>(a, st, agg_grid(N));
        if (rc) return rc;
    }
    if (F <= 128) gat_agg_bwd_dst_kernel<1><<<agg_grid(N), kAggThreads, 0, st>>>(a);
    else if (F <= 256) gat_agg_bwd_dst_kernel<2><<<agg_grid(N), kAggThreads, 0, st>>>(a);
    else if (F <= 512) gat_agg_bwd_dst_kernel<4><<<agg_grid(N), kAggThreads, 0, st>>>(a);
    else gat_agg_bwd_dst_kernel<8><<<agg_grid(N), kAggThreads, 0, st>>>(a);
    SPGNN_LAUNCH_OK();
    if (a.skip_fast) {
        rc = launch_fast<2>(a, st, agg_grid(N));
        if (rc) return rc;
    }
    gat_agg_bwd_src_kernel<<<agg_grid(N), kAggThreads, 0, st>>>(a);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

SPGNN_REGISTER_SALT(gat)

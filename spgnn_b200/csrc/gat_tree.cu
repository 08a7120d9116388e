// GAT layer kernels with ONE CTA PER GRAPH (airway tree) and the graph's z rows staged in shared memory by TMA.
//
// The chunk kernels of gat_layer.cu gather the (<= 4) neighbour rows of every node through L1/L2.  On the synthetic
// airway trees a node's parent and children lie anywhere inside its tree (creation order), a tree's projection rows
// are 0.3 - 1.2 MB, and at 4-5 TB/s the 126 MB L2 turns over every ~25 us: ncu showed 40-50 % more DRAM reads than the
// algorithmic bytes (profiles/r01_ncu_layer_chunk_kernels.txt).  Here a CTA owns a whole graph and walks its z columns
// in slices of 32: one elected thread issues cp.async.bulk.tensor loads of z[tree rows, slice] (boxes of 32 rows x
// 128 B) into a two-stage shared-memory ring two slices ahead; a quarter-warp owns a node (8 lanes x float4), every
// neighbour gather is a shared-memory read, the node's own row operands (residual, incoming gradients) are plain
// coalesced loads issued one slice ahead into registers, and DRAM traffic equals the algorithmic bytes.  Edge
// weights and neighbour ids of the tree are staged once per tree (thread-parallel phase A).
//
// The backward fuses the destination and source sides: the slice of G = g_out * act'(y) computed for the tree's
// nodes stays in shared memory and is gathered right away for dz[u] = sum_{u->v} a * G[v], so G is written once (it
// is the residual part of dY) and never read back; the per-edge dot products accumulate in shared memory across
// slices and the softmax / LeakyReLU backward runs once per tree at the end.
//
// Applies when F % 64 == 0, no head mean, every degree <= 4 and the largest graph has <= 384 nodes; everything else
// takes the chunk kernels of gat_layer.cu.
#include <stdlib.h>
#include "layer_util.cuh"

namespace spgnn {
namespace tree {
using namespace layer;
using namespace ptx;

constexpr int kCS = 32;            // columns per slice (128 B per row)
constexpr int kBoxRows = 32;       // TMA box: 32 rows x 32 columns
constexpr int kThreads = 512;
constexpr int kQW = kThreads / 8;  // 64 quarter-warps; a quarter-warp owns one node of the slice (8 lanes x float4)
constexpr int kPer = 6;            // nodes per quarter-warp per slice
constexpr int kBatch = 3;          // forward: rounds whose shared-memory gathers are issued together
constexpr int kBatchBwd = 4;       // backward source side (same-box A/B at 640 threads x 4 rounds: 2 / 3 / 4 rounds per
                                   // batch -> 1.90 / 1.86 / 1.79 ms per launch, profiles/r02_tree_bwd_variants.txt)
constexpr int kMaxNodes = kQW * kPer;   // 384: every backward launch shape below covers it as well
constexpr size_t kSmemLimit = 232448;

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}

// explicit shared-space accesses with 32-bit addresses (pointers carved out of the dynamic shared array lose their
// address space and would compile to generic LD/ST with 64-bit address arithmetic)
__device__ __forceinline__ float4 lds4(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts4(uint32_t addr, float4 v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

struct TArgs {
    Args a;
    const int64_t* node_off; int64_t B;
    int nmax;                      // rows per z stage (largest graph rounded up to the box)
    int nstages;                   // 1 or 2
    int nslices;                   // H*F / 32
    int split;                     // CTAs per tree: each takes a contiguous range of the tree's slices (small batches)
};

struct short4s { short x, y, z, w; };

// one elected thread: z[tree rows, slice] -> stage
__device__ __forceinline__ void issue_slice(const CUtensorMap* map, uint32_t bar, uint32_t dst, int64_t n0, int n, int col) {
    const int nbox = (n + kBoxRows - 1) / kBoxRows;
    mbar_expect_tx(bar, (uint32_t)nbox * kBoxRows * kCS * 4);
    for (int r = 0; r < nbox; ++r) tma_load_2d(dst + r * (kBoxRows * kCS * 4), map, bar, col, (int)(n0 + r * kBoxRows));
}

// walks the (tree, slice) items of one CTA: slices [s0, s1) of trees first, first + tstep, ...  With t.split == 1 a
// CTA takes whole trees; batches with fewer trees than SMs (the reference trains on 64 scans and infers one scan at a
// time, job_runner.py:1892-1919, :840-911) give every tree to t.split CTAs, each with its own range of slices.
struct Cursor {
    int64_t tr, n0; int n, s; int s0, s1, tstep;
    __device__ __forceinline__ bool valid(const TArgs& t) const { return tr < t.B; }
    __device__ __forceinline__ void load(const TArgs& t) {
        if (tr < t.B) { n0 = t.node_off[tr]; n = (int)(t.node_off[tr + 1] - n0); }
    }
    __device__ __forceinline__ void advance(const TArgs& t) {
        if (++s == s1) { s = s0; tr += tstep; load(t); }
    }
};
__device__ __forceinline__ Cursor first_cursor(const TArgs& t) {
    Cursor c;
    const int sg = (int)(blockIdx.x % (unsigned)t.split);
    c.s0 = (int)((int64_t)sg * t.nslices / t.split);
    c.s1 = (int)((int64_t)(sg + 1) * t.nslices / t.split);
    c.tstep = (int)(gridDim.x / (unsigned)t.split);
    c.tr = blockIdx.x / (unsigned)t.split;
    c.s = c.s0; c.n0 = 0; c.n = 0;
    return c;
}

// activation known at compile time (ACT = SPGNN_ACT_ELU / _TANH), else the runtime code
template <int ACT>
__device__ __forceinline__ float4 act_apply4(float4 p, int act) {
    if (ACT == SPGNN_ACT_ELU)
        return make_float4(p.x > 0.f ? p.x : exp_fast(p.x) - 1.f, p.y > 0.f ? p.y : exp_fast(p.y) - 1.f,
                           p.z > 0.f ? p.z : exp_fast(p.z) - 1.f, p.w > 0.f ? p.w : exp_fast(p.w) - 1.f);
    if (ACT == SPGNN_ACT_TANH)
        return make_float4(1.f - __fdividef(2.f, exp_fast(2.f * p.x) + 1.f), 1.f - __fdividef(2.f, exp_fast(2.f * p.y) + 1.f),
                           1.f - __fdividef(2.f, exp_fast(2.f * p.z) + 1.f), 1.f - __fdividef(2.f, exp_fast(2.f * p.w) + 1.f));
    return act4(p, act);
}

// ------------------------------------------------------------------------------------------------ forward
struct FSmem {
    uint64_t* full; int* deg; short4s* nb; float* w; float* zs;
};
__device__ __forceinline__ FSmem carve_f(uint8_t* base, int nmax, int H) {
    FSmem s;
    s.full = reinterpret_cast<uint64_t*>(base);
    s.deg = reinterpret_cast<int*>(base + 128);
    s.nb = reinterpret_cast<short4s*>(s.deg + nmax);
    s.w = reinterpret_cast<float*>(s.nb + nmax);
    uintptr_t z = reinterpret_cast<uintptr_t>(s.w + (size_t)nmax * H * 4);
    s.zs = reinterpret_cast<float*>((z + 127) & ~(uintptr_t)127);
    return s;
}
static size_t fwd_smem_bytes(int nmax, int H, int nstages) {
    return 128 + (size_t)nmax * (4 + 8 + H * 16) + 128 + (size_t)nstages * nmax * kCS * 4 + 128;
}

template <int ACT, int THREADS, int KPER>
__global__ void __launch_bounds__(THREADS, 1) gat_tree_fwd_kernel(const __grid_constant__ CUtensorMap zmap, const TArgs t) {
    constexpr int kThreads = THREADS, kQW = THREADS / 8;
    extern __shared__ __align__(128) uint8_t smem[];
    const Args& a = t.a;
    const int H = a.H, F = a.F;
    const FSmem st = carve_f(smem, t.nmax, H);
    const int l8 = threadIdx.x & 7, qw = threadIdx.x >> 3;
    const uint32_t zs_u32 = smem_u32(st.zs);
    const uint32_t stage_bytes = (uint32_t)t.nmax * kCS * 4;
    const bool has_res = a.res_mode == 1;

    if (threadIdx.x == 0) {
        mbar_init(smem_u32(&st.full[0]), 1);
        mbar_init(smem_u32(&st.full[1]), 1);
        fence_barrier_init();
        prefetch_tmap(&zmap);
    }
    __syncthreads();

    Cursor cur = first_cursor(t);
    if (!cur.valid(t)) return;
    cur.load(t);
    Cursor nxt = cur;            // item whose z slice was issued last
    nxt.advance(t);
    if (threadIdx.x == 0) {
        issue_slice(&zmap, smem_u32(&st.full[0]), zs_u32, cur.n0, cur.n, cur.s * kCS);
        if (t.nstages == 2 && nxt.valid(t))
            issue_slice(&zmap, smem_u32(&st.full[1]), zs_u32 + stage_bytes, nxt.n0, nxt.n, nxt.s * kCS);
    }
    float4 r[KPER];              // residual rows of the item about to be computed (prefetched one slice ahead)
    float4 bv = a.bias ? ldg4(a.bias + cur.s * kCS + l8 * 4) : zero4();
#pragma unroll
    for (int k = 0; k < KPER; ++k) {
        const int i = qw + k * kQW;
        r[k] = (has_res && i < cur.n) ? ldg4(a.Y + (cur.n0 + i) * a.ldy + a.res_off + cur.s * kCS + l8 * 4) : zero4();
    }

    for (uint32_t item = 0; cur.valid(t); ++item) {
        const int stg = t.nstages == 2 ? (int)(item & 1) : 0;
        const uint32_t par = t.nstages == 2 ? ((item >> 1) & 1) : (item & 1);
        const int64_t n0 = cur.n0;
        const int n = cur.n, s = cur.s;
        if (s == cur.s0) {
            // ---------------- phase A: edge softmax of the tree, one thread per (node, head); the attention weights go
            // to global memory from the CTA that owns the head's first slice
            for (int it = threadIdx.x; it < n * H; it += kThreads) {
                const int i = it / H, h = it - i * H;
                const int64_t v = n0 + i;
                const int beg = __ldg(a.in_ptr + v), deg = __ldg(a.in_ptr + v + 1) - beg;
                const float er = __ldg(a.Y + v * a.ldy + a.er_off + h);
                const int hs = h * (F / kCS);
                const bool own_head = hs >= cur.s0 && hs < cur.s1;
                int u[4];
                float e[4], m = -INFINITY;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    u[j] = deg > 0 ? __ldg(a.in_src + beg + min(j, deg - 1)) : (int)v;
                    e[j] = leaky(__ldg(a.Y + (int64_t)u[j] * a.ldy + a.el_off + h) + er, a.neg_slope);
                    if (j < deg) m = fmaxf(m, e[j]);
                }
                float p[4], sum = 0.f;
#pragma unroll
                for (int j = 0; j < 4; ++j) { p[j] = j < deg ? __expf(e[j] - m) : 0.f; sum += p[j]; }
                const float inv = deg > 0 ? 1.f / sum : 0.f;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float at = p[j] * inv;
                    if (j < deg && own_head) a.att[(int64_t)(beg + j) * H + h] = at;
                    st.w[(i * H + h) * 4 + j] = j < deg ? at * keep_scale(a, beg + j, h) : 0.f;
                }
                if (h == 0) {
                    st.deg[i] = deg;
                    st.nb[i] = short4s{(short)(u[0] - n0), (short)(u[1] - n0), (short)(u[2] - n0), (short)(u[3] - n0)};
                }
            }
            __syncthreads();
        }
        // own rows of this item are in r[]; move them out and start the loads of the next item
        float4 rc[KPER];
#pragma unroll
        for (int k = 0; k < KPER; ++k) rc[k] = r[k];
        const float4 bvc = bv;
        Cursor nn = cur;
        nn.advance(t);
        if (nn.valid(t)) {
            const float* yrow = a.Y + (nn.n0 + qw) * a.ldy + a.res_off + nn.s * kCS + l8 * 4;
            if (a.bias) bv = ldg4(a.bias + nn.s * kCS + l8 * 4);
#pragma unroll
            for (int k = 0; k < KPER; ++k) {
                const int i = qw + k * kQW;
                r[k] = (has_res && i < nn.n) ? ldg4(yrow + (int64_t)(k * kQW) * a.ldy) : zero4();
            }
        }
        if (t.nstages == 1 && item > 0 && threadIdx.x == 0)
            issue_slice(&zmap, smem_u32(&st.full[0]), zs_u32, n0, n, s * kCS);
        mbar_wait(smem_u32(&st.full[stg]), par);
        // ---------------- phase B: one quarter-warp per node, 32 columns of head h
        const uint32_t zs = zs_u32 + stg * stage_bytes + l8 * 16;
        const int c = s * kCS + l8 * 4;                       // column inside [0, H*F)
        const int h = (s * kCS) / F;
        // rounds kBatch at a time, out-of-range nodes clamped to node 0 (see the backward's source side)
#pragma unroll
        for (int k0 = 0; k0 < KPER; k0 += kBatch) {
            constexpr int kB = kBatch;
            const int nb_ = KPER - k0 < kB ? KPER - k0 : kB;   // rounds in this batch (compile-time after unrolling)
            if ((qw & ~3) + k0 * kQW < n) {                    // warp-uniform
                short4s nb[kB];
                float4 w[kB], acc[kB];
#pragma unroll
                for (int j = 0; j < kB; ++j) {
                    if (j < nb_) {
                        const int i = qw + (k0 + j) * kQW;
                        const int ii = i < n ? i : 0;
                        nb[j] = st.nb[ii];
                        w[j] = *reinterpret_cast<const float4*>(st.w + (ii * H + h) * 4);
                    }
                }
#pragma unroll
                for (int j = 0; j < kB; ++j) {
                    if (j < nb_) {
                        acc[j] = add4(rc[k0 + j], bvc);
                        acc[j] = fma4(w[j].x, lds4(zs + nb[j].x * (kCS * 4)), acc[j]);
                        acc[j] = fma4(w[j].y, lds4(zs + nb[j].y * (kCS * 4)), acc[j]);
                        acc[j] = fma4(w[j].z, lds4(zs + nb[j].z * (kCS * 4)), acc[j]);
                        acc[j] = fma4(w[j].w, lds4(zs + nb[j].w * (kCS * 4)), acc[j]);
                    }
                }
#pragma unroll
                for (int j = 0; j < kB; ++j) {
                    if (j < nb_) {
                        const int i = qw + (k0 + j) * kQW;
                        if (i < n) emit(a, n0 + i, c, act_apply4<ACT>(acc[j], a.act));
                    }
                }
            }
        }
        __syncthreads();
        // the stage just consumed takes the slice two items ahead
        cur = nn;
        if (t.nstages == 2) {
            nxt.advance(t);
            if (threadIdx.x == 0 && nxt.valid(t))
                issue_slice(&zmap, smem_u32(&st.full[stg]), zs_u32 + stg * stage_bytes, nxt.n0, nxt.n, nxt.s * kCS);
        }
    }
}

// ------------------------------------------------------------------------------------------------ backward (fused)
struct BSmem {
    uint64_t* full;
    int* deg; int* beg; int* odeg;
    short4s *nb, *onb, *oslot;
    float *w, *at, *dd, *ow;       // [n][H][4]; at carries the LeakyReLU branch in its sign (negative: slope branch)
    float* ds;                     // [4n][H]
    float* part;                   // [kThreads / 32][kCS] bias-gradient partials of the slice, one row per warp
    float* sb;                     // [H*F]
    float* zs; float* gs;
};
__device__ __forceinline__ BSmem carve_b(uint8_t* base, int nmax, int H, int HF, int nstages, int nwarps) {
    BSmem s;
    s.full = reinterpret_cast<uint64_t*>(base);
    s.deg = reinterpret_cast<int*>(base + 128);
    s.beg = s.deg + nmax;
    s.odeg = s.beg + nmax;
    s.nb = reinterpret_cast<short4s*>(s.odeg + nmax);
    s.onb = s.nb + nmax;
    s.oslot = s.onb + nmax;
    s.w = reinterpret_cast<float*>(s.oslot + nmax);
    s.at = s.w + (size_t)nmax * H * 4;
    s.dd = s.at + (size_t)nmax * H * 4;
    s.ow = s.dd + (size_t)nmax * H * 4;
    s.ds = s.ow + (size_t)nmax * H * 4;
    s.part = s.ds + (size_t)nmax * H * 4;
    s.sb = s.part + nwarps * kCS;
    uintptr_t z = reinterpret_cast<uintptr_t>(s.sb + HF);
    s.zs = reinterpret_cast<float*>((z + 127) & ~(uintptr_t)127);
    s.gs = s.zs + (size_t)nstages * nmax * kCS;
    return s;
}
static size_t bwd_smem_bytes(int nmax, int H, int HF, int nstages, int nwarps) {
    return 128 + (size_t)nmax * (12 + 24 + 5 * H * 16) + (size_t)nwarps * kCS * 4 + (size_t)HF * 4 + 128 +
           (size_t)(nstages + 1) * nmax * kCS * 4 + 128;
}

// d act(x) / dx from the pre-activation, for the activation known at compile time (ACT = SPGNN_ACT_ELU / _TANH: one
// exponential and no compare chain on the runtime code; anything else takes the generic pair act / act-grad-from-output)
template <int ACT>
__device__ __forceinline__ float act_slope(float x, int act) {
    if (ACT == SPGNN_ACT_ELU) return x > 0.f ? 1.f : exp_fast(x);
    if (ACT == SPGNN_ACT_TANH) {
        const float y = 1.f - __fdividef(2.f, exp_fast(2.f * x) + 1.f);
        return 1.f - y * y;
    }
    return act_grad_from_out(act_fast(x, act), act, kGatLeakySlope);
}
template <int ACT>
__device__ __forceinline__ float4 act_slope4(float4 p, int act) {
    return make_float4(act_slope<ACT>(p.x, act), act_slope<ACT>(p.y, act), act_slope<ACT>(p.z, act), act_slope<ACT>(p.w, act));
}

// NG gradient sources; ACT: activation known at compile time (0 = read it from the arguments); THREADS / 8 nodes are
// taken per round and a slice takes KPER rounds; PF: how many rounds ahead a node's own-row operands (residual
// projection, gradient sources) are loaded into registers.  PF == KPER is the first generation of this kernel
// (512 threads, everything of the next slice loaded a whole slice ahead: 4 * KPER * (1 + NG) registers, which pinned
// the kernel at 128 registers x 16 warps); PF = 2 with 896 threads keeps 8 * (1 + NG) prefetch registers and lets
// 28 warps share the issue slots (the ncu source view showed neither DRAM nor issue slots saturated at 16 warps).
template <int NG, int ACT, int THREADS, int KPER, int PF>
__global__ void __launch_bounds__(THREADS, 1) gat_tree_bwd_kernel(const __grid_constant__ CUtensorMap zmap, const TArgs t) {
    constexpr int kThreads = THREADS, kQW = THREADS / 8;
    static_assert(PF >= 1 && PF <= KPER, "prefetch depth");
    extern __shared__ __align__(128) uint8_t smem[];
    const Args& a = t.a;
    const int H = a.H, F = a.F, HF = H * F;
    const BSmem st = carve_b(smem, t.nmax, H, HF, t.nstages, THREADS / 32);
    const int l8 = threadIdx.x & 7, qw = threadIdx.x >> 3;
    const uint32_t zs_u32 = smem_u32(st.zs), gs_u32 = smem_u32(st.gs);
    const uint32_t stage_bytes = (uint32_t)t.nmax * kCS * 4;
    const bool has_res = a.res_mode == 1;

    if (threadIdx.x == 0) {
        mbar_init(smem_u32(&st.full[0]), 1);
        mbar_init(smem_u32(&st.full[1]), 1);
        fence_barrier_init();
        prefetch_tmap(&zmap);
    }
    for (int i = threadIdx.x; i < HF; i += kThreads) st.sb[i] = 0.f;
    __syncthreads();

    Cursor cur = first_cursor(t);
    if (cur.valid(t)) cur.load(t);
    Cursor nxt = cur;
    if (cur.valid(t)) {
        nxt.advance(t);
        if (threadIdx.x == 0) {
            issue_slice(&zmap, smem_u32(&st.full[0]), zs_u32, cur.n0, cur.n, cur.s * kCS);
            if (t.nstages == 2 && nxt.valid(t))
                issue_slice(&zmap, smem_u32(&st.full[1]), zs_u32 + stage_bytes, nxt.n0, nxt.n, nxt.s * kCS);
        }
    }
    // own-row operands (residual projection, raw gradient sources) of the rounds about to be computed: a ring of PF
    // rounds in registers, round k of an item lives in slot k % PF (every index below is a compile-time constant)
    float4 r[PF], g[NG][PF];
    float4 bv = zero4();
    auto load_round = [&](const Cursor& it, int k, float4& r_, float4 (&g_)[NG][PF], int slot) {
        const int i = qw + k * kQW;
        const bool on = i < it.n;
        const int64_t v = it.n0 + i;
        const int c = it.s * kCS + l8 * 4;
        r_ = (has_res && on) ? ldg4(a.Y + v * a.ldy + a.res_off + c) : zero4();
#pragma unroll
        for (int q = 0; q < NG; ++q) g_[q][slot] = on ? ldg4(a.gs[q].g + v * a.gs[q].ld + c) : zero4();
    };
    auto load_own = [&](const Cursor& it) {        // the first PF rounds of an item
        if (a.bias) bv = ldg4(a.bias + it.s * kCS + l8 * 4);
#pragma unroll
        for (int k = 0; k < PF; ++k) load_round(it, k, r[k], g, k);
    };
    if (cur.valid(t)) load_own(cur);

    for (uint32_t item = 0; cur.valid(t); ++item) {
        const int stg = t.nstages == 2 ? (int)(item & 1) : 0;
        const uint32_t par = t.nstages == 2 ? ((item >> 1) & 1) : (item & 1);
        const int64_t n0 = cur.n0;
        const int n = cur.n, s = cur.s;
        if (s == cur.s0) {
            // ---------------- phase A: stage both edge directions of the tree, one thread per (node, head)
            const int lb0 = __ldg(a.in_ptr + n0);
            for (int it = threadIdx.x; it < n * H; it += kThreads) {
                const int i = it / H, h = it - i * H;
                const int64_t v = n0 + i;
                const int beg = __ldg(a.in_ptr + v), deg = __ldg(a.in_ptr + v + 1) - beg;
                const float er = __ldg(a.Y + v * a.ldy + a.er_off + h);
                int u[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    u[j] = deg > 0 ? __ldg(a.in_src + beg + min(j, deg - 1)) : (int)v;
                    const float raw = __ldg(a.Y + (int64_t)u[j] * a.ldy + a.el_off + h) + er;
                    const float at = j < deg ? __ldg(a.att + (int64_t)(beg + j) * H + h) : 0.f;
                    const int o = (i * H + h) * 4 + j;
                    st.w[o] = j < deg ? at * keep_scale(a, beg + j, h) : 0.f;
                    st.at[o] = raw > 0.f ? at : -at;
                    st.dd[o] = 0.f;
                }
                const int ob = __ldg(a.out_ptr + v), od = __ldg(a.out_ptr + v + 1) - ob;
                int ov[4], os[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int q = ob + min(j, max(od - 1, 0));
                    os[j] = od > 0 ? __ldg(a.out_slot + q) : lb0;
                    ov[j] = od > 0 ? __ldg(a.out_dst + q) : (int)v;
                    st.ow[(i * H + h) * 4 + j] = j < od ? __ldg(a.att + (int64_t)os[j] * H + h) * keep_scale(a, os[j], h) : 0.f;
                }
                if (h == 0) {
                    st.deg[i] = deg; st.beg[i] = beg - lb0; st.odeg[i] = od;
                    st.nb[i] = short4s{(short)(u[0] - n0), (short)(u[1] - n0), (short)(u[2] - n0), (short)(u[3] - n0)};
                    st.onb[i] = short4s{(short)(ov[0] - n0), (short)(ov[1] - n0), (short)(ov[2] - n0), (short)(ov[3] - n0)};
                    st.oslot[i] = short4s{(short)(os[0] - lb0), (short)(os[1] - lb0), (short)(os[2] - lb0), (short)(os[3] - lb0)};
                }
            }
            __syncthreads();
        }
        if (t.nstages == 1 && item > 0 && threadIdx.x == 0)
            issue_slice(&zmap, smem_u32(&st.full[0]), zs_u32, n0, n, s * kCS);
        mbar_wait(smem_u32(&st.full[stg]), par);
        // ---------------- dst side: g = g_out * act'(y) (y recomputed), G -> smem (+ dY residual part), <g, z_j>
        const uint32_t zs = zs_u32 + stg * stage_bytes + l8 * 16;
        const uint32_t gsm = gs_u32 + l8 * 16;
        const int c = s * kCS + l8 * 4;
        const int h = (s * kCS) / F;
        float4 bsum = zero4();
#pragma unroll
        for (int k = 0; k < KPER; ++k) {
            const int i = qw + k * kQW;
            const float4 rk = r[k % PF];
            float4 gk[NG];
#pragma unroll
            for (int q = 0; q < NG; ++q) gk[q] = g[q][k % PF];
            if (k + PF < KPER) load_round(cur, k + PF, r[k % PF], g, k % PF);     // in flight for PF rounds
            if (i < n) {
                const int64_t v = n0 + i;
                const short4s nb = st.nb[i];
                const float4 w = *reinterpret_cast<const float4*>(st.w + (i * H + h) * 4);
                const float4 z0 = lds4(zs + nb.x * (kCS * 4)), z1 = lds4(zs + nb.y * (kCS * 4));
                const float4 z2 = lds4(zs + nb.z * (kCS * 4)), z3 = lds4(zs + nb.w * (kCS * 4));
                float4 acc = add4(rk, bv);
                acc = fma4(w.x, z0, acc); acc = fma4(w.y, z1, acc); acc = fma4(w.z, z2, acc); acc = fma4(w.w, z3, acc);
                float4 go = zero4();
#pragma unroll
                for (int q = 0; q < NG; ++q) {
                    const GSrc& gq_ = a.gs[q];
                    go = add4(go, drop4(gk[q], gq_.thr, gq_.scale, gq_.seed,
                                        (uint64_t)v * (uint64_t)gq_.nch + (uint64_t)(gq_.ch_off + (c >> 2))));
                }
                const float4 gq = mul4(go, act_slope4<ACT>(acc, a.act));
                sts4(gsm + i * (kCS * 4), gq);
                if (has_res) store_planes4(a.dY + v * a.dld + a.res_off + c, a.dps, gq);
                bsum = add4(bsum, gq);
                float d0 = dot4(gq, z0), d1 = dot4(gq, z1), d2 = dot4(gq, z2), d3 = dot4(gq, z3);
                const unsigned qmask = 0xFFu << (threadIdx.x & 24);
#pragma unroll
                for (int o = 1; o < 8; o <<= 1) {
                    d0 += __shfl_xor_sync(qmask, d0, o); d1 += __shfl_xor_sync(qmask, d1, o);
                    d2 += __shfl_xor_sync(qmask, d2, o); d3 += __shfl_xor_sync(qmask, d3, o);
                }
                if (l8 == 0) {
                    float4* dp = reinterpret_cast<float4*>(st.dd + (i * H + h) * 4);
                    float4 dv = *dp;
                    dv.x += d0; dv.y += d1; dv.z += d2; dv.w += d3;
                    *dp = dv;
                }
            }
        }
        // bias gradient of the slice: the quarter-warps of a warp share their columns -> two shuffle rounds, one
        // staged row per warp (2 KB; the 8 KB of one row per quarter-warp kept a 384-node stage pair from fitting, and
        // shared-memory atomics straight into sb measured 8-20 % slower: 16 warps on the same 32 addresses)
        if (a.dbias_ws) {
#pragma unroll
            for (int o = 8; o < 32; o <<= 1) {
                bsum.x += __shfl_xor_sync(0xFFFFFFFFu, bsum.x, o); bsum.y += __shfl_xor_sync(0xFFFFFFFFu, bsum.y, o);
                bsum.z += __shfl_xor_sync(0xFFFFFFFFu, bsum.z, o); bsum.w += __shfl_xor_sync(0xFFFFFFFFu, bsum.w, o);
            }
            if ((threadIdx.x & 31) < 8) *reinterpret_cast<float4*>(st.part + (threadIdx.x >> 5) * kCS + l8 * 4) = bsum;
        }
        __syncthreads();
        // the z stage is free: slice two items ahead; own rows of the next item
        Cursor nn = cur;
        nn.advance(t);
        if (t.nstages == 2) {
            nxt.advance(t);
            if (threadIdx.x == 0 && nxt.valid(t))
                issue_slice(&zmap, smem_u32(&st.full[stg]), zs_u32 + stg * stage_bytes, nxt.n0, nxt.n, nxt.s * kCS);
        }
        if (nn.valid(t)) load_own(nn);
        if (a.dbias_ws && threadIdx.x < kCS) {
            float acc = 0.f;
#pragma unroll
            for (int q = 0; q < kThreads / 32; ++q) acc += st.part[q * kCS + threadIdx.x];
            st.sb[s * kCS + threadIdx.x] += acc;
        }
        // ---------------- src side: dz[u] = sum over out-edges (u -> v) of a_drop * G[v]
        // Rounds are taken kBatch at a time with the out-of-range nodes clamped to node 0 instead of branched around:
        // the neighbour lists of the whole batch are read first, then all 4 * kBatch gathers are in flight together
        // (the per-round chain list -> gather -> FMA -> store left the 4 warps of a scheduler waiting on shared-memory
        // latency: 18 % of this kernel's stall samples sat on these lines, profiles/r01_ncu_tree_bwd_source.txt).
#pragma unroll
        for (int k0 = 0; k0 < KPER; k0 += kBatchBwd) {
            constexpr int kB = kBatchBwd;
            const int nb_ = KPER - k0 < kB ? KPER - k0 : kB;   // rounds in this batch (compile-time after unrolling)
            if ((qw & ~3) + k0 * kQW < n) {                    // warp-uniform: this warp has a node in round k0
                short4s nb[kB];
                float4 w[kB], acc[kB];
#pragma unroll
                for (int j = 0; j < kB; ++j) {
                    if (j < nb_) {
                        const int i = qw + (k0 + j) * kQW;
                        const int ii = i < n ? i : 0;
                        nb[j] = st.onb[ii];
                        w[j] = *reinterpret_cast<const float4*>(st.ow + (ii * H + h) * 4);
                    }
                }
#pragma unroll
                for (int j = 0; j < kB; ++j) {
                    if (j < nb_) {
                        acc[j] = scale4(w[j].x, lds4(gsm + nb[j].x * (kCS * 4)));
                        acc[j] = fma4(w[j].y, lds4(gsm + nb[j].y * (kCS * 4)), acc[j]);
                        acc[j] = fma4(w[j].z, lds4(gsm + nb[j].z * (kCS * 4)), acc[j]);
                        acc[j] = fma4(w[j].w, lds4(gsm + nb[j].w * (kCS * 4)), acc[j]);
                    }
                }
#pragma unroll
                for (int j = 0; j < kB; ++j) {
                    if (j < nb_) {
                        const int i = qw + (k0 + j) * kQW;
                        if (i < n) store_planes4(a.dY + (n0 + i) * a.dld + c, a.dps, acc[j]);
                    }
                }
            }
        }
        __syncthreads();
        if (s == cur.s1 - 1) {
            // ---------------- phase C: softmax + LeakyReLU backward of the tree, d(er); then d(el) over out-edges — for
            // the heads this CTA walked (all of them unless the tree is split by head)
            const int h_lo = cur.s0 * kCS / F, h_hi = cur.s1 * kCS / F;
            for (int it = threadIdx.x; it < n * H; it += kThreads) {
                const int i = it / H, hh = it - i * H;
                if (hh < h_lo || hh >= h_hi) continue;
                const int deg = st.deg[i], lb = st.beg[i];
                const int o = (i * H + hh) * 4;
                float da[4], at[4], wsum = 0.f, der = 0.f;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    at[j] = fabsf(st.at[o + j]);
                    da[j] = at[j] > 0.f ? st.dd[o + j] * (st.w[o + j] / at[j]) : 0.f;
                    wsum += at[j] * da[j];
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (j < deg) {
                        const float lk = (__float_as_uint(st.at[o + j]) >> 31) ? a.neg_slope : 1.f;
                        const float dsv = at[j] * (da[j] - wsum) * lk;
                        st.ds[(lb + j) * H + hh] = dsv;
                        der += dsv;
                    }
                }
                store_planes1(a.dY + (n0 + i) * a.dld + a.er_off + hh, a.dps, der);
            }
            __syncthreads();
            for (int it = threadIdx.x; it < n * H; it += kThreads) {
                const int i = it / H, hh = it - i * H;
                if (hh < h_lo || hh >= h_hi) continue;
                const int od = st.odeg[i];
                const short4s sl = st.oslot[i];
                float del = 0.f;
                if (od > 0) del += st.ds[sl.x * H + hh];
                if (od > 1) del += st.ds[sl.y * H + hh];
                if (od > 2) del += st.ds[sl.z * H + hh];
                if (od > 3) del += st.ds[sl.w * H + hh];
                store_planes1(a.dY + (n0 + i) * a.dld + a.el_off + hh, a.dps, del);
            }
            __syncthreads();
        }
        cur = nn;
    }
    if (a.dbias_ws)
        for (int i = threadIdx.x; i < HF; i += kThreads) a.dbias_ws[(int64_t)blockIdx.x * HF + i] = st.sb[i];
}

__global__ void tree_dbias_reduce_kernel(const float* __restrict__ part, int64_t nparts, int64_t HF, float* __restrict__ out) {
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < HF; c += (int64_t)gridDim.x * blockDim.x) {
        float s = 0.f;
        for (int64_t p = 0; p < nparts; ++p) s += part[p * HF + c];
        out[c] = s;
    }
}

// ------------------------------------------------------------------------------------------------ host side
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

// fp32 matrix [rows, cols] with leading dimension ld -> 2-D map, box 32 columns x 32 rows, no swizzle
static int make_rows_map(CUtensorMap* m, const float* base, int64_t rows, int64_t cols, int64_t ld) {
    EncodeTiledFn fn = encode_fn();
    SPGNN_REQUIRE(fn, "cuTensorMapEncodeTiled is not available from the driver");
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
    cuuint32_t box[2] = {(cuuint32_t)kCS, (cuuint32_t)kBoxRows};
    cuuint32_t es[2] = {1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, es,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    SPGNN_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d) rows=%lld cols=%lld ld=%lld", (int)r,
                  (long long)rows, (long long)cols, (long long)ld);
    return SPGNN_OK;
}

static bool applicable(const Args& a, const spgnn_gat_layer* L) {
    return L->node_off && L->B > 0 && L->max_nodes > 0 && L->max_nodes <= kMaxNodes && L->max_degree > 0 &&
           L->max_degree <= 4 && !a.mean_heads && a.F % 64 == 0 && a.H <= 8 && (a.ldy * 4) % 16 == 0 &&
           (a.res_mode == 0 || a.res_mode == 1);
}

static int setup(TArgs& t, const Args& a, const spgnn_gat_layer* L, CUtensorMap* zmap) {
    t.a = a; t.node_off = L->node_off; t.B = L->B;
    t.nmax = (int)ceil_div(L->max_nodes, kBoxRows) * kBoxRows;
    t.nslices = a.H * a.F / kCS;
    return make_rows_map(zmap, a.Y, a.N, (int64_t)a.H * a.F, a.ldy);
}

template <int ACT, int THREADS, int KPER>
static int launch_fwd_cfg(const CUtensorMap& zmap, TArgs& t, const Args& a, const spgnn_gat_layer* L, cudaStream_t st,
                          bool* handled) {
    t.nstages = fwd_smem_bytes(t.nmax, a.H, 2) <= kSmemLimit ? 2 : 1;
    const size_t smem = fwd_smem_bytes(t.nmax, a.H, t.nstages);
    if (smem > kSmemLimit) return SPGNN_OK;
    auto fn = gat_tree_fwd_kernel<ACT, THREADS, KPER>;
    static DeviceOnce attr;
    if (attr.pending()) {
        SPGNN_CUDA_OK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemLimit));
        attr.done();
    }
    // fewer trees than SMs: up to nslices CTAs per tree, each with its own slices
    t.split = L->B < sm_count() ? (int)(sm_count() / L->B < t.nslices ? sm_count() / L->B : t.nslices) : 1;
    const unsigned grid = (unsigned)(L->B < sm_count() ? L->B * t.split : sm_count());
    fn<<<grid, THREADS, smem, st>>>(zmap, t);
    SPGNN_LAUNCH_OK();
    *handled = true;
    return SPGNN_OK;
}

// Launch shape of the forward: 512 threads x 5-6 rounds of 64 nodes.  The shapes that help the backward (640 x 4,
// 608 x 4, 896 x 3, 1024 x 3) measured within noise or slower here (0.91 - 0.95 vs 0.92 - 1.04 ms per launch,
// profiles/r02_tree_bwd_variants.txt); SPGNN_TREE_FWD=1 selects 896 x 3-4 for A/B runs.
static int fwd_variant() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("SPGNN_TREE_FWD");
        v = (e && atoi(e) == 1) ? 1 : 0;
    }
    return v;
}

template <int ACT>
static int launch_fwd_act(const CUtensorMap& zmap, TArgs& t, const Args& a, const spgnn_gat_layer* L, cudaStream_t st,
                          bool* handled) {
    const int64_t n = L->max_nodes;
    if (fwd_variant() == 1) {
        if (n <= 3 * 112) return launch_fwd_cfg<ACT, 896, 3>(zmap, t, a, L, st, handled);
        return launch_fwd_cfg<ACT, 896, 4>(zmap, t, a, L, st, handled);
    }
    if (n <= 5 * 64) return launch_fwd_cfg<ACT, 512, 5>(zmap, t, a, L, st, handled);
    return launch_fwd_cfg<ACT, 512, 6>(zmap, t, a, L, st, handled);
}

// returns SPGNN_OK and sets *handled when the tree kernel ran
int launch_fwd(const Args& a, const spgnn_gat_layer* L, cudaStream_t st, bool* handled) {
    *handled = false;
    if (!applicable(a, L)) return SPGNN_OK;
    TArgs t{};
    CUtensorMap zmap;
    int rc = setup(t, a, L, &zmap);
    if (rc) return rc;
    if (a.act == SPGNN_ACT_ELU) return launch_fwd_act<SPGNN_ACT_ELU>(zmap, t, a, L, st, handled);
    if (a.act == SPGNN_ACT_TANH) return launch_fwd_act<SPGNN_ACT_TANH>(zmap, t, a, L, st, handled);
    return launch_fwd_act<0>(zmap, t, a, L, st, handled);
}

// one launch configuration of the backward: threads per CTA, rounds per slice, prefetch depth
template <int NG, int ACT, int THREADS, int KPER, int PF>
static int launch_bwd_cfg(const CUtensorMap& zmap, TArgs& t, const Args& a, const spgnn_gat_layer* L, cudaStream_t st,
                          bool* handled) {
    const int HF = a.H * a.F, nwarps = THREADS / 32;
    t.nstages = bwd_smem_bytes(t.nmax, a.H, HF, 2, nwarps) <= kSmemLimit ? 2 : 1;
    const size_t smem = bwd_smem_bytes(t.nmax, a.H, HF, t.nstages, nwarps);
    if (smem > kSmemLimit) return SPGNN_OK;
    auto fn = gat_tree_bwd_kernel<NG, ACT, THREADS, KPER, PF>;
    static DeviceOnce attr;
    if (attr.pending()) {
        SPGNN_CUDA_OK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemLimit));
        attr.done();
    }
    // fewer than #SMs / H trees: one CTA per (tree, head) — the per-edge dot products of a head accumulate over its
    // slices inside one CTA, so a head is the finest split the backward takes
    t.split = (a.H > 1 && L->B * a.H <= sm_count()) ? a.H : 1;
    const unsigned grid = (unsigned)(L->B < sm_count() ? L->B * t.split : sm_count());
    fn<<<grid, THREADS, smem, st>>>(zmap, t);
    SPGNN_LAUNCH_OK();
    if (L->dbias) {
        tree_dbias_reduce_kernel<<<(unsigned)ceil_div(HF, 128), 128, 0, st>>>(a.dbias_ws, grid, HF, L->dbias);
        SPGNN_LAUNCH_OK();
    }
    *handled = true;
    return SPGNN_OK;
}

// Launch shape of the backward.  Default: 640 threads (20 warps, 96 registers), a slice in 4 rounds of 80 nodes (5 for
// graphs of up to 400 nodes), own rows loaded 3 (2) rounds ahead.  Same-box A/Bs on 4096 trees of 301 nodes
// (profiles/r02_tree_bwd_variants.txt), ms per launch averaged over the step's six launches:
//   512 x 5 rounds, whole-slice prefetch (first generation, 128 registers)  2.04 - 2.09
//   640 x 4, 2 rounds ahead 1.83 - 1.88   |  640 x 4, whole-slice 1.98 - 2.01  |  608 x 4 1.93  |  832 x 3 1.93
//   896 x 3 1.95 - 1.98  |  1024 x 3 (64 registers) 2.10 - 2.14: more warps do not help, the rounds of a slice must
//   divide the tree evenly (301 = 80 + 80 + 80 + 61) because every slice ends in a block barrier.
// SPGNN_TREE_BWD = 0 (first generation) / 1 (896 x 3) / 9 (640 x 4, 2 rounds ahead) keep the alternatives reachable.
static int bwd_variant() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("SPGNN_TREE_BWD");
        v = e ? atoi(e) : 3;
        if (v != 0 && v != 1 && v != 9) v = 3;
    }
    return v;
}

template <int NG, int ACT>
static int launch_bwd_act(const CUtensorMap& zmap, TArgs& t, const Args& a, const spgnn_gat_layer* L, cudaStream_t st,
                          bool* handled) {
    const int64_t n = L->max_nodes;
    switch (bwd_variant()) {
        case 0:
            if (n <= 5 * 64) return launch_bwd_cfg<NG, ACT, 512, 5, 5>(zmap, t, a, L, st, handled);
            return launch_bwd_cfg<NG, ACT, 512, 6, 6>(zmap, t, a, L, st, handled);
        case 1:
            if (n <= 3 * 112) return launch_bwd_cfg<NG, ACT, 896, 3, 2>(zmap, t, a, L, st, handled);
            return launch_bwd_cfg<NG, ACT, 896, 4, 2>(zmap, t, a, L, st, handled);
        case 9:
            if (n <= 4 * 80) return launch_bwd_cfg<NG, ACT, 640, 4, 2>(zmap, t, a, L, st, handled);
            return launch_bwd_cfg<NG, ACT, 640, 5, 2>(zmap, t, a, L, st, handled);
        default:
            if (n <= 4 * 80) return launch_bwd_cfg<NG, ACT, 640, 4, 3>(zmap, t, a, L, st, handled);
            return launch_bwd_cfg<NG, ACT, 640, 5, 2>(zmap, t, a, L, st, handled);
    }
}

int launch_bwd(const Args& a, const spgnn_gat_layer* L, cudaStream_t st, bool* handled) {
    *handled = false;
    if (!applicable(a, L) || a.n_g < 1 || a.n_g > 2) return SPGNN_OK;
    TArgs t{};
    CUtensorMap zmap;
    int rc = setup(t, a, L, &zmap);
    if (rc) return rc;
    if (a.n_g == 1) {
        if (a.act == SPGNN_ACT_ELU) return launch_bwd_act<1, SPGNN_ACT_ELU>(zmap, t, a, L, st, handled);
        if (a.act == SPGNN_ACT_TANH) return launch_bwd_act<1, SPGNN_ACT_TANH>(zmap, t, a, L, st, handled);
        return launch_bwd_act<1, 0>(zmap, t, a, L, st, handled);
    }
    if (a.act == SPGNN_ACT_ELU) return launch_bwd_act<2, SPGNN_ACT_ELU>(zmap, t, a, L, st, handled);
    if (a.act == SPGNN_ACT_TANH) return launch_bwd_act<2, SPGNN_ACT_TANH>(zmap, t, a, L, st, handled);
    return launch_bwd_act<2, 0>(zmap, t, a, L, st, handled);
}

}  // namespace tree
}  // namespace spgnn

SPGNN_REGISTER_SALT(gat_tree)

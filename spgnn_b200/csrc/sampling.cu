// Neighbour sampling and block building for SAGE mini-batches (sampling.DeviceBlockSampler): every layer of
// MultiLayerNeighborSampler.sample_blocks + to_block + Block.__init__ in ONE launch of ONE CTA, plus a row gather for
// the node data.
//
// One CTA because a mini-batch is small (st_sage_3: 64 seeds, fanout 2, 4 layers: at most a few thousand nodes and
// edges per layer) and the layers are a chain of dependent phases (counts -> scan -> draw -> unique -> sort -> CSR):
// a single block separates them with __syncthreads instead of launches or grid barriers.  The two orderings a block
// needs - the extras in ascending global id (torch.unique) and the edges stably by source (the out-CSR) - are both a
// sort of unique 64-bit keys, done by one bitonic sort in shared memory (4096 keys) or, beyond that, the same sort
// over a global scratch buffer: slower, but any size stays correct.
//
// Safety: every global write is checked against the capacity the caller allocated; a miss (or an out-of-range seed,
// a repeated seed, an in_src entry outside [0, N)) sets an error code in sizes[2L] and skips the rest of the work.
// The kernel never traps.  On every path it resets the entries of `pos` it set, so the scratch stays all -1.
#include "common.cuh"

namespace spgnn {
namespace {

constexpr int kThreads = 1024;
constexpr int kWarps = kThreads / kWarp;
constexpr int kSmemKeys = 4096;        // 32 KB of uint64 keys: the whole st_sage_3 envelope sorts in shared memory
constexpr int kMaxLayers = 8;
constexpr uint64_t kPad = ~0ull;

enum : int { kErrNone = 0, kErrCapacity = 1, kErrSeedRange = 2, kErrSeedRepeat = 3, kErrGraph = 4 };

struct LayerOut {
    int32_t *in_ptr, *in_src, *out_ptr, *out_dst, *out_slot;
    int64_t* src_ids;
    int64_t cap_dst, cap_src, cap_e;
    int fanout;
};
struct SampleArgs {
    const int32_t* g_in_ptr; const int32_t* g_in_src; int64_t N;
    const int64_t* seeds; int64_t S;
    int L;
    uint64_t seed, salt;
    int32_t* pos;
    int32_t* edst; int64_t edst_cap;         // destination of every edge of the current layer
    uint64_t* keys_ws; int64_t keys_cap;     // global sort scratch (beyond kSmemKeys)
    int64_t* sizes;                          // [2L + 1]: (num_src, num_edges) per layer, then the error code
    LayerOut layer[kMaxLayers];
};

__device__ __forceinline__ uint64_t layer_base(uint64_t seed, uint64_t salt, int layer) {
    return mix64(seed ^ mix64(salt ^ ((uint64_t)(layer + 1) << 56)));
}
// (key, slot) pairs, ordered lexicographically: the draw keeps the `fanout` smallest
__device__ __forceinline__ bool pair_lt(uint64_t ka, int64_t sa, uint64_t kb, int64_t sb) {
    return ka < kb || (ka == kb && sa < sb);
}

__device__ __forceinline__ void set_err(int* s_err, int code) { atomicCAS(s_err, kErrNone, code); }

// Exclusive scan of v[0..n) in place (one CTA), returns the total.  v holds counts on entry.
__device__ int64_t block_scan_inplace(int32_t* v, int64_t n, int64_t* s_warp) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int64_t carry = 0;
    for (int64_t base = 0; base < n; base += kThreads) {
        const int64_t i = base + threadIdx.x;
        const int64_t x = i < n ? v[i] : 0;
        int64_t inc = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t y = __shfl_up_sync(kFull, inc, o);
            if (lane >= o) inc += y;
        }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            int64_t w = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int64_t y = __shfl_up_sync(kFull, w, o);
                if (lane >= o) w += y;
            }
            s_warp[lane] = w;                     // inclusive over warps
        }
        __syncthreads();
        const int64_t before = carry + (warp > 0 ? s_warp[warp - 1] : 0) + inc - x;
        if (i < n) v[i] = (int32_t)before;
        carry += s_warp[kWarps - 1];
        __syncthreads();
    }
    return carry;
}

// Ascending bitonic sort of a[0..n2), n2 a power of two (generic pointer: shared or global memory).
__device__ void bitonic_sort(uint64_t* a, int64_t n2) {
    for (int64_t k = 2; k <= n2; k <<= 1) {
        for (int64_t j = k >> 1; j > 0; j >>= 1) {
            for (int64_t i = threadIdx.x; i < n2; i += kThreads) {
                const int64_t p = i ^ j;
                if (p > i) {
                    const uint64_t x = a[i], y = a[p];
                    const bool up = (i & k) == 0;
                    if ((x > y) == up) { a[i] = y; a[p] = x; }
                }
            }
            __syncthreads();
        }
    }
}

__device__ __forceinline__ int64_t pow2_at_least(int64_t n) {
    int64_t p = 1;
    while (p < n) p <<= 1;
    return p;
}

__global__ void __launch_bounds__(kThreads, 1) sample_blocks_kernel(const SampleArgs a) {
    __shared__ uint64_t s_keys[kSmemKeys];
    __shared__ int64_t s_warp[kWarps];
    __shared__ int s_err;
    __shared__ int s_nx;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) { s_err = kErrNone; s_nx = 0; }
    for (int i = threadIdx.x; i <= 2 * a.L; i += kThreads) a.sizes[i] = 0;     // a refused call reports empty blocks
    __syncthreads();

    // the current destination list: the seeds, then each layer's source list
    const int64_t* cur = a.seeds;
    int64_t S = a.S;
    // ---- seeds: range check, then pos[seed] = its index (a repeated seed is refused)
    if (S > a.layer[a.L - 1].cap_dst) set_err(&s_err, kErrCapacity);
    __syncthreads();
    if (s_err == kErrNone) {
        for (int64_t i = threadIdx.x; i < S; i += kThreads) {
            const int64_t u = cur[i];
            if (u < 0 || u >= a.N) { set_err(&s_err, kErrSeedRange); continue; }
            if (atomicCAS(a.pos + u, -1, (int32_t)i) != -1) set_err(&s_err, kErrSeedRepeat);
        }
    }
    __syncthreads();
    // extras claimed but not yet written to a source list live in `xkeys[0, nx_live)`; cleanup resets them too
    uint64_t* xkeys = s_keys;
    int64_t nx_live = 0;

    for (int l = a.L - 1; l >= 0 && s_err == kErrNone; --l) {
        const LayerOut& o = a.layer[l];
        const int f = o.fanout;
        // ---- 1. per-destination edge counts -> in_ptr (exclusive scan)
        if (S > o.cap_dst) { set_err(&s_err, kErrCapacity); break; }
        for (int64_t i = threadIdx.x; i < S; i += kThreads) {
            const int64_t u = cur[i];
            const int32_t d = __ldg(a.g_in_ptr + u + 1) - __ldg(a.g_in_ptr + u);
            o.in_ptr[i] = f < 0 ? d : min(d, f);
        }
        __syncthreads();
        const int64_t E = block_scan_inplace(o.in_ptr, S, s_warp);
        if (threadIdx.x == 0) o.in_ptr[S] = (int32_t)min(E, (int64_t)INT32_MAX);
        if (E > o.cap_e || E > a.edst_cap) set_err(&s_err, kErrCapacity);
        __syncthreads();
        if (s_err != kErrNone) break;

        // ---- 2. the draw: one warp per destination; kept edges in ascending CSC slot, global source ids in in_src
        const uint64_t base = layer_base(a.seed, a.salt, l);
        for (int64_t i = warp; i < S; i += kWarps) {
            const int64_t u = cur[i];
            const int64_t beg = __ldg(a.g_in_ptr + u);
            const int64_t d = __ldg(a.g_in_ptr + u + 1) - beg;
            const int64_t e0 = o.in_ptr[i];
            const int64_t k = o.in_ptr[i + 1] - e0;
            if (k == 0) continue;
            // threshold = the k-th smallest (key, slot); keep all when k == d
            uint64_t tk = kPad;
            int64_t ts = INT64_MAX;
            if (k < d) {
                uint64_t pk = 0;
                int64_t ps = -1;                                  // previous round's pick (-inf before the first)
                for (int64_t r = 0; r < k; ++r) {
                    uint64_t bk = kPad;
                    int64_t bs = INT64_MAX;
                    for (int64_t j = lane; j < d; j += 32) {
                        const int64_t s = beg + j;
                        const uint64_t key = mix64(base ^ (uint64_t)s);
                        if (pair_lt(pk, ps, key, s) && pair_lt(key, s, bk, bs)) { bk = key; bs = s; }
                    }
#pragma unroll
                    for (int off = 16; off > 0; off >>= 1) {
                        const uint64_t ok = __shfl_xor_sync(kFull, bk, off);
                        const int64_t os = __shfl_xor_sync(kFull, bs, off);
                        if (pair_lt(ok, os, bk, bs)) { bk = ok; bs = os; }
                    }
                    pk = bk; ps = bs;
                }
                tk = pk; ts = ps;
            }
            int64_t n = 0;
            for (int64_t j0 = 0; j0 < d; j0 += 32) {
                const int64_t j = j0 + lane, s = beg + j;
                bool keep = false;
                if (j < d) keep = k == d || !pair_lt(tk, ts, mix64(base ^ (uint64_t)s), s);
                const unsigned m = __ballot_sync(kFull, keep);
                if (keep) {
                    const int64_t e = e0 + n + __popc(m & ((1u << lane) - 1u));
                    const int32_t src = __ldg(a.g_in_src + s);
                    if (e >= o.cap_e || e >= a.edst_cap || e >= e0 + k) set_err(&s_err, kErrCapacity);
                    else if (src < 0 || src >= a.N) set_err(&s_err, kErrGraph);
                    else { o.in_src[e] = src; a.edst[e] = (int32_t)i; }
                }
                n += __popc(m);
            }
        }
        __syncthreads();
        if (s_err != kErrNone) break;

        // ---- 3. to_block: claim every source not yet in pos (-2 = claimed), collect the claimed ids
        const int64_t cap_x = min(o.cap_src - S, E);        // sources beyond the destinations
        xkeys = pow2_at_least(cap_x) <= kSmemKeys ? s_keys : a.keys_ws;
        const int64_t xcap = xkeys == s_keys ? (int64_t)kSmemKeys : a.keys_cap;
        for (int64_t e = threadIdx.x; e < E; e += kThreads) {
            const int32_t u = o.in_src[e];
            if (*(volatile int32_t*)(a.pos + u) != -1) continue;
            if (atomicCAS(a.pos + u, -1, -2) != -1) continue;
            const int idx = atomicAdd(&s_nx, 1);
            if (idx < xcap && idx < cap_x) xkeys[idx] = (uint64_t)u;
            else { a.pos[u] = -1; set_err(&s_err, kErrCapacity); }
        }
        __syncthreads();
        const int64_t X = min((int64_t)s_nx, min(xcap, max(cap_x, (int64_t)0)));
        nx_live = X;
        if (s_err != kErrNone) break;
        // ---- 4. extras in ascending global id after the destinations
        const int64_t x2 = pow2_at_least(X);
        for (int64_t i = X + threadIdx.x; i < x2; i += kThreads) xkeys[i] = kPad;
        __syncthreads();
        bitonic_sort(xkeys, x2);
        const int64_t n_src = S + X;
        for (int64_t i = threadIdx.x; i < n_src; i += kThreads) {
            const int64_t u = i < S ? cur[i] : (int64_t)xkeys[i - S];
            o.src_ids[i] = u;                                    // n_src <= cap_src: cap_x = cap_src - S
            if (i >= S) a.pos[u] = (int32_t)i;
        }
        __syncthreads();
        nx_live = 0;
        if (threadIdx.x == 0) s_nx = 0;

        // ---- 5. local source ids; out-CSR = stable sort of the edges by source: keys (local src << 32 | slot)
        uint64_t* ek = pow2_at_least(o.cap_e) <= kSmemKeys ? s_keys : a.keys_ws;
        const int64_t ekcap = ek == s_keys ? (int64_t)kSmemKeys : a.keys_cap;
        const int64_t e2 = pow2_at_least(E);
        if (e2 > ekcap) { set_err(&s_err, kErrCapacity); }
        __syncthreads();
        if (s_err != kErrNone) { cur = o.src_ids; S = n_src; break; }
        for (int64_t e = threadIdx.x; e < e2; e += kThreads) {
            if (e < E) {
                const int32_t loc = a.pos[o.in_src[e]];
                o.in_src[e] = loc;
                ek[e] = ((uint64_t)(uint32_t)loc << 32) | (uint64_t)e;
            } else {
                ek[e] = kPad;
            }
        }
        __syncthreads();
        bitonic_sort(ek, e2);
        for (int64_t j = threadIdx.x; j < E; j += kThreads) {
            const uint64_t kv = ek[j];
            const int64_t s = (int64_t)(kv >> 32), e = (int64_t)(kv & 0xffffffffull);
            o.out_slot[j] = (int32_t)e;
            o.out_dst[j] = a.edst[e];
            const int64_t prev = j == 0 ? -1 : (int64_t)(ek[j - 1] >> 32);
            for (int64_t t = prev + 1; t <= s && t <= n_src; ++t) o.out_ptr[t] = (int32_t)j;
        }
        {
            const int64_t last = E == 0 ? -1 : (int64_t)(ek[E - 1] >> 32);
            for (int64_t t = last + 1 + threadIdx.x; t <= n_src; t += kThreads) o.out_ptr[t] = (int32_t)E;
        }
        __syncthreads();
        if (threadIdx.x == 0) { a.sizes[2 * l] = n_src; a.sizes[2 * l + 1] = E; }
        cur = o.src_ids;
        S = n_src;
    }
    __syncthreads();

    // ---- cleanup: pos entries of the last source list (a superset of every earlier one) and of claimed extras
    for (int64_t i = threadIdx.x; i < S; i += kThreads) {
        const int64_t u = cur[i];
        if (u >= 0 && u < a.N) a.pos[u] = -1;
    }
    for (int64_t i = threadIdx.x; i < nx_live; i += kThreads) a.pos[xkeys[i]] = -1;
    if (threadIdx.x == 0) a.sizes[2 * a.L] = s_err;
}

// out[r, :] = x[idx[r], :] as 32-bit words, for r < min(cap, *count) (count == null: r < cap)
__global__ void gather_rows_kernel(const uint32_t* __restrict__ x, int64_t ldx, const int64_t* __restrict__ idx,
                                   const int64_t* __restrict__ count, int64_t cap, int64_t words, int64_t n_rows,
                                   uint32_t* __restrict__ out, int64_t ldo) {
    const int64_t n = count ? min(cap, *count) : cap;
    for (int64_t r = blockIdx.x; r < n; r += gridDim.x) {
        const int64_t u = idx[r];
        if (u < 0 || u >= n_rows) continue;
        const uint32_t* src = x + u * ldx;
        uint32_t* dst = out + r * ldo;
        for (int64_t c = threadIdx.x; c < words; c += blockDim.x) dst[c] = __ldg(src + c);
    }
}

}  // namespace
}  // namespace spgnn

extern "C" int spgnn_sample_blocks(const int32_t* in_ptr, const int32_t* in_src, int64_t N, const int64_t* seeds,
                                   int64_t S, int64_t L, const int64_t* fanouts_host, const int64_t* caps_host,
                                   const int64_t* bufs_host, uint64_t seed, uint64_t salt, int32_t* pos,
                                   int32_t* edst_ws, int64_t edst_cap, uint64_t* keys_ws, int64_t keys_cap,
                                   int64_t* sizes, void* stream) {
    using namespace spgnn;
    SPGNN_REQUIRE(in_ptr && in_src && seeds && fanouts_host && caps_host && bufs_host && pos && edst_ws && sizes,
                  "sample_blocks: null pointer");
    SPGNN_REQUIRE(N > 0 && N <= INT32_MAX && S >= 0 && L >= 1 && L <= kMaxLayers,
                  "sample_blocks: N = %lld, S = %lld, L = %lld out of range", (long long)N, (long long)S, (long long)L);
    SPGNN_REQUIRE(edst_cap >= 0 && edst_cap <= INT32_MAX && keys_cap >= 0 && (keys_cap & (keys_cap - 1)) == 0 &&
                  (keys_cap == 0 || keys_ws), "sample_blocks: bad scratch (keys_cap must be 0 or a power of two)");
    SampleArgs a{};
    a.g_in_ptr = in_ptr; a.g_in_src = in_src; a.N = N; a.seeds = seeds; a.S = S; a.L = (int)L;
    a.seed = seed; a.salt = salt; a.pos = pos; a.edst = edst_ws; a.edst_cap = edst_cap;
    a.keys_ws = keys_ws; a.keys_cap = keys_cap; a.sizes = sizes;
    for (int64_t l = 0; l < L; ++l) {
        LayerOut& o = a.layer[l];
        const int64_t* c = caps_host + 3 * l;
        const int64_t* b = bufs_host + 6 * l;
        SPGNN_REQUIRE(fanouts_host[l] >= -1 && fanouts_host[l] <= INT32_MAX, "sample_blocks: fanout %lld",
                      (long long)fanouts_host[l]);
        for (int k = 0; k < 3; ++k)
            SPGNN_REQUIRE(c[k] >= 0 && c[k] <= INT32_MAX - 1, "sample_blocks: capacity %lld of layer %lld",
                          (long long)c[k], (long long)l);
        SPGNN_REQUIRE(c[1] >= c[0], "sample_blocks: layer %lld has fewer source than destination slots", (long long)l);
        SPGNN_REQUIRE(l == L - 1 || (caps_host + 3 * (l + 1))[1] <= c[0],
                      "sample_blocks: layer %lld cannot take layer %lld's sources as destinations", (long long)l,
                      (long long)(l + 1));
        // in_ptr / out_ptr always hold one entry; an edge or source buffer of capacity 0 may be null
        SPGNN_REQUIRE(b[0] && b[2] && (c[2] == 0 || (b[1] && b[3] && b[4])) && (c[1] == 0 || b[5]),
                      "sample_blocks: null buffer of layer %lld", (long long)l);
        o.in_ptr = (int32_t*)b[0]; o.in_src = (int32_t*)b[1]; o.out_ptr = (int32_t*)b[2];
        o.out_dst = (int32_t*)b[3]; o.out_slot = (int32_t*)b[4]; o.src_ids = (int64_t*)b[5];
        o.cap_dst = c[0]; o.cap_src = c[1]; o.cap_e = c[2];
        o.fanout = fanouts_host[l] < 0 ? -1 : (int)fanouts_host[l];
    }
    cudaStream_t st = as_stream(stream);
    sample_blocks_kernel<<<1, kThreads, 0, st>>>(a);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

extern "C" int spgnn_gather_rows(const void* x, int64_t ldx_words, int64_t n_rows, const int64_t* idx,
                                 const int64_t* count, int64_t cap, int64_t words, void* out, int64_t ldo_words,
                                 void* stream) {
    using namespace spgnn;
    SPGNN_REQUIRE(x && idx && out && n_rows >= 0 && cap >= 0 && words > 0 && ldx_words >= words && ldo_words >= words,
                  "gather_rows: bad argument");
    if (cap == 0) return SPGNN_OK;
    const int threads = words >= 256 ? 256 : 64;
    const int blocks = (int)(cap < 4LL * sm_count() ? cap : 4LL * sm_count());
    gather_rows_kernel<<<blocks, threads, 0, as_stream(stream)>>>((const uint32_t*)x, ldx_words, idx, count, cap,
                                                                 words, n_rows, (uint32_t*)out, ldo_words);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

// Callers of the path kept on device: masked weighted cross-entropy (job_runner.py:1885-1900) and the
// SGD-momentum update over a flat parameter bucket (torch.optim.SGD semantics, job_runner.py:1919), and the
// Adam / AdamW update a settings file can name instead (torch.optim.Adam / AdamW semantics).
#include "common.cuh"

namespace spgnn {

constexpr int kT = 256;

__device__ __forceinline__ bool keep_node(const int64_t* y, const uint8_t* mask, float rate, uint64_t seed, int64_t i) {
    if (mask) return mask[i] != 0;
    return y[i] != 0 || u01(seed, (uint64_t)i) < rate;
}

__global__ void __launch_bounds__(kT) masked_ce_fwd_kernel(const float* __restrict__ logits, int64_t ld, int C,
                                                           const int64_t* __restrict__ y,
                                                           const uint8_t* __restrict__ mask, float rate, uint64_t seed,
                                                           const float* __restrict__ cw, int64_t N,
                                                           double* __restrict__ sums) {
    __shared__ double sh[2][kT / 32];
    double nll = 0.0, wsum = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
        if (!keep_node(y, mask, rate, seed, i)) continue;
        const float* row = logits + i * ld;
        float m = -INFINITY;
        for (int c = 0; c < C; ++c) m = fmaxf(m, __ldg(row + c));
        float s = 0.f;
        for (int c = 0; c < C; ++c) s += expf(__ldg(row + c) - m);
        const int64_t t = y[i];
        const float w = __ldg(cw + t);
        nll += (double)(w * (logf(s) + m - __ldg(row + t)));
        wsum += (double)w;
    }
    nll = warp_sum(nll);
    wsum = warp_sum(wsum);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) { sh[0][wid] = nll; sh[1][wid] = wsum; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, b = 0.0;
        for (int k = 0; k < kT / 32; ++k) { a += sh[0][k]; b += sh[1][k]; }
        atomicAdd(&sums[0], a);
        atomicAdd(&sums[1], b);
    }
}

__global__ void __launch_bounds__(kT) masked_ce_bwd_kernel(const float* __restrict__ logits, int64_t ld, int C,
                                                           const int64_t* __restrict__ y,
                                                           const uint8_t* __restrict__ mask, float rate, uint64_t seed,
                                                           const float* __restrict__ cw,
                                                           const double* __restrict__ sums, float scale, int64_t N,
                                                           float* __restrict__ dl, int64_t ldd) {
    const float k = (float)((double)scale / sums[1]);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
        float* drow = dl + i * ldd;
        if (!keep_node(y, mask, rate, seed, i)) {
            for (int c = 0; c < C; ++c) drow[c] = 0.f;
            continue;
        }
        const float* row = logits + i * ld;
        float m = -INFINITY;
        for (int c = 0; c < C; ++c) m = fmaxf(m, __ldg(row + c));
        float s = 0.f;
        for (int c = 0; c < C; ++c) s += expf(__ldg(row + c) - m);
        const int64_t t = y[i];
        const float w = __ldg(cw + t) * k;
        const float inv = 1.f / s;
        for (int c = 0; c < C; ++c) drow[c] = w * (expf(__ldg(row + c) - m) * inv - (c == t ? 1.f : 0.f));
    }
}

__global__ void sgd_momentum_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ buf,
                                    int64_t n, float lr, float mu, float gs, int first) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float gi = g[i] * gs;
        const float b = first ? gi : fmaf(mu, buf[i], gi);
        buf[i] = b;
        p[i] -= lr * b;
    }
}

// torch.optim.SGD._single_tensor_sgd (torch/optim/sgd.py): g += wd*p; buf = first ? g : mu*buf + (1-damp)*g;
// g = nesterov ? g + mu*buf : buf (only with momentum); p -= lr*g
__global__ void sgd_step_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ buf, int64_t n,
                                float lr, float mu, float damp, float wd, int nesterov, float gs, int first) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float pi = p[i];
        float gi = g[i] * gs;
        if (wd != 0.f) gi = fmaf(wd, pi, gi);
        if (mu != 0.f) {
            const float b = first ? gi : fmaf(mu, buf[i], (1.f - damp) * gi);
            buf[i] = b;
            gi = nesterov ? fmaf(mu, b, gi) : b;
        }
        p[i] = pi - lr * gi;
    }
}

// torch.optim.Adam / AdamW (_single_tensor_adam, torch/optim/adam.py) over the live chunks of a flat bucket.  The step
// counters are per parameter and live in device memory, so a CUDA-graph replay of the step sees the count advance:
// adam_count_kernel bumps the counter of every live parameter, then adam_step_kernel reads it (one block per chunk,
// so all blocks of a parameter see the same t) and forms the bias corrections in fp64, as torch does in Python floats.
struct AdamArgs {
    double lr, beta1, beta2, eps, wd;
    int amsgrad, maximize, decoupled;
};

__global__ void adam_count_kernel(int64_t* __restrict__ steps, const int64_t* __restrict__ live, int64_t n_live) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_live; i += (int64_t)gridDim.x * blockDim.x)
        steps[live[i]] += 1;
}

struct AdamScalars {
    float neg_step_size, bc2_sqrt, beta2, one_m_beta1, one_m_beta2, eps, wd, decay;
};

__device__ __forceinline__ void adam_elem(float& p, float g, float& m, float& v, float* vmax, const AdamScalars& s,
                                          const AdamArgs& a) {
    if (a.maximize) g = -g;
    if (a.wd != 0.0) {
        if (a.decoupled) p *= s.decay;
        else g = fmaf(p, s.wd, g);
    }
    // exp_avg.lerp_(g, 1 - beta1): torch's lerp switches formula at weight 0.5
    m = s.one_m_beta1 < 0.5f ? fmaf(s.one_m_beta1, g - m, m) : g - (g - m) * (1.f - s.one_m_beta1);
    v = fmaf(s.one_m_beta2 * g, g, v * s.beta2);
    float vv = v;
    if (a.amsgrad) { vv = fmaxf(*vmax, v); *vmax = vv; }
    p = fmaf(s.neg_step_size, m / (sqrtf(vv) / s.bc2_sqrt + s.eps), p);
}

// chunks: n_chunks x {offset, length, parameter index}; a chunk lies inside one parameter
__global__ void __launch_bounds__(kT) adam_step_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                       float* __restrict__ m, float* __restrict__ v,
                                                       float* __restrict__ vmax, const int64_t* __restrict__ steps,
                                                       const int64_t* __restrict__ chunks, AdamArgs a) {
    __shared__ AdamScalars sh;
    const int64_t* c = chunks + 3 * (int64_t)blockIdx.x;
    const int64_t off = c[0], len = c[1];
    if (threadIdx.x == 0) {
        const double t = (double)steps[c[2]];
        const double bc1 = 1.0 - pow(a.beta1, t), bc2 = 1.0 - pow(a.beta2, t);
        sh.neg_step_size = (float)(-a.lr / bc1);
        sh.bc2_sqrt = (float)sqrt(bc2);
        sh.beta2 = (float)a.beta2;
        sh.one_m_beta1 = (float)(1.0 - a.beta1);
        sh.one_m_beta2 = (float)(1.0 - a.beta2);
        sh.eps = (float)a.eps;
        sh.wd = (float)a.wd;
        sh.decay = (float)(1.0 - a.lr * a.wd);
    }
    __syncthreads();
    const AdamScalars s = sh;
    // scalar head up to a 16-byte boundary, float4 body, scalar tail
    const int64_t head = min(len, (int64_t)((4 - (off & 3)) & 3));
    const int64_t nvec = (len - head) >> 2, tail0 = head + 4 * nvec;
    for (int64_t k = threadIdx.x; k < head + (len - tail0); k += kT) {
        const int64_t i = off + (k < head ? k : tail0 - head + k);
        float pi = p[i], mi = m[i], vi = v[i];
        adam_elem(pi, g[i], mi, vi, vmax ? vmax + i : nullptr, s, a);
        p[i] = pi; m[i] = mi; v[i] = vi;
    }
    const int64_t b = off + head;
    for (int64_t k = threadIdx.x; k < nvec; k += kT) {
        const int64_t i = b + 4 * k;
        float4 pv = *reinterpret_cast<const float4*>(p + i), mv = *reinterpret_cast<const float4*>(m + i);
        float4 vv = *reinterpret_cast<const float4*>(v + i);
        const float4 gv = ldg4(g + i);
        float4 xv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (a.amsgrad) xv = *reinterpret_cast<const float4*>(vmax + i);
        adam_elem(pv.x, gv.x, mv.x, vv.x, &xv.x, s, a);
        adam_elem(pv.y, gv.y, mv.y, vv.y, &xv.y, s, a);
        adam_elem(pv.z, gv.z, mv.z, vv.z, &xv.z, s, a);
        adam_elem(pv.w, gv.w, mv.w, vv.w, &xv.w, s, a);
        st4(p + i, pv); st4(m + i, mv); st4(v + i, vv);
        if (a.amsgrad) st4(vmax + i, xv);
    }
}

static inline unsigned egrid(int64_t n) {
    int64_t want = ceil_div(n, kT), cap = (int64_t)sm_count() * 8;
    if (want < 1) want = 1;
    return (unsigned)(want < cap ? want : cap);
}

}  // namespace spgnn

using namespace spgnn;

extern "C" int spgnn_masked_ce_fwd(const float* logits, int64_t ld, int64_t n_class, const int64_t* y,
                                   const uint8_t* mask, float rate, uint64_t seed, const float* class_w, int64_t N,
                                   double* sums, void* stream) {
    SPGNN_REQUIRE(logits && y && class_w && sums && N > 0 && n_class > 1 && ld >= n_class, "masked_ce_fwd: bad argument");
    cudaStream_t st = as_stream(stream);
    SPGNN_CUDA_OK(cudaMemsetAsync(sums, 0, 2 * sizeof(double), st));
    masked_ce_fwd_kernel<<<egrid(N), kT, 0, st>>>(logits, ld, (int)n_class, y, mask, rate, seed, class_w, N, sums);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

extern "C" int spgnn_masked_ce_bwd(const float* logits, int64_t ld, int64_t n_class, const int64_t* y,
                                   const uint8_t* mask, float rate, uint64_t seed, const float* class_w,
                                   const double* sums, float scale, int64_t N, float* dlogits, int64_t ldd,
                                   void* stream) {
    SPGNN_REQUIRE(logits && y && class_w && sums && dlogits && N > 0 && n_class > 1 && ld >= n_class && ldd >= n_class,
                  "masked_ce_bwd: bad argument");
    masked_ce_bwd_kernel<<<egrid(N), kT, 0, as_stream(stream)>>>(logits, ld, (int)n_class, y, mask, rate, seed, class_w,
                                                                 sums, scale, N, dlogits, ldd);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

extern "C" int spgnn_sgd_step(float* p, const float* g, float* buf, int64_t n, float lr, float mu, float dampening,
                              float weight_decay, int nesterov, float grad_scale, int first_step, void* stream) {
    SPGNN_REQUIRE(p && g && n > 0 && (buf || mu == 0.f), "sgd_step: bad argument");
    SPGNN_REQUIRE(!nesterov || (mu > 0.f && dampening == 0.f), "sgd_step: nesterov needs momentum > 0 and dampening == 0");
    sgd_step_kernel<<<egrid(n), kT, 0, as_stream(stream)>>>(p, g, buf, n, lr, mu, dampening, weight_decay, nesterov,
                                                           grad_scale, first_step);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

extern "C" int spgnn_adam_step(float* p, const float* g, float* exp_avg, float* exp_avg_sq, float* max_exp_avg_sq,
                               int64_t* steps, const int64_t* chunks, int64_t n_chunks, const int64_t* live,
                               int64_t n_live, double lr, double beta1, double beta2, double eps, double weight_decay,
                               int amsgrad, int maximize, int decoupled, void* stream) {
    SPGNN_REQUIRE(p && g && exp_avg && exp_avg_sq && steps && chunks && live && n_chunks > 0 && n_live > 0 &&
                  n_chunks < (int64_t)INT32_MAX, "adam_step: bad argument");
    SPGNN_REQUIRE(beta1 >= 0.0 && beta1 < 1.0 && beta2 >= 0.0 && beta2 < 1.0, "adam_step: betas must be in [0, 1)");
    SPGNN_REQUIRE(eps >= 0.0 && lr >= 0.0 && weight_decay >= 0.0, "adam_step: lr, eps and weight_decay must be >= 0");
    SPGNN_REQUIRE((max_exp_avg_sq != nullptr) == (amsgrad != 0), "adam_step: max_exp_avg_sq is needed iff amsgrad");
    const uintptr_t align = (uintptr_t)p | (uintptr_t)g | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq |
                            (uintptr_t)max_exp_avg_sq;
    SPGNN_REQUIRE((align & 15) == 0, "adam_step: bucket pointers must be 16-byte aligned");
    cudaStream_t st = as_stream(stream);
    adam_count_kernel<<<(unsigned)ceil_div(n_live, kT), kT, 0, st>>>(steps, live, n_live);
    SPGNN_LAUNCH_OK();
    const AdamArgs a{lr, beta1, beta2, eps, weight_decay, amsgrad != 0, maximize != 0, decoupled != 0};
    adam_step_kernel<<<(unsigned)n_chunks, kT, 0, st>>>(p, g, exp_avg, exp_avg_sq, max_exp_avg_sq, steps, chunks, a);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

extern "C" int spgnn_sgd_momentum(float* p, const float* g, float* buf, int64_t n, float lr, float mu,
                                  float grad_scale, int first_step, void* stream) {
    SPGNN_REQUIRE(p && g && buf && n > 0, "sgd_momentum: bad argument");
    sgd_momentum_kernel<<<egrid(n), kT, 0, as_stream(stream)>>>(p, g, buf, n, lr, mu, grad_scale, first_step);
    SPGNN_LAUNCH_OK();
    return SPGNN_OK;
}

SPGNN_REGISTER_SALT(train)

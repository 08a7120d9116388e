// Shared device/host helpers for libspgnn_b200 (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include "../../include/spgnn_b200.h"

namespace spgnn {

void set_error(const char* fmt, ...);
void count_launch();

#define SPGNN_REQUIRE(cond, ...)                               \
    do {                                                       \
        if (!(cond)) {                                         \
            spgnn::set_error(__VA_ARGS__);                     \
            return SPGNN_E_INVALID;                            \
        }                                                      \
    } while (0)

#define SPGNN_CUDA_OK(expr)                                                                   \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            spgnn::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return SPGNN_E_CUDA;                                                              \
        }                                                                                     \
    } while (0)

// every kernel launch goes through this: counts launches (bench.py's gpu_launches) and checks the launch status
#define SPGNN_LAUNCH_OK()                      \
    do {                                       \
        spgnn::count_launch();                 \
        SPGNN_CUDA_OK(cudaGetLastError());     \
    } while (0)

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
int sm_count();
// One-time per-DEVICE setup (cudaFuncSetAttribute is a per-device property: a process-wide flag would leave a second
// GPU, or the device after a cudaDeviceReset, without the opt-in to > 48 KB of dynamic shared memory).  pending()
// is true until done() was called for the current device; setting an attribute twice from two threads is harmless.
struct DeviceOnce {
    unsigned long long mask = 0;
    bool pending() const;
    void done();
};

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFull, v, o));
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// activation on the pre-activation x
__device__ __forceinline__ float act_fwd(float x, int act, float slope) {
    switch (act) {
        case SPGNN_ACT_ELU: return x > 0.f ? x : expm1f(x);
        case SPGNN_ACT_TANH: return tanhf(x);
        case SPGNN_ACT_RELU: return fmaxf(x, 0.f);
        case SPGNN_ACT_LEAKY: return x > 0.f ? x : slope * x;
        default: return x;
    }
}
// lean variants for the bandwidth-bound aggregation kernels (a handful of instructions instead of the libm
// expansions; absolute error ~1e-7, far inside the 1e-4 parity bar)
// exp(x) as one FMUL + MUFU.EX2 (flush-to-zero; __expf adds a denormal-range fix-up of ~6 instructions per call)
__device__ __forceinline__ float exp_fast(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x * 1.4426950408889634f));
    return y;
}
// Slope of SPGNN_ACT_LEAKY as the activation of a GAT layer (gat.cu, gat_layer.cu, gat_tree.cu and the aggregate-first
// output layer of gemm_tma.cu): GATConv takes its activation as a callable, and F.leaky_relu applies its default
// negative_slope of 0.01.  Kernels whose activation comes with an explicit slope (linear, spmm, max-pool) pass it.
constexpr float kGatLeakySlope = 0.01f;
__device__ __forceinline__ float act_fast(float x, int act) {
    if (act == SPGNN_ACT_ELU) return x > 0.f ? x : exp_fast(x) - 1.f;
    if (act == SPGNN_ACT_TANH) return 1.f - __fdividef(2.f, exp_fast(2.f * x) + 1.f);
    if (act == SPGNN_ACT_RELU) return fmaxf(x, 0.f);
    if (act == SPGNN_ACT_LEAKY) return x > 0.f ? x : kGatLeakySlope * x;
    return x;
}
// derivative expressed through the OUTPUT y = act(x)
__device__ __forceinline__ float act_grad_from_out(float y, int act, float slope) {
    switch (act) {
        case SPGNN_ACT_ELU: return y > 0.f ? 1.f : y + 1.f;
        case SPGNN_ACT_TANH: return 1.f - y * y;
        case SPGNN_ACT_RELU: return y > 0.f ? 1.f : 0.f;
        case SPGNN_ACT_LEAKY: return y > 0.f ? 1.f : slope;
        default: return 1.f;
    }
}

// Per-step salt of every dropout / sampling seed.  Seeds are kernel ARGUMENTS (host-side counters): a training step
// replayed from a CUDA graph would draw the same masks every time.  The salt lives in constant memory (one copy per
// translation unit, read through the constant cache at no cost), is 0 in eager execution and is refreshed by the
// first nodes of a captured step from a device-side counter (spgnn_seed_salt_set: one D2D cudaMemcpyToSymbolAsync
// per translation unit, itself captured), so replay k uses seed + k * golden-ratio for every mask of the step.
static __constant__ unsigned long long g_seed_salt = 0ull;
typedef int (*SaltSetter)(const void* dev_src, cudaStream_t st);
struct SaltRegistrar { explicit SaltRegistrar(SaltSetter fn); };
#define SPGNN_REGISTER_SALT(tag)                                                                              \
    static int set_seed_salt_##tag(const void* dev_src, cudaStream_t st) {                                   \
        return (int)cudaMemcpyToSymbolAsync(spgnn::g_seed_salt, dev_src, sizeof(unsigned long long), 0,      \
                                            cudaMemcpyDeviceToDevice, st);                                   \
    }                                                                                                         \
    static spgnn::SaltRegistrar salt_registrar_##tag(set_seed_salt_##tag);
__host__ __device__ __forceinline__ uint64_t salted(uint64_t seed) {
#ifdef __CUDA_ARCH__
    return seed + g_seed_salt * 0x9E3779B97F4A7C15ull;
#else
    return seed;
#endif
}

// Counter-based hash -> uniform in [0,1): two rounds of a 64-bit finaliser (splitmix64).  Used for
// dropout / node-sampling masks so that backward can regenerate the forward mask from (seed, index).
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
// 64 mask bits for one 4-column chunk of a feat_drop mask (16 bits per element): two murmur3-style 32-bit
// finalisers over (seed, chunk index) — 32-bit multiplies only, a third of the instructions of mix64 on the
// bandwidth-bound plane producers.  Every producer / consumer of a planes dropout mask uses this one function.
__host__ __device__ __forceinline__ uint32_t fmix32(uint32_t h) {
    h ^= h >> 16; h *= 0x85EBCA6Bu;
    h ^= h >> 13; h *= 0xC2B2AE35u;
    return h ^ (h >> 16);
}
__host__ __device__ __forceinline__ uint64_t chunk_hash(uint64_t seed, uint64_t idx) {
    seed = salted(seed);
    const uint32_t lo = (uint32_t)idx, hi = (uint32_t)(idx >> 32);
    const uint32_t a = fmix32(((uint32_t)seed ^ (lo * 0x9E3779B1u)) + hi * 0x85EBCA77u);
    const uint32_t b = fmix32(((uint32_t)(seed >> 32) ^ (lo * 0xC2B2AE3Du) ^ a) + hi * 0x27D4EB2Fu);
    return (uint64_t)a | ((uint64_t)b << 32);
}
__host__ __device__ __forceinline__ float u01(uint64_t seed, uint64_t idx) {
    uint64_t h = mix64(salted(seed) ^ mix64(idx));
    return (float)(uint32_t)(h >> 40) * (1.0f / 16777216.0f);   // 24 random bits
}

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

}  // namespace spgnn

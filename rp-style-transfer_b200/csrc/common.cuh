// Shared device/host helpers for librpst (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <string.h>

#include "../../include/rpst.h"
#ifdef RPST_DEBUG_EXPORTS
#include "../../include/rpst_debug.h"
#endif

namespace rpst {

// ---------------------------------------------------------------- host: error plumbing
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define RPST_CHECK_ARG(cond, ...)                 \
    do {                                          \
        if (!(cond)) {                            \
            ::rpst::set_error(__VA_ARGS__);       \
            return RPST_ERR_INVALID;              \
        }                                         \
    } while (0)

#define RPST_CUDA(call)                                              \
    do {                                                             \
        cudaError_t e__ = (call);                                    \
        if (e__ != cudaSuccess) return ::rpst::cuda_fail(e__, #call);\
    } while (0)

int sm_count();

// cudaFuncSetAttribute is per device: a process that drives several GPUs (one host thread each, SURVEY.md §8b
// threading contract) must configure every kernel once PER DEVICE, not once per process.
struct PerDeviceFlag {
    bool done[64] = {};
    bool& get() {
        int d = 0;
        if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= 64) d = 0;
        return done[d];
    }
};

// WCT covariance kernels (cov.cu / wct.cu): production choice, or one forced (tests)
enum CovPath : int { kCovPathAuto = 0, kCovPathTma = 1, kCovPathStaged = 2, kCovPathPack = 3 };

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ---------------------------------------------------------------- device: memory ops
#ifdef __CUDACC__

__device__ __forceinline__ uint64_t policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}

// 128-bit streaming load that bypasses L1 and carries an L2 eviction policy.
__device__ __forceinline__ float4 ldg_f4_hint(const float* p, uint64_t pol) {
    float4 v;
    asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ float ldg_f1_hint(const float* p, uint64_t pol) {
    float v;
    asm volatile("ld.global.L1::no_allocate.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(v) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ void stg_f4_hint(float* p, float4 v, uint64_t pol) {
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;"
                 :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol) : "memory");
}
__device__ __forceinline__ void stg_f1_hint(float* p, float v, uint64_t pol) {
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.f32 [%0], %1, %2;" :: "l"(p), "f"(v), "l"(pol) : "memory");
}

__device__ __forceinline__ int ld_acquire(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(int* p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}

// ---------------------------------------------------------------- device: running moments
// (count, mean, sum of squared deviations) with Chan's pairwise merge — the numerically safe way
// to get an unbiased variance out of a tree reduction (network/base.py:404 uses torch.var).
struct Moments {
    float n, mean, m2;
};

__device__ __forceinline__ Moments merge(Moments a, Moments b) {
    float n = a.n + b.n;
    float inv = n > 0.f ? 1.f / n : 0.f;
    float d = b.mean - a.mean;
    float w = b.n * inv;
    Moments r;
    r.n = n;
    r.mean = a.mean + d * w;
    r.m2 = a.m2 + b.m2 + d * d * a.n * w;
    return r;
}

__device__ __forceinline__ Moments warp_merge(Moments m) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        Moments other;
        other.n = __shfl_xor_sync(0xffffffffu, m.n, o);
        other.mean = __shfl_xor_sync(0xffffffffu, m.mean, o);
        other.m2 = __shfl_xor_sync(0xffffffffu, m.m2, o);
        m = merge(m, other);
    }
    return m;
}

// Block-wide merge; every thread returns the block total.  `scratch` must hold 32 Moments and is
// safe to reuse after the call only across a __syncthreads() (callers alternate two buffers).
template <int THREADS>
__device__ __forceinline__ Moments block_merge(Moments m, Moments* scratch) {
    constexpr int W = THREADS / 32;
    m = warp_merge(m);
    if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = m;
    __syncthreads();
    Moments t = scratch[0];
#pragma unroll
    for (int w = 1; w < W; ++w) t = merge(t, scratch[w]);
    return t;
}

struct MomentsD {
    double n, mean, m2;
};
__device__ __forceinline__ MomentsD merge(MomentsD a, MomentsD b) {
    double n = a.n + b.n;
    double inv = n > 0.0 ? 1.0 / n : 0.0;
    double d = b.mean - a.mean;
    double w = b.n * inv;
    MomentsD r;
    r.n = n;
    r.mean = a.mean + d * w;
    r.m2 = a.m2 + b.m2 + d * d * a.n * w;
    return r;
}
__device__ __forceinline__ MomentsD warp_merge(MomentsD m) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        MomentsD other;
        other.n = __shfl_xor_sync(0xffffffffu, m.n, o);
        other.mean = __shfl_xor_sync(0xffffffffu, m.mean, o);
        other.m2 = __shfl_xor_sync(0xffffffffu, m.m2, o);
        m = merge(m, other);
    }
    return m;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

#endif  // __CUDACC__

}  // namespace rpst

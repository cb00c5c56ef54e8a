// Register-batch plane I/O and the lag-pipeline schedule shared by the AdaIN-family kernels (adain.cu, seg.cu).
#pragma once
#include "common.cuh"
#include "async.cuh"

namespace rpst {

constexpr int kBatch = 4;          // vectors per load batch
constexpr int kBatches = 2;        // batches per thread per item
constexpr int kPerThread = kBatch * kBatches;
constexpr int kPipeThreads = 256;

template <int VEC>
__device__ __forceinline__ void load_vec(float (&dst)[VEC], const float* p, uint64_t pol, bool hint) {
    if constexpr (VEC == 4) {
        float4 v = hint ? ldg_f4_hint(p, pol) : __ldg(reinterpret_cast<const float4*>(p));
        dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
    } else {
        dst[0] = hint ? ldg_f1_hint(p, pol) : __ldg(p);
    }
}
template <int VEC>
__device__ __forceinline__ void store_vec(float* p, const float (&src)[VEC], uint64_t pol, bool hint) {
    if constexpr (VEC == 4) {
        float4 v = make_float4(src[0], src[1], src[2], src[3]);
        if (hint) stg_f4_hint(p, v, pol); else *reinterpret_cast<float4*>(p) = v;
    } else {
        if (hint) stg_f1_hint(p, src[0], pol); else *p = src[0];
    }
}

// Load one batch (kBatch vectors, strided by THREADS vectors) of a chunk that holds `nvec` vectors.
template <int VEC, int THREADS>
__device__ __forceinline__ void load_batch(float (&v)[kBatch][VEC], const float* base, int batch, int nvec,
                                           uint64_t pol, bool hint, int tid = threadIdx.x) {
#pragma unroll
    for (int j = 0; j < kBatch; ++j) {
        int idx = (batch * kBatch + j) * THREADS + tid;
        if (idx < nvec) {
            load_vec<VEC>(v[j], base + (int64_t)idx * VEC, pol, hint);
        } else {
#pragma unroll
            for (int e = 0; e < VEC; ++e) v[j][e] = 0.f;
        }
    }
}

// Exact two-pass moments of the valid part of a register batch, merged into `acc`.
template <int VEC, int THREADS>
__device__ __forceinline__ void batch_moments(Moments& acc, const float (&v)[kBatch][VEC], int batch, int nvec,
                                              int tid = threadIdx.x) {
    float sum = 0.f;
    int cnt = 0;
#pragma unroll
    for (int j = 0; j < kBatch; ++j) {
        int idx = (batch * kBatch + j) * THREADS + tid;
        if (idx < nvec) {
#pragma unroll
            for (int e = 0; e < VEC; ++e) sum += v[j][e];
            cnt += VEC;
        }
    }
    if (cnt == 0) return;
    Moments m;
    m.n = (float)cnt;
    m.mean = sum / m.n;
    float m2 = 0.f;
#pragma unroll
    for (int j = 0; j < kBatch; ++j) {
        int idx = (batch * kBatch + j) * THREADS + tid;
        if (idx < nvec) {
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
                float d = v[j][e] - m.mean;
                m2 = fmaf(d, d, m2);
            }
        }
    }
    m.m2 = m2;
    acc = merge(acc, m);
}

__device__ __forceinline__ float std_from(const Moments& m, float hw, float eps) {
    // unbiased: divide by HW-1 (0/0 -> NaN for HW==1, like torch.var)
    return sqrtf(m.m2 / (hw - 1.f) + eps);
}

// ---------------------------------------------------------------- lag pipelines
// Persistent CTAs take tickets in order.  The statistics items of plane r+lag run interleaved with the apply items of
// plane r, so that a plane's content is still in L2 when its apply items read it again.

// Planes between a plane's statistics and its apply (host): enough planes to cover `lag_bytes`, at least 3, at most
// `planes`.
inline int lag_planes(int64_t lag_bytes, int64_t plane_bytes, int64_t planes) {
    int64_t lag = (lag_bytes + plane_bytes - 1) / plane_bytes;
    if (lag < 3) lag = 3;
    return (int)(lag < planes ? lag : planes);
}

struct LagItem {
    int kind;        // 0 statistics, 1 apply
    int64_t plane;
    int chunk;       // among the plane's statistics items, or among its apply items
};

// Ticket t -> item.  Prologue: the statistics items of planes [0, lag).  Steady round r: [the statistics items of
// plane r+lag][the apply items of plane r].  Epilogue: the apply items of the last `lag` planes.  lag == planes is a
// statistics-only schedule.  32-bit arithmetic: callers keep the ticket count below 2^31.
__device__ __forceinline__ LagItem decode_lag(unsigned t, unsigned planes, unsigned lag, unsigned stats_pp,
                                              unsigned apply_pp) {
    LagItem it;
    const unsigned pro = lag * stats_pp;
    if (t < pro) {
        it.kind = 0; it.plane = t / stats_pp; it.chunk = (int)(t % stats_pp);
        return it;
    }
    t -= pro;
    const unsigned round = stats_pp + apply_pp;
    const unsigned steady = (planes - lag) * round;
    if (t < steady) {
        const unsigned r = t / round, u = t % round;
        it.kind = u >= stats_pp;
        it.chunk = (int)(it.kind ? u - stats_pp : u);
        it.plane = it.kind ? r : r + lag;
        return it;
    }
    t -= steady;
    it.kind = 1; it.plane = (planes - lag) + t / apply_pp; it.chunk = (int)(t % apply_pp);
    return it;
}

// Plane gate of the register-staged lag pipelines whose last statistics item finishes the plane: each statistics
// item arrives on done[plane]; the last arriver combines the plane's partial results and publishes ready[plane];
// the plane's apply items wait for it.  Both counters are zeroed before the launch.
//
// gate_arrive: CTA-wide; returns to every thread whether this item was the last of the plane's `items`.
//  * Before the call, the item's partial results are visible GPU-wide: each thread that wrote some fenced, and when
//    threads other than thread 0 wrote, a barrier follows their fences.
//  * After a true return, the threads that read the other items' partial results fence before reading.
__device__ __forceinline__ bool gate_arrive(int* done, int items, int& s_last) {
    if (threadIdx.x == 0) s_last = atomicAdd(done, 1) == items - 1;
    __syncthreads();
    return s_last;
}
// gate_publish: one thread, once the plane's result is visible GPU-wide (every writer fenced; other threads' writes are
// also ordered before the call by a barrier).
__device__ __forceinline__ void gate_publish(int* ready) {
    st_release(ready, 1);
}
// gate_wait: one thread; the plane's result may be read after the wait.
__device__ __forceinline__ void gate_wait(const int* ready) {
    int v = ld_acquire(ready);
    spin_wait(100, [&] { v = ld_acquire(ready); }, [&] { return v != 0; });
}

}  // namespace rpst

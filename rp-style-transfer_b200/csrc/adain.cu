// AdaIN family (SURVEY.md §8 a1/a2/a3/a8/a15): per-(n,c) plane statistics, normalise-affine,
// multiscale blend, concat-write — hand-written for sm_100a, HBM-bound by design.
//
// Two kernels:
//  * adain_direct_kernel  — planes that fit one CTA's registers (<= 32 floats/thread, <= 512 threads): one CTA per
//    plane, content is read ONCE from HBM and stays in registers between the statistics and the
//    apply phase.
//  * adain_pipe_kernel    — larger planes (512x512 = 1 MiB, 1024x2048 = 8 MiB ...): a persistent
//    kernel whose warps each walk a static, ordered list of 4 KiB work items.  Statistics items of
//    plane p+D are interleaved with apply items of plane p, so that the second read of the content
//    (apply) is served by the 126 MB L2 (the content lines are loaded with an evict_last policy,
//    every other stream with evict_first) and HBM sees each tensor exactly once: the algorithmic
//    3*E*4 (AdaIN) / 4*E*4 (blend) bytes of SURVEY.md §8d.  An apply item waits on a per-plane
//    release/acquire flag set by the CTA that finished the plane's last statistics item; items
//    are walked in order by co-resident warps and statistics items never block, so the wait cannot deadlock.
//
// Numerics (SURVEY.md Appendix B): unbiased variance, eps inside the sqrt (network/base.py:404-405);
// moments are accumulated as (count, mean, M2) with a two-pass evaluation over each thread's
// registers and Chan merges above that, never as raw sum/sum-of-squares.
#include "common.cuh"
#include "plane_io.cuh"
#include "async.cuh"
#include "tuning.cuh"

namespace rpst {
namespace {

constexpr int kItemElems = 4096;  // one work item: 16 KiB of each tensor (256 threads x 4 float4)

// Unsigned 32-bit division by a launch-time constant (Granlund-Montgomery round-up method): two multiplies and
// shifts instead of the ~20-instruction software division; the ticket decode of the TMA kernel does up to eight
// of them per batch on the producer's critical path.
struct FastDiv {
    uint32_t d, m, sh1, sh2;
};
inline FastDiv make_fastdiv(uint32_t d) {
    FastDiv f;
    f.d = d < 1u ? 1u : d;
    uint32_t l = 0;
    while ((1ull << l) < f.d) ++l;                                   // ceil(log2 d)
    f.m = (uint32_t)((((1ull << l) - f.d) << 32) / f.d + 1ull);
    f.sh1 = l < 1u ? l : 1u;
    f.sh2 = l > 0u ? l - 1u : 0u;
    return f;
}
__device__ __forceinline__ uint32_t fdiv(uint32_t n, const FastDiv& f) {
    const uint32_t t = __umulhi(f.m, n);
    return (t + ((n - t) >> f.sh1)) >> f.sh2;
}

struct AdainParams {
    const float* content;
    const float* style;  // may be null
    const float* prev;   // may be null
    float* out;
    float* mean_out;     // stats-only mode
    float* std_out;
    float* saved;        // [planes,4] or null
    int64_t planes, hw, channels, out_batch_stride;
    float eps;
    int stats_only;
    int hints;
    // pipelined kernel only
    int ipp;             // items (chunks) per plane
    int ips;             // TMA kernel: statistics items per plane (ipp with a style tensor; ceil(ipp/2) without:
                         // the item then carries two content chunks — calc_mean_std / mean_variance_norm)
    int ipa;             // TMA kernel: apply items per plane (ipp with prev; ceil(ipp/2) without: an apply item
                         // then carries two content chunks, so every stage moves 32 KiB whatever the item kind)
    int spp;             // statistics slots per plane
    int slot_elems;      // elements summarised by one slot (last slot of a plane may be short)
    int lag;             // planes between statistics and apply
    unsigned total_items;
    unsigned* ticket;    // starts at 0xFFFFFFFF
    float4* coef;        // [planes] (mu_c hi, a, mu_s, mu_c lo); 0xFF-filled = not merged yet
    float4* part;        // [planes*ipp] (mean_c, m2_c, mean_s, m2_s); 0xFF-filled = not written yet
    // channel shuffle / sort folded into the loads (network/adain_rp.py:230-249,304-311): output plane p
    // takes its content from plane cmap[p] and its style from plane smap[p] (null = identity)
    const int* cmap;
    const int* smap;
    FastDiv div_s, div_s1, div_s1a, div_a1, div_a;   // by ips, ips+1, ips+1+ipa, ipa+1, ipa (decode_tma)
    int group_merge_min_spp;   // TMA kernel: planes with at least this many statistics slots are merged by the whole group
    int merge_lead;            // TMA kernel: planes between a plane's MERGE ticket and its first APPLY ticket (1 .. lag-1)
};

__device__ __forceinline__ int64_t src_plane(const int* map, int64_t plane) {
    return map ? (int64_t)__ldg(map + plane) : plane;
}

// ------------------------------------------------------------------------------------------
// direct kernel: one CTA per plane, content stays in registers
// ------------------------------------------------------------------------------------------
template <int VEC, int THREADS>
__global__ void __launch_bounds__(THREADS) adain_direct_kernel(AdainParams p) {
    __shared__ Moments scratch[2][32];
    const uint64_t pol_first = policy_evict_first();
    const bool hint = p.hints != 0;
    const int nvec = (int)(p.hw / VEC);
    const float hwf = (float)p.hw;

    for (int64_t plane = blockIdx.x; plane < p.planes; plane += gridDim.x) {
        const float* cbase = p.content + src_plane(p.cmap, plane) * p.hw;
        float c[kBatches][kBatch][VEC];
        Moments mc = {0.f, 0.f, 0.f}, ms = {0.f, 0.f, 0.f};
#pragma unroll
        for (int b = 0; b < kBatches; ++b) load_batch<VEC, THREADS>(c[b], cbase, b, nvec, pol_first, hint);
        if (p.style != nullptr) {
            const float* sbase = p.style + src_plane(p.smap, plane) * p.hw;
#pragma unroll
            for (int b = 0; b < kBatches; ++b) {
                float s[kBatch][VEC];
                load_batch<VEC, THREADS>(s, sbase, b, nvec, pol_first, hint);
                batch_moments<VEC, THREADS>(ms, s, b, nvec);
            }
        }
#pragma unroll
        for (int b = 0; b < kBatches; ++b) batch_moments<VEC, THREADS>(mc, c[b], b, nvec);

        mc = block_merge<THREADS>(mc, scratch[0]);
        float mu_c = mc.mean, sd_c = std_from(mc, hwf, p.eps);
        float mu_s = 0.f, sd_s = 1.f;
        if (p.style != nullptr) {
            ms = block_merge<THREADS>(ms, scratch[1]);
            mu_s = ms.mean;
            sd_s = std_from(ms, hwf, p.eps);
        }
        if (threadIdx.x == 0) {
            if (p.mean_out) p.mean_out[plane] = mu_c;
            if (p.std_out) p.std_out[plane] = sd_c;
            if (p.saved) reinterpret_cast<float4*>(p.saved)[plane] = make_float4(mu_c, sd_c, mu_s, sd_s);
        }
        if (!p.stats_only) {
            const float a = sd_s / sd_c;
            const int64_t n_idx = plane / p.channels, ch = plane % p.channels;
            float* obase = p.out + n_idx * p.out_batch_stride + ch * p.hw;
            const float* pbase = p.prev ? p.prev + plane * p.hw : nullptr;
#pragma unroll
            for (int b = 0; b < kBatches; ++b) {
                float pv[kBatch][VEC];
                if (pbase) load_batch<VEC, THREADS>(pv, pbase, b, nvec, pol_first, hint);
#pragma unroll
                for (int j = 0; j < kBatch; ++j) {
                    int idx = (b * kBatch + j) * THREADS + threadIdx.x;
                    if (idx < nvec) {
                        float o[VEC];
#pragma unroll
                        for (int e = 0; e < VEC; ++e) {
                            float y = fmaf(c[b][j][e] - mu_c, a, mu_s);
                            o[e] = pbase ? y + pv[j][e] : y;
                        }
                        store_vec<VEC>(obase + (int64_t)idx * VEC, o, pol_first, hint);
                    }
                }
            }
        }
        __syncthreads();  // scratch reuse across the grid-stride loop
    }
}

// ------------------------------------------------------------------------------------------
// pipelined kernel: persistent CTAs + ticket counter, statistics D planes ahead of apply
// ------------------------------------------------------------------------------------------
struct Item {
    int kind;  // 0 statistics, 1 apply
    int64_t plane;
    int chunk;
};

__device__ __forceinline__ Item decode_ticket(unsigned t, const AdainParams& p) {
    Item it;
    const int64_t ipp = p.ipp;
    if (p.stats_only) {
        it.kind = 0; it.plane = t / ipp; it.chunk = (int)(t % ipp);
        return it;
    }
    const int64_t lag = p.lag < p.planes ? p.lag : p.planes;
    int64_t tt = t;
    if (tt < lag * ipp) {  // prologue: statistics only
        it.kind = 0; it.plane = tt / ipp; it.chunk = (int)(tt % ipp);
        return it;
    }
    tt -= lag * ipp;
    const int64_t steady = (p.planes - lag) * 2 * ipp;
    if (tt < steady) {  // steady state: alternate statistics(plane r+lag) / apply(plane r)
        int64_t r = tt / (2 * ipp), u = tt % (2 * ipp);
        it.kind = (int)(u & 1);
        it.chunk = (int)(u >> 1);
        it.plane = it.kind ? r : r + lag;
        return it;
    }
    tt -= steady;  // epilogue: apply only
    it.kind = 1; it.plane = (p.planes - lag) + tt / ipp; it.chunk = (int)(tt % ipp);
    return it;
}

// Hand-off without fences or atomics.  A statistics item publishes its chunk moments as ONE
// 16-byte slot {mean_c, M2_c, mean_s, M2_s}; the slot array is memset to 0xFF before the launch and a
// component whose bits are still 0xFFFFFFFF means "not written yet" (a computed value is never that
// bit pattern: results are canonicalised).  Data and "valid" marker being the same word, no ordering
// between separate locations is needed, hence no __threadfence / counter / last-arriver logic.  An
// apply item first looks at the plane's merged-coefficient slot (same sentinel scheme); on a miss its
// warp 0 polls the plane's partial slots, merges them in fp64 and publishes the coefficients (every
// merger computes bit-identical values, so concurrent publication is benign and deterministic).
// Items are handed out in schedule order by a ticket counter (one atomic per item, prefetched);
// statistics items never wait, so polling always terminates.  Exactly one __syncthreads per item.
__device__ __forceinline__ bool slot_valid(const float4& v) {
    return __float_as_uint(v.x) != 0xffffffffu && __float_as_uint(v.y) != 0xffffffffu &&
           __float_as_uint(v.z) != 0xffffffffu && __float_as_uint(v.w) != 0xffffffffu;
}
__device__ __forceinline__ float canon(float v) {
    return __float_as_uint(v) == 0xffffffffu ? __uint_as_float(0x7fc00000u) : v;
}
__device__ __forceinline__ float4 ld_slot(const float4* p) {
    float4 v;
    asm volatile("ld.relaxed.gpu.global.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_slot(float4* p, float4 v) {
    asm volatile("st.relaxed.gpu.global.v4.f32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "f"(canon(v.x)), "f"(canon(v.y)), "f"(canon(v.z)), "f"(canon(v.w)) : "memory");
}

// schedule: prologue = statistics of the first `lag` planes; steady round r = [statistics of plane
// r+lag][apply of plane r]; epilogue = apply of the last `lag` planes.
__device__ __forceinline__ Item decode_item(unsigned t, const AdainParams& p) {
    Item it;
    const unsigned ipp = (unsigned)p.ipp;
    if (p.stats_only) {
        it.kind = 0; it.plane = t / ipp; it.chunk = (int)(t % ipp);
        return it;
    }
    const unsigned planes = (unsigned)p.planes;
    const unsigned lag = (unsigned)p.lag < planes ? (unsigned)p.lag : planes;
    const unsigned pro = lag * ipp;
    if (t < pro) {
        it.kind = 0; it.plane = t / ipp; it.chunk = (int)(t % ipp);
        return it;
    }
    t -= pro;
    const unsigned steady = (planes - lag) * 2u * ipp;
    if (t < steady) {
        const unsigned r = t / (2u * ipp), u = t % (2u * ipp);
        it.kind = u >= ipp;
        it.chunk = (int)(it.kind ? u - ipp : u);
        it.plane = it.kind ? r : r + lag;
        return it;
    }
    t -= steady;
    it.kind = 1; it.plane = (planes - lag) + t / ipp; it.chunk = (int)(t % ipp);
    return it;
}

// Merge the chunk moments of one plane (full warp).  All arithmetic is fp32 but relative to the
// first chunk's mean K, so the result keeps the plane mean to better than fp32 (returned as hi+lo):
//   mean = K + d,  d = sum n_k (mean_k - K) / N,   M2 = sum M2_k + sum n_k (mean_k - K - d)^2
// Every caller computes bit-identical values (fixed lane assignment, fixed reduction tree).
// Up to 256 slots (planes of <= 256 Ki elements, e.g. 512x512): every lane keeps its <= 8 slots in registers —
// all loads in flight at once instead of one validity branch (= one L2 round trip) per slot, and the second
// pass needs no reload.  Same arithmetic in the same order as the generic path below: bit-identical results.
__device__ __forceinline__ float4 merge_plane_coef_small(const AdainParams& p, int64_t plane, int lane) {
    const float4* slots = p.part + plane * p.spp;
    float4 v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        const int k = lane + 32 * u;
        v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (k < p.spp) v[u] = ld_slot(slots + k);
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        const int k = lane + 32 * u;
        if (k < p.spp && !slot_valid(v[u])) {   // straggling statistics item: wait for it
            const uint64_t t0 = global_timer_ns();
            do {
                __nanosleep(40);
                v[u] = ld_slot(slots + k);
                if (watchdog_expired(t0)) __trap();
            } while (!slot_valid(v[u]));
        }
    }
    const float kc = __shfl_sync(0xffffffffu, v[0].x, 0), ks = __shfl_sync(0xffffffffu, v[0].z, 0);
    float dc = 0.f, ds = 0.f;
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        const int k = lane + 32 * u;
        if (k < p.spp) {
            const int64_t rem = p.hw - (int64_t)k * p.slot_elems;
            const float n = (float)(rem < p.slot_elems ? rem : p.slot_elems);
            dc = fmaf(n, v[u].x - kc, dc);
            ds = fmaf(n, v[u].z - ks, ds);
        }
    }
    const float inv_n = 1.f / (float)p.hw;
    dc = warp_sum(dc) * inv_n;
    ds = warp_sum(ds) * inv_n;
    float m2c = 0.f, m2s = 0.f;
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        const int k = lane + 32 * u;
        if (k < p.spp) {
            const int64_t rem = p.hw - (int64_t)k * p.slot_elems;
            const float n = (float)(rem < p.slot_elems ? rem : p.slot_elems);
            const float ec = v[u].x - kc - dc, es = v[u].z - ks - ds;
            m2c += fmaf(n * ec, ec, v[u].y);
            m2s += fmaf(n * es, es, v[u].w);
        }
    }
    m2c = warp_sum(m2c);
    m2s = warp_sum(m2s);
    const float mu_hi = kc + dc;
    const float mu_lo = (kc - mu_hi) + dc;
    const float denom = (float)p.hw - 1.f;
    const float sd_c = sqrtf(m2c / denom + p.eps);
    float mu_s = 0.f, sd_s = 1.f;
    if (p.style != nullptr) {
        mu_s = ks + ds;
        sd_s = sqrtf(m2s / denom + p.eps);
    }
    const float4 cf = make_float4(mu_hi, sd_s / sd_c, mu_s, mu_lo);
    if (lane == 0) {
        st_slot(&p.coef[plane], cf);
        if (p.saved) reinterpret_cast<float4*>(p.saved)[plane] = make_float4(mu_hi, sd_c, mu_s, sd_s);
    }
    return cf;
}

__device__ __forceinline__ float4 merge_plane_coef(const AdainParams& p, int64_t plane, int lane) {
    const float4* slots = p.part + plane * p.spp;
    // pass 1 (polling): K = first chunk's means, d = sum n_k (mean_k - K) / N
    float4 v0 = ld_slot(slots);
    if (!slot_valid(v0)) {
        const uint64_t t0 = global_timer_ns();
        do {
            __nanosleep(40);
            v0 = ld_slot(slots);
            if (watchdog_expired(t0)) __trap();
        } while (!slot_valid(v0));
    }
    const float kc = v0.x, ks = v0.z;
    float dc = 0.f, ds = 0.f;
    for (int k = lane; k < p.spp; k += 32) {
        float4 v = ld_slot(slots + k);
        if (!slot_valid(v)) {  // straggling statistics item: wait for it
            const uint64_t t0 = global_timer_ns();
            do {
                __nanosleep(40);
                v = ld_slot(slots + k);
                if (watchdog_expired(t0)) __trap();
            } while (!slot_valid(v));
        }
        const int64_t rem = p.hw - (int64_t)k * p.slot_elems;
        const float n = (float)(rem < p.slot_elems ? rem : p.slot_elems);
        dc = fmaf(n, v.x - kc, dc);
        ds = fmaf(n, v.z - ks, ds);
    }
    const float inv_n = 1.f / (float)p.hw;
    dc = warp_sum(dc) * inv_n;
    ds = warp_sum(ds) * inv_n;
    // pass 2 (all slots are valid now; L2 hits)
    float m2c = 0.f, m2s = 0.f;
    for (int k = lane; k < p.spp; k += 32) {
        const float4 v = ld_slot(slots + k);
        const int64_t rem = p.hw - (int64_t)k * p.slot_elems;
        const float n = (float)(rem < p.slot_elems ? rem : p.slot_elems);
        const float ec = v.x - kc - dc, es = v.z - ks - ds;
        m2c += fmaf(n * ec, ec, v.y);
        m2s += fmaf(n * es, es, v.w);
    }
    m2c = warp_sum(m2c);
    m2s = warp_sum(m2s);
    const float mu_hi = kc + dc;
    const float mu_lo = (kc - mu_hi) + dc;  // Fast2Sum remainder (|kc| >= |dc| in all but degenerate planes)
    const float denom = (float)p.hw - 1.f;
    const float sd_c = sqrtf(m2c / denom + p.eps);
    float mu_s = 0.f, sd_s = 1.f;
    if (p.style != nullptr) {
        mu_s = ks + ds;
        sd_s = sqrtf(m2s / denom + p.eps);
    }
    const float4 cf = make_float4(mu_hi, sd_s / sd_c, mu_s, mu_lo);
    if (lane == 0) {
        st_slot(&p.coef[plane], cf);
        if (p.saved) reinterpret_cast<float4*>(p.saved)[plane] = make_float4(mu_hi, sd_c, mu_s, sd_s);
    }
    return cf;
}

template <int VEC, int MINB>
__global__ void __launch_bounds__(kPipeThreads, MINB) adain_pipe_kernel(AdainParams p) {
    constexpr int T = kPipeThreads;
    constexpr int NB = kItemElems / (T * kBatch * VEC);  // register batches per thread per tensor
    static_assert(NB >= 1, "item too small");
    __shared__ Moments scratch[2][2][T / 32];
    __shared__ float4 s_coef[2];
    __shared__ unsigned s_next[2];

    const uint64_t pol_first = policy_evict_first();
    const uint64_t pol_last = policy_evict_last();
    const bool hint = p.hints != 0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool has_style = p.style != nullptr;
    unsigned parity = 0;

    // dynamic schedule: the ticket word starts at 0xFFFFFFFF (workspace memset), so old+1 counts from 0.
    // The ticket of the NEXT item is requested at the top of an item (latency hidden behind the data
    // loads) and broadcast through the item's single barrier.
    if (threadIdx.x == 0) s_next[0] = atomicAdd(p.ticket, 1u) + 1u;
    __syncthreads();
    unsigned t = s_next[0];

    for (; t < p.total_items; t = s_next[parity ^ 1u], parity ^= 1u) {
        unsigned nxt = 0;
        if (threadIdx.x == 0) nxt = atomicAdd(p.ticket, 1u) + 1u;
        const Item it = decode_item(t, p);
        const int64_t e0 = (int64_t)it.chunk * kItemElems;
        const int64_t rem = p.hw - e0;
        const int nvec = (int)((rem < kItemElems ? rem : kItemElems) / VEC);
        const float* cbase = p.content + src_plane(p.cmap, it.plane) * p.hw + e0;

        if (it.kind == 0) {
            // ---------------- statistics item
            float c[NB][kBatch][VEC], s[NB][kBatch][VEC];
            const uint64_t cpol = p.stats_only ? pol_first : pol_last;
#pragma unroll
            for (int b = 0; b < NB; ++b) load_batch<VEC, T>(c[b], cbase, b, nvec, cpol, hint);
            if (has_style) {
                const float* sbase = p.style + src_plane(p.smap, it.plane) * p.hw + e0;
#pragma unroll
                for (int b = 0; b < NB; ++b) load_batch<VEC, T>(s[b], sbase, b, nvec, pol_first, hint);
            }
            Moments mc = {0.f, 0.f, 0.f}, ms = {0.f, 0.f, 0.f};
#pragma unroll
            for (int b = 0; b < NB; ++b) batch_moments<VEC, T>(mc, c[b], b, nvec);
            mc = warp_merge(mc);
            if (has_style) {
#pragma unroll
                for (int b = 0; b < NB; ++b) batch_moments<VEC, T>(ms, s[b], b, nvec);
                ms = warp_merge(ms);
            }
            if (lane == 0) {
                scratch[parity][0][warp] = mc;
                scratch[parity][1][warp] = ms;
            }
            if (threadIdx.x == 0) s_next[parity ^ 1u] = nxt;
            __syncthreads();
            if (threadIdx.x == 0) {
                Moments tc = scratch[parity][0][0], ts = scratch[parity][1][0];
#pragma unroll
                for (int w = 1; w < T / 32; ++w) {
                    tc = merge(tc, scratch[parity][0][w]);
                    ts = merge(ts, scratch[parity][1][w]);
                }
                st_slot(&p.part[it.plane * p.spp + it.chunk], make_float4(tc.mean, tc.m2, ts.mean, ts.m2));
            }
        } else {
            // ---------------- apply item: content comes back from L2, prev streams from HBM
            const float* pbase = p.prev ? p.prev + it.plane * p.hw + e0 : nullptr;
            const int64_t n_idx = it.plane / p.channels, ch = it.plane % p.channels;
            float* obase = p.out + n_idx * p.out_batch_stride + ch * p.hw + e0;
            float c[NB][kBatch][VEC], pv[NB][kBatch][VEC];
#pragma unroll
            for (int b = 0; b < NB; ++b) {
                load_batch<VEC, T>(c[b], cbase, b, nvec, pol_first, hint);
                if (pbase) load_batch<VEC, T>(pv[b], pbase, b, nvec, pol_first, hint);
            }
            if (warp == 0) {
                float4 cf = ld_slot(&p.coef[it.plane]);
                if (!slot_valid(cf)) cf = merge_plane_coef(p, it.plane, lane);
                if (lane == 0) {
                    s_coef[parity] = cf;
                    s_next[parity ^ 1u] = nxt;
                }
            }
            __syncthreads();
            const float4 cf = s_coef[parity];
            const float mu_hi = cf.x, a = cf.y, mu_s = cf.z, mu_lo = cf.w;
#pragma unroll
            for (int b = 0; b < NB; ++b) {
#pragma unroll
                for (int j = 0; j < kBatch; ++j) {
                    int idx = (b * kBatch + j) * T + threadIdx.x;
                    if (idx < nvec) {
                        float o[VEC];
#pragma unroll
                        for (int e = 0; e < VEC; ++e) {
                            float y = fmaf((c[b][j][e] - mu_hi) - mu_lo, a, mu_s);
                            o[e] = pbase ? y + pv[b][j][e] : y;
                        }
                        store_vec<VEC>(obase + (int64_t)idx * VEC, o, pol_first, hint);
                    }
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// TMA-staged pipelined kernel (the default for 16-byte-aligned planes).
//
// One persistent CTA per SM.  Warp 0 is the PRODUCER: one thread takes tickets (two at a time, the
// next request always in flight), decodes them and streams the item's 16 KiB chunks into a ring of
// shared-memory stages with cp.async.bulk (TMA, 1-D: planes are contiguous), completion counted on
// the stage's `full` mbarrier.  So the bytes in flight live in shared memory (STAGES x 32 KiB, up to
// 224 KiB per SM), not in registers, and nobody blocks on a global load.  Each stage has its own
// CONSUMER group of four warps: statistics items reduce the chunk(s) to (mean, M2) and publish the
// 16-byte slot; apply items read content (L2 hit) and prev from the stage, the plane coefficients
// from the descriptor (the producer bulk-copied the 16-byte coefficient slot along with the data)
// and store the result with 128-bit evict-first stores; the group then hands the stage back through
// the `empty` mbarrier.  A third item kind, MERGE (one per plane, scheduled between the plane's
// statistics and apply items), turns the chunk slots into the coefficient slot so that apply items
// almost never have to wait.
// ------------------------------------------------------------------------------------------
constexpr int kTmaGroupWarps = 4;
constexpr int kTmaGroupThreads = kTmaGroupWarps * 32;
constexpr int kTmaSlotElems = kItemElems / kTmaGroupWarps;   // one warp summarises 1024 contiguous elements
constexpr int kTmaVecs = kTmaSlotElems / 4 / 32;             // float4 per lane per tensor per item (8)
constexpr int kTicketBatch = 8;   // 4 was measured: mean_variance_norm 4.7 -> 5.8 TB/s (a plane's last statistics ticket
                                  // waits behind fewer items of its SM's batch) but plain 6.4 -> 6.1 and blend 6.9 -> 6.2

// moments of 4*kTmaVecs register values per lane, then a warp tree.  `full` (warp-uniform): every lane
// holds exactly 4*kTmaVecs valid values, so every merge joins equal counts and needs no division.
__device__ __forceinline__ Moments warp_moments(const float4 (&v)[kTmaVecs], int valid_vecs, bool full) {
    Moments m = {0.f, 0.f, 0.f};
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < kTmaVecs; ++j)
        if (j < valid_vecs) sum += (v[j].x + v[j].y) + (v[j].z + v[j].w);
    m.n = 4.f * (float)valid_vecs;
    m.mean = valid_vecs > 0 ? sum / m.n : 0.f;
#pragma unroll
    for (int j = 0; j < kTmaVecs; ++j) {
        if (j < valid_vecs) {
            const float d0 = v[j].x - m.mean, d1 = v[j].y - m.mean, d2 = v[j].z - m.mean, d3 = v[j].w - m.mean;
            m.m2 = fmaf(d0, d0, m.m2);
            m.m2 = fmaf(d1, d1, m.m2);
            m.m2 = fmaf(d2, d2, m.m2);
            m.m2 = fmaf(d3, d3, m.m2);
        }
    }
    if (full) {
        float half_n = 2.f * kTmaVecs;  // n/2 of the two sides being joined
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const float om = __shfl_xor_sync(0xffffffffu, m.mean, o);
            const float o2 = __shfl_xor_sync(0xffffffffu, m.m2, o);
            const float d = om - m.mean;
            m.mean = fmaf(d, 0.5f, m.mean);
            m.m2 = fmaf(d * d, half_n, m.m2 + o2);
            half_n *= 2.f;
        }
        m.n = 128.f * kTmaVecs;
        return m;
    }
    return warp_merge(m);
}

struct __align__(16) StageDesc {
    float4 coef;    // apply items: written by TMA
    int64_t plane;
    int kind;       // 0 statistics, 1 apply, 2 merge, -1 stop
    int chunk;
    int nvec;       // valid float4 in buffer a
    int nvec2;      // apply items without prev: valid float4 of the SECOND content chunk in buffer b
    int pad[2];
};

struct DecodedItem {
    int64_t plane, cplane, splane;   // output plane, source planes of content / style
    int kind, chunk;
};

__device__ __forceinline__ void decode_tma(unsigned t, const AdainParams& p, int& kind, int64_t& plane, int& chunk) {
    const unsigned I = (unsigned)p.ips;    // statistics items per plane
    if (p.stats_only) { const unsigned q = fdiv(t, p.div_s); kind = 0; plane = q; chunk = (int)(t - q * I); return; }
    const unsigned P = (unsigned)p.planes, L = (unsigned)p.lag, Lm = (unsigned)p.merge_lead, A = (unsigned)p.ipa;
    // rounds: [S only] x (L-Lm), [S,M] x Lm, [S,M,A] x (P-L), [M,A] x (L-Lm), [A] x Lm
    unsigned n = (L - Lm) * I;
    if (t < n) { const unsigned q = fdiv(t, p.div_s); kind = 0; plane = q; chunk = (int)(t - q * I); return; }
    t -= n; n = Lm * (I + 1);
    if (t < n) {
        const unsigned j = fdiv(t, p.div_s1), u = t - j * (I + 1);
        if (u < I) { kind = 0; plane = (L - Lm) + j; chunk = (int)u; }
        else { kind = 2; plane = j; chunk = 0; }
        return;
    }
    t -= n; n = (P - L) * (I + 1 + A);
    if (t < n) {
        const unsigned j = fdiv(t, p.div_s1a), u = t - j * (I + 1 + A);
        if (u < I) { kind = 0; plane = L + j; chunk = (int)u; }
        else if (u == I) { kind = 2; plane = Lm + j; chunk = 0; }
        else { kind = 1; plane = j; chunk = (int)(u - I - 1); }
        return;
    }
    t -= n; n = (L - Lm) * (A + 1);
    if (t < n) {
        const unsigned j = fdiv(t, p.div_a1), u = t - j * (A + 1);
        if (u == 0) { kind = 2; plane = (P - L + Lm) + j; chunk = 0; }
        else { kind = 1; plane = (P - L) + j; chunk = (int)(u - 1); }
        return;
    }
    t -= n;
    const unsigned q = fdiv(t, p.div_a);
    kind = 1; plane = (P - Lm) + q; chunk = (int)(t - q * A);
}

// Plane merge by a whole consumer group (128 threads), used by the TMA kernel's MERGE items.  A plane of
// 1024x2048 has 2048 statistics slots; folded by one warp in two dependent passes that was ~64 serialized
// round trips per pass (2.25 TB/s forward at that plane size).  Here thread t takes slots t, t+128, ... with
// all of its loads in flight at once, folds them with Chan's update in fp64 (no common shift needed, so a
// single pass), and the 128 partials are merged by a fixed shuffle tree + a fixed 4-warp order: one memory
// round trip per plane, bit-reproducible.
struct MomD {
    double n, mc, m2c, ms, m2s;
};
__device__ __forceinline__ MomD momd_merge(const MomD& a, const MomD& b) {
    MomD r;
    r.n = a.n + b.n;
    if (r.n == 0.0) { r.mc = r.m2c = r.ms = r.m2s = 0.0; return r; }
    const double w = b.n / r.n, k = a.n * w;
    const double dc = b.mc - a.mc, ds = b.ms - a.ms;
    r.mc = a.mc + dc * w;
    r.ms = a.ms + ds * w;
    r.m2c = a.m2c + b.m2c + dc * dc * k;
    r.m2s = a.m2s + b.m2s + ds * ds * k;
    return r;
}
constexpr int kMergeSlotsPerThread = 8;    // loads in flight per thread (128 threads x 8 = 1024 slots per round)
__device__ __noinline__ void merge_plane_coef_group(const AdainParams& p, int64_t plane, int gt, int barrier_id,
                                                       double (*scratch)[5]) {
    const float4* slots = p.part + plane * p.spp;
    MomD acc = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (int k0 = gt; k0 < p.spp; k0 += kTmaGroupThreads * kMergeSlotsPerThread) {
        float4 v[kMergeSlotsPerThread];
#pragma unroll
        for (int u = 0; u < kMergeSlotsPerThread; ++u) {
            const int k = k0 + u * kTmaGroupThreads;
            if (k < p.spp) v[u] = ld_slot(slots + k);
        }
#pragma unroll
        for (int u = 0; u < kMergeSlotsPerThread; ++u) {
            const int k = k0 + u * kTmaGroupThreads;
            if (k < p.spp) {
                if (!slot_valid(v[u])) {   // straggling statistics item: wait for it
                    const uint64_t t0 = global_timer_ns();
                    do {
                        __nanosleep(40);
                        v[u] = ld_slot(slots + k);
                        if (watchdog_expired(t0)) __trap();
                    } while (!slot_valid(v[u]));
                }
                const int64_t rem = p.hw - (int64_t)k * p.slot_elems;
                const MomD b = {(double)(rem < p.slot_elems ? rem : p.slot_elems), (double)v[u].x, (double)v[u].y,
                                (double)v[u].z, (double)v[u].w};
                acc = momd_merge(acc, b);
            }
        }
    }
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        MomD other;
        other.n = __shfl_xor_sync(0xffffffffu, acc.n, o);
        other.mc = __shfl_xor_sync(0xffffffffu, acc.mc, o);
        other.m2c = __shfl_xor_sync(0xffffffffu, acc.m2c, o);
        other.ms = __shfl_xor_sync(0xffffffffu, acc.ms, o);
        other.m2s = __shfl_xor_sync(0xffffffffu, acc.m2s, o);
        // the lower lane of a pair is always the left operand: both lanes compute the same value
        acc = ((gt & 31) & o) ? momd_merge(other, acc) : momd_merge(acc, other);
    }
    const int gw = gt >> 5;
    if ((gt & 31) == 0) {
        scratch[gw][0] = acc.n; scratch[gw][1] = acc.mc; scratch[gw][2] = acc.m2c; scratch[gw][3] = acc.ms; scratch[gw][4] = acc.m2s;
    }
    named_bar_sync((uint32_t)barrier_id, kTmaGroupThreads);
    if (gt == 0) {
        MomD t = {scratch[0][0], scratch[0][1], scratch[0][2], scratch[0][3], scratch[0][4]};
#pragma unroll
        for (int w = 1; w < kTmaGroupWarps; ++w) {
            const MomD b = {scratch[w][0], scratch[w][1], scratch[w][2], scratch[w][3], scratch[w][4]};
            t = momd_merge(t, b);
        }
        const double denom = (double)p.hw - 1.0;
        const float mu_hi = (float)t.mc;
        const float mu_lo = (float)(t.mc - (double)mu_hi);
        const float sd_c = (float)sqrt(t.m2c / denom + (double)p.eps);
        float mu_s = 0.f, sd_s = 1.f;
        if (p.style != nullptr) {
            mu_s = (float)t.ms;
            sd_s = (float)sqrt(t.m2s / denom + (double)p.eps);
        }
        st_slot(&p.coef[plane], make_float4(mu_hi, sd_s / sd_c, mu_s, mu_lo));
        if (p.saved) reinterpret_cast<float4*>(p.saved)[plane] = make_float4(mu_hi, sd_c, mu_s, sd_s);
    }
    named_bar_sync((uint32_t)barrier_id, kTmaGroupThreads);   // scratch is reused by the group's next merge item
}

// STAGES == number of consumer groups: group g owns stage g for the whole kernel, so the uses of a
// stage are consumed in order by one group and the single-bit mbarrier parity can never alias (a group
// that ran two phases ahead of a shared stage would pass the parity wait on stale data).
// GROUP_MERGE is a separate instantiation so that the small-plane kernel (the benchmark's) carries neither the
// call nor its register/barrier footprint: with a run-time switch the 512x512 path lost 10 % (5.66 vs 6.3 TB/s).
template <int STAGES, bool GROUP_MERGE>
__global__ void __launch_bounds__(64 + STAGES * kTmaGroupThreads, 1) adain_tma_kernel(AdainParams p) {
    constexpr int kTmaGroups = STAGES;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* bufs = reinterpret_cast<float*>(smem_raw);
    StageDesc* desc = reinterpret_cast<StageDesc*>(smem_raw + (size_t)STAGES * 2 * kItemElems * sizeof(float));
    uint64_t* full = reinterpret_cast<uint64_t*>(desc + STAGES);
    uint64_t* empty = full + STAGES;
    DecodedItem* dec = reinterpret_cast<DecodedItem*>(empty + STAGES);
    __shared__ double merge_scratch[GROUP_MERGE ? STAGES : 1][kTmaGroupWarps][5];
    // MERGE tickets of the single-warp merge bypass the stage ring: the producer posts the plane id into a
    // mailbox served by a dedicated merge warp (the last warp of the CTA).  Through the ring a merge queued
    // behind ~7 us of data items, twice per plane (statistics -> merge, merge -> apply), and that latency — not
    // HBM — set the time per plane: mean_variance_norm ran as slowly as full AdaIN.
    constexpr int kMailbox = 8;
    __shared__ uint64_t mfull[kMailbox], mempty[kMailbox];
    __shared__ int64_t mbox[kMailbox];
    constexpr bool mailbox = !GROUP_MERGE;   // small planes: always; the consumer loop then carries no merge code at all

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kTmaGroupWarps);
        }
        for (int s = 0; s < kMailbox; ++s) {
            mbar_init(&mfull[s], 1);
            mbar_init(&mempty[s], 1);
        }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp == 0) {
        // ================================================================ producer warp
        // Tickets are taken kTicketBatch at a time (the next request is always in flight); lanes
        // 0..kTicketBatch-1 decode one ticket each in parallel, lane 0 then issues them in order.
        const uint64_t pol_first = policy_evict_first();
        const uint64_t pol_last = policy_evict_last();
        unsigned next_base = 0;
        if (lane == 0) next_base = atomicAdd(p.ticket, (unsigned)kTicketBatch) + 1u;
        unsigned seq = 0, mseq = 0;
        auto post_merge = [&](int64_t plane_or_stop) {
            const int ms = (int)(mseq % kMailbox);
            mbar_wait(&mempty[ms], ((mseq / kMailbox) & 1u) ^ 1u);
            mbox[ms] = plane_or_stop;
            mbar_arrive(&mfull[ms]);
            ++mseq;
        };
        for (;;) {
            const unsigned base = __shfl_sync(0xffffffffu, next_base, 0);
            if (lane == 0) next_base = atomicAdd(p.ticket, (unsigned)kTicketBatch) + 1u;
            if (lane < kTicketBatch) {
                int kind = -1, chunk = 0;
                int64_t plane = 0;
                const unsigned t = base + (unsigned)lane;
                if (t < p.total_items) decode_tma(t, p, kind, plane, chunk);
                dec[lane].kind = kind; dec[lane].chunk = chunk; dec[lane].plane = plane;
                dec[lane].cplane = (kind == 0 || kind == 1) ? src_plane(p.cmap, plane) : plane;
                dec[lane].splane = kind == 0 ? src_plane(p.smap, plane) : plane;
            }
            __syncwarp();
            bool finished = false;
            if (lane == 0) {
                for (int i = 0; i < kTicketBatch; ++i) {
                    const int kind = dec[i].kind;
                    if (kind < 0) {
                        // out of work: one stop descriptor per consumer group (= per stage)
                        for (int g = 0; g < kTmaGroups; ++g, ++seq) {
                            const int stage = (int)(seq % STAGES);
                            mbar_wait(&empty[stage], ((seq / STAGES) & 1u) ^ 1u);
                            desc[stage].kind = -1;
                            mbar_arrive(&full[stage]);
                        }
                        post_merge(-1);
                        finished = true;
                        break;
                    }
                    if (kind == 2 && mailbox) {   // merge ticket: straight to the merge warp, no stage
                        post_merge(dec[i].plane);
                        continue;
                    }
                    const int chunk = dec[i].chunk;
                    const int64_t plane = dec[i].plane;
                    const int stage = (int)(seq % STAGES);
                    mbar_wait(&empty[stage], ((seq / STAGES) & 1u) ^ 1u);
                    StageDesc* d = &desc[stage];
                    // twin items carry two consecutive content chunks (apply without prev; statistics without style)
                    const bool twin = (kind == 1 && p.ipa != p.ipp) || (kind == 0 && p.ips != p.ipp);
                    const int64_t e0 = (int64_t)chunk * (twin ? 2 * kItemElems : kItemElems);
                    const int64_t rem = p.hw - e0;
                    const int nvec = (int)((rem < kItemElems ? rem : kItemElems) / 4);
                    const int64_t rem2 = rem - kItemElems;
                    const int nvec2 = twin && rem2 > 0 ? (int)((rem2 < kItemElems ? rem2 : kItemElems) / 4) : 0;
                    const uint32_t bytes = (uint32_t)nvec * 16u;
                    d->plane = plane; d->kind = kind; d->chunk = chunk; d->nvec = nvec; d->nvec2 = nvec2;
                    float* buf_a = bufs + (size_t)(stage * 2 + 0) * kItemElems;
                    float* buf_b = bufs + (size_t)(stage * 2 + 1) * kItemElems;
                    const float* csrc = p.content + dec[i].cplane * p.hw + e0;
                    if (kind == 0) {
                        const bool has_style = p.style != nullptr;
                        const uint64_t cpol = p.stats_only ? pol_first : pol_last;
                        mbar_arrive_expect_tx(&full[stage], (has_style ? 2u * bytes : bytes) + (uint32_t)nvec2 * 16u);
                        tma_load_1d(buf_a, csrc, bytes, &full[stage], cpol);
                        if (has_style) tma_load_1d(buf_b, p.style + dec[i].splane * p.hw + e0, bytes, &full[stage], pol_first);
                        if (nvec2 > 0) tma_load_1d(buf_b, csrc + kItemElems, (uint32_t)nvec2 * 16u, &full[stage], cpol);
                    } else if (kind == 1) {
                        const bool has_prev = p.prev != nullptr;
                        mbar_arrive_expect_tx(&full[stage], (has_prev ? 2u * bytes : bytes) + (uint32_t)nvec2 * 16u + 16u);
                        tma_load_1d(buf_a, csrc, bytes, &full[stage], pol_first);
                        if (has_prev) tma_load_1d(buf_b, p.prev + plane * p.hw + e0, bytes, &full[stage], pol_first);
                        if (nvec2 > 0) tma_load_1d(buf_b, csrc + kItemElems, (uint32_t)nvec2 * 16u, &full[stage], pol_first);
                        tma_load_1d(&d->coef, &p.coef[plane], 16u, &full[stage], pol_last);
                    } else {
                        mbar_arrive(&full[stage]);
                    }
                    ++seq;
                }
            }
            finished = __shfl_sync(0xffffffffu, (int)finished, 0) != 0;
            if (finished) return;
            __syncwarp();
        }
    }

    if (warp == 1 + STAGES * kTmaGroupWarps) {
        // ================================================================ merge warp (mailbox)
        for (unsigned mseq = 0;; ++mseq) {
            const int ms = (int)(mseq % kMailbox);
            mbar_wait(&mfull[ms], (mseq / kMailbox) & 1u);
            const int64_t plane = mbox[ms];
            __syncwarp();
            if (lane == 0) mbar_arrive(&mempty[ms]);
            if (plane < 0) break;
            if (p.spp <= 256) merge_plane_coef_small(p, plane, lane);
            else merge_plane_coef(p, plane, lane);
        }
        return;
    }

    // ==================================================================== consumers
    // Warp `gw` of a group owns vectors [gw*256, gw*256+256) of the item (a contiguous 4 KiB of each
    // tensor) and publishes its own statistics slot: consumer warps never synchronise with each other.
    const int group = (warp - 1) / kTmaGroupWarps;
    const int gw = (warp - 1) % kTmaGroupWarps;
    const uint64_t pol_first = policy_evict_first();
    const bool has_style = p.style != nullptr;
    const bool has_prev = p.prev != nullptr;

    for (unsigned seq = group;; seq += kTmaGroups) {
        const int stage = (int)(seq % STAGES);
        const unsigned ph = (seq / STAGES) & 1u;
        mbar_wait(&full[stage], ph);  // every lane observes the phase (async-proxy writes become visible to waiters)
        const StageDesc* d = &desc[stage];
        const int kind = d->kind;           // copy everything out of the descriptor: once the stage is
        if (kind < 0) break;                // released the producer may overwrite it
        const int64_t plane = d->plane;
        const int chunk = d->chunk;
        const int wvec = min(max(d->nvec - gw * (kTmaSlotElems / 4), 0), kTmaSlotElems / 4);  // this warp's vectors
        const float4* a4 = reinterpret_cast<const float4*>(bufs + (size_t)(stage * 2 + 0) * kItemElems) + gw * (kTmaSlotElems / 4);
        const float4* b4 = reinterpret_cast<const float4*>(bufs + (size_t)(stage * 2 + 1) * kItemElems) + gw * (kTmaSlotElems / 4);
        // lane's vectors: j*32 + lane, j < kTmaVecs; valid while < wvec
        const int my_vecs = wvec > lane ? min((wvec - lane + 31) / 32, kTmaVecs) : 0;
        const bool full_warp = wvec == kTmaSlotElems / 4;

        if (kind == 0) {
            // ---------------- statistics: moments of this warp's 4 KiB of content (and style)
            float4 v[kTmaVecs];
#pragma unroll
            for (int j = 0; j < kTmaVecs; ++j) v[j] = j < my_vecs ? a4[j * 32 + lane] : make_float4(0.f, 0.f, 0.f, 0.f);
            const Moments mc = warp_moments(v, my_vecs, full_warp);
            Moments ms = {0.f, 0.f, 0.f};
            const bool twin_s = !has_style && p.ips != p.ipp;   // buffer b holds the NEXT content chunk
            int wvec2 = 0;
            if (has_style) {
#pragma unroll
                for (int j = 0; j < kTmaVecs; ++j) v[j] = j < my_vecs ? b4[j * 32 + lane] : make_float4(0.f, 0.f, 0.f, 0.f);
                ms = warp_moments(v, my_vecs, full_warp);
            } else if (twin_s) {
                wvec2 = min(max(d->nvec2 - gw * (kTmaSlotElems / 4), 0), kTmaSlotElems / 4);
                const int my_vecs2 = wvec2 > lane ? min((wvec2 - lane + 31) / 32, kTmaVecs) : 0;
#pragma unroll
                for (int j = 0; j < kTmaVecs; ++j) v[j] = j < my_vecs2 ? b4[j * 32 + lane] : make_float4(0.f, 0.f, 0.f, 0.f);
                ms = warp_moments(v, my_vecs2, wvec2 == kTmaSlotElems / 4);   // moments of the second chunk's 4 KiB
            }
            // the stage has been consumed (the moments depend on every value read from it)
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&empty[stage]);
                const int64_t slot_chunk = twin_s ? 2 * (int64_t)chunk : chunk;
                if (wvec > 0)
                    st_slot(&p.part[plane * p.spp + slot_chunk * kTmaGroupWarps + gw],
                            twin_s ? make_float4(mc.mean, mc.m2, 0.f, 0.f) : make_float4(mc.mean, mc.m2, ms.mean, ms.m2));
                if (wvec2 > 0)
                    st_slot(&p.part[plane * p.spp + (slot_chunk + 1) * kTmaGroupWarps + gw], make_float4(ms.mean, ms.m2, 0.f, 0.f));
            }
        } else if (kind == 1) {
            // ---------------- apply: out = (c - mu_c) * a + mu_s (+ prev)
            float4 cf = d->coef;
            if (!slot_valid(cf)) {  // merge item still running somewhere: wait for its result
                if (lane == 0) {
                    const uint64_t t0 = global_timer_ns();
                    do {
                        __nanosleep(40);
                        cf = ld_slot(&p.coef[plane]);
                        if (watchdog_expired(t0)) __trap();
                    } while (!slot_valid(cf));
                }
                cf.x = __shfl_sync(0xffffffffu, cf.x, 0);
                cf.y = __shfl_sync(0xffffffffu, cf.y, 0);
                cf.z = __shfl_sync(0xffffffffu, cf.z, 0);
                cf.w = __shfl_sync(0xffffffffu, cf.w, 0);
            }
            const float mu_hi = cf.x, a = cf.y, mu_s = cf.z, mu_lo = cf.w;
            const int64_t n_idx = plane / p.channels, ch = plane % p.channels;
            const bool twin = p.ipa != p.ipp;   // no prev: the item carries two content chunks (buffers a and b)
            float4* o4 = reinterpret_cast<float4*>(p.out + n_idx * p.out_batch_stride + ch * p.hw +
                                                   (int64_t)chunk * (twin ? 2 * kItemElems : kItemElems)) + gw * (kTmaSlotElems / 4);
#pragma unroll
            for (int j = 0; j < kTmaVecs; ++j) {
                if (j < my_vecs) {
                    const float4 c = a4[j * 32 + lane];
                    float4 o;
                    o.x = fmaf((c.x - mu_hi) - mu_lo, a, mu_s);
                    o.y = fmaf((c.y - mu_hi) - mu_lo, a, mu_s);
                    o.z = fmaf((c.z - mu_hi) - mu_lo, a, mu_s);
                    o.w = fmaf((c.w - mu_hi) - mu_lo, a, mu_s);
                    if (has_prev) {
                        const float4 q = b4[j * 32 + lane];
                        o.x += q.x; o.y += q.y; o.z += q.z; o.w += q.w;
                    }
                    stg_f4_hint(reinterpret_cast<float*>(o4 + j * 32 + lane), o, pol_first);
                }
            }
            if (twin) {
                const int wvec2 = min(max(d->nvec2 - gw * (kTmaSlotElems / 4), 0), kTmaSlotElems / 4);
                const int my_vecs2 = wvec2 > lane ? min((wvec2 - lane + 31) / 32, kTmaVecs) : 0;
                float4* o4b = o4 + kItemElems / 4;
#pragma unroll
                for (int j = 0; j < kTmaVecs; ++j) {
                    if (j < my_vecs2) {
                        const float4 c = b4[j * 32 + lane];
                        float4 o;
                        o.x = fmaf((c.x - mu_hi) - mu_lo, a, mu_s);
                        o.y = fmaf((c.y - mu_hi) - mu_lo, a, mu_s);
                        o.z = fmaf((c.z - mu_hi) - mu_lo, a, mu_s);
                        o.w = fmaf((c.w - mu_hi) - mu_lo, a, mu_s);
                        stg_f4_hint(reinterpret_cast<float*>(o4b + j * 32 + lane), o, pol_first);
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[stage]);
        } else {
            // ---------------- merge: statistics slots of one plane -> coefficient slot
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[stage]);
            // few slots (512x512 planes: 256): one warp folds them while the other three go on to the next item;
            // many slots (1024x2048: 2048): the whole group takes one round trip instead of 2 x 64 serialized ones
            if constexpr (GROUP_MERGE) merge_plane_coef_group(p, plane, gw * 32 + lane, 1 + group, merge_scratch[group]);
        }
    }
}

// statistics-only finalisation (calc_mean_std on large planes): one warp per plane merges the
// chunk partials written by the preceding adain_pipe_kernel launch (stream order, no flags).
__global__ void __launch_bounds__(256) stats_finalize_kernel(AdainParams p) {
    const int lane = threadIdx.x & 31;
    const int64_t plane = (int64_t)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
    if (plane >= p.planes) return;
    // generic in ipp: two passes over the slots (they are final: previous launch in stream order)
    const float4* slots = p.part + plane * p.spp;
    const float k0 = __ldcg(slots).x;
    float d = 0.f;
#pragma unroll 8   // independent loads: keep 8 in flight (2048 slots per plane at 1024x2048)
    for (int k = lane; k < p.spp; k += 32) {
        const int64_t rem = p.hw - (int64_t)k * p.slot_elems;
        d = fmaf((float)(rem < p.slot_elems ? rem : p.slot_elems), __ldcg(slots + k).x - k0, d);
    }
    d = warp_sum(d) / (float)p.hw;
    float m2 = 0.f;
#pragma unroll 8
    for (int k = lane; k < p.spp; k += 32) {
        const float4 v = __ldcg(slots + k);
        const int64_t rem = p.hw - (int64_t)k * p.slot_elems;
        const float e = v.x - k0 - d;
        m2 += v.y + (float)(rem < p.slot_elems ? rem : p.slot_elems) * e * e;
    }
    m2 = warp_sum(m2);
    if (lane == 0) {
        if (p.mean_out) p.mean_out[plane] = k0 + d;
        if (p.std_out) p.std_out[plane] = sqrtf(m2 / ((float)p.hw - 1.f) + p.eps);
    }
}

// ------------------------------------------------------------------------------------------
// backward.  With x^ = (c-mu_c)/sd_c, G1 = sum(dy), G2 = sum(dy*x^) over the plane (HW = n):
//   dc = (sd_s/sd_c) * (dy - G1/n - x^ * G2/(n-1))        (unbiased variance => n-1)
//   ds = G1/n + (s-mu_s)/((n-1)*sd_s) * G2
// Same two-phase structure as the forward: reduce items (dy, c from HBM, kept in L2) run D planes
// ahead of write items (dy, c from L2; s from HBM; dc, ds to HBM): 5*E*4 algorithmic bytes.
// ------------------------------------------------------------------------------------------
struct BwdParams {
    const float* dy;
    const float* content;
    const float* style;   // may be null
    const float4* saved;  // [planes] (mu_c, sd_c, mu_s, sd_s)
    float* dcontent;
    float* dstyle;        // may be null
    int64_t planes, hw;
    int hints;
    int ipp, lag;
    unsigned total_items;
    unsigned* ticket;
    int* done;
    int* ready;
    float2* sums;         // [planes] (G1, G2)
    float2* part;         // [planes*ipp]
};

template <int THREADS>
__device__ __forceinline__ float2 block_sum2(float2 v, float2* scratch) {
    constexpr int W = THREADS / 32;
    v.x = warp_sum(v.x);
    v.y = warp_sum(v.y);
    if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
    __syncthreads();
    float2 t = scratch[0];
#pragma unroll
    for (int w = 1; w < W; ++w) { t.x += scratch[w].x; t.y += scratch[w].y; }
    return t;
}

template <int VEC, int THREADS>
__device__ __forceinline__ void bwd_write_batch(const float (&dy)[kBatch][VEC], const float (&c)[kBatch][VEC],
                                                const float* sbase, float* dcbase, float* dsbase, int b, int nvec,
                                                float4 st, float2 g, float hwf, uint64_t pol, bool hint) {
    const float inv_sd_c = 1.f / st.y;
    const float a = st.w * inv_sd_c;
    const float g1n = g.x / hwf;
    const float g2n = g.y / (hwf - 1.f);
    float sv[kBatch][VEC];
    if (dsbase) load_batch<VEC, THREADS>(sv, sbase, b, nvec, pol, hint);
#pragma unroll
    for (int j = 0; j < kBatch; ++j) {
        int idx = (b * kBatch + j) * THREADS + threadIdx.x;
        if (idx < nvec) {
            float o[VEC];
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
                float xh = (c[j][e] - st.x) * inv_sd_c;
                o[e] = a * (dy[j][e] - g1n - xh * g2n);
            }
            store_vec<VEC>(dcbase + (int64_t)idx * VEC, o, pol, hint);
            if (dsbase) {
                const float k = g2n / st.w;
#pragma unroll
                for (int e = 0; e < VEC; ++e) o[e] = fmaf(sv[j][e] - st.z, k, g1n);
                store_vec<VEC>(dsbase + (int64_t)idx * VEC, o, pol, hint);
            }
        }
    }
}

template <int VEC, int THREADS>
__device__ __forceinline__ float2 bwd_partial(const float (&dy)[kBatch][VEC], const float (&c)[kBatch][VEC], int b,
                                              int nvec, float4 st) {
    const float inv_sd_c = 1.f / st.y;
    float2 acc = make_float2(0.f, 0.f);
#pragma unroll
    for (int j = 0; j < kBatch; ++j) {
        int idx = (b * kBatch + j) * THREADS + threadIdx.x;
        if (idx < nvec) {
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
                acc.x += dy[j][e];
                acc.y = fmaf(dy[j][e], (c[j][e] - st.x) * inv_sd_c, acc.y);
            }
        }
    }
    return acc;
}

template <int VEC, int THREADS>
__global__ void __launch_bounds__(THREADS) adain_bwd_direct_kernel(BwdParams p) {
    __shared__ float2 scratch[32];
    const uint64_t pol = policy_evict_first();
    const bool hint = p.hints != 0;
    const int nvec = (int)(p.hw / VEC);
    const float hwf = (float)p.hw;
    for (int64_t plane = blockIdx.x; plane < p.planes; plane += gridDim.x) {
        const float4 st = __ldg(&p.saved[plane]);
        const float* dybase = p.dy + plane * p.hw;
        const float* cbase = p.content + plane * p.hw;
        float dy[kBatches][kBatch][VEC], c[kBatches][kBatch][VEC];
        float2 acc = make_float2(0.f, 0.f);
#pragma unroll
        for (int b = 0; b < kBatches; ++b) {
            load_batch<VEC, THREADS>(dy[b], dybase, b, nvec, pol, hint);
            load_batch<VEC, THREADS>(c[b], cbase, b, nvec, pol, hint);
        }
#pragma unroll
        for (int b = 0; b < kBatches; ++b) {
            float2 t = bwd_partial<VEC, THREADS>(dy[b], c[b], b, nvec, st);
            acc.x += t.x; acc.y += t.y;
        }
        const float2 g = block_sum2<THREADS>(acc, scratch);
#pragma unroll
        for (int b = 0; b < kBatches; ++b)
            bwd_write_batch<VEC, THREADS>(dy[b], c[b], p.style ? p.style + plane * p.hw : nullptr,
                                          p.dcontent + plane * p.hw, p.dstyle ? p.dstyle + plane * p.hw : nullptr,
                                          b, nvec, st, g, hwf, pol, hint);
        __syncthreads();
    }
}

template <int VEC>
__global__ void __launch_bounds__(kPipeThreads, 3) adain_bwd_pipe_kernel(BwdParams p) {
    constexpr int T = kPipeThreads;
    constexpr int CHUNK = T * kPerThread * VEC;
    __shared__ float2 scratch[32];
    __shared__ unsigned s_ticket;
    __shared__ int s_last;
    __shared__ float2 s_sums;
    const uint64_t pol_first = policy_evict_first();
    const uint64_t pol_last = policy_evict_last();
    const bool hint = p.hints != 0;
    const float hwf = (float)p.hw;

    AdainParams dec{};  // reuse the ticket decoder
    dec.planes = p.planes; dec.ipp = p.ipp; dec.lag = p.lag; dec.stats_only = 0;

    if (threadIdx.x == 0) s_ticket = atomicAdd(p.ticket, 1u);
    __syncthreads();
    unsigned t = s_ticket;
    while (t < p.total_items) {
        unsigned next = 0;
        if (threadIdx.x == 0) next = atomicAdd(p.ticket, 1u);
        const Item it = decode_ticket(t, dec);
        const int64_t e0 = (int64_t)it.chunk * CHUNK;
        const int64_t rem = p.hw - e0;
        const int nvec = (int)((rem < CHUNK ? rem : CHUNK) / VEC);
        const int64_t off = it.plane * p.hw + e0;
        const float4 st = __ldg(&p.saved[it.plane]);
        if (it.kind == 0) {
            float2 acc = make_float2(0.f, 0.f);
#pragma unroll
            for (int b = 0; b < kBatches; ++b) {
                float dy[kBatch][VEC], c[kBatch][VEC];
                load_batch<VEC, T>(dy, p.dy + off, b, nvec, pol_last, hint);
                load_batch<VEC, T>(c, p.content + off, b, nvec, pol_last, hint);
                float2 tt = bwd_partial<VEC, T>(dy, c, b, nvec, st);
                acc.x += tt.x; acc.y += tt.y;
            }
            const float2 g = block_sum2<T>(acc, scratch);
            if (threadIdx.x == 0) {
                __stcg(&p.part[it.plane * p.ipp + it.chunk], g);
                __threadfence();
                int old = atomicAdd(&p.done[it.plane], 1);
                s_last = (old == p.ipp - 1);
            }
            __syncthreads();
            if (s_last && threadIdx.x < 32) {
                __threadfence();
                float2 tot = make_float2(0.f, 0.f);
                for (int k = threadIdx.x; k < p.ipp; k += 32) {
                    float2 v = __ldcg(&p.part[it.plane * p.ipp + k]);
                    tot.x += v.x; tot.y += v.y;
                }
                tot.x = warp_sum(tot.x);
                tot.y = warp_sum(tot.y);
                if (threadIdx.x == 0) {
                    __stcg(&p.sums[it.plane], tot);
                    __threadfence();
                    st_release(&p.ready[it.plane], 1);
                }
            }
        } else {
            float dy[kBatch][VEC], c[kBatch][VEC];
            load_batch<VEC, T>(dy, p.dy + off, 0, nvec, pol_first, hint);
            load_batch<VEC, T>(c, p.content + off, 0, nvec, pol_first, hint);
            if (threadIdx.x == 0) {
                while (ld_acquire(&p.ready[it.plane]) == 0) __nanosleep(100);
                s_sums = __ldcg(&p.sums[it.plane]);
            }
            __syncthreads();
            const float2 g = s_sums;
#pragma unroll
            for (int b = 0; b < kBatches; ++b) {
                if (b > 0) {
                    load_batch<VEC, T>(dy, p.dy + off, b, nvec, pol_first, hint);
                    load_batch<VEC, T>(c, p.content + off, b, nvec, pol_first, hint);
                }
                bwd_write_batch<VEC, T>(dy, c, p.style ? p.style + off : nullptr, p.dcontent + off,
                                        p.dstyle ? p.dstyle + off : nullptr, b, nvec, st, g, hwf, pol_first, hint);
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) s_ticket = next;
        __syncthreads();
        t = s_ticket;
    }
}

// ------------------------------------------------------------------------------------------
// plane affine: out = x*scale[p] + shift[p]   (SELayer gating, network/attention.py:22)
// ------------------------------------------------------------------------------------------
template <int VEC>
__global__ void __launch_bounds__(256) plane_affine_kernel(const float* __restrict__ x, const float* __restrict__ scale,
                                                           const float* __restrict__ shift, float* __restrict__ out,
                                                           int64_t planes, int64_t hw, int chunks_per_plane) {
    constexpr int CHUNK = 256 * kPerThread * VEC;
    const uint64_t pol = policy_evict_first();
    const int64_t items = planes * chunks_per_plane;
    for (int64_t item = blockIdx.x; item < items; item += gridDim.x) {
        int64_t plane = item / chunks_per_plane;
        int64_t e0 = (item % chunks_per_plane) * CHUNK;
        int64_t rem = hw - e0;
        int nvec = (int)((rem < CHUNK ? rem : CHUNK) / VEC);
        const float a = __ldg(scale + plane);
        const float b = shift ? __ldg(shift + plane) : 0.f;
        const float* xb = x + plane * hw + e0;
        float* ob = out + plane * hw + e0;
#pragma unroll
        for (int bt = 0; bt < kBatches; ++bt) {
            float v[kBatch][VEC];
            load_batch<VEC, 256>(v, xb, bt, nvec, pol, true);
#pragma unroll
            for (int j = 0; j < kBatch; ++j) {
                int idx = (bt * kBatch + j) * 256 + threadIdx.x;
                if (idx < nvec) {
                    float o[VEC];
#pragma unroll
                    for (int e = 0; e < VEC; ++e) o[e] = fmaf(v[j][e], a, b);
                    store_vec<VEC>(ob + (int64_t)idx * VEC, o, pol, true);
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------

struct PipeLayout {
    size_t coef_off, part_off, total;  // ticket, coef, partial slots; everything is memset to 0xFF
};

PipeLayout pipe_layout(int64_t planes, int64_t hw) {
    const int64_t spp = (hw + kTmaSlotElems - 1) / kTmaSlotElems;
    PipeLayout l;
    l.coef_off = 256;
    l.part_off = align_up(l.coef_off + (size_t)planes * sizeof(float4), 256);
    l.total = align_up(l.part_off + (size_t)planes * spp * sizeof(float4), 256);
    return l;
}

template <int VEC>
int launch_direct(const AdainParams& p, cudaStream_t stream) {
    const int64_t nvec = p.hw / VEC;
    const int64_t grid64 = p.planes < (int64_t)sm_count() * 32 ? p.planes : (int64_t)sm_count() * 32;
    const int grid = (int)grid64;
    if (nvec <= 128 * kPerThread) adain_direct_kernel<VEC, 128><<<grid, 128, 0, stream>>>(p);
    else if (nvec <= 256 * kPerThread) adain_direct_kernel<VEC, 256><<<grid, 256, 0, stream>>>(p);
    else adain_direct_kernel<VEC, 512><<<grid, 512, 0, stream>>>(p);
    RPST_CUDA(cudaGetLastError());
    return RPST_OK;
}

template <int VEC, int MINB>
int launch_pipe_variant(const AdainParams& p, cudaStream_t stream) {
    // every CTA must be co-resident (apply items poll slots written by other CTAs)
    static int blocks_per_sm = 0;
    if (blocks_per_sm == 0) {
        int nb = 0;
        RPST_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, adain_pipe_kernel<VEC, MINB>, kPipeThreads, 0));
        blocks_per_sm = nb > 0 ? nb : 1;
    }
    const int per_sm = blocks_per_sm < MINB ? blocks_per_sm : MINB;
    int64_t grid = (int64_t)sm_count() * per_sm;
    if (grid > (int64_t)p.total_items) grid = p.total_items;
    adain_pipe_kernel<VEC, MINB><<<(int)grid, kPipeThreads, 0, stream>>>(p);
    RPST_CUDA(cudaGetLastError());
    return RPST_OK;
}

template <int STAGES, bool GROUP_MERGE>
int launch_tma_variant2(const AdainParams& p, cudaStream_t stream);

template <int STAGES>
int launch_tma_variant(const AdainParams& p, cudaStream_t stream) {
    return (!p.stats_only && p.spp >= p.group_merge_min_spp) ? launch_tma_variant2<STAGES, true>(p, stream)
                                                             : launch_tma_variant2<STAGES, false>(p, stream);
}

template <int STAGES, bool GROUP_MERGE>
int launch_tma_variant2(const AdainParams& p, cudaStream_t stream) {
    constexpr size_t smem = (size_t)STAGES * 2 * kItemElems * sizeof(float) + STAGES * sizeof(StageDesc) +
                            2 * STAGES * sizeof(uint64_t) + kTicketBatch * sizeof(DecodedItem);
    static PerDeviceFlag configured_on;
    bool& configured = configured_on.get();
    if (!configured) {
        RPST_CUDA(cudaFuncSetAttribute(adain_tma_kernel<STAGES, GROUP_MERGE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = true;
    }
    int64_t grid = sm_count();
    if (grid > (int64_t)p.total_items) grid = p.total_items;
    adain_tma_kernel<STAGES, GROUP_MERGE><<<(int)grid, 64 + STAGES * kTmaGroupThreads, smem, stream>>>(p);
    RPST_CUDA(cudaGetLastError());
    return RPST_OK;
}

// Item geometry and ticket schedule of the pipelined kernels for one call (host side): chunks per plane, lag,
// merge lead, twin items, the decode's division constants.  Returns the number of tickets.
int64_t plan_schedule(AdainParams& p, bool use_tma) {
    p.ipp = (int)((p.hw + kItemElems - 1) / kItemElems);
    const int64_t plane_bytes = p.hw * (int64_t)sizeof(float);
    // planes of >= 4 MiB: the statistics -> merge -> apply chain (>= 3 dependent global round trips of ~4.5 us
    // each under load) no longer fits the ~32 MiB L2 window, and a short lag stalls the apply items instead;
    // measured at 1x256x1024x2048: 32 MiB 3.03 TB/s, 64 MiB 4.92, 128 MiB 5.22 (tools/big_plane_sweep.py)
    // mean_variance_norm (no style stream): the statistics items drain 1.5x faster in bytes, so the same chain latency
    // spans more planes; 8x256x512x512: 32 MiB 4.2 TB/s, 40 MiB 5.07, 44 MiB 5.18, 48 MiB 4.99 (L2 misses set in), 56 MiB 4.75
    // (tools/mvn_sweep.py)
    const bool mvn = p.style == nullptr && !p.stats_only;
    const int64_t lag_bytes = plane_bytes >= (4ll << 20) ? g_knobs.adain_big_lag_bytes
                              : mvn                      ? g_knobs.adain_mvn_lag_bytes
                                                         : g_knobs.adain_lag_bytes;
    int64_t lag = (lag_bytes + plane_bytes - 1) / plane_bytes;
    if (lag < 3) lag = 3;
    p.lag = (int)(lag < p.planes ? lag : p.planes);
    p.slot_elems = use_tma ? kTmaSlotElems : kItemElems;
    p.spp = (int)((p.hw + p.slot_elems - 1) / p.slot_elems);
    {
        int64_t lead = g_knobs.adain_merge_lead > 0 ? g_knobs.adain_merge_lead : p.lag / 2;
        if (lead > p.lag - 1) lead = p.lag - 1;
        if (lead < 1) lead = 1;
        p.merge_lead = (int)lead;
    }
    p.ipa = (use_tma && !p.stats_only && p.prev == nullptr && g_knobs.adain_twin_apply) ? (p.ipp + 1) / 2 : p.ipp;
    p.ips = (use_tma && p.style == nullptr && g_knobs.adain_twin_apply) ? (p.ipp + 1) / 2 : p.ipp;
    p.div_s = make_fastdiv((uint32_t)p.ips);
    p.div_s1 = make_fastdiv((uint32_t)p.ips + 1u);
    p.div_s1a = make_fastdiv((uint32_t)p.ips + 1u + (uint32_t)p.ipa);
    p.div_a1 = make_fastdiv((uint32_t)p.ipa + 1u);
    p.div_a = make_fastdiv((uint32_t)p.ipa);
    return p.stats_only ? p.planes * p.ips : p.planes * ((int64_t)p.ips + p.ipa + (use_tma ? 1 : 0));
}

template <int VEC>
int launch_pipe(AdainParams p, void* ws, size_t ws_bytes, cudaStream_t stream) {
    const PipeLayout l = pipe_layout(p.planes, p.hw);
    if (ws == nullptr || ws_bytes < l.total) {
        set_error("adain: workspace too small (%zu < %zu bytes)", ws_bytes, l.total);
        return RPST_ERR_WORKSPACE;
    }
    RPST_CHECK_ARG(aligned16(ws), "adain: workspace must be 16-byte aligned");
    char* base = static_cast<char*>(ws);
    const bool use_tma = VEC == 4 && g_knobs.adain_path == 0;
    const int64_t total = plan_schedule(p, use_tma);
    RPST_CHECK_ARG(total < (1ll << 31), "adain: too many work items (%lld); split the call", (long long)total);
    p.total_items = (unsigned)total;
    p.ticket = reinterpret_cast<unsigned*>(base);
    p.coef = reinterpret_cast<float4*>(base + l.coef_off);
    p.part = reinterpret_cast<float4*>(base + l.part_off);
    RPST_CUDA(cudaMemsetAsync(base, 0xff, l.part_off + (size_t)p.planes * p.spp * sizeof(float4), stream));
    int rc;
    if (use_tma) {
        switch ((int)g_knobs.adain_stages) {
            case 2: rc = launch_tma_variant<2>(p, stream); break;
            case 3: rc = launch_tma_variant<3>(p, stream); break;
            case 4: rc = launch_tma_variant<4>(p, stream); break;
            case 5: rc = launch_tma_variant<5>(p, stream); break;
            case 7: rc = launch_tma_variant<7>(p, stream); break;
            default: rc = launch_tma_variant<6>(p, stream); break;
        }
    } else {
        switch ((int)g_knobs.adain_ctas_per_sm) {
            case 2: rc = launch_pipe_variant<VEC, 2>(p, stream); break;
            case 3: rc = launch_pipe_variant<VEC, 3>(p, stream); break;
            case 5: rc = launch_pipe_variant<VEC, 5>(p, stream); break;
            case 6: rc = launch_pipe_variant<VEC, 6>(p, stream); break;
            default: rc = launch_pipe_variant<VEC, 4>(p, stream); break;
        }
    }
    if (rc != RPST_OK) return rc;
    if (p.stats_only) {
        stats_finalize_kernel<<<(unsigned)((p.planes + 7) / 8), 256, 0, stream>>>(p);
        RPST_CUDA(cudaGetLastError());
    }
    return RPST_OK;
}

struct BwdLayout {
    size_t counters_bytes, sums_off, part_off, total;
};
BwdLayout bwd_layout(int64_t planes, int64_t hw) {
    const int64_t chunk = (int64_t)kPipeThreads * kPerThread;
    const int64_t ipp = (hw + chunk - 1) / chunk;
    BwdLayout l;
    l.counters_bytes = align_up(256 + (size_t)planes * 2 * sizeof(int), 256);
    l.sums_off = l.counters_bytes;
    l.part_off = align_up(l.sums_off + (size_t)planes * sizeof(float2), 256);
    l.total = align_up(l.part_off + (size_t)planes * ipp * sizeof(float2), 256);
    return l;
}

template <int VEC>
int launch_bwd(BwdParams p, void* ws, size_t ws_bytes, cudaStream_t stream) {
    const int64_t nvec = p.hw / VEC;
    if (nvec <= 512 * kPerThread) {
        const int64_t g64 = p.planes < (int64_t)sm_count() * 32 ? p.planes : (int64_t)sm_count() * 32;
        const int grid = (int)g64;
        if (nvec <= 128 * kPerThread) adain_bwd_direct_kernel<VEC, 128><<<grid, 128, 0, stream>>>(p);
        else if (nvec <= 256 * kPerThread) adain_bwd_direct_kernel<VEC, 256><<<grid, 256, 0, stream>>>(p);
        else adain_bwd_direct_kernel<VEC, 512><<<grid, 512, 0, stream>>>(p);
        RPST_CUDA(cudaGetLastError());
        return RPST_OK;
    }
    constexpr int64_t CHUNK = (int64_t)kPipeThreads * kPerThread * VEC;
    const BwdLayout l = bwd_layout(p.planes, p.hw);
    if (ws == nullptr || ws_bytes < l.total) {
        set_error("adain_bwd: workspace too small (%zu < %zu bytes)", ws_bytes, l.total);
        return RPST_ERR_WORKSPACE;
    }
    char* base = static_cast<char*>(ws);
    p.ipp = (int)((p.hw + CHUNK - 1) / CHUNK);
    const int64_t plane_bytes = 2 * p.hw * (int64_t)sizeof(float);  // dy and content stay resident
    int64_t lag = (g_knobs.adain_lag_bytes + plane_bytes - 1) / plane_bytes;
    if (lag < 3) lag = 3;
    p.lag = (int)(lag < p.planes ? lag : p.planes);
    const int64_t total = p.planes * p.ipp * 2;
    RPST_CHECK_ARG(total < (1ll << 31), "adain_bwd: too many work items (%lld); split the call", (long long)total);
    p.total_items = (unsigned)total;
    p.ticket = reinterpret_cast<unsigned*>(base);
    p.done = reinterpret_cast<int*>(base + 256);
    p.ready = p.done + p.planes;
    p.sums = reinterpret_cast<float2*>(base + l.sums_off);
    p.part = reinterpret_cast<float2*>(base + l.part_off);
    RPST_CUDA(cudaMemsetAsync(base, 0, l.counters_bytes, stream));
    int64_t grid = (int64_t)sm_count() * 3;
    if (grid > total) grid = total;
    adain_bwd_pipe_kernel<VEC><<<(int)grid, kPipeThreads, 0, stream>>>(p);
    RPST_CUDA(cudaGetLastError());
    return RPST_OK;
}

// Schedule dump for tests: ticket t -> (kind, plane, chunk) through the REAL decode of the TMA kernel.
__global__ void schedule_dump_kernel(AdainParams p, int32_t* out) {
    const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.total_items) return;
    int kind = -1, chunk = 0;
    int64_t plane = 0;
    decode_tma(t, p, kind, plane, chunk);
    out[3 * (size_t)t + 0] = kind;
    out[3 * (size_t)t + 1] = (int32_t)plane;
    out[3 * (size_t)t + 2] = chunk;
}

int run_adain(AdainParams p, void* ws, size_t ws_bytes, cudaStream_t stream) {
    if (p.planes == 0 || p.hw == 0) return RPST_OK;
    p.hints = (int)g_knobs.adain_hints;
    p.group_merge_min_spp = (int)g_knobs.adain_group_merge_min_spp;
    bool vec = (p.hw % 4 == 0) && aligned16(p.content) && (!p.style || aligned16(p.style)) &&
               (!p.prev || aligned16(p.prev)) && (!p.out || (aligned16(p.out) && p.out_batch_stride % 4 == 0));
    if (vec) {
        if (p.hw / 4 <= 512 * kPerThread) return launch_direct<4>(p, stream);
        return launch_pipe<4>(p, ws, ws_bytes, stream);
    }
    if (p.hw <= 512 * kPerThread) return launch_direct<1>(p, stream);
    return launch_pipe<1>(p, ws, ws_bytes, stream);
}

}  // namespace

}  // namespace rpst

using namespace rpst;

extern "C" size_t rpst_stats_workspace_bytes(int64_t planes, int64_t hw) {
    if (planes <= 0 || hw <= 0) return 256;
    return pipe_layout(planes, hw).total;
}

extern "C" int rpst_stats_nchw(const float* x, int64_t planes, int64_t hw, float eps, float* mean, float* std,
                               void* workspace, size_t workspace_bytes, void* stream) {
    RPST_CHECK_ARG(planes >= 0 && hw >= 0, "stats: negative size");
    RPST_CHECK_ARG(planes == 0 || hw == 0 || x != nullptr, "stats: null input");
    AdainParams p{};
    p.content = x;
    p.mean_out = mean;
    p.std_out = std;
    p.planes = planes;
    p.hw = hw;
    p.channels = 1;
    p.eps = eps;
    p.stats_only = 1;
    return run_adain(p, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

extern "C" size_t rpst_adain_workspace_bytes(int64_t n, int64_t c, int64_t hw) {
    if (n <= 0 || c <= 0 || hw <= 0) return 256;
    return pipe_layout(n * c, hw).total;
}

namespace {
int adain_fwd_impl(const float* content, const float* style, const float* prev, float* out, int64_t n, int64_t c,
                   int64_t hw, int64_t out_batch_stride, float eps, const int* content_map, const int* style_map,
                   float* saved_stats, void* workspace, size_t workspace_bytes, void* stream);
}

extern "C" int rpst_adain_fwd(const float* content, const float* style, const float* prev, float* out,
                              int64_t n, int64_t c, int64_t hw, int64_t out_batch_stride, float eps,
                              float* saved_stats, void* workspace, size_t workspace_bytes, void* stream) {
    return adain_fwd_impl(content, style, prev, out, n, c, hw, out_batch_stride, eps, nullptr, nullptr, saved_stats,
                          workspace, workspace_bytes, stream);
}

extern "C" int rpst_adain_fwd_mapped(const float* content, const float* style, const float* prev, float* out,
                                     int64_t n, int64_t c, int64_t hw, int64_t out_batch_stride, float eps,
                                     const int32_t* content_map, const int32_t* style_map, void* workspace,
                                     size_t workspace_bytes, void* stream) {
    RPST_CHECK_ARG(n * c < (1ll << 31), "adain_mapped: plane index does not fit int32");
    return adain_fwd_impl(content, style, prev, out, n, c, hw, out_batch_stride, eps, content_map, style_map, nullptr,
                          workspace, workspace_bytes, stream);
}

namespace {
int adain_fwd_impl(const float* content, const float* style, const float* prev, float* out, int64_t n, int64_t c,
                   int64_t hw, int64_t out_batch_stride, float eps, const int* content_map, const int* style_map,
                   float* saved_stats, void* workspace, size_t workspace_bytes, void* stream) {
    RPST_CHECK_ARG(n >= 0 && c >= 0 && hw >= 0, "adain: negative size");
    if (n == 0 || c == 0 || hw == 0) return RPST_OK;
    RPST_CHECK_ARG(content != nullptr && out != nullptr, "adain: null content/out");
    RPST_CHECK_ARG(out_batch_stride >= c * hw, "adain: out_batch_stride (%lld) < c*hw (%lld)",
                   (long long)out_batch_stride, (long long)(c * hw));
    RPST_CHECK_ARG(out != content && out != style && out != prev, "adain: out must not alias an input");
    AdainParams p{};
    p.content = content;
    p.style = style;
    p.prev = prev;
    p.out = out;
    p.saved = saved_stats;
    p.planes = n * c;
    p.hw = hw;
    p.channels = c;
    p.out_batch_stride = out_batch_stride;
    p.eps = eps;
    p.cmap = content_map;
    p.smap = style_map;
    return run_adain(p, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}
}  // namespace

#ifdef RPST_DEBUG_EXPORTS   // white-box test hooks: only in librpst_debug.so (loaded by tests alone), never in the product library
// Test hook: the ticket schedule the TMA kernel would walk for this call shape.  info = {tickets, stats items
// per plane, apply items per plane, lag, merge lead}; tickets [max_tickets,3] receives (kind, plane, chunk) with
// kind 0 statistics, 1 apply, 2 merge.  Used by tests/test_schedule_gpu.py to check the schedule's invariants
// for shapes that no data test covers.
extern "C" int rpst_debug_adain_schedule(int64_t planes, int64_t hw, int has_style, int has_prev, int stats_only,
                                         int32_t* tickets, int64_t max_tickets, int64_t* info, void* stream) {
    RPST_CHECK_ARG(planes > 0 && hw > 0 && info != nullptr, "debug_schedule: bad arguments");
    AdainParams p{};
    p.planes = planes; p.hw = hw; p.channels = 1; p.stats_only = stats_only;
    p.content = reinterpret_cast<const float*>(16);            // only null-ness is inspected
    p.style = has_style ? reinterpret_cast<const float*>(16) : nullptr;
    p.prev = has_prev ? reinterpret_cast<const float*>(16) : nullptr;
    const int64_t total = plan_schedule(p, true);
    RPST_CHECK_ARG(total < (1ll << 31), "debug_schedule: too many tickets");
    p.total_items = (unsigned)total;
    info[0] = total; info[1] = p.ips; info[2] = p.ipa; info[3] = p.lag; info[4] = p.merge_lead;
    if (tickets != nullptr) {
        RPST_CHECK_ARG(max_tickets >= total, "debug_schedule: ticket buffer too small (%lld < %lld)", (long long)max_tickets, (long long)total);
        schedule_dump_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(p, tickets);
        RPST_CUDA(cudaGetLastError());
    }
    return RPST_OK;
}
#endif  // RPST_DEBUG_EXPORTS

extern "C" size_t rpst_adain_bwd_workspace_bytes(int64_t n, int64_t c, int64_t hw) {
    if (n <= 0 || c <= 0 || hw <= 0) return 256;
    return bwd_layout(n * c, hw).total;
}

extern "C" int rpst_adain_bwd(const float* grad_out, const float* content, const float* style,
                              const float* saved_stats, float* grad_content, float* grad_style,
                              int64_t n, int64_t c, int64_t hw, void* workspace, size_t workspace_bytes,
                              void* stream) {
    RPST_CHECK_ARG(n >= 0 && c >= 0 && hw >= 0, "adain_bwd: negative size");
    if (n == 0 || c == 0 || hw == 0) return RPST_OK;
    RPST_CHECK_ARG(grad_out && content && saved_stats && grad_content, "adain_bwd: null pointer");
    RPST_CHECK_ARG(grad_style == nullptr || style != nullptr, "adain_bwd: grad_style requested without style");
    RPST_CHECK_ARG(aligned16(saved_stats), "adain_bwd: saved_stats must be 16-byte aligned");
    BwdParams p{};
    p.dy = grad_out;
    p.content = content;
    p.style = grad_style ? style : nullptr;
    p.saved = reinterpret_cast<const float4*>(saved_stats);
    p.dcontent = grad_content;
    p.dstyle = grad_style;
    p.planes = n * c;
    p.hw = hw;
    p.hints = (int)g_knobs.adain_hints;
    const bool vec = hw % 4 == 0 && aligned16(grad_out) && aligned16(content) && aligned16(grad_content) &&
                     (!grad_style || (aligned16(style) && aligned16(grad_style)));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    return vec ? launch_bwd<4>(p, workspace, workspace_bytes, st) : launch_bwd<1>(p, workspace, workspace_bytes, st);
}

extern "C" int rpst_plane_affine(const float* x, const float* scale, const float* shift, float* out,
                                 int64_t planes, int64_t hw, void* stream) {
    RPST_CHECK_ARG(planes >= 0 && hw >= 0, "plane_affine: negative size");
    if (planes == 0 || hw == 0) return RPST_OK;
    RPST_CHECK_ARG(x && scale && out, "plane_affine: null pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool vec = hw % 4 == 0 && aligned16(x) && aligned16(out);
    const int64_t chunk = 256ll * kPerThread * (vec ? 4 : 1);
    const int cpp = (int)((hw + chunk - 1) / chunk);
    int64_t items = planes * cpp;
    int64_t grid = (int64_t)sm_count() * 8;
    if (grid > items) grid = items;
    if (vec) plane_affine_kernel<4><<<(int)grid, 256, 0, st>>>(x, scale, shift, out, planes, hw, cpp);
    else plane_affine_kernel<1><<<(int)grid, 256, 0, st>>>(x, scale, shift, out, planes, hw, cpp);
    RPST_CUDA(cudaGetLastError());
    return RPST_OK;
}

RPST_WATCHDOG_SETTER(adain)

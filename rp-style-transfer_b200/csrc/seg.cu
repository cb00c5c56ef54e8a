// Segment (mask-label) AdaIN — SURVEY.md §8 a4; reference: network/base.py:421-530 and the batch
// loop network/adain_rp.py:313-319.
//
// The reference walks the label set on the host (np.where per label, index_select gather, ~12
// launches, index_copy_ scatter; per label, per level, per sample).  Here the whole batch is:
//   seg_hist_kernel   per sample: pixel count and first pixel index of every label value (0..255) in the
//                     content and in the style map (labels are shared by all channels)
//   seg_dense_kernel  dense ids of the usable labels (validity rule evaluated on the device)
//   seg_shift_kernel  per (plane, tensor, label) shift K_l = first pixel of the label in that plane
//   seg_tma_kernel    TMA-staged pipeline (16-byte aligned planes, <= 64 usable labels per sample);
//                     statistics are per-label shifted sums S1 = sum(x-K_l), S2 = sum((x-K_l)^2)
//   seg_pipe_kernel   register-staged fallback (unaligned shapes, or > 64 usable labels: chosen on the
//                     device through a flag, without host synchronisation)
// The validity rule (network/base.py:435: label taken from the CONTENT map; cnt_c>10, cnt_s>10,
// cnt_c/cnt_s<100, cnt_s/cnt_c<100) uses exact integer comparisons; pixels of unusable labels are
// copied through bit-exactly.
#include "common.cuh"
#include "tuning.cuh"
#include "plane_io.cuh"
#include "async.cuh"

namespace rpst {
namespace {

constexpr int kLabels = 256;
constexpr int kNoIndex = 0x7f7f7f7f;  // memset(0x7f) pattern = "no pixel seen"

struct SegParams {
    const float* content;
    const float* style;
    const uint8_t* c_lab;   // [n, hw_c]
    const uint8_t* s_lab;   // [n, hw_s]
    const float* prev;      // may be null; indexed by the output plane
    float* out;             // plane (i, ch) at out + i*out_batch_stride + ch*hw_c
    const int* cmap;        // source plane of content / style per output plane (null: identity)
    const int* smap;
    int64_t n, channels, hw_c, hw_s, out_batch_stride;
    float eps;
    int hints;
    int ipp_c, ipp_s, lag;
    unsigned total_items;
    // workspace
    unsigned* ticket;
    int* done;              // [planes]
    int* ready;             // [planes]
    int* cnt;               // [n][2][256]
    int* first;             // [n][2][256]
    float2* gsum;           // [planes][2][256] (S1, S2)
    float4* coef;           // [planes][256] (mu_c, a, mu_s, valid)
    const int* run_flag;    // null: always run; else run only if *run_flag != 0 (slot-path overflow)
};

__global__ void __launch_bounds__(256) seg_hist_kernel(const uint8_t* __restrict__ c_lab, const uint8_t* __restrict__ s_lab,
                                                       int64_t hw_c, int64_t hw_s, int* __restrict__ cnt,
                                                       int* __restrict__ first) {
    __shared__ int h[kLabels];
    __shared__ int f[kLabels];
    const int which = blockIdx.z;  // 0 content, 1 style
    const int64_t n = blockIdx.y;
    const int64_t hw = which ? hw_s : hw_c;
    const uint8_t* lab = (which ? s_lab : c_lab) + n * hw;
    h[threadIdx.x] = 0;
    f[threadIdx.x] = kNoIndex;
    __syncthreads();
    const int64_t per_block = (hw + gridDim.x - 1) / gridDim.x;
    const int64_t beg = blockIdx.x * per_block;
    const int64_t end = beg + per_block < hw ? beg + per_block : hw;
    for (int64_t i = beg + threadIdx.x; i < end; i += blockDim.x) {
        int l = lab[i];
        atomicAdd(&h[l], 1);
        atomicMin(&f[l], (int)i);
    }
    __syncthreads();
    const int64_t slot = (n * 2 + which) * kLabels + threadIdx.x;
    if (h[threadIdx.x]) {
        atomicAdd(&cnt[slot], h[threadIdx.x]);
        atomicMin(&first[slot], f[threadIdx.x]);
    }
}

// plane maps (rpst_seg_adain_fwd_mapped): output plane -> plane of the content / style tensor that feeds it.
// Everything else (labels, validity, slots, coefficients, prev) stays indexed by the output plane.
__device__ __forceinline__ int64_t src_plane(const int* map, int64_t plane) {
    return map ? (int64_t)__ldg(map + plane) : plane;
}

__device__ __forceinline__ bool label_usable(int nc, int ns) {
    // network/base.py:435 with the float ratios written as exact integer comparisons
    return nc > 10 && ns > 10 && (int64_t)nc < 100ll * ns && (int64_t)ns < 100ll * nc;
}

struct SegItem {
    int kind;  // 0 content statistics, 1 style statistics, 2 apply
    int64_t plane;
    int chunk;
};

__device__ __forceinline__ SegItem seg_decode(unsigned t, const SegParams& p) {
    const int64_t planes = p.n * p.channels;
    const int64_t st = p.ipp_c + p.ipp_s;  // statistics items per plane
    const int64_t lag = p.lag < planes ? p.lag : planes;
    SegItem it;
    int64_t tt = t;
    auto stats = [&](int64_t plane, int64_t u) {
        it.plane = plane;
        if (u < p.ipp_c) { it.kind = 0; it.chunk = (int)u; }
        else { it.kind = 1; it.chunk = (int)(u - p.ipp_c); }
    };
    if (tt < lag * st) { stats(tt / st, tt % st); return it; }
    tt -= lag * st;
    const int64_t round = st + p.ipp_c;
    const int64_t steady = (planes - lag) * round;
    if (tt < steady) {
        int64_t r = tt / round, u = tt % round;
        if (u < st) stats(r + lag, u);
        else { it.kind = 2; it.plane = r; it.chunk = (int)(u - st); }
        return it;
    }
    tt -= steady;
    it.kind = 2; it.plane = (planes - lag) + tt / p.ipp_c; it.chunk = (int)(tt % p.ipp_c);
    return it;
}

template <int VEC>
__device__ __forceinline__ void load_labels(int (&lab)[VEC], const uint8_t* p) {
    if constexpr (VEC == 4) {
        uchar4 v = __ldg(reinterpret_cast<const uchar4*>(p));
        lab[0] = v.x; lab[1] = v.y; lab[2] = v.z; lab[3] = v.w;
    } else {
        lab[0] = __ldg(p);
    }
}

template <int VEC>
__global__ void __launch_bounds__(kPipeThreads, 3) seg_pipe_kernel(SegParams p) {
    constexpr int T = kPipeThreads;
    constexpr int CHUNK = T * kPerThread * VEC;
    static_assert(T == kLabels, "one thread per label value");
    __shared__ float s_shift[kLabels];
    __shared__ float s_acc[kLabels][2];
    __shared__ float4 s_coef[kLabels];
    __shared__ unsigned char s_use[kLabels];
    __shared__ unsigned s_ticket;
    __shared__ int s_last;

    const uint64_t pol_first = policy_evict_first();
    const uint64_t pol_last = policy_evict_last();
    const bool hint = p.hints != 0;
    const int lane = threadIdx.x & 31;
    if (p.run_flag != nullptr && __ldg(p.run_flag) == 0) return;

    if (threadIdx.x == 0) s_ticket = atomicAdd(p.ticket, 1u);
    __syncthreads();
    unsigned t = s_ticket;

    while (t < p.total_items) {
        unsigned next = 0;
        if (threadIdx.x == 0) next = atomicAdd(p.ticket, 1u);
        const SegItem it = seg_decode(t, p);
        const int64_t sample = it.plane / p.channels;
        const int* cnt_c = p.cnt + (sample * 2 + 0) * kLabels;
        const int* cnt_s = p.cnt + (sample * 2 + 1) * kLabels;

        if (it.kind < 2) {
            // ------------------------------------------------ statistics item (content or style)
            const bool is_style = it.kind == 1;
            const int64_t hw = is_style ? p.hw_s : p.hw_c;
            const float* x = is_style ? p.style + src_plane(p.smap, it.plane) * hw : p.content + src_plane(p.cmap, it.plane) * hw;
            const uint8_t* labels = (is_style ? p.s_lab : p.c_lab) + sample * hw;
            const int* first = p.first + (sample * 2 + it.kind) * kLabels;
            const int64_t e0 = (int64_t)it.chunk * CHUNK;
            const int64_t rem = hw - e0;
            const int nvec = (int)((rem < CHUNK ? rem : CHUNK) / VEC);
            {
                const int l = threadIdx.x;
                const bool use = label_usable(__ldg(cnt_c + l), __ldg(cnt_s + l));
                s_use[l] = use;
                s_shift[l] = use ? __ldg(x + __ldg(first + l)) : 0.f;
                s_acc[l][0] = 0.f;
                s_acc[l][1] = 0.f;
            }
            __syncthreads();
            int cur = -1;
            float shift = 0.f, a1 = 0.f, a2 = 0.f;
            const uint64_t xpol = is_style ? pol_first : pol_last;
#pragma unroll
            for (int b = 0; b < kBatches; ++b) {
                float v[kBatch][VEC];
                load_batch<VEC, T>(v, x + e0, b, nvec, xpol, hint);
#pragma unroll
                for (int j = 0; j < kBatch; ++j) {
                    const int idx = (b * kBatch + j) * T + threadIdx.x;
                    if (idx < nvec) {
                        int lab[VEC];
                        load_labels<VEC>(lab, labels + e0 + (int64_t)idx * VEC);
#pragma unroll
                        for (int e = 0; e < VEC; ++e) {
                            const int l = lab[e];
                            if (l != cur) {
                                if (cur >= 0) {  // rare mid-item flush (label run ended)
                                    atomicAdd(&s_acc[cur][0], a1);
                                    atomicAdd(&s_acc[cur][1], a2);
                                }
                                if (s_use[l]) { cur = l; shift = s_shift[l]; }
                                else cur = -1;
                                a1 = 0.f; a2 = 0.f;
                            }
                            if (cur >= 0) {
                                const float d = v[j][e] - shift;
                                a1 += d;
                                a2 = fmaf(d, d, a2);
                            }
                        }
                    }
                }
            }
            // final flush, aggregated per distinct label inside the warp
            unsigned remaining = __ballot_sync(0xffffffffu, cur >= 0);
            while (remaining) {
                const int leader = __ffs(remaining) - 1;
                const int l = __shfl_sync(0xffffffffu, cur, leader);
                const bool mine = cur == l;
                const float r1 = warp_sum(mine ? a1 : 0.f);
                const float r2 = warp_sum(mine ? a2 : 0.f);
                if (lane == leader) {
                    atomicAdd(&s_acc[l][0], r1);
                    atomicAdd(&s_acc[l][1], r2);
                }
                remaining &= ~__ballot_sync(0xffffffffu, mine);
            }
            __syncthreads();
            {
                const int l = threadIdx.x;
                const float r1 = s_acc[l][0], r2 = s_acc[l][1];
                if (r1 != 0.f || r2 != 0.f) {
                    float2* g = p.gsum + (it.plane * 2 + it.kind) * kLabels + l;
                    atomicAdd(&g->x, r1);
                    atomicAdd(&g->y, r2);
                }
            }
            __threadfence();
            __syncthreads();
            if (threadIdx.x == 0) {
                int old = atomicAdd(&p.done[it.plane], 1);
                s_last = (old == p.ipp_c + p.ipp_s - 1);
            }
            __syncthreads();
            if (s_last) {
                // last statistics item of the plane: turn the sums into per-label AdaIN coefficients
                __threadfence();
                const int l = threadIdx.x;
                const int nc = __ldg(cnt_c + l), ns = __ldg(cnt_s + l);
                float4 cf = make_float4(0.f, 1.f, 0.f, 0.f);  // identity for unusable labels
                if (label_usable(nc, ns)) {
                    const float kc = __ldg(p.content + src_plane(p.cmap, it.plane) * p.hw_c + __ldg(p.first + (sample * 2 + 0) * kLabels + l));
                    const float ks = __ldg(p.style + src_plane(p.smap, it.plane) * p.hw_s + __ldg(p.first + (sample * 2 + 1) * kLabels + l));
                    const float2 gc = __ldcg(p.gsum + (it.plane * 2 + 0) * kLabels + l);
                    const float2 gs = __ldcg(p.gsum + (it.plane * 2 + 1) * kLabels + l);
                    const float fnc = (float)nc, fns = (float)ns;
                    const float mu_c = kc + gc.x / fnc;
                    const float mu_s = ks + gs.x / fns;
                    const float m2c = fmaxf(gc.y - gc.x * gc.x / fnc, 0.f);
                    const float m2s = fmaxf(gs.y - gs.x * gs.x / fns, 0.f);
                    const float sd_c = sqrtf(m2c / (fnc - 1.f) + p.eps);
                    const float sd_s = sqrtf(m2s / (fns - 1.f) + p.eps);
                    cf = make_float4(mu_c, sd_s / sd_c, mu_s, 1.f);
                }
                __stcg(&p.coef[it.plane * kLabels + l], cf);
                __threadfence();
                __syncthreads();
                if (threadIdx.x == 0) st_release(&p.ready[it.plane], 1);
            }
        } else {
            // ------------------------------------------------ apply item
            const int64_t e0 = (int64_t)it.chunk * CHUNK;
            const int64_t rem = p.hw_c - e0;
            const int nvec = (int)((rem < CHUNK ? rem : CHUNK) / VEC);
            const float* cbase = p.content + src_plane(p.cmap, it.plane) * p.hw_c + e0;
            const float* pbase = p.prev ? p.prev + it.plane * p.hw_c + e0 : nullptr;
            float* obase = p.out + sample * p.out_batch_stride + (it.plane - sample * p.channels) * p.hw_c + e0;
            const uint8_t* labels = p.c_lab + sample * p.hw_c + e0;
            float c[kBatch][VEC], pv[kBatch][VEC];
            load_batch<VEC, T>(c, cbase, 0, nvec, pol_first, hint);
            if (pbase) load_batch<VEC, T>(pv, pbase, 0, nvec, pol_first, hint);
            if (threadIdx.x == 0) {
                while (ld_acquire(&p.ready[it.plane]) == 0) __nanosleep(100);
            }
            __syncthreads();
            s_coef[threadIdx.x] = __ldcg(&p.coef[it.plane * kLabels + threadIdx.x]);
            __syncthreads();
#pragma unroll
            for (int b = 0; b < kBatches; ++b) {
                if (b > 0) {
                    load_batch<VEC, T>(c, cbase, b, nvec, pol_first, hint);
                    if (pbase) load_batch<VEC, T>(pv, pbase, b, nvec, pol_first, hint);
                }
#pragma unroll
                for (int j = 0; j < kBatch; ++j) {
                    const int idx = (b * kBatch + j) * T + threadIdx.x;
                    if (idx < nvec) {
                        int lab[VEC];
                        load_labels<VEC>(lab, labels + (int64_t)idx * VEC);
                        float o[VEC];
#pragma unroll
                        for (int e = 0; e < VEC; ++e) {
                            const float4 cf = s_coef[lab[e]];
                            // unusable label: (c-0)*1+0 == c bit-exactly (pass-through)
                            const float y = fmaf(c[j][e] - cf.x, cf.y, cf.z);
                            o[e] = pbase ? y + pv[j][e] : y;
                        }
                        store_vec<VEC>(obase + (int64_t)idx * VEC, o, pol_first, hint);
                    }
                }
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) s_ticket = next;
        __syncthreads();
        t = s_ticket;
    }
}

// ------------------------------------------------------------------------------------------
// TMA-staged segment kernel (16-byte aligned planes): the structure of adain_tma_kernel — producer
// warp + one shared-memory stage per consumer group — with three differences:
//  * an item also carries its 4 KiB label chunk; per-lane (label, S1, S2) run accumulation with a
//    whole-float4 fast path when the four labels equal the running label (real maps are blocky);
//  * the four warps of a group add their runs into a shared-memory table indexed by dense label id and
//    publish one self-validating 8-byte slot per usable label and item (no fence, no global atomic);
//  * MERGE tickets bypass the stage ring: two dedicated merge warps per CTA (one thread per dense label)
//    sum a plane's slots in fp64 in a fixed order (deterministic) and publish the per-plane coefficient
//    table [256]; merges therefore never queue behind apply items that wait for them;
//  * apply items cache the coefficient table in shared memory per group, re-loaded when the plane changes.
//  The statistics->apply lag is long (seg_lag_bytes, 256 MiB) because a plane's merge walks ~1000 slots;
//  at 1024x2048 the content re-read therefore comes from HBM (4E instead of 3E bytes): next round's item.
// ------------------------------------------------------------------------------------------
// Item geometry.  A full item is kSegItemElems pixels of one tensor + its labels; an apply item that also
// carries `prev` is kSegPrevElems pixels.  (8192-pixel items were measured: 2.79 ms vs 2.18 ms at config #5 —
// the kernel is bound by per-item consumer latency, not by the producer's item rate, so smaller items on
// more groups win.)
constexpr int kSegItemElems = 4096;
constexpr int kSegPrevElems = 2048;
constexpr int kSegHalfElems = kSegPrevElems;                        // byte offset / 4 of the prev region
constexpr int kSegDataBytes = (kSegItemElems > 2 * kSegPrevElems ? kSegItemElems : 2 * kSegPrevElems) * 4;
constexpr int kSegStageBytes = kSegDataBytes + kSegItemElems;       // data (+prev) region, then the label bytes
// D stages per consumer group (owned by that group alone, used alternately): the next item's TMA is in
// flight while the current one is processed.  ncu on the single-stage version: 45 % of consumer samples sat
// in the wait for the stage's `full` barrier (fetch latency + producer turnaround) and the rest in processing,
// strictly one after the other.
constexpr int kSegDepth = 2;
constexpr int kSegGroups = 4;   // consumer groups of seg_tma_kernel: 4 x kSegDepth stages of 20 KiB
constexpr int kSegGroupWarps = 4;
constexpr int kSegGroupThreads = kSegGroupWarps * 32;
constexpr int kSegWarpVecs = kSegItemElems / 4 / kSegGroupWarps;   // 512 float4 per warp per full item
constexpr int kSegLaneVecs = kSegWarpVecs / 32;                    // 16
constexpr int kSegTicketBatch = 8;
constexpr int kMaxDense = 64;    // usable labels per sample handled by the slot path

struct SegTmaParams {
    const float* content;
    const float* style;
    const uint8_t* c_lab;
    const uint8_t* s_lab;
    const float* prev;           // indexed by the output plane
    float* out;                  // plane (i, ch) at out + i*out_batch_stride + ch*hw_c
    const int* cmap;             // source plane of content / style per output plane (null: identity)
    const int* smap;
    int64_t n, channels, hw_c, hw_s, out_batch_stride;
    float eps;
    int ic, is, lag;             // content / style statistics chunks per plane, statistics lead in planes
    int ia, apply_elems;         // apply chunks per plane and their size (kSegHalfElems with prev, else kSegItemElems)
    unsigned total_items;
    unsigned* ticket;            // starts at 0xFFFFFFFF
    int* ready;                  // [planes] coefficient table published
    const int* cnt;              // [n][2][256]
    const int* first;            // [n][2][256]
    float* shift;                // [planes][2][256]  K_l = first pixel of label l in that plane
    const unsigned char* dense;  // [n][256] dense id of a usable label (255: unusable)
    const unsigned char* label_of;  // [n][kMaxDense] inverse map
    const int* dense_count;      // [n] usable labels of the sample
    const int* overflow;         // != 0: some sample has more than kMaxDense usable labels -> fallback kernel runs
    float2* slots;               // [planes][2][imax][kMaxDense] (S1, S2) per item; 0xFF-filled = not written
    int imax;                    // max(ic, is)
    float4* coef;                // [planes][256] (mu_c, a, mu_s, usable)
};

struct __align__(16) SegDesc {
    int64_t plane;
    int kind;      // 0 content statistics, 1 style statistics, 2 apply, 3 merge, -1 stop
    int chunk;
    int nvec;
    int pad;
};

struct SegDecoded {
    int64_t plane;
    int kind, chunk;
};

// one block per sample: dense ids of the usable labels (increasing label order), inverse map, count
__global__ void __launch_bounds__(kLabels) seg_dense_kernel(const int* __restrict__ cnt, unsigned char* __restrict__ dense,
                                                            unsigned char* __restrict__ label_of,
                                                            int* __restrict__ dense_count, int* __restrict__ overflow) {
    __shared__ int warp_cnt[kLabels / 32];
    const int sample = blockIdx.x, l = threadIdx.x, lane = l & 31, w = l >> 5;
    const bool use = label_usable(cnt[(sample * 2 + 0) * kLabels + l], cnt[(sample * 2 + 1) * kLabels + l]);
    const unsigned m = __ballot_sync(0xffffffffu, use);
    if (lane == 0) warp_cnt[w] = __popc(m);
    __syncthreads();
    int base = 0, total = 0;
    for (int i = 0; i < kLabels / 32; ++i) {
        if (i < w) base += warp_cnt[i];
        total += warp_cnt[i];
    }
    const int id = base + __popc(m & ((1u << lane) - 1u));
    dense[sample * kLabels + l] = (use && id < kMaxDense) ? (unsigned char)id : (unsigned char)255;
    if (use && id < kMaxDense) label_of[sample * kMaxDense + id] = (unsigned char)l;
    if (l == 0) {
        dense_count[sample] = total < kMaxDense ? total : kMaxDense;
        if (total > kMaxDense) atomicOr(overflow, 1);
    }
}

__global__ void seg_shift_kernel(SegTmaParams p) {
    const int64_t planes = p.n * p.channels;
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= planes * 2 * kLabels) return;
    const int l = (int)(idx % kLabels), which = (int)((idx / kLabels) & 1);
    const int64_t plane = idx / (2 * kLabels), sample = plane / p.channels;
    const int slot = (int)((sample * 2 + which) * kLabels + l);
    float v = 0.f;
    if (p.cnt[slot] > 0) {
        v = which ? p.style[src_plane(p.smap, plane) * p.hw_s + p.first[slot]]
                  : p.content[src_plane(p.cmap, plane) * p.hw_c + p.first[slot]];
    }
    p.shift[idx] = v;
}

__device__ __forceinline__ bool slot2_valid(double2 v) {
    return (unsigned)(__double_as_longlong(v.x) >> 32) != 0xffffffffu && (unsigned)(__double_as_longlong(v.y) >> 32) != 0xffffffffu;
}
__device__ __forceinline__ double2 ld_slot2(const double2* p) {
    double2 v;
    asm volatile("ld.global.cg.v2.f64 {%0,%1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float2 ld_slot1(const float2* p) {
    float2 v;
    asm volatile("ld.global.cg.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ bool slot1_valid(float2 v) {
    return __float_as_uint(v.x) != 0xffffffffu && __float_as_uint(v.y) != 0xffffffffu;
}

__device__ __forceinline__ float canon_f(float v) {
    return __float_as_uint(v) == 0xffffffffu ? __uint_as_float(0x7fc00000u) : v;
}

__device__ __forceinline__ void seg_decode(unsigned t, const SegTmaParams& p, int& kind, int64_t& plane, int& chunk) {
    // the merge of a plane follows its statistics by one plane; the apply trails by L planes
    const unsigned P = (unsigned)(p.n * p.channels), L = (unsigned)p.lag, Lm = L - 1;
    const unsigned Ic = (unsigned)p.ic, St = (unsigned)(p.ic + p.is), Ia = (unsigned)p.ia;
    auto stat = [&](unsigned pl, unsigned u) {
        plane = pl;
        if (u < Ic) { kind = 0; chunk = (int)u; } else { kind = 1; chunk = (int)(u - Ic); }
    };
    unsigned n = (L - Lm) * St;
    if (t < n) { stat(t / St, t % St); return; }
    t -= n; n = Lm * (St + 1);
    if (t < n) {
        const unsigned j = t / (St + 1), u = t % (St + 1);
        if (u < St) stat((L - Lm) + j, u); else { kind = 3; plane = j; chunk = 0; }
        return;
    }
    t -= n; n = (P - L) * (St + 1 + Ia);
    if (t < n) {
        const unsigned j = t / (St + 1 + Ia), u = t % (St + 1 + Ia);
        if (u < St) stat(L + j, u);
        else if (u == St) { kind = 3; plane = Lm + j; chunk = 0; }
        else { kind = 2; plane = j; chunk = (int)(u - St - 1); }
        return;
    }
    t -= n; n = (L - Lm) * (1 + Ia);
    if (t < n) {
        const unsigned j = t / (1 + Ia), u = t % (1 + Ia);
        if (u == 0) { kind = 3; plane = (P - L + Lm) + j; chunk = 0; }
        else { kind = 2; plane = (P - L) + j; chunk = (int)(u - 1); }
        return;
    }
    t -= n;
    kind = 2; plane = (P - Lm) + t / Ia; chunk = (int)(t % Ia);
}

// per-group shared-memory cache: coefficient table by DENSE id (+1 identity entry), shift table and dense-id
// map by label value, atomics accumulators [2][64][2], flush staging [4 warps][32 lanes] and per-warp label
// totals [2][4 warps][32 labels][2]
constexpr int kSegCoefBytes = (kMaxDense + 2) * 16;                                  // 1056
constexpr int kSegCacheBytes = (kSegCoefBytes + kLabels * 4 + kLabels + 2 * kMaxDense * 2 * 4 +
                                kSegGroupWarps * 32 * 16 + 2 * kSegGroupWarps * 32 * 2 * 4 + 127) / 128 * 128;
constexpr int kSegMergeThreads = 64;   // two dedicated merge warps per CTA (one thread per dense label)
constexpr int kSegMailbox = 8;

// Open runs of a warp -> per-label totals tab[d] for dense label d (atomic-free, fixed order; needs <= 32 usable
// labels).  Lanes holding the same label form a group (match.any); its lowest lane adds the others in lane order
// (one shuffle pair per step, as many steps as the largest group has members) and stores the group's total.
// A third of the instructions of the scan it replaces (every lane reading all 32 staged runs).
__device__ __forceinline__ void seg_warp_totals(float2* tab, int lane, int cur, float a1, float a2) {
    const int key = cur >= 0 ? cur : -1;
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    const int steps = (int)__reduce_max_sync(0xffffffffu, (unsigned)__popc(peers));
    float s1 = a1, s2 = a2;
    unsigned rem = peers & (peers - 1u);   // the group without its lowest lane
    const bool leader = (peers & ((1u << lane) - 1u)) == 0u;
    for (int k = 1; k < steps; ++k) {
        const int src = rem ? __ffs(rem) - 1 : lane;
        const float x1 = __shfl_sync(0xffffffffu, a1, src), x2 = __shfl_sync(0xffffffffu, a2, src);
        if (rem) { s1 += x1; s2 += x2; }
        rem &= rem - 1u;
    }
    tab[lane] = make_float2(0.f, 0.f);
    __syncwarp();
    if (leader && key >= 0) tab[key] = make_float2(s1, s2);
    __syncwarp();
}

__global__ void __launch_bounds__(32 + kSegGroups * kSegGroupThreads + kSegMergeThreads, 1) seg_tma_kernel(SegTmaParams p) {
    constexpr int S = kSegGroups * kSegDepth;   // stages; group g owns stages g*kSegDepth .. +kSegDepth-1
    constexpr int STAGE_BYTES = kSegStageBytes;
    constexpr int CACHE_BYTES = kSegCacheBytes;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    unsigned char* stages = smem_raw;
    unsigned char* caches = smem_raw + (size_t)S * STAGE_BYTES;
    SegDesc* desc = reinterpret_cast<SegDesc*>(caches + (size_t)kSegGroups * ((CACHE_BYTES + 127) / 128 * 128));
    uint64_t* full = reinterpret_cast<uint64_t*>(desc + S);
    uint64_t* empty = full + S;
    uint64_t* mfull = empty + S;              // merge mailbox: producer -> merge warps
    uint64_t* mempty = mfull + kSegMailbox;
    int64_t* mbox = reinterpret_cast<int64_t*>(mempty + kSegMailbox);   // plane id, -1 = stop
    SegDecoded* dec = reinterpret_cast<SegDecoded*>(mbox + kSegMailbox);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (__ldg(p.overflow) != 0) return;   // more usable labels than slot capacity: the fallback kernel handles the call
    if (threadIdx.x == 0) {
        for (int s = 0; s < S; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kSegGroupWarps);
        }
        for (int s = 0; s < kSegMailbox; ++s) {
            mbar_init(&mfull[s], 1);
            mbar_init(&mempty[s], kSegMergeThreads / 32);
        }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp == 0) {
        // ================================================================ producer warp
        const uint64_t pol_first = policy_evict_first();
        const uint64_t pol_last = policy_evict_last();
        unsigned next_base = 0;
        if (lane == 0) next_base = atomicAdd(p.ticket, (unsigned)kSegTicketBatch) + 1u;
        unsigned seq = 0, mseq = 0;
        for (;;) {
            const unsigned base = __shfl_sync(0xffffffffu, next_base, 0);
            if (lane == 0) next_base = atomicAdd(p.ticket, (unsigned)kSegTicketBatch) + 1u;
            // Lane i decodes AND issues ticket base+i: the eight items of a batch go to eight different stages
            // (consecutive sequence numbers, kSegGroups * kSegDepth >= kSegTicketBatch), so their empty-waits,
            // descriptors and TMA issues run in SIMT lock-step instead of one after the other on a single thread (which
            // capped both TMA kernels at ~1.3 M items/s per SM).
            static_assert(kSegGroups * kSegDepth >= kSegTicketBatch, "a batch must not reuse a stage");
            int kind = 3, chunk = 0;    // lanes >= batch: treated like a merge (skipped)
            int64_t plane = 0, splane = 0;   // output plane; source plane of the tensor the item streams
            if (lane < kSegTicketBatch) {
                kind = -1;
                const unsigned t = base + (unsigned)lane;
                if (t < p.total_items) seg_decode(t, p, kind, plane, chunk);
                dec[lane].kind = kind; dec[lane].chunk = chunk; dec[lane].plane = plane;
                // the lane that decodes a ticket also issues it: the map load overlaps the empty-stage wait below
                if (kind == 1) splane = src_plane(p.smap, plane);
                else if (kind == 0 || kind == 2) splane = src_plane(p.cmap, plane);
            }
            __syncwarp();
            const unsigned stopmask = __ballot_sync(0xffffffffu, kind < 0);
            const int nvalid = stopmask ? __ffs(stopmask) - 1 : kSegTicketBatch;   // tickets before the end of work
            if (lane == 0) {
                // merges first: they bypass the stage ring and must never wait behind a busy stage (their own
                // dependencies, the plane's statistics items, are a whole round older than this batch)
                for (int i = 0; i < nvalid; ++i) {
                    if (dec[i].kind == 3) {
                        const int ms = (int)(mseq % kSegMailbox);
                        mbar_wait_quiet(&mempty[ms], ((mseq / kSegMailbox) & 1u) ^ 1u);
                        mbox[ms] = dec[i].plane;
                        mbar_arrive(&mfull[ms]);
                        ++mseq;
                    }
                }
            }
            const bool is_item = lane < nvalid && kind != 3;
            const unsigned itemmask = __ballot_sync(0xffffffffu, is_item);
            const int my_pos = __popc(itemmask & ((1u << lane) - 1u));
            if (is_item) {
                const unsigned my_seq = seq + (unsigned)my_pos;
                const unsigned k = my_seq / kSegGroups;
                const int stage = (int)(my_seq % kSegGroups) * kSegDepth + (int)(k % kSegDepth);
                mbar_wait_quiet(&empty[stage], ((k / kSegDepth) & 1u) ^ 1u);
                SegDesc* d = &desc[stage];
                d->plane = plane; d->kind = kind; d->chunk = chunk;
                const bool is_style = kind == 1;
                const int64_t hw = is_style ? p.hw_s : p.hw_c;
                const int item_elems = kind == 2 ? p.apply_elems : kSegItemElems;
                const int64_t e0 = (int64_t)chunk * item_elems;
                const int64_t rem = hw - e0;
                const int nvec = (int)((rem < item_elems ? rem : item_elems) / 4);
                d->nvec = nvec;
                const uint32_t bytes = (uint32_t)nvec * 16u;
                unsigned char* st = stages + (size_t)stage * STAGE_BYTES;
                const int64_t sample = (int)plane / (int)p.channels;
                const float* src = (is_style ? p.style : p.content) + splane * hw + e0;
                const uint8_t* lab = (is_style ? p.s_lab : p.c_lab) + sample * hw + e0;
                const bool has_prev = kind == 2 && p.prev != nullptr;
                mbar_arrive_expect_tx(&full[stage], bytes + (has_prev ? bytes : 0u) + (uint32_t)nvec * 4u);
                tma_load_1d(st, src, bytes, &full[stage], kind == 0 ? pol_last : pol_first);
                if (has_prev)
                    tma_load_1d(st + kSegHalfElems * 4, p.prev + plane * hw + e0, bytes, &full[stage], pol_first);
                tma_load_1d(st + kSegDataBytes, lab, (uint32_t)nvec * 4u, &full[stage], pol_last);
            }
            __syncwarp();
            seq += (unsigned)__popc(itemmask);
            bool finished = false;
            if (stopmask != 0u) {
                if (lane == 0) {
                    for (int g = 0; g < kSegGroups; ++g, ++seq) {   // one stop descriptor per consumer group
                        const unsigned k = seq / kSegGroups;
                        const int stage = (int)(seq % kSegGroups) * kSegDepth + (int)(k % kSegDepth);
                        mbar_wait_quiet(&empty[stage], ((k / kSegDepth) & 1u) ^ 1u);
                        desc[stage].kind = -1;
                        mbar_arrive(&full[stage]);
                    }
                    const int ms = (int)(mseq % kSegMailbox);
                    mbar_wait_quiet(&mempty[ms], ((mseq / kSegMailbox) & 1u) ^ 1u);
                    mbox[ms] = -1;
                    mbar_arrive(&mfull[ms]);
                }
                finished = true;
            }
            if (finished) return;
            __syncwarp();
        }
    }

    if (warp > kSegGroups * kSegGroupWarps) {
        // ================================================================ merge warps
        // The 64 merge threads split a plane's slot rows as (dense label, part): with d usable labels there are
        // 64/d parts per label, each summing a contiguous range of item slots (content then style, fixed
        // order, fp64, 32 loads in flight); part 0 then adds the parts in index order (deterministic) and
        // writes the label's coefficients.  19 labels => 3 parts => a plane's ~1000 slots take ~11 load rounds.
        __shared__ double s_merge[kSegMergeThreads][4];
        const int t = threadIdx.x - (32 + kSegGroups * kSegGroupThreads);
        for (unsigned mseq = 0;; ++mseq) {
            const int ms = (int)(mseq % kSegMailbox);
            mbar_wait_quiet(&mfull[ms], (mseq / kSegMailbox) & 1u, 64);
            const int64_t plane = mbox[ms];
            __syncwarp();
            if (lane == 0) mbar_arrive(&mempty[ms]);
            if (plane < 0) break;
            const int64_t sample = plane / p.channels;
            const int dcount = __ldg(p.dense_count + sample);
            const int parts = dcount > 0 ? kSegMergeThreads / dcount : 1;
            const int dn = dcount > 0 ? t % dcount : 0;
            const int part = dcount > 0 ? t / dcount : parts;
            double s4[4] = {0.0, 0.0, 0.0, 0.0};
            if (part < parts) {
#pragma unroll
                for (int which = 0; which < 2; ++which) {
                    const int items = which ? p.is : p.ic;
                    const int per = (items + parts - 1) / parts;
                    const int lo = part * per, hi = min(items, lo + per);
                    const float2* base = p.slots + ((plane * 2 + which) * p.imax) * kMaxDense + dn;
                    constexpr int kUnroll = 32;
                    for (int c0 = lo; c0 < hi; c0 += kUnroll) {
                        float2 v[kUnroll];
#pragma unroll
                        for (int u = 0; u < kUnroll; ++u) {
                            v[u] = make_float2(0.f, 0.f);
                            if (c0 + u < hi) v[u] = ld_slot1(base + (int64_t)(c0 + u) * kMaxDense);
                        }
#pragma unroll
                        for (int u = 0; u < kUnroll; ++u) {
                            if (c0 + u < hi) {
                                if (!slot1_valid(v[u])) {
                                    const float2* sp = base + (int64_t)(c0 + u) * kMaxDense;
                                    const uint64_t t0 = global_timer_ns();
                                    do {   // straggling statistics item
                                        __nanosleep(64);
                                        v[u] = ld_slot1(sp);
                                        if (watchdog_expired(t0)) __trap();
                                    } while (!slot1_valid(v[u]));
                                }
                                s4[which * 2 + 0] += (double)v[u].x;
                                s4[which * 2 + 1] += (double)v[u].y;
                            }
                        }
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) s_merge[t][q] = s4[q];
            named_bar_sync(15, kSegMergeThreads);
            if (t < dcount) {   // part 0 of label dn == t
                for (int q = 1; q < parts; ++q) {
#pragma unroll
                    for (int e = 0; e < 4; ++e) s4[e] += s_merge[q * dcount + t][e];
                }
                const int l = __ldg(p.label_of + sample * kMaxDense + dn);
                const double dnc = (double)__ldg(p.cnt + (sample * 2 + 0) * kLabels + l);
                const double dns = (double)__ldg(p.cnt + (sample * 2 + 1) * kLabels + l);
                const double kc = (double)__ldg(p.shift + (plane * 2 + 0) * kLabels + l);
                const double ks = (double)__ldg(p.shift + (plane * 2 + 1) * kLabels + l);
                const double mu_c = kc + s4[0] / dnc, mu_s = ks + s4[2] / dns;
                const double m2c = fmax(s4[1] - s4[0] * s4[0] / dnc, 0.0), m2s = fmax(s4[3] - s4[2] * s4[2] / dns, 0.0);
                const double sd_c = sqrt(m2c / (dnc - 1.0) + (double)p.eps), sd_s = sqrt(m2s / (dns - 1.0) + (double)p.eps);
                __stcg(&p.coef[plane * kLabels + l], make_float4((float)mu_c, (float)(sd_s / sd_c), (float)mu_s, 1.f));
            }
            // identity for every unusable label: (c-0)*1+0 == c bit-exactly
            for (int l = t; l < kLabels; l += kSegMergeThreads)
                if (__ldg(p.dense + sample * kLabels + l) == 255) __stcg(&p.coef[plane * kLabels + l], make_float4(0.f, 1.f, 0.f, 0.f));
            __threadfence();
            named_bar_sync(15, kSegMergeThreads);
            if (t == 0) st_release(&p.ready[plane], 1);
        }
        return;
    }

    // ==================================================================== consumers
    const int group = (warp - 1) / kSegGroupWarps;
    const int gw = (warp - 1) % kSegGroupWarps;
    const int gt = gw * 32 + lane;
    unsigned char* cache = caches + (size_t)group * ((CACHE_BYTES + 127) / 128 * 128);
    float4* c_coef = reinterpret_cast<float4*>(cache);                                  // [kMaxDense + 1] by dense id; last = identity
    float* c_shift = reinterpret_cast<float*>(cache + kSegCoefBytes);                    // [256] by label
    unsigned char* c_dense = cache + kSegCoefBytes + kLabels * 4;                        // [256] by label
    float* c_acc = reinterpret_cast<float*>(c_dense + kLabels);                          // [2][kMaxDense][2]
    float4* c_stage = reinterpret_cast<float4*>(c_acc + 2 * kMaxDense * 2);              // [4 warps][32 lanes]
    float* c_wtot = reinterpret_cast<float*>(c_stage + kSegGroupWarps * 32);             // [2][4 warps][32][2]
    const uint64_t pol_first = policy_evict_first();
    int64_t cached_stat = -1;    // plane*2+which whose shift table is in the cache
    int64_t cached_apply = -1;   // plane whose coefficient table is in the cache
    int64_t cached_sample = -1;  // sample whose dense-id map is in the cache
    int dcount = 0;
    unsigned sparity = 0;        // accumulator double buffering (per statistics item)
    for (int i = gt; i < 2 * kMaxDense * 2; i += kSegGroupThreads) c_acc[i] = 0.f;
    named_bar_sync(1 + group, kSegGroupThreads);

    for (unsigned seq = group;; seq += kSegGroups) {
        const unsigned k = seq / kSegGroups;
        const int stage = group * kSegDepth + (int)(k % kSegDepth);
        mbar_wait_quiet(&full[stage], (k / kSegDepth) & 1u);
        const SegDesc* d = &desc[stage];
        const int kind = d->kind;
        if (kind < 0) break;
        const int64_t plane = d->plane;
        const int chunk = d->chunk;
        // vectors per warp: a full item gives each warp 512 (16 per lane), a half item (apply with prev) 256
        const int warp_vecs = (kind == 2 ? p.apply_elems : kSegItemElems) / 4 / kSegGroupWarps;
        const int wvec = min(max(d->nvec - gw * warp_vecs, 0), warp_vecs);
        const int64_t sample = (int)plane / (int)p.channels;   // planes < 2^31 (checked by the host): 32-bit division
        unsigned char* st = stages + (size_t)stage * STAGE_BYTES;
        const float4* a4 = reinterpret_cast<const float4*>(st) + gw * warp_vecs;
        const float4* b4 = reinterpret_cast<const float4*>(st + kSegHalfElems * 4) + gw * warp_vecs;
        const uint32_t* l4 = reinterpret_cast<const uint32_t*>(st + kSegDataBytes) + gw * warp_vecs;

        {
            if (sample != cached_sample) {   // group-uniform: dense-id map of this sample
                named_bar_sync(1 + group, kSegGroupThreads);
                for (int l = gt; l < kLabels; l += kSegGroupThreads) c_dense[l] = __ldg(p.dense + sample * kLabels + l);
                dcount = __ldg(p.dense_count + sample);
                named_bar_sync(1 + group, kSegGroupThreads);
                cached_sample = sample;
            }
        }

        if (kind <= 1) {
            // ---------------- statistics of this group's 4096 pixels, per (dense) label
            const int64_t key = plane * 2 + kind;
            if (key != cached_stat) {     // group-uniform: shift table of this plane/tensor
                named_bar_sync(1 + group, kSegGroupThreads);
                for (int l = gt; l < kLabels; l += kSegGroupThreads) c_shift[l] = __ldg(p.shift + key * kLabels + l);
                named_bar_sync(1 + group, kSegGroupThreads);
                cached_stat = key;
            }
            float* acc = c_acc + sparity * (kMaxDense * 2);
            int cur = -1;                  // dense id of the running label (-1: unusable, skipped)
            uint32_t cur4 = 0xffffffffu;   // its label value replicated x4; never matches while cur < 0
            float shift = 0.f, a1 = 0.f, a2 = 0.f;
            // Each lane owns 32 CONTIGUOUS pixels (8 float4) so that label runs stay long on blocky maps;
            // the 8 vectors are visited in a lane-rotated order, which keeps the 128-byte-strided
            // shared-memory reads of a quarter warp on distinct banks.
            // all of the lane's vectors and label words are fetched first (16 independent shared-memory loads),
            // the run logic below then works from registers instead of paying one LDS latency per step
            float4 vv[kSegLaneVecs];
            uint32_t lww[kSegLaneVecs];
#pragma unroll
            for (int j = 0; j < kSegLaneVecs; ++j) {
                const int idx = lane * kSegLaneVecs + ((j + lane) & (kSegLaneVecs - 1));
                if (idx < wvec) { vv[j] = a4[idx]; lww[j] = l4[idx]; }
            }
            // the stage has been consumed (everything is in registers): hand it back before the arithmetic
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[stage]);
#pragma unroll
            for (int j = 0; j < kSegLaneVecs; ++j) {
                const int idx = lane * kSegLaneVecs + ((j + lane) & (kSegLaneVecs - 1));
                if (idx < wvec) {
                    const float4 v = vv[j];
                    const uint32_t lw = lww[j];
                    if (lw == cur4 && cur >= 0) {
                        const float d0 = v.x - shift, d1 = v.y - shift, d2 = v.z - shift, d3 = v.w - shift;
                        a1 += (d0 + d1) + (d2 + d3);
                        a2 = fmaf(d0, d0, a2); a2 = fmaf(d1, d1, a2); a2 = fmaf(d2, d2, a2); a2 = fmaf(d3, d3, a2);
                    } else {
                        const float e[4] = {v.x, v.y, v.z, v.w};
                        int curl = cur >= 0 ? (int)(cur4 & 0xffu) : -1;
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int l = (int)((lw >> (8 * q)) & 0xffu);
                            if (l != curl) {
                                if (cur >= 0) {   // label run ended inside the item: flush it
                                    atomicAdd(&acc[cur * 2 + 0], a1);
                                    atomicAdd(&acc[cur * 2 + 1], a2);
                                }
                                const int dn = c_dense[l];
                                curl = l;
                                if (dn != 255) { cur = dn; shift = c_shift[l]; cur4 = (uint32_t)l * 0x01010101u; }
                                else { cur = -1; cur4 = 0xffffffffu; }
                                a1 = 0.f; a2 = 0.f;
                            }
                            if (cur >= 0) {
                                const float dd = e[q] - shift;
                                a1 += dd;
                                a2 = fmaf(dd, dd, a2);
                            }
                        }
                    }
                }
            }
            // final flush of the open runs into the group's accumulators: with <= 32 usable labels a staged gather
            // (atomic-free and deterministic: the warp's totals per dense label, lane-ordered sums; the publishing
            // thread below adds the four warps in warp order), above that one shared-memory atomic per lane (one pass
            // per distinct address, which beats a shuffle tree per distinct label on fine-grained maps)
            const bool staged = dcount <= 32;
            float* wt = c_wtot + (sparity * kSegGroupWarps + gw) * 64;
            if (staged) {
                seg_warp_totals(reinterpret_cast<float2*>(wt), lane, cur, a1, a2);
            } else if (cur >= 0) {
                atomicAdd(&acc[cur * 2 + 0], a1);
                atomicAdd(&acc[cur * 2 + 1], a2);
            }
            named_bar_sync(1 + group, kSegGroupThreads);
            // publish: one self-validating 8-byte slot per usable label (no fence, no atomic, no counter)
            if (gt < dcount) {
                float t1 = acc[gt * 2 + 0], t2 = acc[gt * 2 + 1];   // mid-item flushes (label change inside a lane's run)
                if (staged) {
                    const float* w0 = c_wtot + sparity * kSegGroupWarps * 64;
#pragma unroll
                    for (int q = 0; q < kSegGroupWarps; ++q) { t1 += w0[q * 64 + gt * 2 + 0]; t2 += w0[q * 64 + gt * 2 + 1]; }
                }
                const float s1 = canon_f(t1), s2 = canon_f(t2);
                acc[gt * 2 + 0] = 0.f;
                acc[gt * 2 + 1] = 0.f;
                float2* slot = p.slots + ((key * p.imax + chunk) * kMaxDense + gt);
                asm volatile("st.global.cg.v2.f32 [%0], {%1,%2};" :: "l"(slot), "f"(s1), "f"(s2) : "memory");
            }
            sparity ^= 1u;
        } else if (kind == 2) {
            // ---------------- apply
            if (plane != cached_apply) {   // group-uniform: wait for the merge item, cache the coefficient table
                if (lane == 0 && ld_acquire(&p.ready[plane]) == 0) {
                    const uint64_t t0 = global_timer_ns();
                    while (ld_acquire(&p.ready[plane]) == 0) {
                        __nanosleep(64);
                        if (watchdog_expired(t0)) __trap();
                    }
                }
                named_bar_sync(1 + group, kSegGroupThreads);
                if (gt < dcount) c_coef[gt] = __ldcg(&p.coef[plane * kLabels + __ldg(p.label_of + sample * kMaxDense + gt)]);
                if (gt == kSegGroupThreads - 1) c_coef[kMaxDense] = make_float4(0.f, 1.f, 0.f, 0.f);   // unusable labels: (c-0)*1+0 == c
                named_bar_sync(1 + group, kSegGroupThreads);
                cached_apply = plane;
            }
            const bool has_prev = p.prev != nullptr;
            float4* o4 = reinterpret_cast<float4*>(p.out + sample * p.out_batch_stride + (plane - sample * p.channels) * p.hw_c +
                                                   (int64_t)chunk * p.apply_elems) + gw * warp_vecs;
            uint32_t last_w = 0;
            float4 cf = c_coef[kMaxDense];
            bool have = false;
            auto coef_of = [&](uint32_t l) -> float4 { const int dn = c_dense[l]; return c_coef[dn < kMaxDense ? dn : kMaxDense]; };
#pragma unroll 8
            for (int j = 0; j < kSegLaneVecs; ++j) {
                const int idx = j * 32 + lane;
                if (idx < wvec) {
                    const float4 v = a4[idx];
                    const uint32_t lw = l4[idx];
                    float4 o;
                    const uint32_t b0 = lw & 0xffu;
                    if (lw == b0 * 0x01010101u) {   // all four pixels carry the same label
                        if (!have || lw != last_w) { cf = coef_of(b0); last_w = lw; have = true; }
                        o.x = fmaf(v.x - cf.x, cf.y, cf.z);
                        o.y = fmaf(v.y - cf.x, cf.y, cf.z);
                        o.z = fmaf(v.z - cf.x, cf.y, cf.z);
                        o.w = fmaf(v.w - cf.x, cf.y, cf.z);
                    } else {
                        const float4 c0 = coef_of(b0), c1 = coef_of((lw >> 8) & 0xffu), c2 = coef_of((lw >> 16) & 0xffu),
                                     c3 = coef_of(lw >> 24);
                        o.x = fmaf(v.x - c0.x, c0.y, c0.z);
                        o.y = fmaf(v.y - c1.x, c1.y, c1.z);
                        o.z = fmaf(v.z - c2.x, c2.y, c2.z);
                        o.w = fmaf(v.w - c3.x, c3.y, c3.z);
                    }
                    if (has_prev) {
                        const float4 q = b4[idx];
                        o.x += q.x; o.y += q.y; o.z += q.z; o.w += q.w;
                    }
                    stg_f4_hint(reinterpret_cast<float*>(o4 + idx), o, pol_first);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[stage]);
        }
    }
}

__global__ void seg_export_info_kernel(const int* __restrict__ cnt, int32_t* __restrict__ info, int64_t n) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n * kLabels) return;
    const int64_t s = i / kLabels, l = i % kLabels;
    const int nc = cnt[(s * 2 + 0) * kLabels + l], ns = cnt[(s * 2 + 1) * kLabels + l];
    info[i * 3 + 0] = nc;
    info[i * 3 + 1] = ns;
    info[i * 3 + 2] = label_usable(nc, ns) ? 1 : 0;
}

struct SegLayout {
    size_t zero_bytes;   // ticket, done, ready, cnt, gsum (memset 0)
    size_t first_off, first_bytes, coef_off, total;
    size_t done_off, cnt_off, gsum_off;
};

SegLayout seg_layout(int64_t n, int64_t c) {
    const size_t planes = (size_t)(n * c);
    SegLayout l;
    l.done_off = 256;
    l.cnt_off = align_up(l.done_off + planes * 2 * sizeof(int), 256);
    l.gsum_off = align_up(l.cnt_off + (size_t)n * 2 * kLabels * sizeof(int), 256);
    l.zero_bytes = align_up(l.gsum_off + planes * 2 * kLabels * sizeof(float2), 256);
    l.first_off = l.zero_bytes;
    l.first_bytes = align_up((size_t)n * 2 * kLabels * sizeof(int), 256);
    l.coef_off = l.first_off + l.first_bytes;
    l.total = align_up(l.coef_off + planes * kLabels * sizeof(float4), 256);
    return l;
}

inline bool aligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }

struct SegTmaLayout {
    size_t ticket, zero_beg, ready, cnt, dcount, overflow, zero_end, first, first_bytes, shift, dense, label_of, coef,
        slots, slots_bytes, total;
};
SegTmaLayout seg_tma_layout(int64_t n, int64_t c, int64_t hw_c, int64_t hw_s) {
    const size_t planes = (size_t)(n * c);
    const size_t ic = (size_t)((hw_c + kSegItemElems - 1) / kSegItemElems), is = (size_t)((hw_s + kSegItemElems - 1) / kSegItemElems);
    const size_t imax = ic > is ? ic : is;
    SegTmaLayout l;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o += align_up(bytes, 256); return at; };
    l.ticket = take(256);
    l.zero_beg = o;
    l.ready = take(planes * sizeof(int));
    l.cnt = take((size_t)n * 2 * kLabels * sizeof(int));
    l.dcount = take((size_t)n * sizeof(int));
    l.overflow = take(sizeof(int));
    l.zero_end = o;
    l.first_bytes = align_up((size_t)n * 2 * kLabels * sizeof(int), 256);
    l.first = take(l.first_bytes);
    l.shift = take(planes * 2 * kLabels * sizeof(float));
    l.dense = take((size_t)n * kLabels);
    l.label_of = take((size_t)n * kMaxDense);
    l.coef = take(planes * kLabels * sizeof(float4));
    l.slots_bytes = planes * 2 * imax * kMaxDense * sizeof(float2);
    l.slots = take(l.slots_bytes);
    l.total = o;
    return l;
}

int launch_seg_tma(const SegTmaParams& p, cudaStream_t st) {
    constexpr size_t stage = kSegStageBytes;
    constexpr size_t cache = kSegCacheBytes;
    constexpr size_t smem = kSegGroups * (kSegDepth * stage + cache) + kSegGroups * kSegDepth * sizeof(SegDesc) +
                            2 * kSegGroups * kSegDepth * sizeof(uint64_t) + 2 * kSegMailbox * sizeof(uint64_t) +
                            kSegMailbox * sizeof(int64_t) +
                            kSegTicketBatch * sizeof(SegDecoded);
    static PerDeviceFlag configured_on;
    bool& configured = configured_on.get();
    if (!configured) {
        RPST_CUDA(cudaFuncSetAttribute(seg_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = true;
    }
    int64_t grid = sm_count();
    if (grid > (int64_t)p.total_items) grid = p.total_items;
    seg_tma_kernel<<<(int)grid, 32 + kSegGroups * kSegGroupThreads + kSegMergeThreads, smem, st>>>(p);
    RPST_CUDA(cudaGetLastError());
    return RPST_OK;
}

}  // namespace
}  // namespace rpst

namespace rpst {
namespace {
// item geometry and ticket schedule of seg_tma_kernel for one call (q.n, q.channels, q.hw_c, q.hw_s set); returns the ticket count
int64_t seg_plan_schedule(SegTmaParams& q, bool has_prev) {
    const int64_t planes = q.n * q.channels;
    q.ic = (int)((q.hw_c + kSegItemElems - 1) / kSegItemElems);
    q.is = (int)((q.hw_s + kSegItemElems - 1) / kSegItemElems);
    q.imax = q.ic > q.is ? q.ic : q.is;
    q.apply_elems = has_prev ? kSegPrevElems : kSegItemElems;
    q.ia = (int)((q.hw_c + q.apply_elems - 1) / q.apply_elems);
    const int64_t plane_bytes = q.hw_c * (int64_t)sizeof(float);
    int64_t lag = (g_knobs.seg_lag_bytes + plane_bytes - 1) / plane_bytes;
    if (lag < 3) lag = 3;
    q.lag = (int)(lag < planes ? lag : planes);
    return planes * ((int64_t)q.ic + q.is + 1 + q.ia);
}

__global__ void seg_schedule_dump_kernel(SegTmaParams p, int32_t* out) {
    const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.total_items) return;
    int kind = -1, chunk = 0;
    int64_t plane = 0;
    seg_decode(t, p, kind, plane, chunk);
    out[3 * (size_t)t + 0] = kind;
    out[3 * (size_t)t + 1] = (int32_t)plane;
    out[3 * (size_t)t + 2] = chunk;
}
}  // namespace
}  // namespace rpst

using namespace rpst;

#ifdef RPST_DEBUG_EXPORTS   // white-box test hooks: only in librpst_debug.so (loaded by tests alone), never in the product library
// Test hook, see rpst_debug_adain_schedule: kind 0 content statistics, 1 style statistics, 2 apply, 3 merge;
// info = {tickets, content items, style items, apply items, lag}.
extern "C" int rpst_debug_seg_schedule(int64_t n, int64_t c, int64_t hw_c, int64_t hw_s, int has_prev, int32_t* tickets,
                                       int64_t max_tickets, int64_t* info, void* stream) {
    RPST_CHECK_ARG(n > 0 && c > 0 && hw_c > 0 && hw_s > 0 && info != nullptr, "debug_seg_schedule: bad arguments");
    SegTmaParams q{};
    q.n = n; q.channels = c; q.hw_c = hw_c; q.hw_s = hw_s;
    const int64_t total = seg_plan_schedule(q, has_prev != 0);
    RPST_CHECK_ARG(total < (1ll << 31), "debug_seg_schedule: too many tickets");
    q.total_items = (unsigned)total;
    info[0] = total; info[1] = q.ic; info[2] = q.is; info[3] = q.ia; info[4] = q.lag;
    if (tickets != nullptr) {
        RPST_CHECK_ARG(max_tickets >= total, "debug_seg_schedule: ticket buffer too small");
        seg_schedule_dump_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(q, tickets);
        RPST_CUDA(cudaGetLastError());
    }
    return RPST_OK;
}
#endif  // RPST_DEBUG_EXPORTS

extern "C" size_t rpst_seg_adain_workspace_bytes(int64_t n, int64_t c, int64_t hw_c, int64_t hw_s) {
    if (n <= 0 || c <= 0) return 256;
    return seg_layout(n, c).total + seg_tma_layout(n, c, hw_c, hw_s).total;   // slot path + fallback path

}

namespace {
int seg_adain_fwd_impl(const float* content, const float* style, const uint8_t* c_labels, const uint8_t* s_labels,
                       const float* prev, float* out, int64_t n, int64_t c, int64_t hw_c, int64_t hw_s,
                       int64_t out_batch_stride, float eps, const int* content_map, const int* style_map,
                       int32_t* label_info, void* workspace, size_t workspace_bytes, void* stream);
}

extern "C" int rpst_seg_adain_fwd(const float* content, const float* style, const uint8_t* c_labels,
                                  const uint8_t* s_labels, const float* prev, float* out, int64_t n, int64_t c,
                                  int64_t hw_c, int64_t hw_s, float eps, int32_t* label_info, void* workspace,
                                  size_t workspace_bytes, void* stream) {
    return seg_adain_fwd_impl(content, style, c_labels, s_labels, prev, out, n, c, hw_c, hw_s, c * hw_c, eps, nullptr,
                              nullptr, label_info, workspace, workspace_bytes, stream);
}

extern "C" int rpst_seg_adain_fwd_mapped(const float* content, const float* style, const uint8_t* c_labels,
                                         const uint8_t* s_labels, const float* prev, float* out, int64_t n, int64_t c,
                                         int64_t hw_c, int64_t hw_s, int64_t out_batch_stride, float eps,
                                         const int32_t* content_map, const int32_t* style_map, int32_t* label_info,
                                         void* workspace, size_t workspace_bytes, void* stream) {
    RPST_CHECK_ARG(n * c < (1ll << 31), "seg_adain_mapped: plane index does not fit int32");
    return seg_adain_fwd_impl(content, style, c_labels, s_labels, prev, out, n, c, hw_c, hw_s, out_batch_stride, eps,
                              content_map, style_map, label_info, workspace, workspace_bytes, stream);
}

namespace {
int seg_adain_fwd_impl(const float* content, const float* style, const uint8_t* c_labels, const uint8_t* s_labels,
                       const float* prev, float* out, int64_t n, int64_t c, int64_t hw_c, int64_t hw_s,
                       int64_t out_batch_stride, float eps, const int* content_map, const int* style_map,
                       int32_t* label_info, void* workspace, size_t workspace_bytes, void* stream) {
    RPST_CHECK_ARG(n >= 0 && c >= 0 && hw_c >= 0 && hw_s >= 0, "seg_adain: negative size");
    if (n == 0 || c == 0 || hw_c == 0) return RPST_OK;
    RPST_CHECK_ARG(content && style && c_labels && s_labels && out, "seg_adain: null pointer");
    RPST_CHECK_ARG(hw_s > 0, "seg_adain: empty style map");
    RPST_CHECK_ARG(hw_c < (1ll << 31) && hw_s < (1ll << 31), "seg_adain: plane too large");
    RPST_CHECK_ARG(out_batch_stride >= c * hw_c, "seg_adain: out_batch_stride (%lld) < c*hw_c (%lld)",
                   (long long)out_batch_stride, (long long)(c * hw_c));
    RPST_CHECK_ARG(out != content && out != style && out != prev, "seg_adain: out must not alias an input");
    const size_t need = rpst_seg_adain_workspace_bytes(n, c, hw_c, hw_s);
    if (workspace == nullptr || workspace_bytes < need) {
        set_error("seg_adain: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
        return RPST_ERR_WORKSPACE;
    }
    RPST_CHECK_ARG(aligned(workspace, 256), "seg_adain: workspace must be 256-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    char* base = static_cast<char*>(workspace);
    const int64_t hw_max0 = hw_c > hw_s ? hw_c : hw_s;
    int hist_blocks0 = (int)((hw_max0 + 16383) / 16384);
    if (hist_blocks0 > 256) hist_blocks0 = 256;
    const bool tma_ok = g_knobs.adain_path == 0 && hw_c % 16 == 0 && hw_s % 16 == 0 &&
                        aligned(content, 16) && aligned(style, 16) && aligned(out, 16) && out_batch_stride % 4 == 0 &&
                        (!prev || aligned(prev, 16)) && aligned(c_labels, 16) && aligned(s_labels, 16);
    const int* run_flag = nullptr;
    if (tma_ok) {
        const SegTmaLayout t = seg_tma_layout(n, c, hw_c, hw_s);
        SegTmaParams q{};
        q.content = content; q.style = style; q.c_lab = c_labels; q.s_lab = s_labels; q.prev = prev; q.out = out;
        q.cmap = content_map; q.smap = style_map;
        q.n = n; q.channels = c; q.hw_c = hw_c; q.hw_s = hw_s; q.out_batch_stride = out_batch_stride; q.eps = eps;
        q.ticket = reinterpret_cast<unsigned*>(base + t.ticket);
        q.ready = reinterpret_cast<int*>(base + t.ready);
        int* cnt = reinterpret_cast<int*>(base + t.cnt);
        int* first = reinterpret_cast<int*>(base + t.first);
        int* dcount = reinterpret_cast<int*>(base + t.dcount);
        int* overflow = reinterpret_cast<int*>(base + t.overflow);
        unsigned char* dense = reinterpret_cast<unsigned char*>(base + t.dense);
        unsigned char* label_of = reinterpret_cast<unsigned char*>(base + t.label_of);
        q.cnt = cnt; q.first = first; q.dense = dense; q.label_of = label_of; q.dense_count = dcount; q.overflow = overflow;
        q.shift = reinterpret_cast<float*>(base + t.shift);
        q.coef = reinterpret_cast<float4*>(base + t.coef);
        q.slots = reinterpret_cast<float2*>(base + t.slots);
        RPST_CUDA(cudaMemsetAsync(base + t.ticket, 0xff, 256, st));
        RPST_CUDA(cudaMemsetAsync(base + t.zero_beg, 0, t.zero_end - t.zero_beg, st));
        RPST_CUDA(cudaMemsetAsync(base + t.first, 0x7f, t.first_bytes, st));
        RPST_CUDA(cudaMemsetAsync(base + t.slots, 0xff, t.slots_bytes, st));
        seg_hist_kernel<<<dim3(hist_blocks0, (unsigned)n, 2), 256, 0, st>>>(c_labels, s_labels, hw_c, hw_s, cnt, first);
        RPST_CUDA(cudaGetLastError());
        seg_dense_kernel<<<(unsigned)n, kLabels, 0, st>>>(cnt, dense, label_of, dcount, overflow);
        RPST_CUDA(cudaGetLastError());
        if (label_info) {
            const int64_t tot = n * kLabels;
            seg_export_info_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(cnt, label_info, n);
            RPST_CUDA(cudaGetLastError());
            label_info = nullptr;   // the fallback path below must not export it again
        }
        const int64_t planes = n * c;
        seg_shift_kernel<<<(unsigned)((planes * 2 * kLabels + 255) / 256), 256, 0, st>>>(q);
        RPST_CUDA(cudaGetLastError());
        const int64_t total = seg_plan_schedule(q, prev != nullptr);
        RPST_CHECK_ARG(total < (1ll << 31), "seg_adain: too many work items (%lld); split the call", (long long)total);
        q.total_items = (unsigned)total;
        const int rc = launch_seg_tma(q, st);
        if (rc) return rc;
        // a sample with more than kMaxDense usable labels makes the slot kernel exit at once and the
        // register-staged kernel below run instead (device-side decision: no host synchronisation)
        run_flag = overflow;
        base += t.total;
    }
    const SegLayout l = seg_layout(n, c);
    SegParams p{};
    p.content = content; p.style = style; p.c_lab = c_labels; p.s_lab = s_labels; p.prev = prev; p.out = out;
    p.cmap = content_map; p.smap = style_map;
    p.n = n; p.channels = c; p.hw_c = hw_c; p.hw_s = hw_s; p.out_batch_stride = out_batch_stride; p.eps = eps;
    p.hints = (int)g_knobs.adain_hints;
    p.ticket = reinterpret_cast<unsigned*>(base);
    p.done = reinterpret_cast<int*>(base + l.done_off);
    p.ready = p.done + n * c;
    p.cnt = reinterpret_cast<int*>(base + l.cnt_off);
    p.gsum = reinterpret_cast<float2*>(base + l.gsum_off);
    p.first = reinterpret_cast<int*>(base + l.first_off);
    p.coef = reinterpret_cast<float4*>(base + l.coef_off);
    p.run_flag = run_flag;
    RPST_CUDA(cudaMemsetAsync(base, 0, l.zero_bytes, st));
    RPST_CUDA(cudaMemsetAsync(base + l.first_off, 0x7f, l.first_bytes, st));

    const int64_t hw_max = hw_c > hw_s ? hw_c : hw_s;
    int hist_blocks = (int)((hw_max + 16383) / 16384);
    if (hist_blocks > 256) hist_blocks = 256;
    seg_hist_kernel<<<dim3(hist_blocks, (unsigned)n, 2), 256, 0, st>>>(c_labels, s_labels, hw_c, hw_s, p.cnt, p.first);
    RPST_CUDA(cudaGetLastError());
    if (label_info) {
        const int64_t tot = n * kLabels;
        seg_export_info_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(p.cnt, label_info, n);
        RPST_CUDA(cudaGetLastError());
    }

    const bool vec = hw_c % 4 == 0 && hw_s % 4 == 0 && aligned(content, 16) && aligned(style, 16) && aligned(out, 16) &&
                     out_batch_stride % 4 == 0 && (!prev || aligned(prev, 16)) && aligned(c_labels, 4) && aligned(s_labels, 4);
    const int64_t chunk = (int64_t)kPipeThreads * kPerThread * (vec ? 4 : 1);
    p.ipp_c = (int)((hw_c + chunk - 1) / chunk);
    p.ipp_s = (int)((hw_s + chunk - 1) / chunk);
    const int64_t plane_bytes = hw_c * (int64_t)sizeof(float);
    int64_t lag = (g_knobs.adain_lag_bytes + plane_bytes - 1) / plane_bytes;
    if (lag < 3) lag = 3;
    const int64_t planes = n * c;
    p.lag = (int)(lag < planes ? lag : planes);
    const int64_t total = planes * (2ll * p.ipp_c + p.ipp_s);
    RPST_CHECK_ARG(total < (1ll << 31), "seg_adain: too many work items (%lld); split the call", (long long)total);
    p.total_items = (unsigned)total;
    int64_t grid = (int64_t)sm_count() * 3;
    if (grid > total) grid = total;
    if (vec) seg_pipe_kernel<4><<<(int)grid, kPipeThreads, 0, st>>>(p);
    else seg_pipe_kernel<1><<<(int)grid, kPipeThreads, 0, st>>>(p);
    RPST_CUDA(cudaGetLastError());
    return RPST_OK;
}
}  // namespace

RPST_WATCHDOG_SETTER(seg)

// Fused centred covariance for WCT — SURVEY.md §2b K5, §8 a6; reference: network/wct_rp.py:85-94
// (`cF - mean`, `cF @ cF.t() / (HW - 1)` [+ I on the content side]).
//
// One kernel reads the fp32 features ONCE and feeds the tensor cores directly: no packed-operand round trip
// (the separate pack pass read 268 MB and wrote 222 MB per operand before the GEMM read them again).
//   warps 1..16 converters in two groups that alternate k-tiles (one group's global loads are in flight while the
//               other converts): 128-bit loads of a [C x 64 positions] k-tile, subtract a per-channel SHIFT,
//               split into bf16 hi + lo, store into the K-major SWIZZLE_128B operand tile in shared memory
//               (A and B of the SYRK are the same tile), and keep fp32 row sums of the shifted values
//   warp 0      one thread issues tcgen05.mma: X X^T over this CTA's slice of H*W (split-K over all SMs) into TMEM;
//               only the blocks on and above the diagonal are computed (SYRK symmetry: 3 of 4 128x128 blocks)
//   epilogue    TMEM -> per-CTA fp32 partial Gram; a fixed-order fp64 reduction kernel forms
//               cov = (G - S S^T / HW) / (HW - 1) (+ diag) and the exact means mu = shift + S / HW
// The shift is a cheap sub-sampled mean: centring with ANY shift is exact after the rank-1 correction, and a shift
// close to the mean keeps the correction small (no cancellation), so no full statistics pass is needed.
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"
#include "tuning.cuh"
#include "umma.cuh"

namespace rpst {
namespace {

constexpr int kCovGroupWarps = 8;                            // converter warps per group: warp w owns rows [32 w, 32 w + 32)
constexpr int kCovGroups = 2;
constexpr int kCovConvWarps = kCovGroupWarps * kCovGroups;
constexpr int kCovThreads = 32 * (1 + kCovConvWarps);
constexpr int kCovMaxC = 256;
constexpr uint32_t kCovPartBytes = 2 * kTileBytes;          // [256 rows x 64 positions] bf16 = 32 KiB

struct CovParams {
    const float* x;          // [c, hw] one sample, row stride hw
    float* shift;            // [cp] per-channel shift (rows >= c: 0); written by the TMA kernel itself
    float* partial;          // [grid, cp, cp] per-CTA partial Gram (blocks on/above the diagonal only)
    float* rowsum;           // [grid * 2, cp] per-CTA and converter-group sums of (x - shift)
    int64_t hw;
    int c, cp;               // channels, padded to 128 / 256
    int k_tiles;             // ceil(hw / 64)
    int passes;              // 1: bf16, 3: bf16x3
    // TMA kernel only: the whole covariance in ONE launch (shift in the prologue, grid barrier, distributed fp64 finalize)
    int* barrier;            // zeroed before the launch
    double* s_sum;           // [cp] column sums of the shifted values (exchange buffer)
    double* cov;             // [c, c] result
    float* mean;             // [c] exact means or null
    double diag_add;
    const float* shift_in;      // per-channel shifts computed ahead of the launch (cov_shifts_batched) or null: sample here
    unsigned long long* prof;   // optional [8 x 2] %globaltimer stamps of CTA 0 and the last CTA (tuning knob "wct_cov_prof")
};

// {lo, hi} -> packed bf16x2 with round-to-nearest-even: lo in bits 0..15 (the element at the lower address)
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

template <int PARTS>   // 1: hi only, 2: hi + lo
__global__ void __launch_bounds__(kCovThreads, 1) cov_fused_kernel(CovParams p) {
    constexpr int NST = PARTS == 2 ? 3 : 6;
    constexpr uint32_t kStage = kCovPartBytes * PARTS;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    __shared__ uint64_t full[NST], empty[NST], acc_full;
    __shared__ uint32_t tmem_slot;
    __shared__ float s_shift[kCovMaxC];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m_tiles = p.cp / 128;
    // k-tiles are dealt round-robin: at any moment the co-running CTAs read ADJACENT 256-byte pieces of every channel
    // row (contiguous ranges per CTA scattered 256-byte accesses over DRAM pages: 3.0 TB/s)
    const int nkt = blockIdx.x < p.k_tiles ? (p.k_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NST; ++s) {
            mbar_init(&full[s], kCovGroupWarps);
            mbar_init(&empty[s], 1);
        }
        mbar_init(&acc_full, 1);
        mbar_fence_init();
    }
    if (warp == 0) tmem_alloc(&tmem_slot, 512);
    for (int r = threadIdx.x; r < kCovMaxC; r += blockDim.x) s_shift[r] = r < p.cp ? __ldg(p.shift + r) : 0.f;
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = tmem_slot;

    if (warp == 0) {
        if (lane == 0 && nkt > 0) {
            // SYRK: M-tile 0 against all columns, M-tile 1 against columns 128..255 only
            const uint32_t idesc0 = umma_idesc_bf16(128, p.cp);
            const uint32_t idesc1 = umma_idesc_bf16(128, 128);
            for (int it = 0; it < nkt; ++it) {
                const int s = it % NST;
                mbar_wait(&full[s], (uint32_t)(it / NST) & 1u);
                tcgen05_fence_after();
                const uint32_t hi = smem_u32(smem + (size_t)s * kStage), lo = hi + kCovPartBytes;
#pragma unroll
                for (int k = 0; k < kTileK / kUmmaK; ++k) {
                    const uint32_t ko = k * kUmmaK * 2;
                    const bool acc = it > 0 || k > 0;
                    umma_bf16_ss(tmem_base, umma_desc_k_sw128(hi + ko), umma_desc_k_sw128(hi + ko), idesc0, acc);
                    if (PARTS == 2) {
                        umma_bf16_ss(tmem_base, umma_desc_k_sw128(hi + ko), umma_desc_k_sw128(lo + ko), idesc0, true);
                        umma_bf16_ss(tmem_base, umma_desc_k_sw128(lo + ko), umma_desc_k_sw128(hi + ko), idesc0, true);
                    }
                    if (m_tiles == 2) {
                        const uint32_t h1 = hi + kTileBytes + ko, l1 = lo + kTileBytes + ko;
                        umma_bf16_ss(tmem_base + 256, umma_desc_k_sw128(h1), umma_desc_k_sw128(h1), idesc1, acc);
                        if (PARTS == 2) {
                            umma_bf16_ss(tmem_base + 256, umma_desc_k_sw128(h1), umma_desc_k_sw128(l1), idesc1, true);
                            umma_bf16_ss(tmem_base + 256, umma_desc_k_sw128(l1), umma_desc_k_sw128(h1), idesc1, true);
                        }
                    }
                }
                umma_commit(&empty[s]);
            }
            umma_commit(&acc_full);
        }
    } else {
        // ------------------------------------------------------------------ converters: group grp takes k-tiles grp, grp+2, ...
        const int grp = (warp - 1) / kCovGroupWarps;
        const int cw = (warp - 1) % kCovGroupWarps;
        const int sub = lane >> 4;                 // which of the two rows of a load
        const int p4 = (lane & 15) * 4;            // first of this lane's 4 positions inside the k-tile
        float acc[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) acc[i] = 0.f;
        const bool rows_used = cw * 32 < p.cp;     // C <= 128: the upper converter warps only keep the handshake going
        for (int it = grp; it < nkt; it += kCovGroups) {
            const int64_t pos = ((int64_t)blockIdx.x + (int64_t)it * gridDim.x) * kTileK + p4;
            float4 v[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const int row = cw * 32 + 2 * i + sub;
                if (rows_used && row < p.c && pos < p.hw) {               // hw % 4 == 0: a float4 is inside or outside
                    v[i] = __ldcs(reinterpret_cast<const float4*>(p.x + (int64_t)row * p.hw + pos));
                } else {
                    const float sh = s_shift[row];
                    v[i] = make_float4(sh, sh, sh, sh);                   // padding: (x - shift) = 0
                }
            }
            const int s = it % NST;
            mbar_wait(&empty[s], ((uint32_t)(it / NST) & 1u) ^ 1u);
            unsigned char* hi = smem + (size_t)s * kStage;
            unsigned char* lo = hi + kCovPartBytes;
            if (rows_used) {
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int row = cw * 32 + 2 * i + sub;
                    const float sh = s_shift[row];
                    const float a = v[i].x - sh, b = v[i].y - sh, c2 = v[i].z - sh, d = v[i].w - sh;
                    acc[i] += (a + b) + (c2 + d);
                    // two elements per instruction: hi = bf16x2(a, b); the bf16 -> fp32 widening is a shift / mask
                    const uint32_t h01 = pack_bf16x2(a, b), h23 = pack_bf16x2(c2, d);
                    const uint32_t off = (uint32_t)row * 128u + (uint32_t)((((p4 >> 3) ^ (row & 7)) << 4) + ((lane & 1) << 3));
                    *reinterpret_cast<uint2*>(hi + off) = make_uint2(h01, h23);
                    if (PARTS == 2) {
                        const uint32_t l01 = pack_bf16x2(a - __uint_as_float(h01 << 16), b - __uint_as_float(h01 & 0xffff0000u));
                        const uint32_t l23 = pack_bf16x2(c2 - __uint_as_float(h23 << 16), d - __uint_as_float(h23 & 0xffff0000u));
                        *reinterpret_cast<uint2*>(lo + off) = make_uint2(l01, l23);
                    }
                }
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&full[s]);
        }
        // row sums of the shifted values: the 16 lanes sharing a row add up, fixed order
        if (rows_used) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                float a = acc[i];
#pragma unroll
                for (int o = 8; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
                const int row = cw * 32 + 2 * i + sub;
                if ((lane & 15) == 0 && row < p.cp) p.rowsum[((size_t)blockIdx.x * kCovGroups + grp) * p.cp + row] = a;
            }
        }
        // ------------------------------------------------------------------ epilogue (warps 1..4 = TMEM quarters 1,2,3,0)
        if (warp <= 4) {                                         // first four warps of group 0
            const int q = warp & 3;
            const int r = q * 32 + lane;
            float* out = p.partial + (size_t)blockIdx.x * p.cp * p.cp;
            if (nkt > 0) {
                mbar_wait(&acc_full, 0);
                tcgen05_fence_after();
            }
            float vals[32];
            for (int c0 = 0; c0 < p.cp; c0 += 32) {              // M-tile 0: rows 0..127, all columns
                if (nkt > 0) tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, vals);
                else
#pragma unroll
                    for (int j = 0; j < 32; ++j) vals[j] = 0.f;
                float4* dst = reinterpret_cast<float4*>(out + (size_t)r * p.cp + c0);
#pragma unroll
                for (int j = 0; j < 8; ++j) dst[j] = make_float4(vals[4 * j], vals[4 * j + 1], vals[4 * j + 2], vals[4 * j + 3]);
            }
            if (m_tiles == 2) {
                for (int c0 = 0; c0 < 128; c0 += 32) {           // M-tile 1: rows 128..255, columns 128..255
                    if (nkt > 0) tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + 256u + (uint32_t)c0, vals);
                    else
#pragma unroll
                        for (int j = 0; j < 32; ++j) vals[j] = 0.f;
                    float4* dst = reinterpret_cast<float4*>(out + (size_t)(128 + r) * p.cp + 128 + c0);
#pragma unroll
                    for (int j = 0; j < 8; ++j) dst[j] = make_float4(vals[4 * j], vals[4 * j + 1], vals[4 * j + 2], vals[4 * j + 3]);
                }
            }
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 0) {
        tcgen05_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// ---- TMA-staged variant ----------------------------------------------------------------------------------------------
// The register-staged kernel above is bound by the latency of its global loads (16 float4 in flight per converter
// thread: 2.9 TB/s, ncu long_scoreboard 24 %).  Here a producer thread brings [128 channels x 64 positions] fp32 boxes
// into a shared-memory ring with 2-D tensor-map TMA (cp.async.bulk.tensor.2d: 96-128 KiB in flight per SM, no
// registers involved); the converter warps read the boxes with conflict-free 128-bit shared loads and build the same
// bf16 hi/lo operand stages.  Out-of-range channels come back as zeros from the TMA unit (shift 0 there), out-of-range
// positions are masked by the converters.
//   warp 0       TMEM allocation; lane 0 = TMA producer
//   warp 1       lane 0 = MMA issuer (same SYRK block schedule as above)
//   warps 2..17  converters: warp w owns rows [8 w, 8 w + 8) of every box; warps 2..5 also run the epilogue
constexpr int kCovBoxRows = 128;
constexpr uint32_t kCovBoxBytes = kCovBoxRows * kTileK * sizeof(float);    // 32 KiB
constexpr int kCovTmaConvWarps = 16;
constexpr int kCovTmaThreads = 32 * (2 + kCovTmaConvWarps);

// The in-kernel finalize sums the per-CTA partial Grams with every warp of a CTA taking one slice of them and up to
// kCovFinalizeLoads partials per slice: it covers kCovMaxParts partials, so the cooperative grid is clamped to that.
constexpr int kCovFinalizeSlices = kCovTmaThreads / 32;
constexpr int kCovFinalizeLoads = 9;
constexpr int kCovMaxParts = kCovFinalizeSlices * kCovFinalizeLoads;   // 162 >= 148 SMs of a B200
static_assert(kCovFinalizeSlices == 18 && kCovMaxParts == 162, "finalize slice layout (red[2][18][8][32]) out of date");

template <int PARTS> struct CovTmaCfg {
    static constexpr int fstages = PARTS == 2 ? 3 : 4;          // fp32 boxes
    static constexpr int ostages = PARTS == 2 ? 2 : 3;          // operand stages (hi [+ lo], 256 rows)
    static constexpr uint32_t ostage = kCovPartBytes * PARTS;
    static constexpr size_t smem = 1024 + (size_t)fstages * kCovBoxBytes + (size_t)ostages * ostage;   // 225 KiB
};

// k-th grid-wide barrier of a cooperative launch (every CTA resident): the counter was zeroed before the launch
__device__ __forceinline__ void grid_barrier(int* counter, int k) {
    __threadfence();                                   // this thread's global writes before the arrival
    __syncthreads();
    if (threadIdx.x == 0) {
        atomicAdd(counter, 1);
        const int target = k * (int)gridDim.x;
        const uint64_t t0 = global_timer_ns();
        while (ld_acquire(counter) < target) {
            __nanosleep(32);
            if (watchdog_expired(t0)) __trap();
        }
    }
    __syncthreads();
}

template <int PARTS>
__global__ void __launch_bounds__(kCovTmaThreads, 1) cov_tma_kernel(const __grid_constant__ CUtensorMap tmap, CovParams p) {
    using Cfg = CovTmaCfg<PARTS>;
    constexpr int NF = Cfg::fstages, NO = Cfg::ostages;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* fring = smem;
    unsigned char* oring = smem + (size_t)NF * kCovBoxBytes;
    __shared__ uint64_t ffull[NF], fempty[NF], ofull[NO], oempty[NO], acc_full;
    __shared__ uint32_t tmem_slot;
    __shared__ float s_shift[kCovMaxC];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m_tiles = p.cp / 128;
    const int nkt = blockIdx.x < p.k_tiles ? (p.k_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NF; ++s) {
            mbar_init(&ffull[s], 1);
            mbar_init(&fempty[s], kCovTmaConvWarps);
        }
        for (int s = 0; s < NO; ++s) {
            mbar_init(&ofull[s], kCovTmaConvWarps);
            mbar_init(&oempty[s], 1);
        }
        mbar_init(&acc_full, 1);
        mbar_fence_init();
    }
    if (warp == 0) tmem_alloc(&tmem_slot, 512);
    // the producer thread (the one that initialised the barriers) starts the first boxes at once: they fly while the
    // converter warps compute the shift
    const bool prof = p.prof != nullptr && threadIdx.x == 64 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1);
    unsigned long long* pr = p.prof + (blockIdx.x == 0 ? 0 : 8);
    if (prof) pr[0] = global_timer_ns();
    const int total_boxes = nkt * m_tiles;
    const int pre_boxes = total_boxes < NF ? total_boxes : NF;
    auto issue_box = [&](int u) {
        const int it = u / m_tiles, h = u - it * m_tiles;
        const int pos0 = (int)(((int64_t)blockIdx.x + (int64_t)it * gridDim.x) * kTileK);
        const uint32_t sl = (uint32_t)u % NF;
        mbar_arrive_expect_tx(&ffull[sl], kCovBoxBytes);
        tma_load_box_2d(fring + (size_t)sl * kCovBoxBytes, &tmap, pos0, h * kCovBoxRows, &ffull[sl]);
    };
    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" :: "l"(&tmap) : "memory");
        for (int u = 0; u < pre_boxes; ++u) issue_box(u);
    }
    int bar_k = 0;                                         // grid barriers passed so far (uniform over the grid)
    if (p.shift_in) {
        // shifts of every tensor of the batch came from ONE small launch ahead of the covariance launches: no exchange here
        for (int r = threadIdx.x; r < kCovMaxC; r += blockDim.x) s_shift[r] = r < p.cp ? __ldg(p.shift_in + r) : 0.f;
    } else {
    if (warp >= 2) {
        // Centring shift = mean of up to 32 segments of 64 positions spread over the plane.  The channels are dealt over
        // the CTAs (one warp per channel, every load independent) and exchanged through global memory: when every CTA
        // sampled every channel itself, 148 CTAs asked the same L2 lines at the same moment (10.8 us).  Any shift is exact
        // after the rank-1 correction; it only has to be within a few sigma of the mean.
        const int segs = (int)(p.hw / 64 > 32 ? 32 : p.hw / 64);      // hw >= 64
        const int64_t stride = (p.hw / segs) & ~(int64_t)3;            // >= 64, keeps the 8-byte loads aligned
        for (int ch = (int)blockIdx.x + (warp - 2) * (int)gridDim.x; ch < p.cp; ch += kCovTmaConvWarps * (int)gridDim.x) {
            float a = 0.f;
            if (ch < p.c) {
                const float* xr = p.x + (int64_t)ch * p.hw + 2 * lane;
#pragma unroll 8
                for (int sg = 0; sg < segs; ++sg) {
                    const float2 v = __ldg(reinterpret_cast<const float2*>(xr + sg * stride));
                    a += v.x + v.y;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
                a /= (float)(segs * 64);
            }
            if (lane == 0) p.shift[ch] = a;
        }
    }
    grid_barrier(p.barrier, ++bar_k);
    for (int r = threadIdx.x; r < kCovMaxC; r += blockDim.x) s_shift[r] = r < p.cp ? __ldcg(p.shift + r) : 0.f;
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = tmem_slot;
    if (prof) pr[1] = global_timer_ns();

    if (warp == 0) {
        if (lane == 0) {
            for (int u = pre_boxes; u < total_boxes; ++u) {
                mbar_wait(&fempty[(uint32_t)u % NF], (((uint32_t)u / NF) & 1u) ^ 1u);
                issue_box(u);
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && nkt > 0) {
            const uint32_t idesc0 = umma_idesc_bf16(128, p.cp);
            const uint32_t idesc1 = umma_idesc_bf16(128, 128);
            for (int it = 0; it < nkt; ++it) {
                const int s = it % NO;
                mbar_wait(&ofull[s], (uint32_t)(it / NO) & 1u);
                tcgen05_fence_after();
                const uint32_t hi = smem_u32(oring + (size_t)s * Cfg::ostage), lo = hi + kCovPartBytes;
#pragma unroll
                for (int k = 0; k < kTileK / kUmmaK; ++k) {
                    const uint32_t ko = k * kUmmaK * 2;
                    const bool acc = it > 0 || k > 0;
                    umma_bf16_ss(tmem_base, umma_desc_k_sw128(hi + ko), umma_desc_k_sw128(hi + ko), idesc0, acc);
                    if (PARTS == 2) {
                        umma_bf16_ss(tmem_base, umma_desc_k_sw128(hi + ko), umma_desc_k_sw128(lo + ko), idesc0, true);
                        umma_bf16_ss(tmem_base, umma_desc_k_sw128(lo + ko), umma_desc_k_sw128(hi + ko), idesc0, true);
                    }
                    if (m_tiles == 2) {
                        const uint32_t h1 = hi + kTileBytes + ko, l1 = lo + kTileBytes + ko;
                        umma_bf16_ss(tmem_base + 256, umma_desc_k_sw128(h1), umma_desc_k_sw128(h1), idesc1, acc);
                        if (PARTS == 2) {
                            umma_bf16_ss(tmem_base + 256, umma_desc_k_sw128(h1), umma_desc_k_sw128(l1), idesc1, true);
                            umma_bf16_ss(tmem_base + 256, umma_desc_k_sw128(l1), umma_desc_k_sw128(h1), idesc1, true);
                        }
                    }
                }
                umma_commit(&oempty[s]);
            }
            umma_commit(&acc_full);
        }
    } else {
        const int cw = warp - 2;
        const int sub = lane >> 4;                 // which of the two rows of a shared-memory load
        const int p4 = (lane & 15) * 4;            // first of this lane's 4 positions inside the k-tile
        float acc[2][4];
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[h][i] = 0.f;
        uint32_t use = 0;
        for (int it = 0; it < nkt; ++it) {
            const int64_t pos = ((int64_t)blockIdx.x + (int64_t)it * gridDim.x) * kTileK + p4;
            const bool valid = pos < p.hw;                                   // hw % 4 == 0: a float4 is inside or outside
            const int os = it % NO;
            unsigned char* hi = oring + (size_t)os * Cfg::ostage;
            unsigned char* lo = hi + kCovPartBytes;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                if (h < m_tiles) {
                    const uint32_t fs = use % NF;
                    mbar_wait(&ffull[fs], (use / NF) & 1u);
                    ++use;
                    const unsigned char* box = fring + (size_t)fs * kCovBoxBytes;
                    float4 v[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        v[i] = *reinterpret_cast<const float4*>(box + (size_t)(cw * 8 + 2 * i + sub) * (kTileK * 4) + p4 * 4);
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&fempty[fs]);                 // the box may be overwritten
                    if (h == 0) mbar_wait(&oempty[os], ((uint32_t)(it / NO) & 1u) ^ 1u);
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int row = h * kCovBoxRows + cw * 8 + 2 * i + sub;
                        const float sh = s_shift[row];
                        const float a = valid ? v[i].x - sh : 0.f, b = valid ? v[i].y - sh : 0.f;
                        const float c2 = valid ? v[i].z - sh : 0.f, d = valid ? v[i].w - sh : 0.f;
                        acc[h][i] += (a + b) + (c2 + d);
                        const uint32_t h01 = pack_bf16x2(a, b), h23 = pack_bf16x2(c2, d);
                        const uint32_t off = (uint32_t)row * 128u + (uint32_t)((((p4 >> 3) ^ (row & 7)) << 4) + ((lane & 1) << 3));
                        *reinterpret_cast<uint2*>(hi + off) = make_uint2(h01, h23);
                        if (PARTS == 2) {
                            const uint32_t l01 = pack_bf16x2(a - __uint_as_float(h01 << 16), b - __uint_as_float(h01 & 0xffff0000u));
                            const uint32_t l23 = pack_bf16x2(c2 - __uint_as_float(h23 << 16), d - __uint_as_float(h23 & 0xffff0000u));
                            *reinterpret_cast<uint2*>(lo + off) = make_uint2(l01, l23);
                        }
                    }
                }
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&ofull[os]);
        }
        if (prof) pr[2] = global_timer_ns();
        // row sums of the shifted values: the 16 lanes sharing a row add up, fixed order
#pragma unroll
        for (int h = 0; h < 2; ++h) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float a = acc[h][i];
#pragma unroll
                for (int o = 8; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
                const int row = h * kCovBoxRows + cw * 8 + 2 * i + sub;
                if ((lane & 15) == 0 && row < p.cp) p.rowsum[(size_t)blockIdx.x * p.cp + row] = a;
            }
        }
        {
            // epilogue on all 16 converter warps: warp w reads TMEM lane quarter w & 3 (the only one it may access) and
            // every fourth 32-column chunk of it; each lane stores whole 32-byte sectors (256-bit stores)
            const int q = warp & 3, sub = (warp - 2) >> 2;
            const int r = q * 32 + lane;
            float* out = p.partial + (size_t)blockIdx.x * p.cp * p.cp;
            if (nkt > 0) {
                mbar_wait(&acc_full, 0);
                tcgen05_fence_after();
            }
            const int chunks0 = p.cp / 32, chunks = chunks0 + (m_tiles == 2 ? 4 : 0);
            float vals[32];
            for (int ck = sub; ck < chunks; ck += 4) {
                // M-tile 0: rows 0..127, all columns; M-tile 1: rows 128..255, columns 128..255 (TMEM columns 256..383)
                const bool second = ck >= chunks0;
                const int c0 = second ? (ck - chunks0) * 32 : ck * 32;
                if (nkt > 0) tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (second ? 256u : 0u) + (uint32_t)c0, vals);
                else
#pragma unroll
                    for (int j = 0; j < 32; ++j) vals[j] = 0.f;
                float* dst = second ? out + (size_t)(128 + r) * p.cp + 128 + c0 : out + (size_t)r * p.cp + c0;
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                                 :: "l"(dst + 8 * j), "f"(vals[8 * j]), "f"(vals[8 * j + 1]), "f"(vals[8 * j + 2]), "f"(vals[8 * j + 3]),
                                    "f"(vals[8 * j + 4]), "f"(vals[8 * j + 5]), "f"(vals[8 * j + 6]), "f"(vals[8 * j + 7]) : "memory");
            }
        }
    }
    tcgen05_fence_before();
    __threadfence();                                   // partial Gram and row sums visible before the grid barrier
    __syncthreads();
    if (warp == 0) {
        tcgen05_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
    if (prof) pr[3] = global_timer_ns();
    // ---- grid barriers (cooperative launch: every CTA is resident) and the fp64 finalize spread over the CTAs ----
    grid_barrier(p.barrier, ++bar_k);
    if (prof) pr[4] = global_timer_ns();
    const int parts = (int)gridDim.x;
    double* s_S = reinterpret_cast<double*>(smem);                         // [256] column sums of the shifted values
    double* red = s_S + kCovMaxC;                                          // [2 rows][18 slices][8 columns][32 groups]: 72 KiB
    // S[r] = sum over CTAs of the partial row sums: rows dealt over the CTAs, one warp per row, lanes over the CTAs,
    // lane-ordered tree (fixed order); exchanged through global memory (every CTA summing every row itself: 11 us of
    // same-line L2 contention)
    for (int r = (int)blockIdx.x + warp * (int)gridDim.x; r < p.cp; r += (kCovTmaThreads / 32) * (int)gridDim.x) {
        double a = 0.0;
        for (int z = lane; z < parts; z += 32) a += (double)__ldcg(p.rowsum + (size_t)z * p.cp + r);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
        if (lane == 0) {
            p.s_sum[r] = a;
            if (p.mean && r < p.c) p.mean[r] = (float)((double)s_shift[r] + a / (double)p.hw);
        }
    }
    grid_barrier(p.barrier, ++bar_k);
    for (int r = threadIdx.x; r < kCovMaxC; r += blockDim.x) s_S[r] = r < p.cp ? __ldcg(p.s_sum + r) : 0.0;
    __syncthreads();
    if (prof) pr[5] = global_timer_ns();
    const double hw = (double)p.hw;
    // Covariance rows (computed SYRK blocks only) are dealt over the CTAs, two rows in flight at a time (a CTA owns one or
    // two rows at C = 256 and the phase is latency-bound): thread (jg, zs) sums 8 columns of every 18th partial.
    for (int ibase = blockIdx.x; ibase < p.cp; ibase += 2 * gridDim.x) {
        const int jg = threadIdx.x & 31, zs = threadIdx.x >> 5;          // 32 groups of eight columns x 18 slices of the partials
        double a[2][8];
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
            const int i = ibase + rr * (int)gridDim.x;
            const int j0 = (i >= 128 ? 128 : 0) + 8 * jg;                // rows >= 128 start at column 128
            const bool live = i < p.cp && j0 < p.cp && (i < 128 || jg < 16);
#pragma unroll
            for (int e = 0; e < 8; ++e) a[rr][e] = 0.0;
            if (live) {
                const float* src = p.partial + (size_t)i * p.cp + j0;
                const size_t zstride = (size_t)p.cp * p.cp;
#pragma unroll 1
                for (int k0 = 0; k0 < kCovFinalizeLoads; k0 += 5) {      // 5 + 4 sector loads in flight (up to 162 partials)
                    float t[5][8];
#pragma unroll
                    for (int k = 0; k < 5; ++k) {
                        const int z = zs + kCovFinalizeSlices * (k0 + k);
                        if (k0 + k < kCovFinalizeLoads && z < parts) {
                            asm volatile("ld.global.cg.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                                         : "=f"(t[k][0]), "=f"(t[k][1]), "=f"(t[k][2]), "=f"(t[k][3]), "=f"(t[k][4]), "=f"(t[k][5]),
                                           "=f"(t[k][6]), "=f"(t[k][7]) : "l"(src + (size_t)z * zstride) : "memory");
                        } else {
#pragma unroll
                            for (int e = 0; e < 8; ++e) t[k][e] = 0.f;
                        }
                    }
#pragma unroll
                    for (int k = 0; k < 5; ++k)
#pragma unroll
                        for (int e = 0; e < 8; ++e) a[rr][e] += (double)t[k][e];
                }
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) red[(((size_t)rr * kCovFinalizeSlices + zs) * 8 + e) * 32 + jg] = a[rr][e];   // [row][slice][column][group]
        }
        __syncthreads();
        if (zs < 16) {                                                   // thread (jg, rr = zs / 8, e = zs % 8) finishes one column
            const int rr = zs >> 3, e = zs & 7;
            const int i = ibase + rr * (int)gridDim.x;
            const int j = (i >= 128 ? 128 : 0) + 8 * jg + e;
            if (i < p.c && j < p.c && (i < 128 || jg < 16)) {
                double g = 0.0;
#pragma unroll
                for (int q = 0; q < kCovFinalizeSlices; ++q) g += red[(((size_t)rr * kCovFinalizeSlices + q) * 8 + e) * 32 + jg];   // fixed order
                const double v = (g - s_S[i] * s_S[j] / hw) / (hw - 1.0);
                p.cov[(size_t)i * p.c + j] = v + (i == j ? p.diag_add : 0.0);
                if (i < 128 && j >= 128) p.cov[(size_t)j * p.c + i] = v;        // block (1,0) is the mirror of block (0,1)
            }
        }
        __syncthreads();
    }
    if (prof) pr[6] = global_timer_ns();
}

// sub-sampled per-channel mean (up to 32 segments of 64 positions spread over the plane): the centring shift.
// One warp per channel, every load independent.
__global__ void __launch_bounds__(256) cov_shift_kernel(const float* __restrict__ x, int c, int cp, int64_t hw,
                                                        float* __restrict__ shift) {
    x += (int64_t)blockIdx.y * c * hw;                 // blockIdx.y: tensor of a batch (contiguous [n, c, hw]), shifts [n, cp]
    shift += (int64_t)blockIdx.y * cp;
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= cp) return;
    if (row >= c) {
        if (lane == 0) shift[row] = 0.f;
        return;
    }
    const int segs = (int)(hw / 64 > 32 ? 32 : hw / 64);      // hw >= 64
    const int64_t stride = (hw / segs) & ~(int64_t)3;          // >= 64, keeps the 8-byte loads aligned
    const float* xr = x + (int64_t)row * hw + 2 * lane;
    float a = 0.f;
#pragma unroll 8
    for (int sgi = 0; sgi < segs; ++sgi) {
        const float2 v = __ldg(reinterpret_cast<const float2*>(xr + sgi * stride));   // hw % 4 == 0 keeps this 8-byte aligned
        a += v.x + v.y;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) shift[row] = a / (float)(segs * 64);
}

// S[r] = sum over CTAs and converter groups of the partial row sums (fp64, fixed order); exact means.
// Thread (e, r): entry slice e of 8, row r; the 8 slice sums are folded in index order through shared memory.
__global__ void __launch_bounds__(256) cov_rowsum_kernel(const float* __restrict__ rowsum, const float* __restrict__ shift,
                                                         int entries, int c, int cp, double hw, double* __restrict__ s_sum,
                                                         float* __restrict__ mean) {
    __shared__ double red[8][32];
    const int rl = threadIdx.x & 31, e = threadIdx.x >> 5;
    const int r = blockIdx.x * 32 + rl;
    const int per = (entries + 7) / 8;
    const int z0 = e * per, z1 = min(entries, z0 + per);
    double a = 0.0;
    if (r < cp) {
        for (int z = z0; z < z1; z += 8) {             // 8 independent loads in flight, added in index order
            float t[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) t[k] = z + k < z1 ? __ldg(rowsum + (size_t)(z + k) * cp + r) : 0.f;
#pragma unroll
            for (int k = 0; k < 8; ++k) a += (double)t[k];
        }
    }
    red[e][rl] = a;
    __syncthreads();
    if (e == 0 && r < cp) {
        double t = red[0][rl];
#pragma unroll
        for (int k = 1; k < 8; ++k) t += red[k][rl];
        s_sum[r] = t;
        if (mean && r < c) mean[r] = (float)((double)shift[r] + t / hw);
    }
}

// Fixed-order fp64 reduction of the per-CTA partial Grams + rank-1 centring correction.  A block owns 64 groups of
// four consecutive columns of one row; its 4 thread rows split the partials and are folded in index order.
__global__ void __launch_bounds__(256) cov_finalize_kernel(const float* __restrict__ partial, const double* __restrict__ s_sum,
                                                           int parts, int c, int cp, double hw, double diag_add,
                                                           double* __restrict__ cov) {
    __shared__ double red[4][64][4];
    const int i = blockIdx.x;                                   // covariance row (computed blocks only: see below)
    const int jg = threadIdx.x & 63, zs = threadIdx.x >> 6;
    const int j0 = (i >= 128 ? 128 : 0) + 4 * jg + 256 * blockIdx.y;   // rows >= 128 start at column 128 (SYRK blocks)
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    const bool live = j0 < cp;
    if (live) {
        const float* src = partial + (size_t)i * cp + j0;
        const int per = (parts + 3) / 4;
        const int z0 = zs * per, z1 = min(parts, z0 + per);
#pragma unroll 4
        for (int z = z0; z < z1; ++z) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(src + (size_t)z * cp * cp));
            a0 += (double)v.x; a1 += (double)v.y; a2 += (double)v.z; a3 += (double)v.w;
        }
    }
    red[zs][jg][0] = a0; red[zs][jg][1] = a1; red[zs][jg][2] = a2; red[zs][jg][3] = a3;
    __syncthreads();
    if (zs == 0 && live) {
        const double si = s_sum[i];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int j = j0 + e;
            if (i < c && j < c) {
                const double g = ((red[0][jg][e] + red[1][jg][e]) + red[2][jg][e]) + red[3][jg][e];
                const double v = (g - si * s_sum[j] / hw) / (hw - 1.0);
                cov[(size_t)i * c + j] = v + (i == j ? diag_add : 0.0);
                if (i < 128 && j >= 128) cov[(size_t)j * c + i] = v;    // block (1,0) is the mirror of block (0,1)
            }
        }
    }
}

}  // namespace

bool cov_fused_supported(const float* x, int64_t c, int64_t hw) {
    return c >= 1 && c <= kCovMaxC && hw >= 64 && hw % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 15u) == 0;
}

size_t cov_fused_workspace_bytes(int64_t c) {
    const size_t cp = c <= 128 ? 128 : 256;
    const size_t g = (size_t)sm_count();
    return align_up(g * cp * cp * sizeof(float), 256) + align_up(g * kCovGroups * cp * sizeof(float), 256) +
           align_up(cp * sizeof(float), 256) + align_up(cp * sizeof(double), 256) + 256;   // + the grid-barrier counter
}

namespace {
// cuTensorMapEncodeTiled through the runtime's driver entry-point query: librpst.so does not link libcuda
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = [] {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            f = nullptr;
        return reinterpret_cast<EncodeTiledFn>(f);
    }();
    return fn;
}
}  // namespace

// 2-D fp32 tensor map [outer rows, inner elements] (row pitch = inner * 4 bytes) with boxes of box_outer x box_inner;
// false when the driver entry point is not available.  `map` points at a CUtensorMap.
bool tmap_encode_2d_f32(void* map, const float* base, uint64_t inner, uint64_t outer, uint32_t box_inner, uint32_t box_outer) {
    EncodeTiledFn encode = encode_tiled_fn();
    if (!encode) return false;
    const cuuint64_t gdim[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
    const cuuint64_t gstride[1] = {(cuuint64_t)inner * sizeof(float)};
    const cuuint32_t box[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_outer};
    const cuuint32_t estr[2] = {1, 1};
    return encode(static_cast<CUtensorMap*>(map), CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstride, box,
                  estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// cov [c,c] fp64 = centred covariance of x [c,hw] (+ diag_add on the diagonal); mean [c] fp32 exact channel means
// shifts [n, cp] (cp = 128 or 256) of n contiguous [c, hw] tensors in one launch: what cov_fused takes as `shift_in`
int cov_shifts_batched(const float* x, int64_t n, int64_t c, int64_t hw, float* shifts, cudaStream_t st) {
    const int cp = c <= 128 ? 128 : 256;
    cov_shift_kernel<<<dim3((unsigned)((cp + 7) / 8), (unsigned)n), 256, 0, st>>>(x, (int)c, cp, hw, shifts);
    RPST_CUDA(cudaGetLastError());
    return RPST_OK;
}

// path: 0 picks the kernel (the one-launch TMA kernel when the device grants a cooperative launch and the plane has at
// least 64 k-tiles, the register-staged kernel + finalize launches otherwise); kCovPathTma / kCovPathStaged force one
// (tests).  *taken (may be null) receives the kernel that ran.
int cov_fused(const float* x, int64_t c, int64_t hw, int passes, double diag_add, double* cov, float* mean, void* workspace,
              cudaStream_t st, const float* shift_in, int path, int* taken) {
    const int cp = c <= 128 ? 128 : 256;
    const int g = sm_count();
    char* w = static_cast<char*>(workspace);
    float* partial = reinterpret_cast<float*>(w);
    float* rowsum = reinterpret_cast<float*>(w + align_up((size_t)g * cp * cp * sizeof(float), 256));
    float* shift = reinterpret_cast<float*>(reinterpret_cast<char*>(rowsum) + align_up((size_t)g * kCovGroups * cp * sizeof(float), 256));
    double* s_sum = reinterpret_cast<double*>(reinterpret_cast<char*>(shift) + align_up((size_t)cp * sizeof(float), 256));
    CovParams p{};
    p.x = x; p.shift = shift; p.partial = partial; p.rowsum = rowsum; p.hw = hw; p.c = (int)c; p.cp = cp;
    p.k_tiles = (int)((hw + kTileK - 1) / kTileK);
    p.passes = passes;
    const int grid = g < p.k_tiles ? g : p.k_tiles;
    static PerDeviceFlag configured_on;
    bool& configured = configured_on.get();
    constexpr size_t smem = 1024 + 3 * 2 * kCovPartBytes;   // 193 KiB for both instantiations
    if (!configured) {
        RPST_CUDA(cudaFuncSetAttribute(cov_fused_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        RPST_CUDA(cudaFuncSetAttribute(cov_fused_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        RPST_CUDA(cudaFuncSetAttribute(cov_tma_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CovTmaCfg<1>::smem));
        RPST_CUDA(cudaFuncSetAttribute(cov_tma_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CovTmaCfg<2>::smem));
        configured = true;
    }
    // the one-launch kernel needs a cooperative launch with every CTA resident (grid barriers): one CTA per SM; a device
    // (or MIG slice / MPS share) that cannot grant that takes the register-staged kernel + separate finalize launches
    static int coop_ok[64] = {};     // 0 unknown, 1 yes, -1 no
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
    if (coop_ok[dev] == 0) {
        int coop = 0, per_sm = 0;
        cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, cov_tma_kernel<2>, kCovTmaThreads, CovTmaCfg<2>::smem) != cudaSuccess)
            per_sm = 0;
        coop_ok[dev] = (coop && per_sm >= 1) ? 1 : -1;
    }
    // small planes (fewer k-tiles than ~half the SMs): the in-kernel finalize would run on a handful of CTAs (a 64-position
    // plane: ONE CTA walking 128 rows, 0.3 ms); they keep the separate, fully parallel finalize launches
    const bool tma_ok = coop_ok[dev] == 1 && hw < (1ll << 31) - 64;
    EncodeTiledFn encode = nullptr;
    if (path == kCovPathTma) {
        encode = tma_ok ? encode_tiled_fn() : nullptr;
        if (!encode) {
            set_error("wct covariance: the one-launch TMA kernel is not available on this device");
            return RPST_ERR_UNSUPPORTED;
        }
    } else if (path == 0 && g_knobs.wct_cov_tma && tma_ok && grid >= 64) {
        encode = encode_tiled_fn();
    }
    if (encode) {
        // x as a 2-D tensor [c rows, hw positions]; boxes of 128 rows x 64 positions (256-byte row pieces)
        CUtensorMap tmap;
        const cuuint64_t gdim[2] = {(cuuint64_t)hw, (cuuint64_t)c};
        const cuuint64_t gstride[1] = {(cuuint64_t)hw * sizeof(float)};
        const cuuint32_t box[2] = {(cuuint32_t)kTileK, (cuuint32_t)kCovBoxRows};
        const cuuint32_t estr[2] = {1, 1};
        const CUresult r = encode(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(x), gdim, gstride, box, estr,
                                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            set_error("wct covariance: cuTensorMapEncodeTiled failed (%d)", (int)r);
            return RPST_ERR_CUDA;
        }
        // one cooperative launch: shift, SYRK, grid barrier, fp64 finalize (every CTA must be resident for the barrier)
        int* barrier = reinterpret_cast<int*>(reinterpret_cast<char*>(s_sum) + align_up((size_t)cp * sizeof(double), 256));
        RPST_CUDA(cudaMemsetAsync(barrier, 0, sizeof(int), st));
        p.barrier = barrier; p.cov = cov; p.mean = mean; p.diag_add = diag_add; p.s_sum = s_sum; p.shift = shift;
        p.shift_in = shift_in;
        p.prof = reinterpret_cast<unsigned long long*>(g_knobs.wct_cov_prof);
        cudaLaunchConfig_t cfg{};
        // every partial Gram must be inside the finalize's reach: at most kCovMaxParts CTAs (k-tiles are dealt round-robin
        // over whatever grid runs)
        cfg.gridDim = dim3((unsigned)(grid < kCovMaxParts ? grid : kCovMaxParts));
        cfg.blockDim = dim3(kCovTmaThreads);
        cfg.dynamicSmemBytes = passes == 3 ? CovTmaCfg<2>::smem : CovTmaCfg<1>::smem;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeCooperative;
        attr[0].val.cooperative = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        if (passes == 3) RPST_CUDA(cudaLaunchKernelEx(&cfg, cov_tma_kernel<2>, tmap, p));
        else RPST_CUDA(cudaLaunchKernelEx(&cfg, cov_tma_kernel<1>, tmap, p));
        if (taken) *taken = kCovPathTma;
        return RPST_OK;
    }
    cov_shift_kernel<<<(cp + 7) / 8, 256, 0, st>>>(x, (int)c, cp, hw, shift);
    RPST_CUDA(cudaGetLastError());
    p.shift = shift;
    const int entries = grid * kCovGroups;
    if (passes == 3) cov_fused_kernel<2><<<grid, kCovThreads, smem, st>>>(p);
    else cov_fused_kernel<1><<<grid, kCovThreads, smem, st>>>(p);
    RPST_CUDA(cudaGetLastError());
    cov_rowsum_kernel<<<(cp + 31) / 32, 256, 0, st>>>(rowsum, shift, entries, (int)c, cp, (double)hw, s_sum, mean);
    RPST_CUDA(cudaGetLastError());
    cov_finalize_kernel<<<dim3((unsigned)cp, 1), 256, 0, st>>>(partial, s_sum, grid, (int)c, cp, (double)hw, diag_add, cov);
    RPST_CUDA(cudaGetLastError());
    if (taken) *taken = kCovPathStaged;
    return RPST_OK;
}

}  // namespace rpst

RPST_WATCHDOG_SETTER(cov)

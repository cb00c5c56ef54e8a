// Pointwise (1x1) convolution on the 5th-gen tensor cores with fused prologue / epilogue — the contraction over
// CHANNELS that surrounds the statistics transforms:
//   * WCT colouring apply  out = T (x - mu_c) + mu_s                         network/wct_rp.py:110,113   (a6)
//   * SANet projections    F = f(mean_variance_norm(c)), G = g(mvn(s)), H = h(s), out_conv(O) + content
//                          with the instance normalisation folded into the operand conversion and Q / K emitted
//                          directly as packed bf16 operand tiles of the attention kernel     network/sanet.py:82-99 (f2)
//   * RP-encoder 1x1 conv + LeakyReLU with the AdaIN statistics (sum, sum of squares per (n,c)) emitted from the
//     epilogue, so the transform that follows needs no statistics pass            network/base.py:170-198 (f4)
//
//   D[n, o] = sum_c W[o, c] * ((x[c, n] - sub[c]) * mul[c])      M = 128 positions per tile, N <= 256 output channels
//
// The accumulator lanes are POSITIONS, so fp32 stores are contiguous in `out` and packed tiles get one 128-byte row
// per thread.  The A operand is x in its native orientation — positions contiguous = an MN-MAJOR tcgen05 operand
// (SWIZZLE_128B atoms of 64 positions x 8 channels): converter warps read fp32 x with 128-bit position-coalesced loads
// (one 512-byte channel row of the tile per warp instruction, three register buffers deep), apply (x - sub) * mul,
// split into bf16 hi + lo and store 8 bytes — no transposition and no packed-operand round trip through HBM.  W is
// small (<= 1 MiB packed) and streams from L2 by TMA, one k-block of 64 input channels per stage.
//
//   warp 0        TMA producer of the W k-blocks            warps 2..5   epilogue (TMEM -> bias / act / residual /
//   warp 1        tcgen05.mma issuer + TMEM owner                        statistics -> fp32 or packed tiles)
//                                                            warps 6..13  converters
// Two 256-column TMEM accumulators: the epilogue of item i overlaps the MMAs of item i+1.
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"
#include "tuning.cuh"
#include "umma.cuh"

namespace rpst {

size_t packed_operand_bytes(int64_t rows, int64_t k);
bool tmap_encode_2d_f32(void* map, const float* base, uint64_t inner, uint64_t outer, uint32_t box_inner, uint32_t box_outer);   // cov.cu

namespace {

constexpr int kPwConvWarps = 8;
constexpr int kPwThreads = 32 * (6 + kPwConvWarps);
constexpr int kPwMaxC = 512;

struct PwParams {
    const float* x;          // [b, cin, hw]
    const float* sub;        // [b, cin] or null
    const float* mul;        // [b, cin] or null
    const char* w_hi;        // packed W tiles: rows = output channels (coutp / 128 row blocks), K = input channels (kb tiles)
    const char* w_lo;
    int64_t w_batch;         // bytes between per-sample weights (0: shared by the batch)
    const float* bias;       // [cout] (+ bias_batch per sample) or null
    int64_t bias_batch;
    const float* residual;   // [b, cout, hw] or null
    float* out;              // fp32 [b, cout, hw] or null
    char* out_hi;            // packed tiles, rows = positions, K = output channels (the attention kernel's Q / K format) or null
    char* out_lo;
    int64_t tile_batch;      // bytes between samples of the packed output
    float* stats;            // [b, grid * 4, cout, 2] per-CTA-and-warp partial (sum, sum of squares) of the stored values (zeroed by the host) or null
    float slope;             // LeakyReLU slope when act == 1
    int act;
    int64_t hw;
    int cin, cout, coutp;    // coutp: cout padded to a multiple of 128
    int kb;                  // k-blocks of 64 input channels
    int col_tiles;           // column tiles of <= 256 output channels
    int tiles;               // position tiles of 128
    int batch;
    int vec_ok;              // x 16-byte aligned and hw % 4 == 0: 128-bit loads
    int parts;
    int stat_ctas;           // CTA slots per sample in `stats` (= SM count >= grid)
};

// A tile of one k-block: [8 K-atoms (8 channels each)][2 MN-atoms (64 positions each)][8 channel rows][128 B]
constexpr uint32_t kPwLBO = 1024;    // between the two 64-position atoms
constexpr uint32_t kPwSBO = 2048;    // between groups of 8 channels

// shared-memory descriptor: MN-major, SWIZZLE_128B (leading byte offset = MN-atom stride, stride byte offset = K-atom stride)
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3fffu);
    d |= (uint64_t)(kPwLBO >> 4) << 16;
    d |= (uint64_t)(kPwSBO >> 4) << 32;
    d |= (uint64_t)1u << 46;
    d |= (uint64_t)2u << 61;
    return d;
}
constexpr uint32_t kIdescAMajorMN = 1u << 15;

__device__ __forceinline__ uint32_t pw_pack_bf16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

struct PwItem {
    int sample, t, ct, ncol;
};
__device__ __forceinline__ PwItem pw_item(const PwParams& p, int item) {
    PwItem it;
    it.ct = item % p.col_tiles;
    const int rest = item / p.col_tiles;
    it.t = rest % p.tiles;
    it.sample = rest / p.tiles;
    it.ncol = min(256, p.coutp - 256 * it.ct);
    return it;
}

// VEC: hw % 4 == 0, x 16-byte aligned, cin % 8 == 0 (128-bit loads, no ragged-edge code in the hot loop);
// EPI: 0 fp32 output only, 1 packed operand tiles (+ optional fp32), 2 fp32 output + epilogue statistics.
// Separate instantiations keep each kernel's code small: the warp roles run different code at the same time and
// a 64 KiB kernel thrashed the instruction cache (12 % of the stalls were "no instruction").
//
// XTMA (VEC, cin % 64 == 0, EPI 0 / 1): the fp32 x tile of a k-block ([64 channels x 128 positions], 32 KiB) comes in by
// 2-D tensor-map TMA into a two-deep ring and the converter warps read it from shared memory.  The register-staged
// converters (three buffers of 8 float4 per thread) were bound by global-load latency: ncu long_scoreboard 45 %,
// 3.1 TB/s over read + write.  Shared memory then holds ONE A stage (converting a k-block takes a quarter of its MMA
// time, and convert + MMA in series still fit under the k-block's HBM time), the B ring and the x ring: 224 KiB.
constexpr int XTMA_NX = 2;   // x boxes in flight: 2 with one A stage (134 us for the WCT colouring); 1 with two A stages measured 150 us
template <int PARTS, bool VEC, int EPI, bool XTMA>
__global__ void __launch_bounds__(kPwThreads, 1) pw_conv_kernel(const __grid_constant__ CUtensorMap xmap, PwParams p) {
    // stage: A hi [128 pos x 64 ch] 16 KiB (+ lo 16 KiB), B hi [256 out x 64 ch] 32 KiB (+ lo 32 KiB)
    constexpr uint32_t kA = kTileBytes, kB = 2 * kTileBytes;
    constexpr uint32_t kStage = PARTS * (kA + kB);
    constexpr int NST = PARTS == 2 ? 2 : 4;
    constexpr int NX = XTMA_NX;
    constexpr int NA = XTMA ? 3 - NX : 1;                       // A stages on the XTMA layout: 224 KiB either way
    constexpr uint32_t kXBox = 64 * 128 * sizeof(float);        // 32 KiB
    static_assert(!XTMA || (VEC && EPI != 2), "XTMA: vector path, no epilogue statistics (their static arrays need the room)");
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    // XTMA layout: [A stage 0 .. NA-1 (PARTS * kA each)][B stage 0 .. NST-1 (PARTS * kB each)][x box 0 .. NX-1]
    unsigned char* const xring = smem + (size_t)NA * PARTS * kA + (size_t)NST * PARTS * kB;
    auto a_stage = [&](int s) -> unsigned char* { return XTMA ? smem + (size_t)s * PARTS * kA : smem + (size_t)s * kStage; };
    auto b_stage = [&](int s) -> unsigned char* {
        return XTMA ? smem + (size_t)NA * PARTS * kA + (size_t)s * PARTS * kB : smem + (size_t)s * kStage + PARTS * kA;
    };
    __shared__ uint64_t full_a[NST], full_b[NST], empty[NST], acc_full[2], acc_empty[2];
    __shared__ uint64_t xfull[2], xempty[2], a_empty[2];
    __shared__ uint32_t tmem_slot;
    __shared__ float stat_tile[EPI == 2 ? 4 * 32 * 33 : 1];
    __shared__ float stat_acc[EPI == 2 ? 4 * kPwMaxC * 2 : 1];   // running per-warp column sums of the current sample
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int items = p.batch * p.tiles * p.col_tiles;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NST; ++s) {
            mbar_init(&full_a[s], kPwConvWarps);
            mbar_init(&full_b[s], 1);
            mbar_init(&empty[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&acc_full[b], 1);
            mbar_init(&acc_empty[b], 4);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&xfull[b], 1);
            mbar_init(&xempty[b], kPwConvWarps);
            mbar_init(&a_empty[b], 1);
        }
        mbar_fence_init();
    }
    if (warp == 1) tmem_alloc(&tmem_slot, 512);
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            const uint64_t pol = policy_evict_last();
            uint32_t it = 0;
            for (int item = blockIdx.x; item < items; item += gridDim.x) {
                const PwItem w = pw_item(p, item);
                const int n_sub = w.ncol / 128;
                for (int kb = 0; kb < p.kb; ++kb, ++it) {
                    if (XTMA) {                              // x box of this k-block: positions 128 t .., channel rows sample * cin + 64 kb ..
                        const uint32_t xs = it % NX;
                        mbar_wait(&xempty[xs], ((it / NX) & 1u) ^ 1u);
                        mbar_arrive_expect_tx(&xfull[xs], kXBox);
                        tma_load_box_2d(xring + (size_t)xs * kXBox, &xmap, w.t * 128, w.sample * p.cin + kb * 64, &xfull[xs]);
                    }
                    const int s = it % NST;
                    mbar_wait(&empty[s], ((it / NST) & 1u) ^ 1u);
                    unsigned char* st = b_stage(s) - PARTS * kA;   // the loads below add PARTS * kA back
                    mbar_arrive_expect_tx(&full_b[s], (uint32_t)(PARTS * n_sub) * kTileBytes);
                    for (int part = 0; part < PARTS; ++part)
                        for (int sub = 0; sub < n_sub; ++sub)
                            tma_load_1d(st + PARTS * kA + part * kB + sub * kTileBytes,
                                        (part ? p.w_lo : p.w_hi) + (int64_t)w.sample * p.w_batch +
                                            ((int64_t)(2 * w.ct + sub) * p.kb + kb) * kTileBytes,
                                        kTileBytes, &full_b[s], pol);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            uint32_t it = 0;
            int ti = 0;
            for (int item = blockIdx.x; item < items; item += gridDim.x, ++ti) {
                const PwItem w = pw_item(p, item);
                const uint32_t idesc = umma_idesc_bf16(128, w.ncol) | kIdescAMajorMN;
                const int buf = ti & 1;
                mbar_wait(&acc_empty[buf], ((ti >> 1) & 1) ^ 1);
                tcgen05_fence_after();
                const uint32_t d = tmem_base + (uint32_t)(buf * 256);
                for (int kb = 0; kb < p.kb; ++kb, ++it) {
                    const int s = it % NST;
                    const int as = XTMA ? (int)(it % NA) : s;
                    if (XTMA) mbar_wait(&full_a[as], (it / NA) & 1u);
                    else mbar_wait(&full_a[s], (it / NST) & 1u);
                    mbar_wait(&full_b[s], (it / NST) & 1u);
                    tcgen05_fence_after();
                    const uint32_t a_hi = smem_u32(a_stage(as)), a_lo = a_hi + kA;
                    const uint32_t b_hi = smem_u32(b_stage(s)), b_lo = b_hi + kB;
#pragma unroll
                    for (int k = 0; k < kTileK / kUmmaK; ++k) {
                        const uint32_t ko = k * kUmmaK * 2;            // B: 16 channels = 32 bytes along its K-major rows
                        const uint32_t ka = k * 2 * kPwSBO;            // A: 16 channels = two 8-channel atoms
                        umma_bf16_ss(d, umma_desc_mn_sw128(a_hi + ka), umma_desc_k_sw128(b_hi + ko), idesc, kb > 0 || k > 0);
                        if (PARTS == 2) {
                            umma_bf16_ss(d, umma_desc_mn_sw128(a_hi + ka), umma_desc_k_sw128(b_lo + ko), idesc, true);
                            umma_bf16_ss(d, umma_desc_mn_sw128(a_lo + ka), umma_desc_k_sw128(b_hi + ko), idesc, true);
                        }
                    }
                    umma_commit(&empty[s]);
                    if (XTMA) umma_commit(&a_empty[as]);             // this A stage may be rewritten
                    if (kb == p.kb - 1) umma_commit(&acc_full[buf]);
                }
            }
        }
    } else if (warp < 6) {
        // ------------------------------------------------------------------ epilogue
        const int q = warp & 3;
        const int r = q * 32 + lane;                       // row of the position tile
        int ti = 0;
        float* acc = stat_acc + (warp - 2) * (kPwMaxC * 2);
        int acc_sample = -1;
        auto flush_stats = [&](int sample) {               // this warp's sums of `sample` -> global partial, then clear
            if (EPI != 2 || !p.stats || sample < 0) return;
            float* dst = p.stats + (((int64_t)sample * p.stat_ctas + blockIdx.x) * 4 + (warp - 2)) * p.cout * 2;
            for (int o = lane; o < p.cout; o += 32) {
                dst[2 * o] = acc[2 * o];
                dst[2 * o + 1] = acc[2 * o + 1];
            }
        };
        for (int item = blockIdx.x; item < items; item += gridDim.x, ++ti) {
            const PwItem w = pw_item(p, item);
            if (EPI == 2 && p.stats && w.sample != acc_sample) {
                flush_stats(acc_sample);
                for (int o = lane; o < 2 * kPwMaxC; o += 32) acc[o] = 0.f;
                __syncwarp();
                acc_sample = w.sample;
            }
            const int buf = ti & 1;
            mbar_wait(&acc_full[buf], (ti >> 1) & 1);
            tcgen05_fence_after();
            const int64_t n = (int64_t)w.t * 128 + r;
            const bool inside = n < p.hw;
            const float* bias = p.bias ? p.bias + (int64_t)w.sample * p.bias_batch : nullptr;
            float v[32];
#pragma unroll 1
            for (int c0 = 0; c0 < w.ncol; c0 += 32) {
                const int o0 = 256 * w.ct + c0;            // first output channel of this chunk
                tmem_ld_32x32(tmem_base + (uint32_t)(buf * 256) + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, v);
                if (o0 + 32 <= p.cout) {
                    // whole chunk inside the channel range: uniform branches hoisted out of the 32-element loops (the
                    // per-element predicated form cost ~30 instructions per value and made the epilogue the bottleneck)
                    if (bias) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] += __ldg(bias + o0 + j);
                    }
                    if (p.act == 1) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] = v[j] >= 0.f ? v[j] : p.slope * v[j];
                    }
                    if (inside) {
                        if (p.residual) {
                            const float* res = p.residual + ((int64_t)w.sample * p.cout + o0) * p.hw + n;
#pragma unroll
                            for (int j = 0; j < 32; ++j) v[j] += __ldcs(res + (int64_t)j * p.hw);
                        }
                        if (p.out) {
                            float* dst = p.out + ((int64_t)w.sample * p.cout + o0) * p.hw + n;
#pragma unroll
                            for (int j = 0; j < 32; ++j) __stcs(dst + (int64_t)j * p.hw, v[j]);
                        }
                    } else if (EPI != 0) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] = 0.f;
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const bool ok = inside && o0 + j < p.cout;
                        float y = v[j] + ((bias && o0 + j < p.cout) ? __ldg(bias + o0 + j) : 0.f);
                        if (p.act == 1) y = y >= 0.f ? y : p.slope * y;
                        if (p.residual && ok) y += __ldcs(p.residual + ((int64_t)w.sample * p.cout + o0 + j) * p.hw + n);
                        v[j] = ok ? y : 0.f;
                        if (p.out && ok) __stcs(p.out + ((int64_t)w.sample * p.cout + o0 + j) * p.hw + n, y);
                    }
                }
                if (EPI == 1 && p.out_hi) {
                    // packed tile (position tile t, 64-channel block o0 / 64): this thread's row, four 16-byte chunks
                    const int kbo = o0 >> 6, ko_tiles = p.coutp >> 6;
                    char* base = p.out_hi + (int64_t)w.sample * p.tile_batch + ((int64_t)w.t * ko_tiles + kbo) * kTileBytes +
                                 (uint32_t)r * 128u;
                    char* base_lo = p.out_lo ? p.out_lo + (base - p.out_hi) : nullptr;
                    const uint32_t c16 = (uint32_t)(o0 & 63) >> 3;
#pragma unroll
                    for (int q4 = 0; q4 < 4; ++q4) {
                        uint32_t h[4], l[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const float a = v[q4 * 8 + 2 * e], b = v[q4 * 8 + 2 * e + 1];
                            h[e] = pw_pack_bf16x2(a, b);
                            l[e] = pw_pack_bf16x2(a - __uint_as_float(h[e] << 16), b - __uint_as_float(h[e] & 0xffff0000u));
                        }
                        const uint32_t off = ((c16 + q4) ^ (uint32_t)(r & 7)) << 4;
                        *reinterpret_cast<uint4*>(base + off) = make_uint4(h[0], h[1], h[2], h[3]);
                        if (base_lo) *reinterpret_cast<uint4*>(base_lo + off) = make_uint4(l[0], l[1], l[2], l[3]);
                    }
                }
                if (EPI == 2 && p.stats) {
                    // per-channel (sum, sum of squares) over this warp's 32 positions: transpose the 32 x 32 chunk through
                    // a padded shared-memory tile (32 stores + 32 conflict-free loads per thread; the shuffle butterfly
                    // cost ~6k cycles per chunk), lane j then owns column j
                    float* tile = stat_tile + (warp - 2) * (32 * 33);
#pragma unroll
                    for (int j = 0; j < 32; ++j) tile[lane * 33 + j] = v[j];
                    __syncwarp();
                    float t1 = 0.f, t2 = 0.f;
#pragma unroll
                    for (int r2 = 0; r2 < 32; ++r2) {
                        const float y = tile[r2 * 33 + lane];
                        t1 += y;
                        t2 = fmaf(y, y, t2);
                    }
                    __syncwarp();
                    if (o0 + lane < p.cout) {              // lane owns column o0 + lane: plain read-modify-write, fixed order
                        acc[2 * (o0 + lane)] += t1;
                        acc[2 * (o0 + lane) + 1] += t2;
                    }
                }
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[buf]);
        }
        __syncwarp();
        flush_stats(acc_sample);
    } else {
        // ------------------------------------------------------------------ converters: (x - sub) * mul as bf16 hi / lo, MN-major tile
        const int cw = warp - 6;                           // warp cw converts channels [8 cw, 8 cw + 8) of every k-block
        // lane -> positions 4 lane .. 4 lane + 3 of the tile: MN-atom lane / 16, 16-byte chunk (lane % 16) / 2, half lane & 1
        const uint32_t lane_off = (uint32_t)(lane >> 4) * kPwLBO + ((uint32_t)lane & 1u) * 8u;
        const uint32_t chunk = ((uint32_t)lane & 15u) >> 1;
        if (XTMA) {
            uint32_t u = 0;
            for (int item = blockIdx.x; item < items; item += gridDim.x) {
                const PwItem w = pw_item(p, item);
                for (int kb = 0; kb < p.kb; ++kb, ++u) {
                    const uint32_t xs = u % NX;
                    mbar_wait(&xfull[xs], (u / NX) & 1u);
                    const unsigned char* box = xring + (size_t)xs * kXBox + (size_t)(cw * 8) * 512 + lane * 16;
                    float4 v[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[j] = *reinterpret_cast<const float4*>(box + j * 512);
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&xempty[xs]);            // the box may be overwritten
                    const int sidx = w.sample * p.cin + kb * 64 + cw * 8;
                    float sb[8], ml[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        sb[j] = p.sub ? __ldg(p.sub + sidx + j) : 0.f;
                        ml[j] = p.mul ? __ldg(p.mul + sidx + j) : 1.f;
                    }
                    const uint32_t as = u % NA;
                    mbar_wait(&a_empty[as], ((u / NA) & 1u) ^ 1u);       // the MMAs that read this A stage last have completed
                    unsigned char* a_hi = a_stage((int)as) + (size_t)cw * kPwSBO + lane_off;
                    unsigned char* a_lo = a_hi + kA;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float a = (v[j].x - sb[j]) * ml[j], b = (v[j].y - sb[j]) * ml[j];
                        const float c2 = (v[j].z - sb[j]) * ml[j], d = (v[j].w - sb[j]) * ml[j];
                        const uint32_t off = (uint32_t)j * 128u + ((chunk ^ (uint32_t)j) << 4);
                        const uint32_t h01 = pw_pack_bf16x2(a, b), h23 = pw_pack_bf16x2(c2, d);
                        *reinterpret_cast<uint2*>(a_hi + off) = make_uint2(h01, h23);
                        if (PARTS == 2) {
                            const uint32_t l01 = pw_pack_bf16x2(a - __uint_as_float(h01 << 16), b - __uint_as_float(h01 & 0xffff0000u));
                            const uint32_t l23 = pw_pack_bf16x2(c2 - __uint_as_float(h23 << 16), d - __uint_as_float(h23 & 0xffff0000u));
                            *reinterpret_cast<uint2*>(a_lo + off) = make_uint2(l01, l23);
                        }
                    }
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&full_a[as]);
                }
            }
        } else {
        // Work units (item, k-block) in issue order; three register buffers rotate so that the loads of two units are in
        // flight while a third is converted (load-latency bound: 8 loads per thread in flight gave 1.7 TB/s).  Two cursors
        // (load / convert) walk the unit sequence incrementally: no divisions in the loop.
        struct Cursor {
            int item, kb;
            const float* xrow;     // x + (sample * cin + cw * 8) * hw + n  (k-block 0, channel row 0 of this warp)
            int soff;              // sample * cin + cw * 8: index of this warp's first channel in sub / mul
            int64_t n;             // first position of this lane (generic path)
            bool vec, live;
        };
        const int64_t kb_stride = 64 * p.hw;
        auto decode = [&](Cursor& c) {
            c.live = c.item < items;
            if (!c.live) return;
            const PwItem w = pw_item(p, c.item);
            const int64_t n = (int64_t)w.t * 128 + 4 * lane;
            c.vec = p.vec_ok && n + 4 <= p.hw;
            c.n = n;
            c.xrow = p.x + ((int64_t)w.sample * p.cin + cw * 8) * p.hw + n;
            c.soff = w.sample * p.cin + cw * 8;
        };
        auto advance = [&](Cursor& c) {
            if (++c.kb == p.kb) {
                c.kb = 0;
                c.item += (int)gridDim.x;
                decode(c);
            }
        };
        auto load_unit = [&](float4 (&v)[8], Cursor& c) {
            if (!c.live) return;
            const int c0 = c.kb * 64 + cw * 8;
            const float* src0 = c.xrow + (int64_t)c.kb * kb_stride;
            if (VEC) {
                if (c.vec && c0 < p.cin) {                  // cin % 8 == 0: a warp's 8 channels are all inside or all padding
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[j] = __ldcs(reinterpret_cast<const float4*>(src0 + (int64_t)j * p.hw));
                } else {                                    // beyond the last position / channel: the rows are discarded or multiply zero weights
                    const float pad = 0.f;
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[j] = make_float4(pad, pad, pad, pad);
                }
            } else {
                const int64_t n = c.n;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    if (c0 + j < p.cin) {
                        const float* src = src0 + (int64_t)j * p.hw;
                        const float pad = p.sub ? __ldg(p.sub + c.soff + c.kb * 64 + j) : 0.f;     // (pad - sub) * mul = 0
                        v[j].x = n + 0 < p.hw ? src[0] : pad;
                        v[j].y = n + 1 < p.hw ? src[1] : pad;
                        v[j].z = n + 2 < p.hw ? src[2] : pad;
                        v[j].w = n + 3 < p.hw ? src[3] : pad;
                    } else {
                        v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                }
            }
            advance(c);
        };
        uint32_t u = 0;
        auto conv_unit = [&](float4 (&v)[8], Cursor& c) {
            if (!c.live) return;
            const int c0 = c.kb * 64 + cw * 8;
            const int sidx = c.soff + c.kb * 64;
            const uint32_t s = u & (NST - 1);
            mbar_wait(&empty[s], ((u / NST) & 1u) ^ 1u);
            unsigned char* a_hi = smem + (size_t)s * kStage + (size_t)cw * kPwSBO + lane_off;
            unsigned char* a_lo = a_hi + kA;
#pragma unroll
            for (int j = 0; j < 8; ++j) {              // channel row j of this warp's 8-channel atom
                const bool ok = c0 + j < p.cin;
                const float sb = (p.sub && ok) ? __ldg(p.sub + sidx + j) : 0.f;
                const float ml = (p.mul && ok) ? __ldg(p.mul + sidx + j) : 1.f;
                const float a = (v[j].x - sb) * ml, b = (v[j].y - sb) * ml, c2 = (v[j].z - sb) * ml, d = (v[j].w - sb) * ml;
                const uint32_t off = (uint32_t)j * 128u + ((chunk ^ (uint32_t)j) << 4);
                const uint32_t h01 = pw_pack_bf16x2(a, b), h23 = pw_pack_bf16x2(c2, d);
                *reinterpret_cast<uint2*>(a_hi + off) = make_uint2(h01, h23);
                if (PARTS == 2) {
                    const uint32_t l01 = pw_pack_bf16x2(a - __uint_as_float(h01 << 16), b - __uint_as_float(h01 & 0xffff0000u));
                    const uint32_t l23 = pw_pack_bf16x2(c2 - __uint_as_float(h23 << 16), d - __uint_as_float(h23 & 0xffff0000u));
                    *reinterpret_cast<uint2*>(a_lo + off) = make_uint2(l01, l23);
                }
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&full_a[s]);
            ++u;
            advance(c);
        };
        Cursor ld, cv;
        ld.item = cv.item = (int)blockIdx.x;
        ld.kb = cv.kb = 0;
        decode(ld);
        cv = ld;
        float4 v0[8], v1[8], v2[8];
        load_unit(v0, ld);
        load_unit(v1, ld);
        while (cv.live) {
            load_unit(v2, ld);
            conv_unit(v0, cv);
            load_unit(v0, ld);
            conv_unit(v1, cv);
            load_unit(v1, ld);
            conv_unit(v2, cv);
        }
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 1) {
        tcgen05_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// mean / std of the stored values from the epilogue partials: fp64, fixed order (unbiased variance, eps inside the
// square root like calc_mean_std, network/base.py:404-405)
__global__ void __launch_bounds__(128) pw_stats_finalize_kernel(const float* __restrict__ partial, int entries, int cout, double hw,
                                                                double eps, float* __restrict__ mean, float* __restrict__ stdv) {
    const int o = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
    if (o >= cout) return;
    const float* src = partial + ((int64_t)b * entries * cout + o) * 2;
    double s1 = 0.0, s2 = 0.0;
    for (int z = 0; z < entries; ++z) {
        const float2 v = __ldg(reinterpret_cast<const float2*>(src + (int64_t)z * cout * 2));
        s1 += (double)v.x;
        s2 += (double)v.y;
    }
    const double mu = s1 / hw;
    const double var = (s2 - s1 * mu) / (hw - 1.0);
    mean[(int64_t)b * cout + o] = (float)mu;
    stdv[(int64_t)b * cout + o] = (float)sqrt((var > 0.0 ? var : 0.0) + eps);
}

}  // namespace

bool pw_conv_supported(int64_t cin, int64_t cout) { return cin >= 1 && cin <= kPwMaxC && cout >= 1 && cout <= kPwMaxC; }

struct PwArgs {
    const float* x; const float* sub; const float* mul;
    const void* w_hi; const void* w_lo; int64_t w_batch;
    const float* bias; int64_t bias_batch;
    const float* residual;
    float* out; void* out_hi; void* out_lo; int64_t tile_batch;
    float* stats;
    int act; float slope;
    int64_t b, cin, cout, hw;
    int passes;
};

int pw_conv(const PwArgs& a, cudaStream_t st) {
    PwParams p{};
    p.x = a.x; p.sub = a.sub; p.mul = a.mul;
    p.w_hi = static_cast<const char*>(a.w_hi); p.w_lo = static_cast<const char*>(a.w_lo); p.w_batch = a.w_batch;
    p.bias = a.bias; p.bias_batch = a.bias_batch; p.residual = a.residual;
    p.out = a.out; p.out_hi = static_cast<char*>(a.out_hi); p.out_lo = static_cast<char*>(a.out_lo); p.tile_batch = a.tile_batch;
    p.stats = a.stats; p.act = a.act; p.slope = a.slope;
    p.hw = a.hw; p.cin = (int)a.cin; p.cout = (int)a.cout;
    p.coutp = (int)((a.cout + 127) / 128 * 128);
    p.kb = (int)((a.cin + kTileK - 1) / kTileK);
    p.col_tiles = (p.coutp + 255) / 256;
    p.tiles = (int)((a.hw + 127) / 128);
    p.batch = (int)a.b;
    p.stat_ctas = sm_count();
    p.vec_ok = (a.hw % 4 == 0 && (reinterpret_cast<uintptr_t>(a.x) & 15u) == 0) ? 1 : 0;
    const int64_t items = (int64_t)p.batch * p.tiles * p.col_tiles;
    if (items == 0) return RPST_OK;
    RPST_CHECK_ARG(items < (1ll << 30), "conv1x1: too many work items");
    constexpr size_t smem = 1024 + 2 * 2 * (kTileBytes + 2 * kTileBytes);   // 193 KiB for every register-staged instantiation
    constexpr size_t smem_x = 1024 + 2 * kTileBytes + 2 * 2 * 2 * kTileBytes + 2 * 64 * 128 * sizeof(float);   // 225 KiB (XTMA)
    const bool vec = p.vec_ok && a.cin % 8 == 0;
    const int epi = p.out_hi ? 1 : (p.stats ? 2 : 0);
    RPST_CHECK_ARG(!(p.out_hi && p.stats), "conv1x1: packed output and epilogue statistics are separate modes");
    int grid = sm_count();
    if (grid > items) grid = (int)items;
    CUtensorMap xmap;
    memset(&xmap, 0, sizeof(xmap));
    const bool xtma = g_knobs.pw_x_tma && vec && epi != 2 && a.cin % 64 == 0 && a.hw < (1ll << 31) - 128 &&
                      a.b * a.cin < (1ll << 31) && tmap_encode_2d_f32(&xmap, a.x, (uint64_t)a.hw, (uint64_t)(a.b * a.cin), 128, 64);
    static PerDeviceFlag configured_on[24];
#define RPST_PW_CASE(PARTS, VEC, EPI, XT)                                                                                 \
    {                                                                                                                     \
        bool& configured = configured_on[(((PARTS) - 1) * 6 + (VEC) * 3 + (EPI)) * 2 + (XT)].get();                       \
        if (!configured) {                                                                                                \
            RPST_CUDA(cudaFuncSetAttribute(pw_conv_kernel<PARTS, VEC, EPI, XT>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                           (int)((XT) ? smem_x : smem)));                                                 \
            configured = true;                                                                                            \
        }                                                                                                                 \
        pw_conv_kernel<PARTS, VEC, EPI, XT><<<grid, kPwThreads, (XT) ? smem_x : smem, st>>>(xmap, p);                     \
    }
#define RPST_PW_EPI(PARTS, VEC)                                                    \
    if (epi == 0) RPST_PW_CASE(PARTS, VEC, 0, false) else if (epi == 1) RPST_PW_CASE(PARTS, VEC, 1, false) else RPST_PW_CASE(PARTS, VEC, 2, false)
#define RPST_PW_EPI_X(PARTS)                                                       \
    if (epi == 0) RPST_PW_CASE(PARTS, true, 0, true) else RPST_PW_CASE(PARTS, true, 1, true)
    if (a.passes == 3) {
        if (xtma) { RPST_PW_EPI_X(2) } else if (vec) { RPST_PW_EPI(2, true) } else { RPST_PW_EPI(2, false) }
    } else {
        if (xtma) { RPST_PW_EPI_X(1) } else if (vec) { RPST_PW_EPI(1, true) } else { RPST_PW_EPI(1, false) }
    }
#undef RPST_PW_EPI_X
#undef RPST_PW_EPI
#undef RPST_PW_CASE
    RPST_CUDA(cudaGetLastError());
    return RPST_OK;
}

// ---- WCT colouring (wct.cu): out = T (x - mu_c) + mu_s with T given as packed tiles (rows = output channels).
// (A dedicated copy of this kernel without the general epilogue measured 1.80 vs 1.83 ms per sample end to end: dropped.)
bool wct_apply_fused_supported(int64_t c, int64_t hw) { return c >= 1 && c <= kPwMaxC && hw >= 1; }

// n samples in one persistent launch: x / out [n,c,hw], mu_* [n,c], packed transforms t_batch_bytes apart
int wct_apply_fused(const float* x, const float* mu_c, const float* mu_s, const void* t_hi, const void* t_lo, float* out,
                    int64_t n, int64_t t_batch_bytes, int64_t c, int64_t hw, int passes, cudaStream_t st) {
    PwArgs a{};
    a.x = x; a.sub = mu_c; a.w_hi = t_hi; a.w_lo = t_lo; a.w_batch = t_batch_bytes; a.bias = mu_s; a.bias_batch = c; a.out = out;
    a.b = n; a.cin = c; a.cout = c; a.hw = hw; a.passes = passes;
    return pw_conv(a, st);
}

}  // namespace rpst

using namespace rpst;

// per sample: one (sum, sum of squares) pair per channel, CTA and epilogue warp
static int pw_stat_entries() { return sm_count() * 4; }

extern "C" size_t rpst_conv1x1_stats_bytes(int64_t b, int64_t cout, int64_t hw) {
    if (b <= 0 || cout <= 0 || hw <= 0) return 256;
    return align_up((size_t)b * pw_stat_entries() * cout * 2 * sizeof(float), 256);
}

extern "C" int rpst_conv1x1(const float* x, const void* w_hi, const void* w_lo, const float* bias, const float* sub,
                            const float* mul, const float* residual, float* out, void* out_hi, void* out_lo,
                            float* stats_partial, int64_t b, int64_t cin, int64_t cout, int64_t hw, int act, float slope,
                            int passes, void* stream) {
    RPST_CHECK_ARG(b >= 0 && cin >= 0 && cout >= 0 && hw >= 0, "conv1x1: negative size");
    if (b == 0 || cout == 0 || hw == 0) return RPST_OK;
    RPST_CHECK_ARG(pw_conv_supported(cin, cout), "conv1x1: at most 512 input and output channels (got %lld -> %lld)",
                   (long long)cin, (long long)cout);
    RPST_CHECK_ARG(x && w_hi && (out || out_hi), "conv1x1: null pointer");
    RPST_CHECK_ARG(passes == 1 || passes == 3, "conv1x1: passes must be 1 (bf16) or 3 (bf16x3, fp32-grade)");
    RPST_CHECK_ARG(passes == 1 || w_lo, "conv1x1: bf16x3 needs the lo part of the packed weight");
    RPST_CHECK_ARG(act == 0 || act == 1, "conv1x1: act must be 0 (none) or 1 (LeakyReLU)");
    RPST_CHECK_ARG(!out_hi || hw % 128 == 0, "conv1x1: packed output needs H*W to be a multiple of 128");
    RPST_CHECK_ARG(!out_hi || cout % 64 == 0, "conv1x1: packed output needs a multiple of 64 output channels");
    PwArgs a{};
    a.x = x; a.sub = sub; a.mul = mul; a.w_hi = w_hi; a.w_lo = w_lo; a.bias = bias; a.residual = residual;
    a.out = out; a.out_hi = out_hi; a.out_lo = out_lo;
    a.tile_batch = (int64_t)align_up(packed_operand_bytes(hw, cout), 256);
    a.stats = stats_partial; a.act = act; a.slope = slope;
    a.b = b; a.cin = cin; a.cout = cout; a.hw = hw; a.passes = passes;
    if (stats_partial)      // CTAs that never touch a sample leave their entries at zero
        RPST_CUDA(cudaMemsetAsync(stats_partial, 0, rpst_conv1x1_stats_bytes(b, cout, hw), static_cast<cudaStream_t>(stream)));
    return pw_conv(a, static_cast<cudaStream_t>(stream));
}

extern "C" int rpst_conv1x1_stats_finalize(const float* stats_partial, int64_t b, int64_t cout, int64_t hw, float eps,
                                           float* mean, float* std, void* stream) {
    RPST_CHECK_ARG(b >= 0 && cout >= 0 && hw >= 0, "conv1x1_stats: negative size");
    if (b == 0 || cout == 0) return RPST_OK;
    RPST_CHECK_ARG(stats_partial && mean && std, "conv1x1_stats: null pointer");
    const int entries = pw_stat_entries();
    pw_stats_finalize_kernel<<<dim3((unsigned)((cout + 127) / 128), (unsigned)b), 128, 0, static_cast<cudaStream_t>(stream)>>>(
        stats_partial, entries, (int)cout, (double)hw, (double)eps, mean, std);
    RPST_CUDA(cudaGetLastError());
    return RPST_OK;
}

RPST_WATCHDOG_SETTER(pwconv)

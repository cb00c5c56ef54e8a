// Flash-style SANet attention for head dimension C = 512 on the 5th-gen tensor cores — SURVEY.md §2b K8, §8 a9;
// reference: network/sanet.py:85-94 (`S = softmax(F^T G)`, `O = H S^T`, no temperature).
//
// Why a CTA PAIR: O for 128 queries x 512 channels in fp32 is the whole TMEM (512 columns) of one SM, leaving no
// room for S.  With tcgen05.mma.cta_group::2 and M = 128 each CTA of the pair owns 64 query rows, and the
// accumulator layout of that shape spreads a row's N columns over lanes r and r+64 (N/2 TMEM columns): O (64 x 512)
// takes 256 columns, two S tiles (64 x 256 keys each) take 2 x 128 columns — exactly 512.  K and V tiles are the B
// operand, which the hardware shares across the pair: each CTA stages half of every tile.
//
//   TMEM (per CTA)   cols [0,256)  O: d-chunk dc in cols [128 dc, 128 dc + 128); lane r holds d = 256 dc + j,
//                                     lane r + 64 holds d = 256 dc + 128 + j
//                    cols [256,512) S double buffer: tile g in cols 256 + 128 (g & 1); lane r holds keys j,
//                                     lane r + 64 keys 128 + j of the 256-key tile
//   shared memory    Q (64 rows x 512, bf16 hi [+ lo])  64 [128] KiB   resident per work item
//                    P (64 rows x 256 keys, bf16 / f16) 32 KiB         A operand of the P.V product
//                    ring of 16 KiB operand tiles       8 [4] slots    K tiles (128 keys x 64 ch), V tiles (128 ch x 64 keys)
//
// Roles (192 threads, one CTA per SM): warp 0 = TMA producer; warp 1 = MMA issuer in the leader CTA, relay of the
// "tile landed" events in the peer CTA; warps 2-5 = softmax (one TMEM lane per thread): pass 1 row maximum (the two
// halves of a row meet through shared memory), lazy rescale of O (only when the maximum grew by more than 2^8:
// tcgen05.ld -> scale -> tcgen05.st), pass 2 exp2 / row sum / P to swizzled shared memory, and the final 1/l epilogue.
// The tensor pipe runs QK(t+1) while the softmax warps work on tile t and P.V(t-1) drains.
//
// Precision modes: plain bf16 (1 + 1 MMA passes) and fp32-grade X3: bf16x3 on the logits (hi.hi + hi.lo + lo.hi) and
// IEEE-half P and V (11-bit significands; V pre-scaled by a per-sample power of two so that |V| < 2^15).
#include <cuda_fp16.h>

#include "common.cuh"
#include "tuning.cuh"
#include "umma.cuh"

namespace rpst {

size_t packed_operand_bytes(int64_t rows, int64_t k);
int pack_operand_batched(const float* x, int64_t rows, int64_t k, int64_t stride_r, int64_t stride_k,
                         const float* row_scale, const float* row_shift, void* hi, void* lo, int batch, int64_t x_batch,
                         int64_t tile_batch_bytes, int64_t vec_batch, cudaStream_t stream);
int pack_operand_batched_f16(const float* x, int64_t rows, int64_t k, int64_t stride_r, int64_t stride_k,
                             const float* row_scale, void* out, int batch, int64_t x_batch, int64_t tile_batch_bytes,
                             int64_t vec_batch, cudaStream_t stream);

namespace {

constexpr int kFlThreads = 192;
constexpr int kFlD = 512;                          // channels = head dimension
constexpr int kFlRows = 64;                        // query rows per CTA (128 per pair)
constexpr int kFlKeys = 256;                       // keys per S tile
constexpr int kFlQKBlocks = kFlD / kTileK;         // 8 k-blocks of 64 channels in Q K^T
constexpr int kFlPVBlocks = kFlKeys / kTileK;      // 4 key blocks of 64 in P V
constexpr uint32_t kFlHalfTile = kFlRows * 128;    // 8 KiB: 64 rows x 64 16-bit elements, SW128
constexpr uint32_t kFlQPart = kFlQKBlocks * kFlHalfTile;   // 64 KiB
constexpr uint32_t kFlPBytes = kFlPVBlocks * kFlHalfTile;  // 32 KiB
constexpr uint32_t kFlOCols = 256, kFlSCols = 128;
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kRescaleThreshold = 8.f;           // log2 units: P stays below 2^8

template <bool X3> struct FlashCfg {
    static constexpr int parts = X3 ? 2 : 1;
    static constexpr int slots = X3 ? 4 : 8;
    static constexpr uint32_t q_bytes = parts * kFlQPart;
    static constexpr size_t smem = 1024 + (size_t)q_bytes + kFlPBytes + (size_t)slots * kTileBytes;   // 225 KiB
};

struct FlashParams {
    const char* q_hi; const char* q_lo;     // packed [lc x 512] tiles (rows = query positions)
    const char* k_hi; const char* k_lo;     // packed [ls x 512] tiles (rows = key positions)
    const char* v;                          // packed [512 x ls] tiles (rows = channels), bf16 or scaled f16
    int64_t q_batch, k_batch, v_batch;      // byte strides between samples
    const float* v_unscale;                 // [b] 1 / (power-of-two scale applied to V) or null
    float* out;                             // [b, 512, lc]
    int lc, ls;
    int qtiles, ktiles;                     // lc / 128, ls / 256
    int items;                              // b * qtiles
    unsigned long long* prof;               // optional [32] cycle counters of pair 0 (tuning knob "attn_flash_prof")
};

template <bool X3>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kFlThreads, 1) flash_attn_kernel(FlashParams p) {
    using Cfg = FlashCfg<X3>;
    constexpr int NS = Cfg::slots;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* q_smem = smem;
    unsigned char* p_smem = smem + Cfg::q_bytes;
    unsigned char* ring = p_smem + kFlPBytes;
    __shared__ uint64_t full[NS], empty[NS];
    __shared__ uint64_t q_full, q_empty, s_full[2], s_empty[2], p_full, o_done;
    __shared__ uint32_t tmem_slot;
    __shared__ float xch[2][128];           // row maxima / row sums of the two halves of a row

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_rank();
    const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
    const int T = p.ktiles;

    if (threadIdx.x == 0) {
        // In the LEADER a "tile landed" barrier completes when its own TMA bytes have arrived AND the peer's relay thread
        // has reported the other half (count 2): the MMA thread pays one try_wait per tile instead of two (a try_wait
        // costs ~90 cycles even when the phase is already complete: 10.1k -> 8.9k cycles per key tile).
        const uint32_t landed = rank == 0 ? 2u : 1u;
        for (int s = 0; s < NS; ++s) {
            mbar_init(&full[s], landed);
            mbar_init(&empty[s], 1);
        }
        mbar_init(&q_full, landed);
        mbar_init(&q_empty, 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&s_full[i], 1);
            mbar_init(&s_empty[i], 8);      // 4 softmax warps of each CTA (used in the leader only)
        }
        mbar_init(&p_full, 8);
        mbar_init(&o_done, 1);
        mbar_fence_init();
    }
    __syncthreads();
    if (warp == 1) tmem_alloc2(&tmem_slot, 512);
    tcgen05_fence_before();
    cluster_sync_all();       // both CTAs: barriers initialised and TMEM allocated before any remote event
    tcgen05_fence_after();
    const uint32_t tmem_base = tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            // ------------------------------------------------------------------ TMA producer (both CTAs)
            const uint64_t pol = policy_evict_last();    // K / V tiles are re-read by every query tile: keep in L2
            uint32_t use = 0;
            int n = 0;
            for (int item = pair; item < p.items; item += npairs, ++n) {
                const int sample = item / p.qtiles, qt = item % p.qtiles;
                if (n > 0) mbar_wait(&q_empty, (uint32_t)(n - 1) & 1u);
                mbar_arrive_expect_tx(&q_full, Cfg::q_bytes);
                for (int part = 0; part < Cfg::parts; ++part) {
                    const char* src = (part ? p.q_lo : p.q_hi) + (int64_t)sample * p.q_batch +
                                      (int64_t)qt * kFlQKBlocks * kTileBytes + (int64_t)rank * kFlHalfTile;
                    for (int kb = 0; kb < kFlQKBlocks; ++kb)
                        tma_load_1d(q_smem + part * kFlQPart + kb * kFlHalfTile, src + (int64_t)kb * kTileBytes, kFlHalfTile,
                                    &q_full, pol);
                }
                auto load_tile = [&](const char* src) {
                    const uint32_t slot = use % NS;
                    mbar_wait(&empty[slot], ((use / NS) & 1u) ^ 1u);
                    mbar_arrive_expect_tx(&full[slot], kTileBytes);
                    tma_load_1d(ring + (size_t)slot * kTileBytes, src, kTileBytes, &full[slot], pol);
                    ++use;
                };
                const char* kh = p.k_hi + (int64_t)sample * p.k_batch;
                const char* kl = X3 ? p.k_lo + (int64_t)sample * p.k_batch : nullptr;
                const char* vv = p.v + (int64_t)sample * p.v_batch;
                const int64_t v_ktiles = p.ls / kTileK;
                auto load_k = [&](int t) {
                    const int64_t rb = 2 * (int64_t)t + rank;
                    for (int kb = 0; kb < kFlQKBlocks; ++kb) {
                        load_tile(kh + (rb * kFlQKBlocks + kb) * kTileBytes);
                        if (X3) load_tile(kl + (rb * kFlQKBlocks + kb) * kTileBytes);
                    }
                };
                auto load_v = [&](int t) {
                    for (int kbv = 0; kbv < kFlPVBlocks; ++kbv)
                        for (int dc = 0; dc < 2; ++dc)
                            load_tile(vv + ((int64_t)(2 * dc + rank) * v_ktiles + (int64_t)t * kFlPVBlocks + kbv) * kTileBytes);
                };
                load_k(0);
                for (int t = 1; t < T; ++t) {
                    load_k(t);
                    load_v(t - 1);
                }
                load_v(T - 1);
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && rank == 0) {
            // ------------------------------------------------------------------ MMA issuer (leader CTA)
            const uint32_t idesc_qk = umma_idesc_bf16(128, kFlKeys);
            const uint32_t idesc_pv = X3 ? umma_idesc_f16(128, 256) : umma_idesc_bf16(128, 256);
            const uint32_t q_addr = smem_u32(q_smem), p_addr = smem_u32(p_smem), ring_addr = smem_u32(ring);
            uint32_t use = 0, g0 = 0;
            int n = 0;
            uint32_t last_slot = 0;
            const bool prof = p.prof != nullptr && pair == 0;
            long long c_full = 0, c_peer = 0, c_sempty = 0, c_pfull = 0, c_q = 0;
            const long long c_begin = clock64();
            auto wait_slot = [&]() -> uint32_t {
                const uint32_t slot = use % NS, ph = (use / NS) & 1u;
                long long t0 = 0, t1 = 0;
                if (prof) t0 = clock64();
                mbar_wait(&full[slot], ph);            // own bytes + the peer's relayed TMA-completion event
                if (prof) { t1 = clock64(); c_full += t1 - t0; }
                tcgen05_fence_after();
                ++use;
                last_slot = slot;
                return ring_addr + slot * kTileBytes;
            };
            for (int item = pair; item < p.items; item += npairs, ++n) {
                long long tq = prof ? clock64() : 0;
                mbar_wait(&q_full, (uint32_t)n & 1u);
                if (prof) c_q += clock64() - tq;
                tcgen05_fence_after();
                auto issue_qk = [&](int t) {
                    const uint32_t g = g0 + t, buf = g & 1u;
                    long long ts = prof ? clock64() : 0;
                    mbar_wait_cluster(&s_empty[buf], ((g >> 1) & 1u) ^ 1u);
                    if (prof) c_sempty += clock64() - ts;
                    tcgen05_fence_after();
                    const uint32_t d = tmem_base + kFlOCols + buf * kFlSCols;
                    for (int kb = 0; kb < kFlQKBlocks; ++kb) {
                        const uint32_t bh = wait_slot();
                        const uint32_t slot_h = last_slot;
                        uint32_t bl = 0, slot_l = 0;
                        if (X3) { bl = wait_slot(); slot_l = last_slot; }
                        const uint32_t ah = q_addr + kb * kFlHalfTile, al = ah + kFlQPart;
#pragma unroll
                        for (int k = 0; k < kTileK / kUmmaK; ++k) {
                            const uint32_t ko = k * kUmmaK * 2;
                            umma2_ss(d, umma_desc_k_sw128(ah + ko), umma_desc_k_sw128(bh + ko), idesc_qk, kb > 0 || k > 0);
                            if (X3) {
                                umma2_ss(d, umma_desc_k_sw128(ah + ko), umma_desc_k_sw128(bl + ko), idesc_qk, true);
                                umma2_ss(d, umma_desc_k_sw128(al + ko), umma_desc_k_sw128(bh + ko), idesc_qk, true);
                            }
                        }
                        umma2_commit(&empty[slot_h]);
                        if (X3) umma2_commit(&empty[slot_l]);
                    }
                    umma2_commit(&s_full[buf]);
                    if (t == T - 1) umma2_commit(&q_empty);    // Q may be overwritten once these MMAs have read it
                };
                auto issue_pv = [&](int t) {
                    const uint32_t g = g0 + t;
                    long long tp = prof ? clock64() : 0;
                    mbar_wait_cluster(&p_full, g & 1u);
                    if (prof) c_pfull += clock64() - tp;
                    tcgen05_fence_after();
                    for (int kbv = 0; kbv < kFlPVBlocks; ++kbv) {
                        for (int dc = 0; dc < 2; ++dc) {
                            const uint32_t bv = wait_slot();
                            const uint32_t a = p_addr + kbv * kFlHalfTile;
#pragma unroll
                            for (int k = 0; k < kTileK / kUmmaK; ++k) {
                                const uint32_t ko = k * kUmmaK * 2;
                                umma2_ss(tmem_base + dc * 128, umma_desc_k_sw128(a + ko), umma_desc_k_sw128(bv + ko), idesc_pv,
                                         t > 0 || kbv > 0 || k > 0);
                            }
                            umma2_commit(&empty[last_slot]);
                        }
                    }
                    umma2_commit(&o_done);
                };
                issue_qk(0);
                for (int t = 1; t < T; ++t) {
                    issue_qk(t);
                    issue_pv(t - 1);
                }
                issue_pv(T - 1);
                g0 += T;
            }
            if (prof) {
                p.prof[0] = (unsigned long long)(clock64() - c_begin);
                p.prof[1] = (unsigned long long)c_full; p.prof[2] = (unsigned long long)c_peer;
                p.prof[3] = (unsigned long long)c_sempty; p.prof[4] = (unsigned long long)c_pfull;
                p.prof[5] = (unsigned long long)c_q; p.prof[6] = (unsigned long long)g0;
            }
        } else if (lane == 0) {
            // ------------------------------------------------------------------ relay (peer CTA): my half has landed
            const uint32_t uses_per_item = (uint32_t)T * (kFlQKBlocks * Cfg::parts + 2 * kFlPVBlocks);
            const uint32_t peer_full_remote = mapa_u32(smem_u32(&full[0]), 0);      // the leader's barriers (count 2)
            const uint32_t peer_q_remote = mapa_u32(smem_u32(&q_full), 0);
            uint32_t use = 0;
            int n = 0;
            for (int item = pair; item < p.items; item += npairs, ++n) {
                mbar_wait(&q_full, (uint32_t)n & 1u);
                mbar_arrive_cluster_relaxed(peer_q_remote);
                for (uint32_t u = 0; u < uses_per_item; ++u, ++use) {
                    const uint32_t slot = use % NS;
                    mbar_wait(&full[slot], (use / NS) & 1u);
                    mbar_arrive_cluster_relaxed(peer_full_remote + slot * (uint32_t)sizeof(uint64_t));
                }
            }
        }
    } else {
        // ---------------------------------------------------------------------- softmax warps (both CTAs)
        const int quarter = warp & 3;                       // TMEM lanes [32 q, 32 q + 32)
        const int tl = quarter * 32 + lane;                 // this thread's TMEM lane
        const int row = tl & 63, hf = tl >> 6;              // query row within the CTA, column half
        const uint32_t lane_addr = tmem_base + ((uint32_t)(quarter * 32) << 16);
        const uint32_t s_empty_remote = mapa_u32(smem_u32(&s_empty[0]), 0);
        const uint32_t p_full_remote = mapa_u32(smem_u32(&p_full), 0);
        unsigned char* p_row = p_smem + row * 128;
        const uint32_t sw = (uint32_t)(row & 7);
        uint32_t g = 0;
        const bool prof = p.prof != nullptr && pair == 0 && rank == 0 && warp == 2 && lane == 0;
        long long c_sfull = 0, c_p1 = 0, c_bar = 0, c_odone = 0, c_resc = 0, c_p2 = 0, c_epi = 0;
        const long long c_begin = clock64();
        for (int item = pair; item < p.items; item += npairs) {
            const int sample = item / p.qtiles, qt = item % p.qtiles;
            float m_ref = -INFINITY, l = 0.f;
            for (int t = 0; t < T; ++t, ++g) {
                const uint32_t buf = g & 1u;
                long long k0 = prof ? clock64() : 0;
                mbar_wait(&s_full[buf], (g >> 1) & 1u);
                long long k1 = prof ? clock64() : 0;
                tcgen05_fence_after();
                const uint32_t s_addr = lane_addr + kFlOCols + buf * kFlSCols;
                float v[32];
                // pass 1: row maximum over this thread's 128 keys, then over both halves of the row
                float mx = -INFINITY;
#pragma unroll 1
                for (int ch = 0; ch < 4; ++ch) {
                    tmem_ld_32x32(s_addr + ch * 32, v);
#pragma unroll
                    for (int j = 0; j < 32; ++j) mx = fmaxf(mx, v[j]);
                }
                long long k2 = prof ? clock64() : 0;
                xch[g & 1u][tl] = mx;
                named_bar_sync(1, 128);
                mx = fmaxf(mx, xch[g & 1u][tl ^ 64]) * kLog2e;
                long long k3 = prof ? clock64() : 0;
                float scale = 1.f;
                bool need = false;
                if (t == 0) {
                    m_ref = mx;
                } else if (mx > m_ref + kRescaleThreshold) {
                    scale = ex2_approx(m_ref - mx);
                    m_ref = mx;
                    need = true;
                }
                // P buffer free and O quiescent: the previous tile's P.V has completed
                if (g > 0) {
                    mbar_wait(&o_done, (g - 1) & 1u);
                    tcgen05_fence_after();
                }
                long long k4 = prof ? clock64() : 0;
                if (__any_sync(0xffffffffu, need)) {
                    l *= scale;
#pragma unroll 1
                    for (int c0 = 0; c0 < (int)kFlOCols; c0 += 32) {
                        tmem_ld_32x32(lane_addr + c0, v);
                        uint32_t r[32];
#pragma unroll
                        for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(v[j] * scale);
                        tmem_st_32x32(lane_addr + c0, r);
                    }
                }
                long long k5 = prof ? clock64() : 0;
                // pass 2: P = exp2(s log2e - m_ref), row sum, 16-bit P into the swizzled A-operand tile
#pragma unroll 1
                for (int ch = 0; ch < 4; ++ch) {
                    tmem_ld_32x32(s_addr + ch * 32, v);
                    unsigned char* dst = p_row + (2 * hf + (ch >> 1)) * kFlHalfTile;
                    const uint32_t c16 = (uint32_t)(ch & 1) * 4;
#pragma unroll
                    for (int q4 = 0; q4 < 4; ++q4) {
                        float e[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            e[j] = ex2_approx(fmaf(v[q4 * 8 + j], kLog2e, -m_ref));
                            l += e[j];
                        }
                        uint4 w;
                        if (X3) {
                            __half2 h0 = __floats2half2_rn(e[0], e[1]), h1 = __floats2half2_rn(e[2], e[3]);
                            __half2 h2 = __floats2half2_rn(e[4], e[5]), h3 = __floats2half2_rn(e[6], e[7]);
                            w.x = *reinterpret_cast<uint32_t*>(&h0); w.y = *reinterpret_cast<uint32_t*>(&h1);
                            w.z = *reinterpret_cast<uint32_t*>(&h2); w.w = *reinterpret_cast<uint32_t*>(&h3);
                        } else {
                            __nv_bfloat162 h0 = __floats2bfloat162_rn(e[0], e[1]), h1 = __floats2bfloat162_rn(e[2], e[3]);
                            __nv_bfloat162 h2 = __floats2bfloat162_rn(e[4], e[5]), h3 = __floats2bfloat162_rn(e[6], e[7]);
                            w.x = *reinterpret_cast<uint32_t*>(&h0); w.y = *reinterpret_cast<uint32_t*>(&h1);
                            w.z = *reinterpret_cast<uint32_t*>(&h2); w.w = *reinterpret_cast<uint32_t*>(&h3);
                        }
                        *reinterpret_cast<uint4*>(dst + (((c16 + q4) ^ sw) * 16)) = w;
                    }
                }
                // hand S[buf] back to the MMA thread and publish P (generic-proxy writes -> async-proxy reads)
                tcgen05_fence_before();
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) {
                    if (rank == 0) {
                        mbar_arrive(&s_empty[buf]);
                        mbar_arrive(&p_full);
                    } else {
                        mbar_arrive_cluster(s_empty_remote + buf * (uint32_t)sizeof(uint64_t));
                        mbar_arrive_cluster(p_full_remote);
                    }
                }
                if (prof) {
                    const long long k6 = clock64();
                    c_sfull += k1 - k0; c_p1 += k2 - k1; c_bar += k3 - k2; c_odone += k4 - k3; c_resc += k5 - k4; c_p2 += k6 - k5;
                }
            }
            const long long e0 = prof ? clock64() : 0;
            // ---- epilogue of the work item: O / l -> out[sample, d, i]
            mbar_wait(&o_done, (g - 1) & 1u);
            tcgen05_fence_after();
            named_bar_sync(1, 128);                 // everyone is past the last exchange of row maxima
            xch[0][tl] = l;
            named_bar_sync(1, 128);
            float inv = 1.f / (l + xch[0][tl ^ 64]);
            if (p.v_unscale) inv *= __ldg(p.v_unscale + sample);
            float* out = p.out + (int64_t)sample * kFlD * p.lc + (int64_t)qt * 128 + rank * kFlRows + row;
            float v[32];
#pragma unroll 1
            for (int dc = 0; dc < 2; ++dc) {
#pragma unroll 1
                for (int c0 = 0; c0 < 128; c0 += 32) {
                    tmem_ld_32x32(lane_addr + dc * 128 + c0, v);
                    float* o = out + (int64_t)(256 * dc + 128 * hf + c0) * p.lc;
#pragma unroll
                    for (int j = 0; j < 32; ++j) __stcs(o + (int64_t)j * p.lc, v[j] * inv);
                }
            }
            named_bar_sync(1, 128);                 // xch[0] is rewritten by the next item's first tile only after this
            if (prof) c_epi += clock64() - e0;
        }
        if (prof) {
            p.prof[8] = (unsigned long long)(clock64() - c_begin);
            p.prof[9] = (unsigned long long)c_sfull; p.prof[10] = (unsigned long long)c_p1; p.prof[11] = (unsigned long long)c_bar;
            p.prof[12] = (unsigned long long)c_odone; p.prof[13] = (unsigned long long)c_resc; p.prof[14] = (unsigned long long)c_p2;
            p.prof[15] = (unsigned long long)c_epi;
        }
    }
    tcgen05_fence_before();
    cluster_sync_all();      // neither CTA may free TMEM / exit while the other still reads its shared memory
    if (warp == 1) {
        tcgen05_fence_after();
        tmem_dealloc2(tmem_base, 512);
    }
}

// largest |x| of each sample -> power-of-two scale with max|x| * scale < 2^15 (IEEE-half range with head-room)
__global__ void __launch_bounds__(256) absmax_kernel(const float* __restrict__ x, int64_t per_sample, unsigned int* __restrict__ mx) {
    const float* xs = x + blockIdx.y * per_sample;
    float m = 0.f;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nthr = (int64_t)gridDim.x * blockDim.x;
    if ((reinterpret_cast<uintptr_t>(xs) & 15u) == 0 && per_sample % 4 == 0) {
        const float4* x4 = reinterpret_cast<const float4*>(xs);
        for (int64_t i = tid; i < per_sample / 4; i += nthr) {
            const float4 v = __ldg(x4 + i);
            m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
        }
    } else {
        for (int64_t i = tid; i < per_sample; i += nthr) m = fmaxf(m, fabsf(xs[i]));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(mx + blockIdx.y, __float_as_uint(m));   // non-negative floats order like uints
}
__global__ void scale_fill_kernel(const unsigned int* __restrict__ mx, int b, int c, float* __restrict__ row_scale,
                                  float* __restrict__ unscale) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= b * c) return;
    const int s = i / c;
    const float m = __uint_as_float(mx[s]);
    int e = 0;
    float sc = 1.f;
    if (m > 0.f && isfinite(m)) {
        frexpf(m, &e);                      // m < 2^e
        sc = ldexpf(1.f, 15 - e);
    }
    row_scale[i] = sc;
    if (i % c == 0) unscale[s] = 1.f / sc;
}

struct FlashLayout {
    size_t row_scale, unscale, absmax, header;      // small per-sample vectors in front
    size_t q_b, k_b, v_b, per_sample;               // byte strides of the packed operands
};
FlashLayout flash_layout(int64_t lc, int64_t ls, int64_t max_samples) {
    FlashLayout l;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o += align_up(bytes, 256); return at; };
    l.row_scale = take((size_t)max_samples * kFlD * sizeof(float));
    l.unscale = take((size_t)max_samples * sizeof(float));
    l.absmax = take((size_t)max_samples * sizeof(unsigned int));
    l.header = o;
    l.q_b = align_up(packed_operand_bytes(lc, kFlD), 256);
    l.k_b = align_up(packed_operand_bytes(ls, kFlD), 256);
    l.v_b = align_up(packed_operand_bytes(kFlD, ls), 256);
    l.per_sample = 2 * l.q_b + 2 * l.k_b + l.v_b;
    return l;
}

}  // namespace

bool flash_attn_supported(int64_t c, int64_t lc, int64_t ls) {
    return c == kFlD && lc > 0 && ls > 0 && lc % 128 == 0 && ls % kFlKeys == 0;
}

size_t flash_attn_workspace_bytes(int64_t lc, int64_t ls, int64_t samples) {
    const FlashLayout l = flash_layout(lc, ls, samples);
    return l.header + (size_t)samples * l.per_sample;
}

// softmax(F^T G) applied to H for `b` samples, F [b,512,lc], G/H [b,512,ls] -> out [b,512,lc]; samples are processed
// in groups of as many as the workspace holds (one persistent launch per group).  With `q_pre` / `k_pre` the Q / K
// operand tiles come from the caller (pwconv.cu emits them from the 1x1 projections' epilogue: hi at q_pre, lo at
// q_pre + q_pre_lo_offset, sample stride q_pre_batch) and f / g are not read.
struct FlashPrepacked {
    const char* q_hi; const char* q_lo; const char* k_hi; const char* k_lo;
    int64_t q_batch, k_batch;
};

int flash_attn_run(const float* f, const float* g, const float* h, const FlashPrepacked* pre, float* out, int64_t b, int64_t lc,
                   int64_t ls, int passes, void* workspace, size_t workspace_bytes, cudaStream_t st) {
    const bool x3 = passes == 3;
    int64_t kb_max = b;
    while (kb_max > 1 && flash_attn_workspace_bytes(lc, ls, kb_max) > workspace_bytes) --kb_max;
    if (flash_attn_workspace_bytes(lc, ls, kb_max) > workspace_bytes) {
        set_error("flash attention: workspace too small (%zu < %zu bytes)", workspace_bytes, flash_attn_workspace_bytes(lc, ls, 1));
        return RPST_ERR_WORKSPACE;
    }
    const FlashLayout l = flash_layout(lc, ls, kb_max);
    char* w = static_cast<char*>(workspace);
    static PerDeviceFlag configured_on;
    bool& configured = configured_on.get();
    if (!configured) {
        RPST_CUDA(cudaFuncSetAttribute(flash_attn_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FlashCfg<false>::smem));
        RPST_CUDA(cudaFuncSetAttribute(flash_attn_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FlashCfg<true>::smem));
        configured = true;
    }
    for (int64_t i = 0; i < b; i += kb_max) {
        const int kb = (int)(b - i < kb_max ? b - i : kb_max);
        char* q_hi = w + l.header;
        char* q_lo = q_hi + (size_t)kb_max * l.q_b;
        char* k_hi = q_lo + (size_t)kb_max * l.q_b;
        char* k_lo = k_hi + (size_t)kb_max * l.k_b;
        char* vt = k_lo + (size_t)kb_max * l.k_b;
        const float* hi_ = h + i * kFlD * ls;
        int rc;
        if (!pre) {
            const float* fi = f + i * kFlD * lc;
            const float* gi = g + i * kFlD * ls;
            // Q = F^T and K = G^T: rows = positions (unit stride in the source), K = channels
            if ((rc = pack_operand_batched(fi, lc, kFlD, 1, lc, nullptr, nullptr, q_hi, x3 ? q_lo : nullptr, kb, kFlD * lc,
                                           (int64_t)l.q_b, 0, st))) return rc;
            if ((rc = pack_operand_batched(gi, ls, kFlD, 1, ls, nullptr, nullptr, k_hi, x3 ? k_lo : nullptr, kb, kFlD * ls,
                                           (int64_t)l.k_b, 0, st))) return rc;
        }
        float* unscale = nullptr;
        if (x3) {
            // V as IEEE half, pre-scaled by a per-sample power of two (exact) so that it cannot overflow
            unsigned int* amax = reinterpret_cast<unsigned int*>(w + l.absmax);
            float* row_scale = reinterpret_cast<float*>(w + l.row_scale);
            unscale = reinterpret_cast<float*>(w + l.unscale);
            RPST_CUDA(cudaMemsetAsync(amax, 0, (size_t)kb * sizeof(unsigned int), st));
            absmax_kernel<<<dim3((unsigned)(8 * sm_count()), (unsigned)kb), 256, 0, st>>>(hi_, kFlD * ls, amax);   // 64 blocks took 80 us per 32 MB
            RPST_CUDA(cudaGetLastError());
            scale_fill_kernel<<<(unsigned)((kb * kFlD + 255) / 256), 256, 0, st>>>(amax, kb, kFlD, row_scale, unscale);
            RPST_CUDA(cudaGetLastError());
            if ((rc = pack_operand_batched_f16(hi_, kFlD, ls, ls, 1, row_scale, vt, kb, kFlD * ls, (int64_t)l.v_b, kFlD, st))) return rc;
        } else {
            if ((rc = pack_operand_batched(hi_, kFlD, ls, ls, 1, nullptr, nullptr, vt, nullptr, kb, kFlD * ls, (int64_t)l.v_b, 0, st))) return rc;
        }
        FlashParams p{};
        if (pre) {
            p.q_hi = pre->q_hi + i * pre->q_batch; p.q_lo = pre->q_lo ? pre->q_lo + i * pre->q_batch : nullptr;
            p.k_hi = pre->k_hi + i * pre->k_batch; p.k_lo = pre->k_lo ? pre->k_lo + i * pre->k_batch : nullptr;
            p.q_batch = pre->q_batch; p.k_batch = pre->k_batch;
        } else {
            p.q_hi = q_hi; p.q_lo = q_lo; p.k_hi = k_hi; p.k_lo = k_lo;
            p.q_batch = (int64_t)l.q_b; p.k_batch = (int64_t)l.k_b;
        }
        p.v = vt;
        p.v_batch = (int64_t)l.v_b;
        p.v_unscale = unscale;
        p.out = out + i * kFlD * lc;
        p.lc = (int)lc; p.ls = (int)ls;
        p.qtiles = (int)(lc / 128); p.ktiles = (int)(ls / kFlKeys);
        p.items = kb * p.qtiles;
        p.prof = reinterpret_cast<unsigned long long*>(g_knobs.attn_flash_prof);
        int pairs = sm_count() / 2;
        if (pairs > p.items) pairs = p.items;
        if (x3) flash_attn_kernel<true><<<2 * pairs, kFlThreads, FlashCfg<true>::smem, st>>>(p);
        else flash_attn_kernel<false><<<2 * pairs, kFlThreads, FlashCfg<false>::smem, st>>>(p);
        RPST_CUDA(cudaGetLastError());
    }
    return RPST_OK;
}

int flash_attn_fwd(const float* f, const float* g, const float* h, float* out, int64_t b, int64_t lc, int64_t ls,
                   int passes, void* workspace, size_t workspace_bytes, cudaStream_t st) {
    return flash_attn_run(f, g, h, nullptr, out, b, lc, ls, passes, workspace, workspace_bytes, st);
}

}  // namespace rpst

using namespace rpst;

/* Attention core with Q / K already packed (rpst_conv1x1 with out_hi / out_lo): q tiles [b][lc x 512], k tiles
 * [b][ls x 512], sample strides = align_up(packed_operand_bytes(l, 512), 256); h fp32 [b,512,ls] -> out [b,512,lc]. */
extern "C" size_t rpst_sanet_attn_packed_workspace_bytes(int64_t b, int64_t lc, int64_t ls) {
    if (b <= 0 || lc <= 0 || ls <= 0) return 256;
    return flash_attn_workspace_bytes(lc, ls, b);
}

extern "C" int rpst_sanet_attn_fwd_packed(const void* q_hi, const void* q_lo, const void* k_hi, const void* k_lo, const float* h,
                                          float* out, int64_t b, int64_t c, int64_t lc, int64_t ls, int passes, void* workspace,
                                          size_t workspace_bytes, void* stream) {
    RPST_CHECK_ARG(b >= 0, "sanet_packed: negative batch");
    if (b == 0) return RPST_OK;
    RPST_CHECK_ARG(flash_attn_supported(c, lc, ls), "sanet_packed: needs C = 512, Lc %% 128 == 0, Ls %% 256 == 0");
    RPST_CHECK_ARG(q_hi && k_hi && h && out && workspace, "sanet_packed: null pointer");
    RPST_CHECK_ARG(passes == 1 || (passes == 3 && q_lo && k_lo), "sanet_packed: passes must be 1, or 3 with the lo tiles");
    RPST_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, "sanet_packed: workspace must be 256-byte aligned");
    FlashPrepacked pre{};
    pre.q_hi = static_cast<const char*>(q_hi); pre.q_lo = static_cast<const char*>(q_lo);
    pre.k_hi = static_cast<const char*>(k_hi); pre.k_lo = static_cast<const char*>(k_lo);
    pre.q_batch = (int64_t)align_up(packed_operand_bytes(lc, 512), 256);
    pre.k_batch = (int64_t)align_up(packed_operand_bytes(ls, 512), 256);
    return flash_attn_run(nullptr, nullptr, h, &pre, out, b, lc, ls, passes, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

RPST_WATCHDOG_SETTER(flash)
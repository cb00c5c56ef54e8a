// SANet attention core, static and adaptive — SURVEY.md §8 a9/a11; reference: network/sanet.py:82-99
// (`SANet.forward`), :12-18 (`cal_affinity_matrix`), :41-46 / :66-71 (AEA clamps), :114-138
// (`AdaptiveSANet.forward`).  The 1x1 convolutions f/g/h/out_conv stay in cuDNN; this file owns
//   S = F^T G            [Lc,Ls]   tensor cores (tcgen05, packed bf16 / bf16x3 operands)
//   P = softmax_j(S)               one CTA per row; emits P directly as packed bf16 hi/lo operand tiles
//   O = H P^T            [C,Lc]    tensor cores, written in the [C, Lc] layout the module returns
// and for the adaptive variants the cosine affinity, the f_psi MLP (its Linear(L -> L/16) is a
// tensor-core GEMM with a bias epilogue) and the clamped attention
//   'aea' : P' = sigmoid(scale * (P - clamp_i)),  clamp_i = sigmoid(mlp_i) * interval + from   (not renormalised)
//   'relu': P' = softmax_j(relu(P - clamp_i)),    clamp_i = (tanh(mlp_i) + 1) / 2
// Softmax is over the STYLE axis without temperature (network/sanet.py:79,90-91).
#include "common.cuh"
#include "tuning.cuh"
#include "umma.cuh"

namespace rpst {

size_t packed_operand_bytes(int64_t rows, int64_t k);
int pack_operand_shift(const float* x, int64_t rows, int64_t k, int64_t stride_r, int64_t stride_k,
                       const float* row_scale, const float* row_shift, void* hi, void* lo, cudaStream_t stream);
int gemm_packed_to_tiles(const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo, int64_t m, int64_t n, int64_t k,
                         int passes, float alpha, void* out_hi, void* out_lo, cudaStream_t stream);
int gemm_packed_splitk(const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo, float* out, int64_t m,
                       int64_t n, int64_t k, int64_t ldo, int passes, float alpha, const float* row_add,
                       const float* col_add, int splits, int64_t split_stride, cudaStream_t stream);
int pack_operand_batched(const float* x, int64_t rows, int64_t k, int64_t stride_r, int64_t stride_k,
                         const float* row_scale, const float* row_shift, void* hi, void* lo, int batch, int64_t x_batch,
                         int64_t tile_batch_bytes, int64_t vec_batch, cudaStream_t stream);
int gemm_packed_batched(const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo, float* out, int64_t m,
                        int64_t n, int64_t k, int64_t ldo, int passes, float alpha, const float* row_add,
                        const float* col_add, int splits, int64_t split_stride, int batch, int64_t a_batch_bytes,
                        int64_t b_batch_bytes, int64_t out_batch, cudaStream_t stream);
int channel_norms(const float* x, int64_t c, int64_t l, float* sq, float* nrm, float* inv, cudaStream_t st);
// flash.cu: single-kernel attention for C = 512 (S and P never leave the SM)
bool flash_attn_supported(int64_t c, int64_t lc, int64_t ls);
size_t flash_attn_workspace_bytes(int64_t lc, int64_t ls, int64_t samples);
int flash_attn_fwd(const float* f, const float* g, const float* h, float* out, int64_t b, int64_t lc, int64_t ls,
                   int passes, void* workspace, size_t workspace_bytes, cudaStream_t st);

namespace {

constexpr int kRowThreads = 256;

__device__ __forceinline__ float block_max(float v, float* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float r = red[0];
#pragma unroll
    for (int w = 1; w < kRowThreads / 32; ++w) r = fmaxf(r, red[w]);
    __syncthreads();
    return r;
}
__device__ __forceinline__ float block_sum(float v, float* red) {
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float r = red[0];
#pragma unroll
    for (int w = 1; w < kRowThreads / 32; ++w) r += red[w];
    __syncthreads();
    return r;
}

struct RowParams {
    const float* in;      // [rows, cols]
    float* out32;         // [rows, cols] or null (may alias `in`)
    __nv_bfloat16* hi;    // packed [rows x cols(K)] tiles or null
    __nv_bfloat16* lo;    // or null
    const float* clamp;   // [rows] (modes 1, 2)
    int64_t rows, cols;
    int k_tiles;          // ceil(cols / 64)
    int mode;             // 0 softmax(x); 1 sigmoid(scale*(x-clamp)); 2 softmax(relu(x-clamp))
    float scale;
    int pre;              // 1: the input row goes through softmax first (modes 1, 2 then act on the probabilities):
                          //    softmax + clamp of the adaptive attention in ONE pass over the L x L logits
    // blockIdx.y = sample of a group: element strides of in/out32 and clamp, byte stride of the tile buffers
    int64_t in_batch, out_batch, clamp_batch, tile_batch_bytes;
};

// One CTA per row; the row (<= 64 KiB) is re-read from L1/L2 between the passes.
__global__ void __launch_bounds__(kRowThreads) attn_rows_kernel(RowParams p) {
    __shared__ float red[kRowThreads / 32];
    const int64_t row = blockIdx.x;
    const int64_t bi = blockIdx.y;
    const float* x = p.in + bi * p.in_batch + row * p.cols;
    if (p.out32) p.out32 += bi * p.out_batch;
    if (p.hi) p.hi = reinterpret_cast<__nv_bfloat16*>(reinterpret_cast<char*>(p.hi) + bi * p.tile_batch_bytes);
    if (p.lo) p.lo = reinterpret_cast<__nv_bfloat16*>(reinterpret_cast<char*>(p.lo) + bi * p.tile_batch_bytes);
    const float cl = p.clamp ? __ldg(p.clamp + bi * p.clamp_batch + row) : 0.f;
    float mx0 = 0.f, inv0 = 1.f;           // first softmax (pre)
    if (p.pre) {
        float m = -INFINITY;
        for (int64_t j = threadIdx.x; j < p.cols; j += kRowThreads) m = fmaxf(m, x[j]);
        mx0 = block_max(m, red);
        float s = 0.f;
        for (int64_t j = threadIdx.x; j < p.cols; j += kRowThreads) s += expf(x[j] - mx0);
        inv0 = 1.f / block_sum(s, red);
    }
    auto load = [&](int64_t j) { const float v = x[j]; return p.pre ? expf(v - mx0) * inv0 : v; };
    float mx = 0.f, inv_sum = 1.f;
    if (p.mode != 1) {
        float m = -INFINITY;
        for (int64_t j = threadIdx.x; j < p.cols; j += kRowThreads) {
            float v = load(j);
            if (p.mode == 2) v = fmaxf(v - cl, 0.f);
            m = fmaxf(m, v);
        }
        mx = block_max(m, red);
        float s = 0.f;
        for (int64_t j = threadIdx.x; j < p.cols; j += kRowThreads) {
            float v = load(j);
            if (p.mode == 2) v = fmaxf(v - cl, 0.f);
            s += expf(v - mx);
        }
        inv_sum = 1.f / block_sum(s, red);
    }
    const int64_t chunks = (p.cols + 7) / 8;
    const int64_t rb = row / kTileRows;
    const int r = (int)(row % kTileRows);
    for (int64_t q = threadIdx.x; q < chunks; q += kRowThreads) {
        float y[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int64_t j = q * 8 + e;
            float v = 0.f;
            if (j < p.cols) {
                v = load(j);
                if (p.mode == 0) v = expf(v - mx) * inv_sum;
                else if (p.mode == 1) v = 1.f / (1.f + expf(-p.scale * (v - cl)));
                else v = expf(fmaxf(v - cl, 0.f) - mx) * inv_sum;
            }
            y[e] = v;
        }
        if (p.out32) {
#pragma unroll
            for (int e = 0; e < 8; ++e)
                if (q * 8 + e < p.cols) p.out32[row * p.cols + q * 8 + e] = y[e];
        }
        if (p.hi) {
            __align__(16) __nv_bfloat16 h[8];
            __align__(16) __nv_bfloat16 l[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) split_bf16(y[e], h[e], l[e]);
            const int64_t tile = rb * p.k_tiles + (q >> 3);
            const size_t off = (size_t)tile * kTileBytes + tile_chunk_offset(r, (int)(q & 7));
            *reinterpret_cast<uint4*>(reinterpret_cast<char*>(p.hi) + off) = *reinterpret_cast<const uint4*>(h);
            if (p.lo) *reinterpret_cast<uint4*>(reinterpret_cast<char*>(p.lo) + off) = *reinterpret_cast<const uint4*>(l);
        }
    }
}

// Register-resident variant for rows of up to 16384 columns (cols % 4 == 0, 16-byte aligned rows): the row is
// read ONCE with 128-bit loads and stays in registers through max / sum / write (the generic kernel above
// re-reads it three times with 32-bit loads: 483 us per 16384^2 map vs ~1/3 less here).  A thread holds
// float4 #(j*256 + tid); two neighbouring float4 make one 16-byte packed chunk, each thread stores its half.
constexpr int kRowRegVecs = 16;
__global__ void __launch_bounds__(kRowThreads) attn_rows_reg_kernel(RowParams p) {
    __shared__ float red[kRowThreads / 32];
    const int64_t row = blockIdx.x;
    const int64_t bi = blockIdx.y;
    const float4* x4 = reinterpret_cast<const float4*>(p.in + bi * p.in_batch + row * p.cols);
    const int nvec = (int)(p.cols / 4);
    const float cl = p.clamp ? __ldg(p.clamp + bi * p.clamp_batch + row) : 0.f;
    float4 v[kRowRegVecs];
#pragma unroll
    for (int j = 0; j < kRowRegVecs; ++j) {
        const int idx = j * kRowThreads + threadIdx.x;
        if (idx < nvec) v[j] = __ldcs(x4 + idx);
    }
    if (p.pre) {                           // probabilities first, still in registers
        float m = -INFINITY;
#pragma unroll
        for (int j = 0; j < kRowRegVecs; ++j)
            if (j * kRowThreads + (int)threadIdx.x < nvec) m = fmaxf(m, fmaxf(fmaxf(v[j].x, v[j].y), fmaxf(v[j].z, v[j].w)));
        const float mx0 = block_max(m, red);
        float sum = 0.f;
#pragma unroll
        for (int j = 0; j < kRowRegVecs; ++j) {
            if (j * kRowThreads + (int)threadIdx.x < nvec) {
                v[j].x = expf(v[j].x - mx0); v[j].y = expf(v[j].y - mx0);
                v[j].z = expf(v[j].z - mx0); v[j].w = expf(v[j].w - mx0);
                sum += (v[j].x + v[j].y) + (v[j].z + v[j].w);
            }
        }
        const float inv0 = 1.f / block_sum(sum, red);
#pragma unroll
        for (int j = 0; j < kRowRegVecs; ++j) { v[j].x *= inv0; v[j].y *= inv0; v[j].z *= inv0; v[j].w *= inv0; }
    }
    float mx = 0.f, inv_sum = 1.f;
    if (p.mode != 1) {
        float m = -INFINITY;
#pragma unroll
        for (int j = 0; j < kRowRegVecs; ++j) {
            if (j * kRowThreads + (int)threadIdx.x < nvec) {
                if (p.mode == 2) {
                    v[j].x = fmaxf(v[j].x - cl, 0.f); v[j].y = fmaxf(v[j].y - cl, 0.f);
                    v[j].z = fmaxf(v[j].z - cl, 0.f); v[j].w = fmaxf(v[j].w - cl, 0.f);
                }
                m = fmaxf(m, fmaxf(fmaxf(v[j].x, v[j].y), fmaxf(v[j].z, v[j].w)));
            }
        }
        mx = block_max(m, red);
        float sum = 0.f;
#pragma unroll
        for (int j = 0; j < kRowRegVecs; ++j) {
            if (j * kRowThreads + (int)threadIdx.x < nvec) {
                v[j].x = expf(v[j].x - mx); v[j].y = expf(v[j].y - mx);
                v[j].z = expf(v[j].z - mx); v[j].w = expf(v[j].w - mx);
                sum += (v[j].x + v[j].y) + (v[j].z + v[j].w);
            }
        }
        inv_sum = 1.f / block_sum(sum, red);
    }
    float4* o4 = p.out32 ? reinterpret_cast<float4*>(p.out32 + bi * p.out_batch + row * p.cols) : nullptr;
    char* hi = p.hi ? reinterpret_cast<char*>(p.hi) + bi * p.tile_batch_bytes : nullptr;
    char* lo = p.lo ? reinterpret_cast<char*>(p.lo) + bi * p.tile_batch_bytes : nullptr;
    const int64_t rb = row / kTileRows;
    const int r = (int)(row % kTileRows);
#pragma unroll
    for (int j = 0; j < kRowRegVecs; ++j) {
        const int idx = j * kRowThreads + threadIdx.x;
        if (idx < nvec) {
            float4 y = v[j];
            if (p.mode == 1) {
                y.x = 1.f / (1.f + expf(-p.scale * (y.x - cl))); y.y = 1.f / (1.f + expf(-p.scale * (y.y - cl)));
                y.z = 1.f / (1.f + expf(-p.scale * (y.z - cl))); y.w = 1.f / (1.f + expf(-p.scale * (y.w - cl)));
            } else {
                y.x *= inv_sum; y.y *= inv_sum; y.z *= inv_sum; y.w *= inv_sum;
            }
            if (o4) o4[idx] = y;
            if (hi) {
                __align__(8) __nv_bfloat16 h[4];
                __align__(8) __nv_bfloat16 l[4];
                split_bf16(y.x, h[0], l[0]); split_bf16(y.y, h[1], l[1]);
                split_bf16(y.z, h[2], l[2]); split_bf16(y.w, h[3], l[3]);
                const int q = idx >> 1;    // 16-byte chunk (8 columns) this float4 belongs to
                const size_t off = (size_t)(rb * p.k_tiles + (q >> 3)) * kTileBytes + tile_chunk_offset(r, q & 7) + (idx & 1) * 8;
                *reinterpret_cast<uint2*>(hi + off) = *reinterpret_cast<const uint2*>(h);
                if (lo) *reinterpret_cast<uint2*>(lo + off) = *reinterpret_cast<const uint2*>(l);
            }
        }
    }
}

// f_psi head: z_i = sum_h leaky_relu(hidden[i,h], 0.2) * w2[h] + b2 ; clamp per mode. One warp per row.
__global__ void __launch_bounds__(256) psi_head_kernel(const float* __restrict__ hidden, const float* __restrict__ w2,
                                                       const float* __restrict__ b2, int64_t rows, int64_t lh, int mode,
                                                       float from_value, float value_interval, float* __restrict__ clamp) {
    const int lane = threadIdx.x & 31;
    const int64_t row = blockIdx.x * (int64_t)(blockDim.x / 32) + (threadIdx.x >> 5);
    if (row >= rows) return;
    float acc = 0.f;
    for (int64_t h = lane; h < lh; h += 32) {
        float v = hidden[row * lh + h];
        v = v >= 0.f ? v : 0.2f * v;
        acc = fmaf(v, __ldg(w2 + h), acc);
    }
    acc = warp_sum(acc) + __ldg(b2);
    if (lane == 0)
        clamp[row] = mode == 1 ? (1.f / (1.f + expf(-acc))) * value_interval + from_value : (tanhf(acc) + 1.f) * 0.5f;
}

// Workspace of one GROUP of `kb` samples processed by the same launches: every buffer holds kb
// consecutive per-sample slices (byte strides *_b), so total(kb) = kb * total(1) and a caller that passes
// a multiple of the per-sample size gets that many samples per launch.
struct AttnLayout {
    size_t q_hi, q_lo, k_hi, k_lo, v_hi, v_lo, s, p_hi, p_lo, total;
    size_t q_b, k_b, v_b, s_b, p_b;
};
AttnLayout attn_layout(int64_t c, int64_t lc, int64_t ls, int64_t kb = 1) {
    AttnLayout l;
    size_t o = 0;
    auto take = [&](size_t stride) { size_t at = o; o += stride * (size_t)kb; return at; };
    l.q_b = align_up(packed_operand_bytes(lc, c), 256);
    l.k_b = align_up(packed_operand_bytes(ls, c), 256);
    l.v_b = align_up(packed_operand_bytes(c, ls), 256);
    l.s_b = align_up((size_t)lc * ls * sizeof(float), 256);
    l.p_b = align_up(packed_operand_bytes(lc, ls), 256);
    l.q_hi = take(l.q_b); l.q_lo = take(l.q_b);
    l.k_hi = take(l.k_b); l.k_lo = take(l.k_b);
    l.v_hi = take(l.v_b); l.v_lo = take(l.v_b);
    l.s = take(l.s_b);
    l.p_hi = take(l.p_b); l.p_lo = take(l.p_b);
    l.total = o;
    return l;
}

// Backward of the row softmax: dS = P o (dP - sum_j dP o P).  One CTA per row; P and dP rows are read
// twice (second time from L1/L2); dS overwrites dP in fp32 and is emitted as packed operand tiles.
__global__ void __launch_bounds__(kRowThreads) attn_bwd_rows_kernel(const float* __restrict__ prob, float* dp,
                                                                     __nv_bfloat16* hi, __nv_bfloat16* lo,
                                                                     int64_t cols, int k_tiles, int64_t mat_batch,
                                                                     int64_t tile_batch_bytes) {
    __shared__ float red[kRowThreads / 32];
    const int64_t row = blockIdx.x;
    const int64_t bi = blockIdx.y;
    hi = reinterpret_cast<__nv_bfloat16*>(reinterpret_cast<char*>(hi) + bi * tile_batch_bytes);
    if (lo) lo = reinterpret_cast<__nv_bfloat16*>(reinterpret_cast<char*>(lo) + bi * tile_batch_bytes);
    const float* pr = prob + bi * mat_batch + row * cols;
    float* dr = dp + bi * mat_batch + row * cols;
    float acc = 0.f;
    for (int64_t j = threadIdx.x; j < cols; j += kRowThreads) acc = fmaf(pr[j], dr[j], acc);
    const float delta = block_sum(acc, red);
    const int64_t chunks = (cols + 7) / 8;
    const int64_t rb = row / kTileRows;
    const int r = (int)(row % kTileRows);
    for (int64_t q = threadIdx.x; q < chunks; q += kRowThreads) {
        float y[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int64_t j = q * 8 + e;
            y[e] = j < cols ? pr[j] * (dr[j] - delta) : 0.f;
        }
#pragma unroll
        for (int e = 0; e < 8; ++e)
            if (q * 8 + e < cols) dr[q * 8 + e] = y[e];
        __align__(16) __nv_bfloat16 h[8];
        __align__(16) __nv_bfloat16 l[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) split_bf16(y[e], h[e], l[e]);
        const int64_t tile = rb * k_tiles + (q >> 3);
        const size_t off = (size_t)tile * kTileBytes + tile_chunk_offset(r, (int)(q & 7));
        *reinterpret_cast<uint4*>(reinterpret_cast<char*>(hi) + off) = *reinterpret_cast<const uint4*>(h);
        if (lo) *reinterpret_cast<uint4*>(reinterpret_cast<char*>(lo) + off) = *reinterpret_cast<const uint4*>(l);
    }
}

// register-resident variant (see attn_rows_reg_kernel): P and dP rows are read once with 128-bit loads
__global__ void __launch_bounds__(kRowThreads) attn_bwd_rows_reg_kernel(const float* __restrict__ prob, float* dp,
                                                                         __nv_bfloat16* hi, __nv_bfloat16* lo,
                                                                         int64_t cols, int k_tiles, int64_t mat_batch,
                                                                         int64_t tile_batch_bytes) {
    __shared__ float red[kRowThreads / 32];
    const int64_t row = blockIdx.x;
    const int64_t bi = blockIdx.y;
    char* hib = reinterpret_cast<char*>(hi) + bi * tile_batch_bytes;
    char* lob = lo ? reinterpret_cast<char*>(lo) + bi * tile_batch_bytes : nullptr;
    const float4* p4 = reinterpret_cast<const float4*>(prob + bi * mat_batch + row * cols);
    float4* d4 = reinterpret_cast<float4*>(dp + bi * mat_batch + row * cols);
    const int nvec = (int)(cols / 4);
    float4 pv[kRowRegVecs], dv[kRowRegVecs];
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < kRowRegVecs; ++j) {
        const int idx = j * kRowThreads + threadIdx.x;
        if (idx < nvec) {
            pv[j] = __ldcs(p4 + idx);
            dv[j] = d4[idx];
            acc = fmaf(pv[j].x, dv[j].x, acc); acc = fmaf(pv[j].y, dv[j].y, acc);
            acc = fmaf(pv[j].z, dv[j].z, acc); acc = fmaf(pv[j].w, dv[j].w, acc);
        }
    }
    const float delta = block_sum(acc, red);
    const int64_t rb = row / kTileRows;
    const int r = (int)(row % kTileRows);
#pragma unroll
    for (int j = 0; j < kRowRegVecs; ++j) {
        const int idx = j * kRowThreads + threadIdx.x;
        if (idx < nvec) {
            float4 y;
            y.x = pv[j].x * (dv[j].x - delta); y.y = pv[j].y * (dv[j].y - delta);
            y.z = pv[j].z * (dv[j].z - delta); y.w = pv[j].w * (dv[j].w - delta);
            d4[idx] = y;
            __align__(8) __nv_bfloat16 h[4];
            __align__(8) __nv_bfloat16 l[4];
            split_bf16(y.x, h[0], l[0]); split_bf16(y.y, h[1], l[1]);
            split_bf16(y.z, h[2], l[2]); split_bf16(y.w, h[3], l[3]);
            const int q = idx >> 1;
            const size_t off = (size_t)(rb * k_tiles + (q >> 3)) * kTileBytes + tile_chunk_offset(r, q & 7) + (idx & 1) * 8;
            *reinterpret_cast<uint2*>(hib + off) = *reinterpret_cast<const uint2*>(h);
            if (lob) *reinterpret_cast<uint2*>(lob + off) = *reinterpret_cast<const uint2*>(l);
        }
    }
}

// Backward of one row of the CLAMPED attention (network/sanet.py:41-46 'aea', :66-71 'relu') fused with the
// softmax backward.  With U = P - cl (P = softmax row, cl = this row's clamp) and S' the forward result:
//   'aea' : S' = sigmoid(k U)           dU = dS' * k * S' (1 - S')
//   'relu': S' = softmax_j(relu(U))     dR = S' o (dS' - sum_j dS' S'),  dU = dR where U > 0 else 0
//   dcl = -sum_j dU_j ;   dS = P o (dU - sum_j dU P)      (P depends on S through the plain softmax)
// dS overwrites dS' in fp32 and is emitted as packed operand tiles; dcl goes to grad_clamp[row].
__global__ void __launch_bounds__(kRowThreads) attn_clamped_bwd_rows_kernel(const float* __restrict__ prob,
                                                                             const float* __restrict__ sp, float* dp,
                                                                             const float* __restrict__ clamp,
                                                                             float* __restrict__ grad_clamp, int mode, float scale,
                                                                             __nv_bfloat16* hi, __nv_bfloat16* lo, int64_t cols,
                                                                             int k_tiles) {
    __shared__ float red[kRowThreads / 32];
    const int64_t row = blockIdx.x;
    const float* pr = prob + row * cols;
    const float* sr = sp + row * cols;
    float* dr = dp + row * cols;
    const float cl = __ldg(clamp + row);
    float delta1 = 0.f;
    if (mode == 2) {
        float a = 0.f;
        for (int64_t j = threadIdx.x; j < cols; j += kRowThreads) a = fmaf(dr[j], sr[j], a);
        delta1 = block_sum(a, red);
    }
    auto d_u = [&](int64_t j) -> float {
        const float s = sr[j];
        if (mode == 1) return dr[j] * scale * s * (1.f - s);
        return pr[j] - cl > 0.f ? s * (dr[j] - delta1) : 0.f;
    };
    float a1 = 0.f, a2 = 0.f;
    for (int64_t j = threadIdx.x; j < cols; j += kRowThreads) {
        const float du = d_u(j);
        a1 += du;
        a2 = fmaf(du, pr[j], a2);
    }
    const float sum_du = block_sum(a1, red);
    const float delta2 = block_sum(a2, red);
    if (threadIdx.x == 0) grad_clamp[row] = -sum_du;
    const int64_t chunks = (cols + 7) / 8;
    const int64_t rb = row / kTileRows;
    const int r = (int)(row % kTileRows);
    for (int64_t q = threadIdx.x; q < chunks; q += kRowThreads) {
        float y[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int64_t j = q * 8 + e;
            y[e] = j < cols ? pr[j] * (d_u(j) - delta2) : 0.f;
        }
#pragma unroll
        for (int e = 0; e < 8; ++e)
            if (q * 8 + e < cols) dr[q * 8 + e] = y[e];
        __align__(16) __nv_bfloat16 h[8];
        __align__(16) __nv_bfloat16 l[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) split_bf16(y[e], h[e], l[e]);
        const size_t off = (size_t)(rb * k_tiles + (q >> 3)) * kTileBytes + tile_chunk_offset(r, (int)(q & 7));
        *reinterpret_cast<uint4*>(reinterpret_cast<char*>(hi) + off) = *reinterpret_cast<const uint4*>(h);
        if (lo) *reinterpret_cast<uint4*>(reinterpret_cast<char*>(lo) + off) = *reinterpret_cast<const uint4*>(l);
    }
}

// workspace of the backward pass: the forward's buffers (Q/K/V tiles, S) plus dP and two L x L tile sets
struct AttnBwdLayout {
    AttnLayout a;            // q: [lc x c] tiles, k: [ls x c], v: [c x ls], s: P (fp32), p: [lc x ls] tiles (dS)
    size_t dp, t_hi, t_lo, w_hi, w_lo, total;   // dP/dS fp32; [ls x lc] tiles (P^T, dS^T); [c x lc] tiles (dO, F)
    size_t t_b, w_b;
};
AttnBwdLayout attn_bwd_layout(int64_t c, int64_t lc, int64_t ls, int64_t kb = 1) {
    AttnBwdLayout l;
    l.a = attn_layout(c, lc, ls, kb);
    size_t o = l.a.total;
    auto take = [&](size_t stride) { size_t at = o; o += stride * (size_t)kb; return at; };
    l.t_b = align_up(packed_operand_bytes(ls, lc), 256);
    l.w_b = align_up(packed_operand_bytes(c, lc), 256);
    l.dp = take(l.a.s_b);
    l.t_hi = take(l.t_b); l.t_lo = take(l.t_b);
    l.w_hi = take(l.w_b); l.w_lo = take(l.w_b);
    l.total = o;
    return l;
}

struct AdaLayout {
    AttnLayout a;
    size_t aff, w_hi, w_lo, hidden, clamp, vec[6], total;
};
AdaLayout ada_layout(int64_t c, int64_t lc, int64_t ls, int64_t lh) {
    AdaLayout l;
    l.a = attn_layout(c, lc, ls);
    size_t o = l.a.total;
    auto take = [&](size_t bytes) { size_t at = o; o += align_up(bytes, 256); return at; };
    l.aff = take((size_t)lc * ls * sizeof(float));
    l.w_hi = take(packed_operand_bytes(lh, ls)); l.w_lo = take(packed_operand_bytes(lh, ls));
    l.hidden = take((size_t)lc * lh * sizeof(float));
    l.clamp = take((size_t)lc * sizeof(float));
    for (int i = 0; i < 6; ++i) l.vec[i] = take((size_t)(lc > ls ? lc : ls) * sizeof(float));
    l.total = o;
    return l;
}

int launch_rows(const float* in, float* out32, void* hi, void* lo, const float* clamp, int64_t rows, int64_t cols,
                int mode, float scale, cudaStream_t st, int kb = 1, int64_t in_batch = 0, int64_t out_batch = 0,
                int64_t tile_batch_bytes = 0, int64_t clamp_batch = 0, int pre = 0) {
    RowParams p{};
    p.pre = pre;
    p.in = in; p.out32 = out32; p.hi = static_cast<__nv_bfloat16*>(hi); p.lo = static_cast<__nv_bfloat16*>(lo);
    p.clamp = clamp; p.rows = rows; p.cols = cols; p.k_tiles = (int)((cols + kTileK - 1) / kTileK);
    p.mode = mode; p.scale = scale;
    p.in_batch = in_batch; p.out_batch = out_batch; p.tile_batch_bytes = tile_batch_bytes; p.clamp_batch = clamp_batch;
    if (hi && (rows % kTileRows != 0 || cols % kTileK != 0)) {   // zero padding of the partial tiles
        const size_t span = kb > 1 ? (size_t)tile_batch_bytes * kb : packed_operand_bytes(rows, cols);
        RPST_CUDA(cudaMemsetAsync(hi, 0, span, st));
        if (lo) RPST_CUDA(cudaMemsetAsync(lo, 0, span, st));
    }
    // long rows only: at 4096 columns and below the generic kernel's re-reads hit L1 and it measured faster
    const bool reg_path = cols >= 8192 && cols % 4 == 0 && cols / 4 <= (int64_t)kRowRegVecs * kRowThreads && in_batch % 4 == 0 &&
                          out_batch % 4 == 0 && (reinterpret_cast<uintptr_t>(in) & 15u) == 0 &&
                          (reinterpret_cast<uintptr_t>(out32) & 15u) == 0;
    if (reg_path) attn_rows_reg_kernel<<<dim3((unsigned)rows, (unsigned)kb), kRowThreads, 0, st>>>(p);
    else attn_rows_kernel<<<dim3((unsigned)rows, (unsigned)kb), kRowThreads, 0, st>>>(p);
    RPST_CUDA(cudaGetLastError());
    return RPST_OK;
}

// S = F^T G for a group of kb samples into `s` (sample stride s_batch elements)
int scores(const float* f, const float* g, int64_t c, int64_t lc, int64_t ls, int passes, char* w, const AttnLayout& l,
           float* s, cudaStream_t st, int kb = 1, int64_t s_batch = 0) {
    int rc = pack_operand_batched(f, lc, c, 1, lc, nullptr, nullptr, w + l.q_hi, passes == 3 ? w + l.q_lo : nullptr, kb,
                                  c * lc, (int64_t)l.q_b, 0, st);
    if (rc) return rc;
    rc = pack_operand_batched(g, ls, c, 1, ls, nullptr, nullptr, w + l.k_hi, passes == 3 ? w + l.k_lo : nullptr, kb,
                              c * ls, (int64_t)l.k_b, 0, st);
    if (rc) return rc;
    return gemm_packed_batched(w + l.q_hi, w + l.q_lo, w + l.k_hi, w + l.k_lo, s, lc, ls, c, ls, passes, 1.f, nullptr,
                               nullptr, 1, 0, kb, (int64_t)l.q_b, (int64_t)l.k_b, s_batch, st);
}

// O = H P^T for a group of kb samples (P already packed in the workspace)
int weighted_values(const float* h, int64_t c, int64_t lc, int64_t ls, int passes, char* w, const AttnLayout& l,
                    float* out, cudaStream_t st, int kb = 1) {
    int rc = pack_operand_batched(h, c, ls, ls, 1, nullptr, nullptr, w + l.v_hi, passes == 3 ? w + l.v_lo : nullptr, kb,
                                  c * ls, (int64_t)l.v_b, 0, st);
    if (rc) return rc;
    return gemm_packed_batched(w + l.v_hi, w + l.v_lo, w + l.p_hi, w + l.p_lo, out, c, lc, ls, lc, passes, 1.f, nullptr,
                               nullptr, 1, 0, kb, (int64_t)l.v_b, (int64_t)l.p_b, c * lc, st);
}

// samples per launch that fit the caller's workspace (a multiple of the per-sample size buys batching)
int64_t group_size(int64_t b, size_t workspace_bytes, size_t per_sample) {
    int64_t kb = (int64_t)(workspace_bytes / per_sample);
    if (kb > b) kb = b;
    if (kb > 4096) kb = 4096;
    return kb < 1 ? 1 : kb;
}

}  // namespace
}  // namespace rpst

using namespace rpst;

extern "C" size_t rpst_sanet_attn_workspace_bytes(int64_t c, int64_t lc, int64_t ls) {
    if (c <= 0 || lc <= 0 || ls <= 0) return 256;
    return attn_layout(c, lc, ls).total;
}

extern "C" int rpst_sanet_attn_fwd(const float* f, const float* g, const float* h, float* out, int64_t b, int64_t c,
                                   int64_t lc, int64_t ls, int passes, float* attn_out, void* workspace,
                                   size_t workspace_bytes, void* stream) {
    RPST_CHECK_ARG(b >= 0 && c >= 0 && lc >= 0 && ls >= 0, "sanet: negative size");
    if (b == 0 || c == 0 || lc == 0) return RPST_OK;
    RPST_CHECK_ARG(ls > 0, "sanet: empty style map");
    RPST_CHECK_ARG(f && g && h && out, "sanet: null pointer");
    RPST_CHECK_ARG(passes == 1 || passes == 3, "sanet: passes must be 1 (bf16) or 3 (bf16x3, fp32-grade)");
    const size_t per_sample = attn_layout(c, lc, ls).total;
    if (!workspace || workspace_bytes < per_sample) {
        set_error("sanet: workspace too small (%zu < %zu bytes)", workspace_bytes, per_sample);
        return RPST_ERR_WORKSPACE;
    }
    RPST_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, "sanet: workspace must be 256-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    char* w = static_cast<char*>(workspace);
    // C = 512 without a materialised attention map: one flash-style kernel (the per-sample workspace of the
    // three-kernel path below always covers what it needs: packed Q, K, V only)
    if (!attn_out && g_knobs.attn_flash && flash_attn_supported(c, lc, ls) && flash_attn_workspace_bytes(lc, ls, 1) <= workspace_bytes)
        return flash_attn_fwd(f, g, h, out, b, lc, ls, passes, workspace, workspace_bytes, st);
    const int64_t kb_max = group_size(b, workspace_bytes, per_sample);
    for (int64_t i = 0; i < b; i += kb_max) {
        const int kb = (int)(b - i < kb_max ? b - i : kb_max);
        const AttnLayout l = attn_layout(c, lc, ls, kb);
        float* s = attn_out ? attn_out + i * lc * ls : reinterpret_cast<float*>(w + l.s);
        const int64_t s_batch = attn_out ? lc * ls : (int64_t)(l.s_b / sizeof(float));
        int rc = scores(f + i * c * lc, g + i * c * ls, c, lc, ls, passes, w, l, s, st, kb, s_batch);
        if (rc) return rc;
        rc = launch_rows(s, attn_out ? s : nullptr, w + l.p_hi, passes == 3 ? w + l.p_lo : nullptr, nullptr, lc, ls, 0,
                         0.f, st, kb, s_batch, s_batch, (int64_t)l.p_b, 0);
        if (rc) return rc;
        rc = weighted_values(h + i * c * ls, c, lc, ls, passes, w, l, out + i * c * lc, st, kb);
        if (rc) return rc;
    }
    return RPST_OK;
}

extern "C" size_t rpst_sanet_attn_bwd_workspace_bytes(int64_t c, int64_t lc, int64_t ls) {
    if (c <= 0 || lc <= 0 || ls <= 0) return 256;
    return attn_bwd_layout(c, lc, ls).total;
}

// Backward of rpst_sanet_attn_fwd (SURVEY.md §8f rank 2).  With S = F^T G, P = softmax_j(S), O = H P^T:
//   dH = dO P          [C,Ls]      dP = dO^T H   [Lc,Ls]      dS = P o (dP - rowsum(dP o P))
//   dF = G dS^T        [C,Lc]      dG = F dS     [C,Ls]
// P is recomputed (one extra GEMM) instead of being kept from the forward: at L = 16384 it is 1 GiB per
// sample.  Five tcgen05 GEMMs + two row kernels per sample, all on the caller's stream.
extern "C" int rpst_sanet_attn_bwd(const float* f, const float* g, const float* h, const float* grad_out,
                                   float* grad_f, float* grad_g, float* grad_h, int64_t b, int64_t c, int64_t lc,
                                   int64_t ls, int passes, void* workspace, size_t workspace_bytes, void* stream) {
    RPST_CHECK_ARG(b >= 0 && c >= 0 && lc >= 0 && ls >= 0, "sanet_bwd: negative size");
    if (b == 0 || c == 0 || lc == 0) return RPST_OK;
    RPST_CHECK_ARG(ls > 0, "sanet_bwd: empty style map");
    RPST_CHECK_ARG(f && g && h && grad_out && grad_f && grad_g && grad_h, "sanet_bwd: null pointer");
    RPST_CHECK_ARG(passes == 1 || passes == 3, "sanet_bwd: passes must be 1 (bf16) or 3 (bf16x3, fp32-grade)");
    const size_t per_sample = attn_bwd_layout(c, lc, ls).total;
    if (!workspace || workspace_bytes < per_sample) {
        set_error("sanet_bwd: workspace too small (%zu < %zu bytes)", workspace_bytes, per_sample);
        return RPST_ERR_WORKSPACE;
    }
    RPST_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, "sanet_bwd: workspace must be 256-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    char* w = static_cast<char*>(workspace);
    const bool x3 = passes == 3;
    auto lo = [&](size_t off) -> void* { return x3 ? w + off : nullptr; };
    const int64_t kb_max = group_size(b, workspace_bytes, per_sample);
    int rc;
    for (int64_t i = 0; i < b; i += kb_max) {
        const int kb = (int)(b - i < kb_max ? b - i : kb_max);
        const AttnBwdLayout l = attn_bwd_layout(c, lc, ls, kb);
        const AttnLayout& a = l.a;
        float* prob = reinterpret_cast<float*>(w + a.s);
        float* dp = reinterpret_cast<float*>(w + l.dp);
        const int64_t mat = (int64_t)(a.s_b / sizeof(float));    // element stride of the per-sample L x L matrices
        const float* fi = f + i * c * lc;
        const float* gi = g + i * c * ls;
        const float* hi_ = h + i * c * ls;
        const float* doi = grad_out + i * c * lc;
        // 1. P = softmax(F^T G), kept in fp32
        if ((rc = scores(fi, gi, c, lc, ls, passes, w, a, prob, st, kb, mat))) return rc;
        if ((rc = launch_rows(prob, prob, nullptr, nullptr, nullptr, lc, ls, 0, 0.f, st, kb, mat, mat, 0, 0))) return rc;
        // 2. dH[c,j] = sum_i dO[c,i] P[i,j]:  A = dO (rows c, K = i), B = P^T (rows j, K = i)
        if ((rc = pack_operand_batched(doi, c, lc, lc, 1, nullptr, nullptr, w + l.w_hi, lo(l.w_lo), kb, c * lc, (int64_t)l.w_b, 0, st))) return rc;
        if ((rc = pack_operand_batched(prob, ls, lc, 1, ls, nullptr, nullptr, w + l.t_hi, lo(l.t_lo), kb, mat, (int64_t)l.t_b, 0, st))) return rc;
        if ((rc = gemm_packed_batched(w + l.w_hi, w + l.w_lo, w + l.t_hi, w + l.t_lo, grad_h + i * c * ls, c, ls, lc, ls,
                                      passes, 1.f, nullptr, nullptr, 1, 0, kb, (int64_t)l.w_b, (int64_t)l.t_b, c * ls, st))) return rc;
        // 3. dP[i,j] = sum_c dO[c,i] H[c,j]:  A = dO^T (rows i, K = c), B = H^T (rows j, K = c)
        if ((rc = pack_operand_batched(doi, lc, c, 1, lc, nullptr, nullptr, w + a.q_hi, lo(a.q_lo), kb, c * lc, (int64_t)a.q_b, 0, st))) return rc;
        if ((rc = pack_operand_batched(hi_, ls, c, 1, ls, nullptr, nullptr, w + a.k_hi, lo(a.k_lo), kb, c * ls, (int64_t)a.k_b, 0, st))) return rc;
        if ((rc = gemm_packed_batched(w + a.q_hi, w + a.q_lo, w + a.k_hi, w + a.k_lo, dp, lc, ls, c, ls, passes, 1.f,
                                      nullptr, nullptr, 1, 0, kb, (int64_t)a.q_b, (int64_t)a.k_b, mat, st))) return rc;
        // 4. dS = P o (dP - rowsum(dP o P)): fp32 in place of dP + operand tiles (rows i, K = j)
        if (lc % kTileRows != 0 || ls % kTileK != 0) {
            RPST_CUDA(cudaMemsetAsync(w + a.p_hi, 0, a.p_b * kb, st));
            if (x3) RPST_CUDA(cudaMemsetAsync(w + a.p_lo, 0, a.p_b * kb, st));
        }
        if (ls >= 8192 && ls % 4 == 0 && ls / 4 <= (int64_t)kRowRegVecs * kRowThreads)   // workspace matrices are 256-byte aligned
            attn_bwd_rows_reg_kernel<<<dim3((unsigned)lc, (unsigned)kb), kRowThreads, 0, st>>>(
                prob, dp, reinterpret_cast<__nv_bfloat16*>(w + a.p_hi), x3 ? reinterpret_cast<__nv_bfloat16*>(w + a.p_lo) : nullptr,
                ls, (int)((ls + kTileK - 1) / kTileK), mat, (int64_t)a.p_b);
        else
            attn_bwd_rows_kernel<<<dim3((unsigned)lc, (unsigned)kb), kRowThreads, 0, st>>>(
                prob, dp, reinterpret_cast<__nv_bfloat16*>(w + a.p_hi), x3 ? reinterpret_cast<__nv_bfloat16*>(w + a.p_lo) : nullptr,
                ls, (int)((ls + kTileK - 1) / kTileK), mat, (int64_t)a.p_b);
        RPST_CUDA(cudaGetLastError());
        // 5. dF[c,i] = sum_j G[c,j] dS[i,j]:  A = G (rows c, K = j), B = dS (rows i, K = j)
        if ((rc = pack_operand_batched(gi, c, ls, ls, 1, nullptr, nullptr, w + a.v_hi, lo(a.v_lo), kb, c * ls, (int64_t)a.v_b, 0, st))) return rc;
        if ((rc = gemm_packed_batched(w + a.v_hi, w + a.v_lo, w + a.p_hi, w + a.p_lo, grad_f + i * c * lc, c, lc, ls, lc,
                                      passes, 1.f, nullptr, nullptr, 1, 0, kb, (int64_t)a.v_b, (int64_t)a.p_b, c * lc, st))) return rc;
        // 6. dG[c,j] = sum_i F[c,i] dS[i,j]:  A = F (rows c, K = i), B = dS^T (rows j, K = i)
        if ((rc = pack_operand_batched(fi, c, lc, lc, 1, nullptr, nullptr, w + l.w_hi, lo(l.w_lo), kb, c * lc, (int64_t)l.w_b, 0, st))) return rc;
        if ((rc = pack_operand_batched(dp, ls, lc, 1, ls, nullptr, nullptr, w + l.t_hi, lo(l.t_lo), kb, mat, (int64_t)l.t_b, 0, st))) return rc;
        if ((rc = gemm_packed_batched(w + l.w_hi, w + l.w_lo, w + l.t_hi, w + l.t_lo, grad_g + i * c * ls, c, ls, lc, ls,
                                      passes, 1.f, nullptr, nullptr, 1, 0, kb, (int64_t)l.w_b, (int64_t)l.t_b, c * ls, st))) return rc;
    }
    return RPST_OK;
}

// ---- clamped attention with the clamp given (training path of AdaptiveSANet: the clamp MLP and the cosine
//      affinity stay in the caller's autograd graph, the L x L work is here) --------------------------------
extern "C" size_t rpst_sanet_attn_clamped_workspace_bytes(int64_t c, int64_t lc, int64_t ls) {
    if (c <= 0 || lc <= 0 || ls <= 0) return 256;
    return attn_bwd_layout(c, lc, ls).total + align_up((size_t)lc * ls * sizeof(float), 256);   // + S' (fp32)
}

extern "C" int rpst_sanet_attn_clamped_fwd(const float* f, const float* g, const float* h, const float* clamp, int mode,
                                           float scale, float* out, int64_t b, int64_t c, int64_t lc, int64_t ls,
                                           int passes, void* workspace, size_t workspace_bytes, void* stream) {
    RPST_CHECK_ARG(b >= 0 && c > 0 && lc > 0 && ls > 0, "sanet_clamped: bad size");
    if (b == 0) return RPST_OK;
    RPST_CHECK_ARG(f && g && h && clamp && out, "sanet_clamped: null pointer");
    RPST_CHECK_ARG(mode == 1 || mode == 2, "sanet_clamped: mode must be 1 ('aea') or 2 ('relu')");
    RPST_CHECK_ARG(passes == 1 || passes == 3, "sanet_clamped: passes must be 1 or 3");
    const AttnLayout l = attn_layout(c, lc, ls);
    if (!workspace || workspace_bytes < l.total) {
        set_error("sanet_clamped: workspace too small (%zu < %zu bytes)", workspace_bytes, l.total);
        return RPST_ERR_WORKSPACE;
    }
    RPST_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, "sanet_clamped: workspace must be 256-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    char* w = static_cast<char*>(workspace);
    float* s = reinterpret_cast<float*>(w + l.s);
    int rc;
    for (int64_t i = 0; i < b; ++i) {
        if ((rc = scores(f + i * c * lc, g + i * c * ls, c, lc, ls, passes, w, l, s, st))) return rc;
        if ((rc = launch_rows(s, nullptr, w + l.p_hi, passes == 3 ? w + l.p_lo : nullptr, clamp + i * lc, lc, ls, mode,
                              scale, st, 1, 0, 0, 0, 0, 1))) return rc;                  // softmax + clamp -> S' tiles, one pass
        if ((rc = weighted_values(h + i * c * ls, c, lc, ls, passes, w, l, out + i * c * lc, st))) return rc;
    }
    return RPST_OK;
}

extern "C" int rpst_sanet_attn_clamped_bwd(const float* f, const float* g, const float* h, const float* clamp, int mode,
                                           float scale, const float* grad_out, float* grad_f, float* grad_g,
                                           float* grad_h, float* grad_clamp, int64_t b, int64_t c, int64_t lc,
                                           int64_t ls, int passes, void* workspace, size_t workspace_bytes, void* stream) {
    RPST_CHECK_ARG(b >= 0 && c > 0 && lc > 0 && ls > 0, "sanet_clamped_bwd: bad size");
    if (b == 0) return RPST_OK;
    RPST_CHECK_ARG(f && g && h && clamp && grad_out && grad_f && grad_g && grad_h && grad_clamp, "sanet_clamped_bwd: null pointer");
    RPST_CHECK_ARG(mode == 1 || mode == 2, "sanet_clamped_bwd: mode must be 1 ('aea') or 2 ('relu')");
    RPST_CHECK_ARG(passes == 1 || passes == 3, "sanet_clamped_bwd: passes must be 1 or 3");
    const size_t need = rpst_sanet_attn_clamped_workspace_bytes(c, lc, ls);
    if (!workspace || workspace_bytes < need) {
        set_error("sanet_clamped_bwd: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
        return RPST_ERR_WORKSPACE;
    }
    RPST_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, "sanet_clamped_bwd: workspace must be 256-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    char* w = static_cast<char*>(workspace);
    const bool x3 = passes == 3;
    auto lo = [&](size_t off) -> void* { return x3 ? w + off : nullptr; };
    const AttnBwdLayout l = attn_bwd_layout(c, lc, ls);
    const AttnLayout& a = l.a;
    float* prob = reinterpret_cast<float*>(w + a.s);
    float* dp = reinterpret_cast<float*>(w + l.dp);
    float* sp = reinterpret_cast<float*>(w + l.total);
    int rc;
    for (int64_t i = 0; i < b; ++i) {
        const float* fi = f + i * c * lc;
        const float* gi = g + i * c * ls;
        const float* hi_ = h + i * c * ls;
        const float* doi = grad_out + i * c * lc;
        const float* cli = clamp + i * lc;
        // P and S' = act(P - clamp), both kept in fp32
        if ((rc = scores(fi, gi, c, lc, ls, passes, w, a, prob, st))) return rc;
        if ((rc = launch_rows(prob, prob, nullptr, nullptr, nullptr, lc, ls, 0, 0.f, st))) return rc;
        if ((rc = launch_rows(prob, sp, nullptr, nullptr, cli, lc, ls, mode, scale, st))) return rc;
        // dH = dO S'      (A = dO rows c, K = i;  B = S'^T rows j, K = i)
        if ((rc = pack_operand_shift(doi, c, lc, lc, 1, nullptr, nullptr, w + l.w_hi, lo(l.w_lo), st))) return rc;
        if ((rc = pack_operand_shift(sp, ls, lc, 1, ls, nullptr, nullptr, w + l.t_hi, lo(l.t_lo), st))) return rc;
        if ((rc = gemm_packed_splitk(w + l.w_hi, w + l.w_lo, w + l.t_hi, w + l.t_lo, grad_h + i * c * ls, c, ls, lc, ls, passes,
                                     1.f, nullptr, nullptr, 1, 0, st))) return rc;
        // dS' = dO^T H    (A = dO^T rows i, K = c;  B = H^T rows j, K = c)
        if ((rc = pack_operand_shift(doi, lc, c, 1, lc, nullptr, nullptr, w + a.q_hi, lo(a.q_lo), st))) return rc;
        if ((rc = pack_operand_shift(hi_, ls, c, 1, ls, nullptr, nullptr, w + a.k_hi, lo(a.k_lo), st))) return rc;
        if ((rc = gemm_packed_splitk(w + a.q_hi, w + a.q_lo, w + a.k_hi, w + a.k_lo, dp, lc, ls, c, ls, passes, 1.f, nullptr,
                                     nullptr, 1, 0, st))) return rc;
        // clamp + softmax backward: dS (fp32 in place of dS' + tiles rows i, K = j), grad_clamp
        if (lc % kTileRows != 0 || ls % kTileK != 0) {
            RPST_CUDA(cudaMemsetAsync(w + a.p_hi, 0, a.p_b, st));
            if (x3) RPST_CUDA(cudaMemsetAsync(w + a.p_lo, 0, a.p_b, st));
        }
        attn_clamped_bwd_rows_kernel<<<(unsigned)lc, kRowThreads, 0, st>>>(
            prob, sp, dp, cli, grad_clamp + i * lc, mode, scale, reinterpret_cast<__nv_bfloat16*>(w + a.p_hi),
            x3 ? reinterpret_cast<__nv_bfloat16*>(w + a.p_lo) : nullptr, ls, (int)((ls + kTileK - 1) / kTileK));
        RPST_CUDA(cudaGetLastError());
        // dF = G dS^T, dG = F dS
        if ((rc = pack_operand_shift(gi, c, ls, ls, 1, nullptr, nullptr, w + a.v_hi, lo(a.v_lo), st))) return rc;
        if ((rc = gemm_packed_splitk(w + a.v_hi, w + a.v_lo, w + a.p_hi, w + a.p_lo, grad_f + i * c * lc, c, lc, ls, lc, passes,
                                     1.f, nullptr, nullptr, 1, 0, st))) return rc;
        if ((rc = pack_operand_shift(fi, c, lc, lc, 1, nullptr, nullptr, w + l.w_hi, lo(l.w_lo), st))) return rc;
        if ((rc = pack_operand_shift(dp, ls, lc, 1, ls, nullptr, nullptr, w + l.t_hi, lo(l.t_lo), st))) return rc;
        if ((rc = gemm_packed_splitk(w + l.w_hi, w + l.w_lo, w + l.t_hi, w + l.t_lo, grad_g + i * c * ls, c, ls, lc, ls, passes,
                                     1.f, nullptr, nullptr, 1, 0, st))) return rc;
    }
    return RPST_OK;
}

extern "C" size_t rpst_sanet_adaptive_workspace_bytes(int64_t c, int64_t lc, int64_t ls, int64_t lh) {
    if (c <= 0 || lc <= 0 || ls <= 0 || lh <= 0) return 256;
    return ada_layout(c, lc, ls, lh).total;
}

extern "C" int rpst_sanet_attn_adaptive_fwd(const float* f, const float* g, const float* h, const float* content_raw,
                                            const float* style_raw, int64_t c_raw, const float* w0, const float* b0,
                                            const float* w2, const float* b2, int mode, float scale_value,
                                            float from_value, float value_interval, float* out, float* claim_before,
                                            float* claim_after, float* claim_value, int64_t b, int64_t c, int64_t lc,
                                            int64_t ls, int64_t lh, int passes, void* workspace, size_t workspace_bytes,
                                            void* stream) {
    RPST_CHECK_ARG(b >= 0 && c > 0 && lc > 0 && ls > 0 && lh > 0 && c_raw > 0, "sanet_adaptive: bad size");
    if (b == 0) return RPST_OK;
    RPST_CHECK_ARG(f && g && h && content_raw && style_raw && w0 && b0 && w2 && b2 && out, "sanet_adaptive: null pointer");
    RPST_CHECK_ARG(lc == ls, "sanet_adaptive: the reference asserts equal content/style sizes (network/sanet.py:14)");
    RPST_CHECK_ARG(mode == 1 || mode == 2, "sanet_adaptive: mode must be 1 ('aea') or 2 ('relu')");
    RPST_CHECK_ARG(passes == 1 || passes == 3, "sanet_adaptive: passes must be 1 or 3");
    const AdaLayout l = ada_layout(c, lc, ls, lh);
    if (!workspace || workspace_bytes < l.total) {
        set_error("sanet_adaptive: workspace too small (%zu < %zu bytes)", workspace_bytes, l.total);
        return RPST_ERR_WORKSPACE;
    }
    RPST_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, "sanet_adaptive: workspace must be 256-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    char* w = static_cast<char*>(workspace);
    float* vec[6];
    for (int i = 0; i < 6; ++i) vec[i] = reinterpret_cast<float*>(w + l.vec[i]);
    float* aff = reinterpret_cast<float*>(w + l.aff);
    float* hidden = reinterpret_cast<float*>(w + l.hidden);
    int rc;
    // the Linear(L -> L/16) weight is shared by every sample: pack it once (rows = hidden units, K = L)
    if ((rc = pack_operand_shift(w0, lh, ls, ls, 1, nullptr, nullptr, w + l.w_hi, w + l.w_lo, st))) return rc;
    for (int64_t i = 0; i < b; ++i) {
        float* before = claim_before ? claim_before + i * lc * ls : reinterpret_cast<float*>(w + l.a.s);
        float* clampv = claim_value ? claim_value + i * lc : reinterpret_cast<float*>(w + l.clamp);
        // cosine affinity of the RAW features (network/sanet.py:16-18), reusing the Q/K tile buffers
        if ((rc = channel_norms(content_raw + i * c_raw * lc, c_raw, lc, vec[0], vec[1], vec[2], st))) return rc;
        if ((rc = channel_norms(style_raw + i * c_raw * ls, c_raw, ls, vec[3], vec[4], vec[5], st))) return rc;
        if ((rc = pack_operand_shift(content_raw + i * c_raw * lc, lc, c_raw, 1, lc, vec[2], nullptr, w + l.a.q_hi, w + l.a.q_lo, st))) return rc;
        if ((rc = pack_operand_shift(style_raw + i * c_raw * ls, ls, c_raw, 1, ls, vec[5], nullptr, w + l.a.k_hi, w + l.a.k_lo, st))) return rc;
        // the affinity leaves its GEMM as the packed A operand of the f_psi product (rows = content positions, K = style
        // positions): no fp32 L x L map, no pack pass (SURVEY 2b K9; a true back-to-back GEMM would need the
        // [128 x L/16] hidden accumulator next to the affinity tile in TMEM: 1024 + 256 columns of 512 at L = 16384)
        (void)aff;
        if ((rc = gemm_packed_to_tiles(w + l.a.q_hi, w + l.a.q_lo, w + l.a.k_hi, w + l.a.k_lo, lc, ls, c_raw, 3, 1.f,
                                       w + l.a.p_hi, w + l.a.p_lo, st))) return rc;
        // f_psi: hidden = aff @ W0^T + b0 (tensor cores)
        if ((rc = gemm_packed_splitk(w + l.a.p_hi, w + l.a.p_lo, w + l.w_hi, w + l.w_lo, hidden, lc, lh, ls, lh, 3, 1.f,
                                     nullptr, b0, 1, 0, st))) return rc;
        psi_head_kernel<<<(unsigned)((lc + 7) / 8), 256, 0, st>>>(hidden, w2, b2, lc, lh, mode, from_value, value_interval, clampv);
        RPST_CUDA(cudaGetLastError());
        // plain attention first (claim_before), then the clamped one (claim_after) straight into operand tiles
        if ((rc = scores(f + i * c * lc, g + i * c * ls, c, lc, ls, passes, w, l.a, before, st))) return rc;
        if (!claim_before) {
            // softmax and clamp in one pass over the logits (the probabilities are not an output)
            if ((rc = launch_rows(before, claim_after ? claim_after + i * lc * ls : nullptr, w + l.a.p_hi,
                                  passes == 3 ? w + l.a.p_lo : nullptr, clampv, lc, ls, mode, scale_value, st, 1, 0, 0, 0, 0, 1))) return rc;
        } else {
        if ((rc = launch_rows(before, before, nullptr, nullptr, nullptr, lc, ls, 0, 0.f, st))) return rc;
        if ((rc = launch_rows(before, claim_after ? claim_after + i * lc * ls : nullptr, w + l.a.p_hi,
                              passes == 3 ? w + l.a.p_lo : nullptr, clampv, lc, ls, mode, scale_value, st))) return rc;
        }
        if ((rc = weighted_values(h + i * c * ls, c, lc, ls, passes, w, l.a, out + i * c * lc, st))) return rc;
    }
    return RPST_OK;
}

extern "C" size_t rpst_cosine_affinity_workspace_bytes(int64_t c, int64_t lc, int64_t ls) {
    if (c <= 0 || lc <= 0 || ls <= 0) return 256;
    return 2 * align_up(packed_operand_bytes(lc, c), 256) + 2 * align_up(packed_operand_bytes(ls, c), 256) +
           6 * align_up((size_t)(lc > ls ? lc : ls) * sizeof(float), 256);
}

extern "C" int rpst_cosine_affinity(const float* content, const float* style, float* out, int64_t b, int64_t c,
                                    int64_t lc, int64_t ls, void* workspace, size_t workspace_bytes, void* stream) {
    RPST_CHECK_ARG(b >= 0 && c > 0 && lc > 0 && ls > 0, "cosine_affinity: bad size");
    if (b == 0) return RPST_OK;
    RPST_CHECK_ARG(content && style && out, "cosine_affinity: null pointer");
    const size_t need = rpst_cosine_affinity_workspace_bytes(c, lc, ls);
    if (!workspace || workspace_bytes < need) {
        set_error("cosine_affinity: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
        return RPST_ERR_WORKSPACE;
    }
    RPST_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, "cosine_affinity: workspace must be 256-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    char* w = static_cast<char*>(workspace);
    const size_t ta = align_up(packed_operand_bytes(lc, c), 256), tb = align_up(packed_operand_bytes(ls, c), 256);
    const size_t vb = align_up((size_t)(lc > ls ? lc : ls) * sizeof(float), 256);
    char* v = w + 2 * ta + 2 * tb;
    float* vec[6];
    for (int i = 0; i < 6; ++i) vec[i] = reinterpret_cast<float*>(v + i * vb);
    for (int64_t i = 0; i < b; ++i) {
        int rc;
        if ((rc = channel_norms(content + i * c * lc, c, lc, vec[0], vec[1], vec[2], st))) return rc;
        if ((rc = channel_norms(style + i * c * ls, c, ls, vec[3], vec[4], vec[5], st))) return rc;
        if ((rc = pack_operand_shift(content + i * c * lc, lc, c, 1, lc, vec[2], nullptr, w, w + ta, st))) return rc;
        if ((rc = pack_operand_shift(style + i * c * ls, ls, c, 1, ls, vec[5], nullptr, w + 2 * ta, w + 2 * ta + tb, st))) return rc;
        if ((rc = gemm_packed_splitk(w, w + ta, w + 2 * ta, w + 2 * ta + tb, out + i * lc * ls, lc, ls, c, ls, 3, 1.f,
                                     nullptr, nullptr, 1, 0, st))) return rc;
    }
    return RPST_OK;
}

RPST_WATCHDOG_SETTER(sanet)

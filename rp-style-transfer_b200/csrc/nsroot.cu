// Batched symmetric matrix square root and inverse square root by a scaled coupled Newton-Schulz iteration in fp64 —
// SURVEY.md §8 a5/a6; reference: network/wct_rp.py:7-38 (`matrix_sqrt` / `matrix_inv_sqrt`: `A + 1e-4 I`, SVD,
// spectrum cut below 1e-5, V diag(s^+-1/2) V^T).
//
// Why not only the eigensolver: the WCT's matrices are positive definite BY CONSTRUCTION (a covariance plus 1e-4 I,
// the content side plus another I), so the 1e-5 cut of the reference never fires and f(A) = V f(s) V^T is the
// principal root.  A one-sided Jacobi solve of 16 256x256 matrices takes 4.4 ms (latency / issue bound, eig.cu); the
// coupled iteration below needs 9 (content) to ~16 (style) steps of three 256^3 products each, which run at DFMA
// throughput on every SM.
//
//   s = 1 / ||A||_F,  Y_0 = s A,  Z_0 = I,   x in [l_0, 1] with l_0 = sqrt(lmin * s) for the roots of the spectrum
//   T_k = (3 I - a_k^2 Z_k Y_k) / 2,  Y_{k+1} = a_k Y_k T_k,  Z_{k+1} = a_k T_k Z_k         (Y -> (sA)^1/2, Z -> (sA)^-1/2)
//   a_k = sqrt(3 / (1 + l_k + l_k^2)),  l_{k+1} = a_k l_k (3 - a_k^2 l_k^2) / 2             (Chen & Chow's scaling of the
//   Newton-Schulz sign iteration: maps [l_k, 1] onto [l_{k+1}, 1] with both ends at l_{k+1}; 2.6x per step instead of
//   1.5x while l is small), then one unscaled step.  The step count and the a_k depend on ||A||_F only, so they are
//   computed on the device per matrix (no host synchronisation); launches beyond a matrix's count return at once.
//
// Acceptance: ||Z Y - I||_F <= 1e-7 after the last step.  A matrix that fails (not positive definite after rounding,
// smallest eigenvalue far below the bound, count above the cap) is FLAGGED and the caller runs the Jacobi path for the
// flagged matrices only (eig.cu kernels take the flag array), so the reference's |s|-and-cut semantics still hold there.
#include "common.cuh"
#include "tuning.cuh"

namespace rpst {

namespace {

constexpr int kNsMaxIt = 24;
constexpr int kGM = 128, kGN = 64, kGK = 16, kGThreads = 256;

// matrices handed to the Jacobi path since the library was loaded (diagnostics: rpst_get_tuning("wct_ns_flagged"))
__device__ unsigned long long g_ns_flag_count = 0;

enum NsMode : int { kPlain = 0, kStepT = 1, kStepYZ = 2, kCheck = 3 };

struct GemmArgs {
    const double* a; const double* b; double* c;   // kPlain operands
    double* y[2]; double* z[2]; double* t;         // Newton-Schulz ping-pong buffers
    int jobs, n, batch;
    int mode, it;
    const double* alpha;   // [batch, kNsMaxIt]
    const int* nit;        // [batch]
    double* partial;       // kCheck: [batch, tiles] sums of (Z Y - I)^2
};

__device__ __forceinline__ double block_sum_256(double v, double* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0)
        for (int i = 0; i < kGThreads / 32; ++i) t += red[i];      // fixed order
    return t;
}

__device__ __forceinline__ void cp_async_16(void* smem_dst, const void* gmem_src, int src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;"
                 :: "r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" :: "n"(N) : "memory"); }

// C[z] = A[z] B[z] (n x n fp64, row-major, ld n) with the Newton-Schulz epilogues.  128 x 64 tile per CTA, 8 x 4 per
// thread, k-tiles of 16.  kStepT / kStepYZ do nothing from step nit[b] on; the step's parity picks the ping-pong buffer.
//
// The products are computed EXACTLY as written (Y T, T Z, Z Y from the stored operands): the coupled iteration is only
// stable while Y_k = A Z_k holds to rounding.  Reading an operand through its transpose, mirroring the upper triangle
// of a result or averaging a result with its transpose — all "free" for symmetric iterates — made it diverge for
// condition numbers >= 1e6 (rank-deficient covariances + 1e-4 I), so none of those shortcuts is taken.
//
// ASYNC (even n): both tiles go global -> shared with cp.async (zero-fill past the edge), double buffered, A as
// [128 rows][16 k], B as [16 k][64 columns]: no staging registers.  Odd n stages through registers.
template <int MODE, bool ASYNC>
__global__ void __launch_bounds__(kGThreads, 2) ns_gemm_kernel(GemmArgs g) {
    constexpr int kStageDoubles = kGK * kGM + kGK * kGN;                // 3072
    __shared__ __align__(16) double tile_smem[2 * kStageDoubles];       // 48 KiB: two stages (the generic path uses one)
    const int job = (int)blockIdx.z / g.batch, smp = (int)blockIdx.z % g.batch;
    const int n = g.n;
    double alpha = 1.0;
    int par = 0;                                   // operand buffer parity (ping-pong modes)
    if (MODE == kStepT || MODE == kStepYZ) {
        if (g.it >= g.nit[smp]) return;
        alpha = g.alpha[smp * kNsMaxIt + g.it];
        par = g.it & 1;
    } else if (MODE == kCheck) {
        par = g.nit[smp] & 1;
    }
    const size_t off = (size_t)smp * n * n;
    const double *A, *B;
    double* C = nullptr;
    if (MODE == kPlain) {
        A = g.a + off; B = g.b + off; C = g.c + off;
    } else if (MODE == kStepT) {                   // T = 1.5 I - 0.5 a^2 Z Y
        A = g.z[par] + off; B = g.y[par] + off; C = g.t + off;
    } else if (MODE == kStepYZ) {                  // job 0: Y' = a Y T, job 1: Z' = a T Z
        if (job == 0) { A = g.y[par] + off; B = g.t + off; C = g.y[par ^ 1] + off; }
        else          { A = g.t + off; B = g.z[par] + off; C = g.z[par ^ 1] + off; }
    } else {                                       // kCheck: Z Y against I
        A = g.z[par] + off; B = g.y[par] + off;
    }
    const int i0 = blockIdx.y * kGM, j0 = blockIdx.x * kGN;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const bool vec = (n & 1) == 0;                 // 16-byte accesses stay aligned when rows have even length

    double acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;

    auto compute = [&](const double* as, const double* bs) {      // as [128][16], bs [16][64]
#pragma unroll
        for (int k = 0; k < kGK; k += 2) {
            // rows {4 ty .. 4 ty + 3} and {64 + 4 ty ..} (two k values per load), columns {2 tx, 2 tx + 1} and {32 + 2 tx, ..}
            double2 a[8];
#pragma unroll
            for (int i = 0; i < 8; ++i)
                a[i] = *reinterpret_cast<const double2*>(as + ((i < 4 ? 4 * ty + i : 64 + 4 * ty + (i - 4)) * kGK + k));
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
                const double2 b0 = *reinterpret_cast<const double2*>(bs + (k + kk) * kGN + 2 * tx);
                const double2 b1 = *reinterpret_cast<const double2*>(bs + (k + kk) * kGN + 32 + 2 * tx);
                const double b[4] = {b0.x, b0.y, b1.x, b1.y};
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const double av = kk ? a[i].y : a[i].x;
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fma(av, b[j], acc[i][j]);
                }
            }
        }
    };

    if (ASYNC) {
        // A tile: rows i0 + m (128), columns k0 .. k0 + 15: 8 chunks of 16 bytes per row, 4 per thread
        // B tile: rows k0 + k (16), columns j0 .. j0 + 63:  32 chunks per row, 2 per thread
        auto issue = [&](int k0, int stage) {
            double* as = tile_smem + stage * kStageDoubles;
            double* bs = as + kGK * kGM;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int ch = threadIdx.x + q * kGThreads, m = ch >> 3, k = (ch & 7) * 2;
                const bool ok = i0 + m < n && k0 + k < n;
                cp_async_16(as + m * kGK + k, ok ? A + (size_t)(i0 + m) * n + k0 + k : A, ok ? 16 : 0);
            }
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int ch = threadIdx.x + q * kGThreads, k = ch >> 5, c = (ch & 31) * 2;
                const bool ok = k0 + k < n && j0 + c < n;
                cp_async_16(bs + k * kGN + c, ok ? B + (size_t)(k0 + k) * n + j0 + c : B, ok ? 16 : 0);
            }
            cp_async_commit();
        };
        const int nk = (n + kGK - 1) / kGK;
        issue(0, 0);
        for (int kt = 0; kt < nk; ++kt) {
            if (kt + 1 < nk) { issue((kt + 1) * kGK, (kt + 1) & 1); cp_async_wait<1>(); }
            else cp_async_wait<0>();
            __syncthreads();
            const double* as = tile_smem + (kt & 1) * kStageDoubles;
            compute(as, as + kGK * kGM);
            __syncthreads();
        }
    } else {
        // global -> register staging: A tile 128 x 16 (4 double2 per thread), B tile 16 x 64 (2 double2 per thread)
        double* as = tile_smem;
        double* bs = as + kGK * kGM;
        const int ar = threadIdx.x >> 3, ak = (threadIdx.x & 7) * 2;     // rows ar + 32 j
        const int bk = threadIdx.x >> 5, bj = (threadIdx.x & 31) * 2;    // k rows bk + 8 j
        double2 ra[4], rb[2];
        auto load_tiles = [&](int k0) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int r = i0 + ar + 32 * j, k = k0 + ak;
                double2 v = make_double2(0.0, 0.0);
                if (r < n) {
                    const double* src = A + (size_t)r * n + k;
                    if (vec && k + 1 < n) v = *reinterpret_cast<const double2*>(src);
                    else {
                        if (k < n) v.x = src[0];
                        if (k + 1 < n) v.y = src[1];
                    }
                }
                ra[j] = v;
            }
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int k = k0 + bk + 8 * j, c = j0 + bj;
                double2 v = make_double2(0.0, 0.0);
                if (k < n) {
                    const double* src = B + (size_t)k * n + c;
                    if (vec && c + 1 < n) v = *reinterpret_cast<const double2*>(src);
                    else {
                        if (c < n) v.x = src[0];
                        if (c + 1 < n) v.y = src[1];
                    }
                }
                rb[j] = v;
            }
        };
        load_tiles(0);
        for (int k0 = 0; k0 < n; k0 += kGK) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                *reinterpret_cast<double2*>(as + (ar + 32 * j) * kGK + ak) = ra[j];
            }
#pragma unroll
            for (int j = 0; j < 2; ++j) *reinterpret_cast<double2*>(bs + (bk + 8 * j) * kGN + bj) = rb[j];
            __syncthreads();
            if (k0 + kGK < n) load_tiles(k0 + kGK);
            compute(as, bs);
            __syncthreads();
        }
    }

    double mul = 1.0, diag = 0.0;
    if (MODE == kStepT) { mul = -0.5 * alpha * alpha; diag = 1.5; }
    else if (MODE == kStepYZ) mul = alpha;
    double sq = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int r = i0 + (i < 4 ? 4 * ty + i : 64 + 4 * ty + (i - 4));
        if (r >= n) continue;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int c = j0 + 32 * h + 2 * tx;
            const double v0 = acc[i][2 * h] * mul + (r == c ? diag : 0.0);
            const double v1 = acc[i][2 * h + 1] * mul + (r == c + 1 ? diag : 0.0);
            if (MODE == kCheck) {
                if (c < n) { const double d = v0 - (r == c ? 1.0 : 0.0); sq = fma(d, d, sq); }
                if (c + 1 < n) { const double d = v1 - (r == c + 1 ? 1.0 : 0.0); sq = fma(d, d, sq); }
                continue;
            }
            if (vec && c + 1 < n) {
                *reinterpret_cast<double2*>(C + (size_t)r * n + c) = make_double2(v0, v1);
            } else {
                if (c < n) C[(size_t)r * n + c] = v0;
                if (c + 1 < n) C[(size_t)r * n + c + 1] = v1;
            }
        }
    }
    if (MODE == kCheck) {
        const double t = block_sum_256(sq, tile_smem);
        if (threadIdx.x == 0) g.partial[(size_t)smp * gridDim.x * gridDim.y + blockIdx.y * gridDim.x + blockIdx.x] = t;
    }
}

// partial sums of squares of A + d I: kNormParts blocks per matrix
constexpr int kNormParts = 32;
__global__ void __launch_bounds__(kGThreads) ns_norm_kernel(const double* __restrict__ a, int n, double diag_add,
                                                            double* __restrict__ part) {
    __shared__ double red[kGThreads / 32];
    const int b = blockIdx.y;
    const double* A = a + (size_t)b * n * n;
    double sq = 0.0;
    for (int e = blockIdx.x * kGThreads + threadIdx.x; e < n * n; e += kNormParts * kGThreads) {
        const int r = e / n, c = e % n;
        const double v = A[e] + (r == c ? diag_add : 0.0);
        sq = fma(v, v, sq);
    }
    const double t = block_sum_256(sq, red);
    if (threadIdx.x == 0) part[b * kNormParts + blockIdx.x] = t;
}

// per matrix: s = 1 / ||A + d I||_F, the scaling sequence a_k and the step count
__global__ void ns_plan_kernel(const double* __restrict__ part, int batch, double lmin, int maxit, double* __restrict__ scale,
                               double* __restrict__ alpha, int* __restrict__ nit, int* __restrict__ capped) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= batch) return;
    double t = 0.0;
    for (int i = 0; i < kNormParts; ++i) t += part[b * kNormParts + i];      // fixed order
    const double fro = sqrt(t);
    const double s = fro > 0.0 && isfinite(fro) ? 1.0 / fro : 1.0;
    scale[b] = s;
    // lower bound on the roots of the scaled spectrum, with a safety factor of 4 on the eigenvalue bound
    double l = sqrt(0.25 * lmin * s);
    if (!(l < 1.0)) l = 1.0;
    int k = 0;
    while (k < maxit - 1 && 1.0 - l > 1e-7) {
        const double al = sqrt(3.0 / (1.0 + l + l * l));
        alpha[b * kNsMaxIt + k++] = al;
        l = 0.5 * al * l * (3.0 - al * al * l * l);
    }
    capped[b] = 1.0 - l > 1e-7;        // the cap was hit: iterate anyway, flagged at the end
    alpha[b * kNsMaxIt + k++] = 1.0;   // one unscaled step: 1 - l <= 1e-7 -> 1.5e-14 (a second one bought 1e-28 on paper)
    nit[b] = k;
}

// Y_0 = s (A + d I); Z_0 = I makes the first step's T and Z products trivial, so they are written here:
// T_0 = 1.5 I - 0.5 a_0^2 Y_0 and Z_1 = a_0 T_0 (exactly what the products with the identity would give)
__global__ void __launch_bounds__(256) ns_init_kernel(const double* __restrict__ a, int n, double diag_add,
                                                      const double* __restrict__ scale, const double* __restrict__ alpha,
                                                      double* __restrict__ y0, double* __restrict__ t0, double* __restrict__ z1) {
    const int b = blockIdx.y;
    const size_t off = (size_t)b * n * n;
    const double s = scale[b], al = alpha[b * kNsMaxIt];
    for (int e = blockIdx.x * 256 + threadIdx.x; e < n * n; e += gridDim.x * 256) {
        const int r = e / n, c = e % n;
        const double y = s * (a[off + e] + (r == c ? diag_add : 0.0));
        const double t = (r == c ? 1.5 : 0.0) - 0.5 * al * al * y;
        y0[off + e] = y;
        t0[off + e] = t;
        z1[off + e] = al * t;
    }
}

// root = sym(Y) / sqrt(s), iroot = sym(Z) sqrt(s); flag[b] = 1 when the iteration is not accepted
__global__ void __launch_bounds__(256) ns_finish_kernel(const double* __restrict__ ybuf0, const double* __restrict__ ybuf1,
                                                        const double* __restrict__ zbuf0, const double* __restrict__ zbuf1,
                                                        int n, const double* __restrict__ scale, const int* __restrict__ nit,
                                                        const int* __restrict__ capped, const double* __restrict__ partial,
                                                        int tiles, double tol2, int force_flag, double* __restrict__ root,
                                                        double* __restrict__ iroot, int* __restrict__ flag) {
    const int b = blockIdx.y;
    const size_t off = (size_t)b * n * n;
    const int par = nit[b] & 1;
    const double* Y = (par ? ybuf1 : ybuf0) + off;
    const double* Z = (par ? zbuf1 : zbuf0) + off;
    const double rs = sqrt(scale[b]);
    for (int e = blockIdx.x * 256 + threadIdx.x; e < n * n; e += gridDim.x * 256) {
        const int r = e / n, c = e % n;
        if (root) root[off + e] = 0.5 * (Y[e] + Y[(size_t)c * n + r]) / rs;
        if (iroot) iroot[off + e] = 0.5 * (Z[e] + Z[(size_t)c * n + r]) * rs;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < tiles; ++i) t += partial[(size_t)b * tiles + i];
        const int f = (force_flag || capped[b] || !(t <= tol2)) ? 1 : 0;
        flag[b] = f;
        if (f) atomicAdd(&g_ns_flag_count, 1ull);
    }
}

struct NsLayout {
    size_t y[2], z[2], t, alpha, scale, nit, capped, partial, norm, total;
    int tiles;
};
NsLayout ns_layout(int64_t batch, int n) {
    NsLayout l;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o += align_up(bytes, 256); return at; };
    const size_t mat = (size_t)batch * n * n * sizeof(double);
    l.y[0] = take(mat); l.y[1] = take(mat);
    l.z[0] = take(mat); l.z[1] = take(mat);
    l.t = take(mat);
    l.alpha = take((size_t)batch * kNsMaxIt * sizeof(double));
    l.scale = take((size_t)batch * sizeof(double));
    l.nit = take((size_t)batch * sizeof(int));
    l.capped = take((size_t)batch * sizeof(int));
    l.tiles = ((n + 63) / 64) * ((n + kGN - 1) / kGN);            // room for the 64-row tiling of small batches
    l.partial = take((size_t)batch * l.tiles * sizeof(double));
    l.norm = take((size_t)batch * kNormParts * sizeof(double));
    l.total = o;
    return l;
}

// ---- the same products on the fp64 tensor-core path (mma.sync.m8n8k4.f64) --------------------------------------------
// The DFMA kernel above stops at 55-58 % of the fp64 pipe with one CTA per SM or two (three 64-bit register operands per
// FMA); a DMMA carries 8 FMAs per thread on one A and one B register.  Even n only (cp.async tiles).  CTA tile 128 x 64,
// warp tile 32 x 32 = 4 x 4 m8n8 tiles, k-tiles of 16 = four k4 steps.  Shared-memory strides (A rows 20 doubles, B rows
// 68) put the 16 lanes of a half warp on 16 different bank pairs for both fragment loads.
constexpr int kDA = 20, kDB = 68;
constexpr int kDStage = kGM * kDA + kGK * kDB;             // 3648 doubles = 29184 bytes
constexpr size_t kDmmaSmem = 2 * (size_t)kDStage * sizeof(double);

__device__ __forceinline__ void dmma_884(double (&c)[2], double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}

// BM = 128: warps 4 x 2, 32 x 32 per warp; BM = 64 (small batches: twice the CTAs): warps 2 x 4, 32 x 16 per warp.
template <int MODE, int BM>
__global__ void __launch_bounds__(kGThreads, 2) ns_gemm_dmma_kernel(GemmArgs g) {
    constexpr int WM = BM / 32, WN = 8 / WM, WNC = kGN / WN, NT = WNC / 8;     // warp grid, warp columns, n tiles per warp
    constexpr int kStageD = BM * kDA + kGK * kDB;
    extern __shared__ __align__(16) unsigned char dmma_smem[];
    double* tile_smem = reinterpret_cast<double*>(dmma_smem);
    const int job = (int)blockIdx.z / g.batch, smp = (int)blockIdx.z % g.batch;
    const int n = g.n;
    double alpha = 1.0;
    int par = 0;
    if (MODE == kStepT || MODE == kStepYZ) {
        if (g.it >= g.nit[smp]) return;
        alpha = g.alpha[smp * kNsMaxIt + g.it];
        par = g.it & 1;
    } else if (MODE == kCheck) {
        par = g.nit[smp] & 1;
    }
    const size_t off = (size_t)smp * n * n;
    const double *A, *B;
    double* C = nullptr;
    if (MODE == kPlain) {
        A = g.a + off; B = g.b + off; C = g.c + off;
    } else if (MODE == kStepT) {
        A = g.z[par] + off; B = g.y[par] + off; C = g.t + off;
    } else if (MODE == kStepYZ) {
        if (job == 0) { A = g.y[par] + off; B = g.t + off; C = g.y[par ^ 1] + off; }
        else          { A = g.t + off; B = g.z[par] + off; C = g.z[par ^ 1] + off; }
    } else {
        A = g.z[par] + off; B = g.y[par] + off;
    }
    const int i0 = blockIdx.y * BM, j0 = blockIdx.x * kGN;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wm = warp % WM, wn = warp / WM;
    const int gid = lane >> 2, tig = lane & 3;

    double acc[4][NT][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < NT; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }

    auto issue = [&](int k0, int stage) {
        double* as = tile_smem + stage * kStageD;
        double* bs = as + BM * kDA;
#pragma unroll
        for (int q = 0; q < BM / 32; ++q) {
            const int ch = threadIdx.x + q * kGThreads, m = ch >> 3, k = (ch & 7) * 2;
            const bool ok = i0 + m < n && k0 + k < n;
            cp_async_16(as + m * kDA + k, ok ? A + (size_t)(i0 + m) * n + k0 + k : A, ok ? 16 : 0);
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int ch = threadIdx.x + q * kGThreads, k = ch >> 5, c = (ch & 31) * 2;
            const bool ok = k0 + k < n && j0 + c < n;
            cp_async_16(bs + k * kDB + c, ok ? B + (size_t)(k0 + k) * n + j0 + c : B, ok ? 16 : 0);
        }
        cp_async_commit();
    };
    const int nk = (n + kGK - 1) / kGK;
    issue(0, 0);
    for (int kt = 0; kt < nk; ++kt) {
        if (kt + 1 < nk) { issue((kt + 1) * kGK, (kt + 1) & 1); cp_async_wait<1>(); }
        else cp_async_wait<0>();
        __syncthreads();
        const double* as = tile_smem + (kt & 1) * kStageD + (32 * wm + gid) * kDA + tig;
        const double* bs = tile_smem + (kt & 1) * kStageD + BM * kDA + tig * kDB + WNC * wn + gid;
#pragma unroll
        for (int kk = 0; kk < kGK; kk += 4) {
            double a[4], b[NT];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = as[(8 * i) * kDA + kk];
#pragma unroll
            for (int j = 0; j < NT; ++j) b[j] = bs[kk * kDB + 8 * j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < NT; ++j) dmma_884(acc[i][j], a[i], b[j]);
        }
        __syncthreads();
    }

    double mul = 1.0, diag = 0.0;
    if (MODE == kStepT) { mul = -0.5 * alpha * alpha; diag = 1.5; }
    else if (MODE == kStepYZ) mul = alpha;
    double sq = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = i0 + 32 * wm + 8 * i + gid;
        if (r >= n) continue;
#pragma unroll
        for (int j = 0; j < NT; ++j) {
            const int c = j0 + WNC * wn + 8 * j + 2 * tig;
            const double v0 = acc[i][j][0] * mul + (r == c ? diag : 0.0);
            const double v1 = acc[i][j][1] * mul + (r == c + 1 ? diag : 0.0);
            if (MODE == kCheck) {
                if (c < n) { const double d = v0 - (r == c ? 1.0 : 0.0); sq = fma(d, d, sq); }
                if (c + 1 < n) { const double d = v1 - (r == c + 1 ? 1.0 : 0.0); sq = fma(d, d, sq); }
                continue;
            }
            if (c + 1 < n) *reinterpret_cast<double2*>(C + (size_t)r * n + c) = make_double2(v0, v1);   // n even, c even
            else if (c < n) C[(size_t)r * n + c] = v0;
        }
    }
    if (MODE == kCheck) {
        const double t = block_sum_256(sq, tile_smem);
        if (threadIdx.x == 0) g.partial[(size_t)smp * gridDim.x * gridDim.y + blockIdx.y * gridDim.x + blockIdx.x] = t;
    }
}

// rows per CTA tile of the tensor-core GEMM: 64 when the 128-row tiling would leave a third of the SMs without a CTA
int gemm_tile_rows(int n, int batch) {
    if ((n & 1) || !g_knobs.ns_dmma) return kGM;
    const int64_t ctas = (int64_t)((n + kGM - 1) / kGM) * ((n + kGN - 1) / kGN) * batch;
    return ctas < 2 * sm_count() / 3 ? 64 : kGM;
}

int launch_gemm(GemmArgs g, cudaStream_t st) {
    dim3 grid((unsigned)((g.n + kGN - 1) / kGN), (unsigned)((g.n + kGM - 1) / kGM), (unsigned)(g.jobs * g.batch));
    const bool even = (g.n & 1) == 0;
    if (even && g_knobs.ns_dmma) {
        static PerDeviceFlag configured_on;
        bool& configured = configured_on.get();
        if (!configured) {
#define RPST_NS_ATTR(M, B) RPST_CUDA(cudaFuncSetAttribute(ns_gemm_dmma_kernel<M, B>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDmmaSmem))
            RPST_NS_ATTR(kPlain, 128); RPST_NS_ATTR(kStepT, 128); RPST_NS_ATTR(kStepYZ, 128); RPST_NS_ATTR(kCheck, 128);
            RPST_NS_ATTR(kPlain, 64); RPST_NS_ATTR(kStepT, 64); RPST_NS_ATTR(kStepYZ, 64); RPST_NS_ATTR(kCheck, 64);
#undef RPST_NS_ATTR
            configured = true;
        }
        // small batches: 64-row tiles double the CTA count (one 256^2 matrix: 16 / 32 CTAs per product instead of 8 / 16)
        if (gemm_tile_rows(g.n, g.batch) == 64) {
            dim3 grid64(grid.x, (unsigned)((g.n + 63) / 64), grid.z);
            switch (g.mode) {
                case kPlain: ns_gemm_dmma_kernel<kPlain, 64><<<grid64, kGThreads, kDmmaSmem, st>>>(g); break;
                case kStepT: ns_gemm_dmma_kernel<kStepT, 64><<<grid64, kGThreads, kDmmaSmem, st>>>(g); break;
                case kStepYZ: ns_gemm_dmma_kernel<kStepYZ, 64><<<grid64, kGThreads, kDmmaSmem, st>>>(g); break;
                default: ns_gemm_dmma_kernel<kCheck, 64><<<grid64, kGThreads, kDmmaSmem, st>>>(g); break;
            }
        } else {
            switch (g.mode) {
                case kPlain: ns_gemm_dmma_kernel<kPlain, 128><<<grid, kGThreads, kDmmaSmem, st>>>(g); break;
                case kStepT: ns_gemm_dmma_kernel<kStepT, 128><<<grid, kGThreads, kDmmaSmem, st>>>(g); break;
                case kStepYZ: ns_gemm_dmma_kernel<kStepYZ, 128><<<grid, kGThreads, kDmmaSmem, st>>>(g); break;
                default: ns_gemm_dmma_kernel<kCheck, 128><<<grid, kGThreads, kDmmaSmem, st>>>(g); break;
            }
        }
        RPST_CUDA(cudaGetLastError());
        return RPST_OK;
    }
    switch (g.mode) {
        case kPlain:
            if (even) ns_gemm_kernel<kPlain, true><<<grid, kGThreads, 0, st>>>(g);
            else ns_gemm_kernel<kPlain, false><<<grid, kGThreads, 0, st>>>(g);
            break;
        case kStepT:
            if (even) ns_gemm_kernel<kStepT, true><<<grid, kGThreads, 0, st>>>(g);
            else ns_gemm_kernel<kStepT, false><<<grid, kGThreads, 0, st>>>(g);
            break;
        case kStepYZ:
            if (even) ns_gemm_kernel<kStepYZ, true><<<grid, kGThreads, 0, st>>>(g);
            else ns_gemm_kernel<kStepYZ, false><<<grid, kGThreads, 0, st>>>(g);
            break;
        default:
            if (even) ns_gemm_kernel<kCheck, true><<<grid, kGThreads, 0, st>>>(g);
            else ns_gemm_kernel<kCheck, false><<<grid, kGThreads, 0, st>>>(g);
            break;
    }
    RPST_CUDA(cudaGetLastError());
    return RPST_OK;
}

}  // namespace

int64_t ns_flagged_total() {
    unsigned long long v = 0;
    if (cudaMemcpyFromSymbol(&v, g_ns_flag_count, sizeof(v)) != cudaSuccess) return -1;
    return (int64_t)v;
}

size_t ns_roots_workspace_bytes(int64_t batch, int n) { return ns_layout(batch, n).total; }

// C[b] = A[b] B[b], batched n x n fp64 (row-major)
int dgemm_batched(const double* a, const double* b, double* c, int64_t batch, int n, cudaStream_t st) {
    GemmArgs g{};
    g.a = a; g.b = b; g.c = c;
    g.jobs = 1; g.n = n; g.batch = (int)batch; g.mode = kPlain;
    return launch_gemm(g, st);
}

// root[b] = (A[b] + d I)^(1/2), iroot[b] = (A[b] + d I)^(-1/2) (either may be null) for symmetric A whose eigenvalues,
// after the diagonal shift, are bounded below by `lmin` > 0.  flag[b] = 1 where the result must not be used.
int ns_roots(const double* a, int64_t batch, int n, double diag_add, double lmin, double* root, double* iroot, int* flag,
             void* workspace, size_t workspace_bytes, cudaStream_t st) {
    const NsLayout l = ns_layout(batch, n);
    if (workspace_bytes < l.total) {
        set_error("ns_roots: workspace too small (%zu < %zu bytes)", workspace_bytes, l.total);
        return RPST_ERR_WORKSPACE;
    }
    char* w = static_cast<char*>(workspace);
    double* y[2] = {reinterpret_cast<double*>(w + l.y[0]), reinterpret_cast<double*>(w + l.y[1])};
    double* z[2] = {reinterpret_cast<double*>(w + l.z[0]), reinterpret_cast<double*>(w + l.z[1])};
    double* t = reinterpret_cast<double*>(w + l.t);
    double* alpha = reinterpret_cast<double*>(w + l.alpha);
    double* scale = reinterpret_cast<double*>(w + l.scale);
    int* nit = reinterpret_cast<int*>(w + l.nit);
    int* capped = reinterpret_cast<int*>(w + l.capped);
    double* partial = reinterpret_cast<double*>(w + l.partial);
    double* norm = reinterpret_cast<double*>(w + l.norm);
    // Step cap = number of launches (launches past a matrix's own count return at once, ~2 us each).  With l_0 =
    // sqrt(lmin / 4 ||A||_F): lmin >= 0.5 (content side) needs 9 steps at ||A||_F = 2.5e3 and 12 at 1e6; lmin = 1e-4 needs
    // 15 steps at ||A||_F = 1e4 and 19 at 2.5e7.  A matrix beyond the cap is flagged and goes to the Jacobi solver.
    const int maxit = lmin >= 0.5 ? 12 : 20;
    ns_norm_kernel<<<dim3(kNormParts, (unsigned)batch), kGThreads, 0, st>>>(a, n, diag_add, norm);
    RPST_CUDA(cudaGetLastError());
    ns_plan_kernel<<<(unsigned)((batch + 63) / 64), 64, 0, st>>>(norm, (int)batch, lmin, maxit, scale, alpha, nit, capped);
    RPST_CUDA(cudaGetLastError());
    const unsigned eb = (unsigned)(((size_t)n * n + 255) / 256 < 64 ? ((size_t)n * n + 255) / 256 : 64);
    ns_init_kernel<<<dim3(eb, (unsigned)batch), 256, 0, st>>>(a, n, diag_add, scale, alpha, y[0], t, z[1]);
    RPST_CUDA(cudaGetLastError());
    int rc;
    GemmArgs g{};
    g.y[0] = y[0]; g.y[1] = y[1]; g.z[0] = z[0]; g.z[1] = z[1]; g.t = t;
    g.n = n; g.batch = (int)batch; g.alpha = alpha; g.nit = nit; g.partial = partial;
    for (int it = 0; it < maxit; ++it) {
        g.it = it;
        if (it > 0) {                       // step 0: T_0 and Z_1 came from the init kernel, only Y_1 = a_0 Y_0 T_0 is a product
            g.jobs = 1; g.mode = kStepT;
            if ((rc = launch_gemm(g, st))) return rc;
        }
        g.jobs = it > 0 ? 2 : 1; g.mode = kStepYZ;
        if ((rc = launch_gemm(g, st))) return rc;
    }
    g.jobs = 1; g.mode = kCheck;
    if ((rc = launch_gemm(g, st))) return rc;
    const int tiles_used = ((n + gemm_tile_rows(n, (int)batch) - 1) / gemm_tile_rows(n, (int)batch)) * ((n + kGN - 1) / kGN);
    ns_finish_kernel<<<dim3(eb, (unsigned)batch), 256, 0, st>>>(y[0], y[1], z[0], z[1], n, scale, nit, capped, partial, tiles_used,
                                                                1e-14, g_knobs.wct_roots_ns == 2, root, iroot, flag);
    RPST_CUDA(cudaGetLastError());
    return RPST_OK;
}

}  // namespace rpst

using namespace rpst;

#ifdef RPST_DEBUG_EXPORTS   // white-box test hooks: only in librpst_debug.so (loaded by tests alone), never in the product library
// Test hook: c[b] = a[b] b[b] (n x n fp64, row-major) through dgemm_batched, the products of the Newton-Schulz iteration and
// of the WCT transform (DMMA kernel with 64- or 128-row tiles for even n, DFMA kernel for odd n or with ns_dmma = 0).
extern "C" int rpst_debug_dgemm_batched(const double* a, const double* b, double* c, int64_t batch, int64_t n, void* stream) {
    RPST_CHECK_ARG(batch > 0 && n > 0 && n <= 512 && a && b && c, "debug_dgemm_batched: bad arguments");
    return dgemm_batched(a, b, c, batch, (int)n, static_cast<cudaStream_t>(stream));
}
#endif  // RPST_DEBUG_EXPORTS

extern "C" size_t rpst_spd_roots_workspace_bytes(int64_t batch, int64_t n) {
    if (batch <= 0 || n <= 0 || n > 512) return 256;
    return ns_roots_workspace_bytes(batch, (int)n);
}

extern "C" int rpst_spd_roots(const double* a, int64_t batch, int64_t n, double diag_add, double lmin, double* out_sqrt,
                              double* out_inv_sqrt, int32_t* flags, void* workspace, size_t workspace_bytes, void* stream) {
    RPST_CHECK_ARG(batch >= 0 && n >= 0, "spd_roots: negative size");
    if (batch == 0 || n == 0) return RPST_OK;
    RPST_CHECK_ARG(n <= 512, "spd_roots: order must be <= 512 (got %lld)", (long long)n);
    RPST_CHECK_ARG(a != nullptr && flags != nullptr && workspace != nullptr, "spd_roots: null pointer");
    RPST_CHECK_ARG(lmin > 0.0, "spd_roots: the eigenvalue bound lmin must be positive");
    RPST_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, "spd_roots: workspace must be 256-byte aligned");
    return ns_roots(a, batch, (int)n, diag_add, lmin, out_sqrt, out_inv_sqrt, flags, workspace, workspace_bytes,
                    static_cast<cudaStream_t>(stream));
}

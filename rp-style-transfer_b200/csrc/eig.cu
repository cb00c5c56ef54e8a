// Batched symmetric eigensolver + matrix functions for WCT — SURVEY.md §8 a5; reference:
// network/wct_rp.py:7-40 (`matrix_sqrt`, `matrix_inv_sqrt`: +1e-4 on the diagonal, torch.svd on the
// host, a Python loop with one device->host sync per singular value, V diag(s^p) V^T).
//
// Here: one-sided (Hestenes) Jacobi in fp64, entirely on the device, no host synchronisation.
// W starts as A (+diag) and pairs of COLUMNS are rotated until mutually orthogonal; then column j of W
// is lambda_j v_j (A symmetric PSD), so f(A) = V f(L) V^T = W diag(f(l_j)/l_j^2) W^T needs no separate
// eigenvector accumulation.  One matrix = one thread-block CLUSTER: the n x n fp64 matrix lives in the
// cluster's distributed shared memory, two blocks of BC columns per CTA (BC = 32: 64 columns, 1024 threads, a
// whole SM per CTA — a 256 x 256 matrix is a 4-CTA cluster, so the 16 matrices of BASELINE config #3 are all
// co-resident; BC = 16 for order 512 where 64 columns would not fit shared memory), a warp per column pair.
// Block round-robin ordering: within a round a CTA orthogonalises its two column blocks against each
// other (BC steps x BC disjoint pairs; plus the pairs inside each block once per sweep); between rounds
// the blocks move to their next owners through DSMEM (circle-method tournament, two cluster barriers).
// In the cross steps a warp keeps ITS X column in registers for all BC steps (only the Y columns travel through
// shared memory): the steps are shared-memory-bandwidth bound (2 x 2 KiB read + written per pair and step).
// All CTAs of a cluster see the same convergence value, so the sweep loop exits uniformly.
#include "common.cuh"
#include "tuning.cuh"

namespace rpst {
namespace {

// columns per block (BC).  BC = 32 (one whole SM per CTA, 4-CTA clusters at order 256) when many matrices must be
// co-resident; BC = 16 (twice the SMs per matrix) for small batches: a step's cost grows with the pairs per SM
// (measured: order 256, one matrix 3.0 ms with BC = 16 vs 5.3 ms with BC = 32; 16 matrices 5.6 vs 5.4 ms).
constexpr bool eig_wide_ok(int np) { return np >= 64 && np <= 256; }

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_rank(const void* smem_ptr, uint32_t rank) {
    uint32_t local = static_cast<uint32_t>(__cvta_generic_to_shared(smem_ptr)), remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local), "r"(rank));
    return remote;
}
__device__ __forceinline__ double ld_cluster_f64(uint32_t addr) {
    double v;
    asm volatile("ld.shared::cluster.f64 %0, [%1];" : "=d"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// gmax is the largest |cos| between two columns seen BEFORE they were rotated in this sweep; Jacobi converges
// quadratically, so a sweep that saw 1e-8 leaves ~1e-16.  (1e-12 here cost one extra verification sweep in 11.)
constexpr double kEigConverged = 1e-8;

struct EigParams {
    const double* a;      // [batch, n, n] symmetric
    double diag_add;
    int n, np;            // logical / padded (multiple of 32) order
    int ctas;             // cluster size = np / 32
    int max_sweeps;
    double tol;           // stop after a sweep whose largest |cos| between two columns (before rotating them) was below this
    double* w;            // [batch, np, np]: column j at w + j*np (lambda_j v_j)
    double* lam;          // [batch, np]
    int* sweeps;          // [batch] or null
    const int* only;      // [batch] or null: matrices whose entry is 0 are skipped (every CTA of their cluster returns at once)
};

// circle-method tournament over m blocks: position -> block in round r and its inverse
__device__ __forceinline__ int block_at(int pos, int r, int m) { return pos == 0 ? 0 : 1 + (pos - 1 + r) % (m - 1); }
__device__ __forceinline__ int pos_of(int blk, int r, int m) {
    if (blk == 0) return 0;
    int v = (blk - 1 - r) % (m - 1);
    if (v < 0) v += m - 1;
    return 1 + v;
}

// The rotation angle is evaluated in fp32 from the squared column norms aa, bb (~lambda^2), the dot product gg and bb - aa.
// When aa or bb lies outside [2^-60, 2^60] all four are first scaled by a common power of two that brings aa * bb to ~1.
// Scaling by a power of two is exact in fp32 as long as nothing leaves the normal range, so the angle, the convergence
// value and the zero test are the same at every scale of the input either way.  (Unscaled, aa * bb overflowed fp32 for
// lambda_i lambda_j > ~1.8e19, and such pairs counted as converged without being rotated.)  False: aa or bb is not positive.
__device__ __forceinline__ bool angle_inputs(double aa, double bb, double gg, float& aaf, float& bbf, float& ggf, float& dif) {
    aaf = (float)aa; bbf = (float)bb; ggf = (float)gg; dif = (float)(bb - aa);   // difference in fp64: near-degenerate pairs cancel in fp32
    if (aaf >= 0x1p-60f && aaf <= 0x1p60f && bbf >= 0x1p-60f && bbf <= 0x1p60f) return true;
    if (!(aa > 0.0 && bb > 0.0)) return false;
    const int ea = (int)((__double_as_longlong(aa) >> 52) & 0x7ff), eb = (int)((__double_as_longlong(bb) >> 52) & 0x7ff);
    int e = 2046 - ((ea + eb) >> 1);                   // biased exponent of 2^-((ea + eb) / 2 - 1023)
    e = e < 1 ? 1 : (e > 2046 ? 2046 : e);
    const double sc = __longlong_as_double((long long)e << 52);
    aaf = (float)(aa * sc); bbf = (float)(bb * sc); ggf = (float)(gg * sc); dif = (float)((bb - aa) * sc);
    return true;
}

// rotate columns x, y (length 32*ROWS, in shared memory) so that they become orthogonal; returns |cos angle|
template <int ROWS>
__device__ __forceinline__ double rotate_pair(double* x, double* y, int lane) {
    double xv[ROWS], yv[ROWS];
    double aa = 0.0, bb = 0.0, gg = 0.0;
#pragma unroll
    for (int i = 0; i < ROWS; ++i) {
        xv[i] = x[i * 32 + lane];
        yv[i] = y[i * 32 + lane];
        aa = fma(xv[i], xv[i], aa);
        bb = fma(yv[i], yv[i], bb);
        gg = fma(xv[i], yv[i], gg);
    }
    aa = warp_sum_f64(aa);
    bb = warp_sum_f64(bb);
    gg = warp_sum_f64(gg);
    // The rotation ANGLE only steers convergence (Jacobi is self-correcting), so it is evaluated in fp32 (angle_inputs);
    // orthogonality of the rotation (c^2 + s^2 = 1) is what preserves the spectrum, so c, s are fp64.
    float aaf, bbf, ggf, dif;
    if (!angle_inputs(aa, bb, gg, aaf, bbf, ggf, dif)) return 0.0;
    const float prod = aaf * bbf;
    if (!(prod > 0.f)) return 0.0;
    const float relf = fabsf(ggf) * rsqrtf(prod);
    if (relf <= 1e-15f) return (double)relf;
    const float zeta = dif / (2.f * ggf);
    const float tf = copysignf(1.f, zeta) / (fabsf(zeta) + sqrtf(fmaf(zeta, zeta, 1.f)));
    const double t = (double)tf;
    const double c = rsqrt(fma(t, t, 1.0));
    const double s = c * t;
    const double rel = (double)relf;
#pragma unroll
    for (int i = 0; i < ROWS; ++i) {
        x[i * 32 + lane] = c * xv[i] - s * yv[i];
        y[i * 32 + lane] = s * xv[i] + c * yv[i];
    }
    return rel;
}

// Cross-pair step with TRACKED squared norms: aa (this warp's X column, a register) and bb (the Y column, from shared
// memory) are updated analytically after the rotation (|x'|^2 = aa - t g, |y'|^2 = bb + t g: Rutishauser), so a step
// needs ONE dot product and one warp reduction instead of three.  The norms are recomputed from the data at the start
// of every round, so rounding drift is bounded by one round; they only steer the rotation ANGLE (c^2 + s^2 = 1 holds
// exactly), and Jacobi is self-correcting in the angle.
template <int ROWS>
__device__ __forceinline__ double rotate_pair_tracked(double (&xv)[ROWS], double* y, double& aa, double& bb, int lane) {
    double yv[ROWS];
    double gg = 0.0;
#pragma unroll
    for (int i = 0; i < ROWS; ++i) {
        yv[i] = y[i * 32 + lane];
        gg = fma(xv[i], yv[i], gg);
    }
    gg = warp_sum_f64(gg);
    float aaf, bbf, ggf, dif;
    if (!angle_inputs(aa, bb, gg, aaf, bbf, ggf, dif)) return 0.0;
    const float prod = aaf * bbf;
    if (!(prod > 0.f)) return 0.0;
    const float relf = fabsf(ggf) * rsqrtf(prod);
    if (relf <= 1e-15f) return (double)relf;
    const float zeta = dif / (2.f * ggf);
    const float tf = copysignf(1.f, zeta) / (fabsf(zeta) + sqrtf(fmaf(zeta, zeta, 1.f)));
    const double t = (double)tf;
    const double c = rsqrt(fma(t, t, 1.0));
    const double s = c * t;
#pragma unroll
    for (int i = 0; i < ROWS; ++i) {
        const double xo = xv[i];
        xv[i] = c * xo - s * yv[i];
        y[i * 32 + lane] = s * xo + c * yv[i];
    }
    aa = fma(-t, gg, aa);
    bb = fma(t, gg, bb);
    return (double)relf;
}

template <int ROWS, int BC>   // padded order np = 32*ROWS, BC columns per block, cluster of np / (2 BC) CTAs
__global__ void __launch_bounds__(32 * BC, (BC == 16 && ROWS < 16) ? 2 : 1) jacobi_cluster_kernel(EigParams p) {
    constexpr int kBlockCols = BC, kCtaCols = 2 * BC, kEigThreads = 32 * BC;
    extern __shared__ __align__(16) unsigned char eig_smem[];
    double* cols = reinterpret_cast<double*>(eig_smem);            // [32][np]
    double* conv = cols + (size_t)kCtaCols * p.np;                 // [2]: per-sweep local maxima (double buffered)
    __shared__ double warp_max[kBlockCols];
    __shared__ double ynorm[kBlockCols];                           // tracked squared norms of the Y block's columns

    const int B = p.ctas, m = 2 * B;
    const int rank = (int)cluster_ctarank();
    const int batch = blockIdx.x / B;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int np = 32 * ROWS;
    const int n = p.n;
    const double* A = p.a + (size_t)batch * n * n;
    if (p.only && p.only[batch] == 0) return;      // uniform across the cluster: nobody reaches a cluster barrier

    // round-0 arrangement: slot 0 = block `rank`, slot 1 = block m-1-rank (block b = columns 16b..16b+15).
    // Column j of the symmetric input = row j; the padding extends A with an identity block.
    for (int e = threadIdx.x; e < kCtaCols * np; e += kEigThreads) {
        const int lc = e / np, row = e % np;
        const int blk = lc < kBlockCols ? rank : m - 1 - rank;
        const int col = blk * kBlockCols + (lc % kBlockCols);
        double v;
        if (col < n && row < n) v = A[(size_t)col * n + row] + (col == row ? p.diag_add : 0.0);
        else v = (col == row) ? 1.0 : 0.0;
        cols[e] = v;
    }
    if (threadIdx.x < 2) conv[threadIdx.x] = 0.0;
    __syncthreads();
    cluster_sync_all();

    int sweep = 0;
    for (; sweep < p.max_sweeps; ++sweep) {
        double wmax = 0.0;
        for (int r = 0; r < m - 1; ++r) {
            if (r == 0) {
                // pairs inside each block (once per sweep): the lower half of the warps takes block X, the upper block Y
                const int half = warp / (kBlockCols / 2), k = warp % (kBlockCols / 2);
                double* base = cols + (size_t)half * kBlockCols * np;
                for (int t = 0; t < kBlockCols - 1; ++t) {
                    const int c0 = block_at(k, t, kBlockCols), c1 = block_at(kBlockCols - 1 - k, t, kBlockCols);
                    wmax = fmax(wmax, rotate_pair<ROWS>(base + (size_t)c0 * np, base + (size_t)c1 * np, lane));
                    __syncthreads();
                }
            }
            // cross pairs: X_i with Y_(i+s); X_i stays in this warp's registers for the whole round
            {
                double xv[ROWS];
                double* xcol = cols + (size_t)warp * np;
                double* ycol = cols + (size_t)(kBlockCols + warp) * np;
                double aa = 0.0, yy = 0.0;
#pragma unroll
                for (int i = 0; i < ROWS; ++i) {
                    xv[i] = xcol[i * 32 + lane];
                    const double yw = ycol[i * 32 + lane];
                    aa = fma(xv[i], xv[i], aa);
                    yy = fma(yw, yw, yy);
                }
                aa = warp_sum_f64(aa);
                yy = warp_sum_f64(yy);
                if (lane == 0) ynorm[warp] = yy;
                __syncthreads();
                for (int s = 0; s < kBlockCols; ++s) {
                    const int j = (warp + s) & (kBlockCols - 1);
                    double bb = ynorm[j];
                    wmax = fmax(wmax, rotate_pair_tracked<ROWS>(xv, cols + (size_t)(kBlockCols + j) * np, aa, bb, lane));
                    if (lane == 0) ynorm[j] = bb;
                    __syncthreads();
                }
#pragma unroll
                for (int i = 0; i < ROWS; ++i) xcol[i * 32 + lane] = xv[i];
            }
            const bool last_round = r == m - 2;
            if (last_round) {
                if (lane == 0) warp_max[warp] = wmax;
                __syncthreads();
                if (threadIdx.x == 0) {
                    double v = 0.0;
                    for (int w = 0; w < kBlockCols; ++w) v = fmax(v, warp_max[w]);
                    conv[sweep & 1] = v;
                }
                __syncthreads();
            }
            // ---- move the blocks to their owners of the next round (== round 0 after the last one)
            cluster_sync_all();                      // everyone finished rotating / publishing conv
            const int rn = (r + 1) % (m - 1);
            double stage[2][ROWS];                   // 16*np / 512 values per thread and slot
#pragma unroll
            for (int slot = 0; slot < 2; ++slot) {
                const int pos = slot == 0 ? rank : m - 1 - rank;
                const int blk = block_at(pos, rn, m);
                const int old = pos_of(blk, r, m);
                const int src_rank = old < B ? old : m - 1 - old;
                const int src_slot = old < B ? 0 : 1;
                const uint32_t src = map_to_rank(cols + (size_t)src_slot * kBlockCols * np, (uint32_t)src_rank);
#pragma unroll
                for (int i = 0; i < ROWS; ++i)
                    stage[slot][i] = ld_cluster_f64(src + (uint32_t)((i * kEigThreads + threadIdx.x) * 8));
            }
            double gmax = 0.0;
            if (last_round)
                for (int c = 0; c < B; ++c) gmax = fmax(gmax, ld_cluster_f64(map_to_rank(&conv[sweep & 1], (uint32_t)c)));
            cluster_sync_all();                      // everyone finished reading
#pragma unroll
            for (int slot = 0; slot < 2; ++slot)
#pragma unroll
                for (int i = 0; i < ROWS; ++i)
                    cols[(size_t)slot * kBlockCols * np + i * kEigThreads + threadIdx.x] = stage[slot][i];
            __syncthreads();
            if (last_round && gmax < p.tol) { ++sweep; goto done; }   // uniform across the cluster
        }
    }
done:
    // arrangement is round 0 again: slot 0 = block rank, slot 1 = block m-1-rank
    double* W = p.w + (size_t)batch * np * np;
    for (int e = threadIdx.x; e < kCtaCols * np; e += kEigThreads) {
        const int lc = e / np, row = e % np;
        const int blk = lc < kBlockCols ? rank : m - 1 - rank;
        W[(size_t)(blk * kBlockCols + (lc % kBlockCols)) * np + row] = cols[e];
    }
    for (int lc = warp; lc < kCtaCols; lc += kBlockCols) {
        double ss = 0.0;
        for (int i = lane; i < np; i += 32) ss = fma(cols[(size_t)lc * np + i], cols[(size_t)lc * np + i], ss);
        ss = warp_sum_f64(ss);
        const int blk = lc < kBlockCols ? rank : m - 1 - rank;
        if (lane == 0) p.lam[(size_t)batch * np + blk * kBlockCols + (lc % kBlockCols)] = sqrt(ss);
    }
    if (p.sweeps && rank == 0 && threadIdx.x == 0) p.sweeps[batch] = sweep;
    cluster_sync_all();   // no CTA may exit while others still read its shared memory
}

// out[b] (n x n, row-major, ld n) = sum_j g(lam_j) w_j w_j^T restricted to the first n rows,
// g = lam^(power) / lam^2, dropped where lam < cut (network/wct_rp.py:14-17: spectrum truncated at 1e-5)
__global__ void __launch_bounds__(256) matfn_kernel(const double* __restrict__ w, const double* __restrict__ lam, int n,
                                                    int np, double power, double cut, double* __restrict__ out,
                                                    const int* __restrict__ only) {
    __shared__ double wi[16][17], wj[16][17], g[16];
    const int b = blockIdx.z;
    if (only && only[b] == 0) return;
    const double* W = w + (size_t)b * np * np;
    const double* L = lam + (size_t)b * np;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int i = blockIdx.y * 16 + ty, j = blockIdx.x * 16 + tx;
    double acc = 0.0;
    for (int c0 = 0; c0 < np; c0 += 16) {
        // tile of columns c0..c0+15: rows i-tile and j-tile
        const int col = c0 + ty;
        wi[ty][tx] = W[(size_t)col * np + blockIdx.y * 16 + tx];
        wj[ty][tx] = W[(size_t)col * np + blockIdx.x * 16 + tx];
        if (threadIdx.x < 16) {
            const double l = L[c0 + threadIdx.x];
            g[threadIdx.x] = l >= cut ? pow(l, power - 2.0) : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int c = 0; c < 16; ++c) acc = fma(g[c] * wi[c][ty], wj[c][tx], acc);
        __syncthreads();
    }
    if (i < n && j < n) out[(size_t)b * n * n + (size_t)i * n + j] = acc;
}

}  // namespace

// ---- internal host API -------------------------------------------------------------------------
int eig_padded_order(int n) {
    int np = 32;
    while (np < n) np *= 2;   // 32, 64, 128, 256, 512: cluster sizes 1, 2, 4, 8, 16
    return np;
}

size_t eig_workspace_bytes(int64_t batch, int n) {
    const size_t np = eig_padded_order(n);
    return align_up((size_t)batch * np * np * sizeof(double), 256) + align_up((size_t)batch * np * sizeof(double), 256);
}

// a [batch,n,n] -> W/lam in workspace
int eig_decompose(const double* a, int64_t batch, int n, double diag_add, void* ws, size_t ws_bytes, double** w_out,
                  double** lam_out, int* sweeps, cudaStream_t stream, double tol, const int* only) {
    RPST_CHECK_ARG(n >= 1 && n <= 512, "sym_eig: order must be in [1, 512] (got %d)", n);
    const int np = eig_padded_order(n);
    if (ws_bytes < eig_workspace_bytes(batch, n)) {
        set_error("sym_eig: workspace too small (%zu < %zu bytes)", ws_bytes, eig_workspace_bytes(batch, n));
        return RPST_ERR_WORKSPACE;
    }
    double* w = static_cast<double*>(ws);
    double* lam = reinterpret_cast<double*>(static_cast<char*>(ws) + align_up((size_t)batch * np * np * sizeof(double), 256));
    EigParams p{};
    // 16-column blocks (np/32 CTAs per matrix) until they need more than ~one CTA per SM; 15 eight-CTA clusters are
    // co-resident at one CTA per SM (cudaOccupancyMaxActiveClusters), a 16th shares SMs: 16 x 256^2 4.43 ms against
    // 4.77 with 32-column blocks (4 CTAs per matrix, 64 SMs); from 160 CTAs on the wide blocks win (32 x 256^2: 4.94 / 5.31)
    bool wide = eig_wide_ok(np) && batch * (np / 32) > 160;
    if (g_knobs.eig_wide >= 0 && eig_wide_ok(np)) wide = g_knobs.eig_wide == 1;
    const bool spread = g_knobs.eig_wide == 2;   // 16-column blocks, shared memory padded so that one CTA fits per SM
    const int bc = wide ? 32 : 16, cta_cols = 2 * bc;
    p.a = a; p.diag_add = diag_add; p.n = n; p.np = np; p.ctas = np / cta_cols; p.max_sweeps = 20;
    p.tol = tol > 0.0 ? tol : kEigConverged;
    p.w = w; p.lam = lam; p.sweeps = sweeps; p.only = only;
    size_t smem = (size_t)cta_cols * np * sizeof(double) + 2 * sizeof(double);
    if (spread && smem < (120u << 10)) smem = 120u << 10;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(batch * p.ctas));
    cfg.blockDim = dim3(32 * bc);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)p.ctas;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
#define RPST_EIG_CASE(R, BC)                                                                                       \
    case R + 100 * (BC == 32): {                                                                                   \
        static PerDeviceFlag configured_on;                                                                        \
        bool& configured = configured_on.get();                                                                    \
        if (!configured) {                                                                                         \
            RPST_CUDA(cudaFuncSetAttribute(jacobi_cluster_kernel<R, BC>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                           (int)(smem > (120u << 10) ? smem : (120u << 10))));                     \
            if (32 * R / (2 * BC) > 8)                                                                             \
                RPST_CUDA(cudaFuncSetAttribute(jacobi_cluster_kernel<R, BC>,                                       \
                                               cudaFuncAttributeNonPortableClusterSizeAllowed, 1));                \
            configured = true;                                                                                     \
        }                                                                                                          \
        if (g_knobs.eig_wide == -2 || g_knobs.eig_wide == 2) {                                                     \
            int nc = 0;                                                                                            \
            RPST_CUDA(cudaOccupancyMaxActiveClusters(&nc, jacobi_cluster_kernel<R, BC>, &cfg));                    \
            fprintf(stderr, "[rpst] jacobi<%d,%d>: cluster %d, max active clusters %d\n", R, BC, p.ctas, nc);      \
        }                                                                                                          \
        RPST_CUDA(cudaLaunchKernelEx(&cfg, jacobi_cluster_kernel<R, BC>, p));                                      \
        break;                                                                                                     \
    }
    switch (np / 32 + 100 * (bc == 32)) {
        RPST_EIG_CASE(1, 16)
        RPST_EIG_CASE(2, 16)
        RPST_EIG_CASE(4, 16)
        RPST_EIG_CASE(8, 16)
        RPST_EIG_CASE(16, 16)
        RPST_EIG_CASE(2, 32)
        RPST_EIG_CASE(4, 32)
        RPST_EIG_CASE(8, 32)
        default:
            set_error("sym_eig: unsupported padded order %d", np);
            return RPST_ERR_UNSUPPORTED;
    }
#undef RPST_EIG_CASE
    *w_out = w;
    *lam_out = lam;
    return RPST_OK;
}

int eig_matfn(const double* w, const double* lam, int64_t batch, int n, double power, double cut, double* out,
              cudaStream_t stream, const int* only) {
    const int np = eig_padded_order(n);
    dim3 grid((unsigned)((n + 15) / 16), (unsigned)((n + 15) / 16), (unsigned)batch);
    matfn_kernel<<<grid, 256, 0, stream>>>(w, lam, n, np, power, cut, out, only);
    RPST_CUDA(cudaGetLastError());
    return RPST_OK;
}

}  // namespace rpst

using namespace rpst;

extern "C" size_t rpst_sym_eig_fn_workspace_bytes(int64_t batch, int64_t n) {
    if (batch <= 0 || n <= 0 || n > 512) return 256;
    return eig_workspace_bytes(batch, (int)n);
}

extern "C" int rpst_sym_eig_fn(const double* a, int64_t batch, int64_t n, double diag_add, double* out_sqrt,
                               double* out_inv_sqrt, double* eigenvalues, int32_t* sweeps, void* workspace,
                               size_t workspace_bytes, void* stream) {
    RPST_CHECK_ARG(batch >= 0 && n >= 0, "sym_eig: negative size");
    if (batch == 0 || n == 0) return RPST_OK;
    RPST_CHECK_ARG(a != nullptr && workspace != nullptr, "sym_eig: null pointer");
    RPST_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, "sym_eig: workspace must be 256-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    double *w, *lam;
    int rc = eig_decompose(a, batch, (int)n, diag_add, workspace, workspace_bytes, &w, &lam, sweeps, st, 0.0, nullptr);
    if (rc) return rc;
    // network/wct_rp.py:14-17 / 32-35: the spectrum is cut at the first value below 1e-5
    if (out_sqrt && (rc = eig_matfn(w, lam, batch, (int)n, 0.5, 1e-5, out_sqrt, st, nullptr))) return rc;
    if (out_inv_sqrt && (rc = eig_matfn(w, lam, batch, (int)n, -0.5, 1e-5, out_inv_sqrt, st, nullptr))) return rc;
    if (eigenvalues) {
        const int np = eig_padded_order((int)n);
        RPST_CUDA(cudaMemcpy2DAsync(eigenvalues, (size_t)n * sizeof(double), lam, (size_t)np * sizeof(double),
                                    (size_t)n * sizeof(double), (size_t)batch, cudaMemcpyDeviceToDevice, st));
    }
    return RPST_OK;
}

// WCT whitening / colouring — SURVEY.md §8 a6/a7; reference: network/wct_rp.py:82-114
// (`whiten_and_color`) and :157-166 (`fuse`: per-sample Python loop, fp64 inside, three host SVDs with
// 768 `.item()` syncs per sample).
//
// Device pipeline for a whole batch, no host synchronisation:
//   1. channel means of content and style                (TMA-staged statistics kernel, adain.cu)
//   2. per sample and tensor: centred bf16 hi/lo operand tiles, then Xc.Xc^T on the tensor cores
//      (tcgen05, bf16x3 = fp32-grade, split-K over H*W across all SMs), reduced to fp64 covariance
//      (/(HW-1), +I on the content covariance only, network/wct_rp.py:89,94)
//   3. batched over samples: cluster-resident Jacobi eigensolver (eig.cu) -> C^(1/2), C^(-1/2); the
//      closed-form (Lu et al., default) transform T = C^(-1/2) (C^(1/2) S C^(1/2))^(1/2) C^(-1/2) or the
//      original (Li et al.) T = S^(1/2) C^(-1/2), small fp64 products on CUDA cores
//   4. per sample: out = T.X + (mu_s - T.mu_c) as one tensor-core GEMM with a bias epilogue
#include "common.cuh"
#include "tuning.cuh"

namespace rpst {

size_t packed_operand_bytes(int64_t rows, int64_t k);
int pack_operand_shift(const float* x, int64_t rows, int64_t k, int64_t stride_r, int64_t stride_k,
                       const float* row_scale, const float* row_shift, void* hi, void* lo, cudaStream_t stream);
int gemm_packed_splitk(const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo, float* out, int64_t m,
                       int64_t n, int64_t k, int64_t ldo, int passes, float alpha, const float* row_add,
                       const float* col_add, int splits, int64_t split_stride, cudaStream_t stream);
int eig_padded_order(int n);
size_t eig_workspace_bytes(int64_t batch, int n);
int eig_decompose(const double* a, int64_t batch, int n, double diag_add, void* ws, size_t ws_bytes, double** w_out,
                  double** lam_out, int* sweeps, cudaStream_t stream, double tol, const int* only);
int eig_matfn(const double* w, const double* lam, int64_t batch, int n, double power, double cut, double* out,
              cudaStream_t stream, const int* only);
// nsroot.cu: Newton-Schulz roots of positive definite matrices; flag[b] = 1 where the Jacobi path must take over
size_t ns_roots_workspace_bytes(int64_t batch, int n);
int ns_roots(const double* a, int64_t batch, int n, double diag_add, double lmin, double* root, double* iroot, int* flag,
             void* workspace, size_t workspace_bytes, cudaStream_t st);
int dgemm_batched(const double* a, const double* b, double* c, int64_t batch, int n, cudaStream_t st);
// Jacobi stop for the WCT's own decompositions: a sweep that saw |cos| < 1e-5 leaves ~1e-10 (quadratic convergence),
// far below the fp32-grade covariances that go in; the public rpst_sym_eig_fn keeps 1e-8 (-> 1e-16).  One sweep less.
constexpr double kWctEigTol = 1e-5;
// cov.cu: one kernel from fp32 features to the centred covariance (conversion + centring inside the SYRK)
bool cov_fused_supported(const float* x, int64_t c, int64_t hw);
size_t cov_fused_workspace_bytes(int64_t c);
int cov_fused(const float* x, int64_t c, int64_t hw, int passes, double diag_add, double* cov, float* mean, void* workspace,
              cudaStream_t st, const float* shift_in, int path, int* taken);
int cov_shifts_batched(const float* x, int64_t n, int64_t c, int64_t hw, float* shifts, cudaStream_t st);
// gemm.cu / pwconv.cu: out = T (x - mu_c) + mu_s with the transposed bf16 operand built on the fly
int pack_operand_batched(const float* x, int64_t rows, int64_t k, int64_t stride_r, int64_t stride_k,
                         const float* row_scale, const float* row_shift, void* hi, void* lo, int batch, int64_t x_batch,
                         int64_t tile_batch_bytes, int64_t vec_batch, cudaStream_t stream);
bool wct_apply_fused_supported(int64_t c, int64_t hw);
int wct_apply_fused(const float* x, const float* mu_c, const float* mu_s, const void* t_hi, const void* t_lo, float* out,
                    int64_t n, int64_t t_batch_bytes, int64_t c, int64_t hw, int passes, cudaStream_t st);

namespace {

// cov[i][j] = sum_z partial[z][i][j] / (hw-1) (+1 on the diagonal)
__global__ void cov_reduce_kernel(const float* __restrict__ partial, int splits, int c, double inv_dof,
                                  double diag_add, double* __restrict__ cov) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= c * c) return;
    double acc = 0.0;
    for (int z = 0; z < splits; ++z) acc += (double)partial[(size_t)z * c * c + idx];
    const int i = idx / c, j = idx % c;
    cov[idx] = acc * inv_dof + (i == j ? diag_add : 0.0);
}

// t32 = (float) T ; bias[i] = mu_s[i] - sum_j T[i][j] mu_c[j]
__global__ void transform_finalize_kernel(const double* __restrict__ t, const float* __restrict__ mu_c,
                                          const float* __restrict__ mu_s, int c, float* __restrict__ t32,
                                          float* __restrict__ bias) {
    // blockIdx.y: sample (T [n,c,c], mu_* [n,c], t32 [n,c,c], bias [n,c])
    t += (size_t)blockIdx.y * c * c; mu_c += (size_t)blockIdx.y * c; mu_s += (size_t)blockIdx.y * c;
    t32 += (size_t)blockIdx.y * c * c; bias += (size_t)blockIdx.y * c;
    const int i = blockIdx.x;
    double acc = 0.0;
    for (int j = threadIdx.x; j < c; j += blockDim.x) {
        const double v = t[(size_t)i * c + j];
        t32[(size_t)i * c + j] = (float)v;
        acc += v * (double)mu_c[j];
    }
    __shared__ double red[32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
        bias[i] = (float)((double)mu_s[i] - s);
    }
}

struct WctLayout {
    size_t stats, mean_c, mean_s, cov_tiles_hi, cov_tiles_lo, partial, cov_c, cov_s, flag, ns, eig, mats[6], t32, bias,
        t_hi, t_lo, x_hi, x_lo, fused, shifts, t_tile, total;
    int splits;
};

int cov_splits(int64_t c, int64_t hw) {
    const int64_t tiles = ((c + 127) / 128) * ((c + 255) / 256);   // 128 x 256 output tiles of the GEMM
    int64_t s = sm_count() / tiles;
    if (s < 1) s = 1;
    const int64_t kt = (hw + 63) / 64;
    if (s > kt) s = kt;
    const int64_t per = (kt + s - 1) / s;
    return (int)((kt + per - 1) / per);
}

WctLayout wct_layout(int64_t n, int64_t c, int64_t hw_c, int64_t hw_s) {
    WctLayout l;
    const int64_t hw_max = hw_c > hw_s ? hw_c : hw_s;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o += align_up(bytes, 256); return at; };
    l.stats = take(rpst_stats_workspace_bytes(n * c, hw_max));
    l.mean_c = take((size_t)n * c * sizeof(float));
    l.mean_s = take((size_t)n * c * sizeof(float));
    l.cov_tiles_hi = take(packed_operand_bytes(c, hw_max));
    l.cov_tiles_lo = take(packed_operand_bytes(c, hw_max));
    const int sc = cov_splits(c, hw_c), ss = cov_splits(c, hw_s);
    l.splits = sc > ss ? sc : ss;
    l.partial = take((size_t)l.splits * c * c * sizeof(float));
    l.cov_c = take((size_t)n * c * c * sizeof(double));
    l.cov_s = take((size_t)n * c * c * sizeof(double));
    l.flag = take((size_t)n * sizeof(int));
    l.ns = take(ns_roots_workspace_bytes(n, (int)c));
    l.eig = take(eig_workspace_bytes(n, (int)c));
    for (int i = 0; i < 6; ++i) l.mats[i] = take((size_t)n * c * c * sizeof(double));
    l.t_tile = align_up(packed_operand_bytes(c, c), 256);          // per-sample stride of the packed transforms
    l.t32 = take((size_t)n * c * c * sizeof(float));
    l.bias = take((size_t)n * c * sizeof(float));
    l.t_hi = take((size_t)n * l.t_tile);
    l.t_lo = take((size_t)n * l.t_tile);
    l.x_hi = take(packed_operand_bytes(hw_c, c));
    l.x_lo = take(packed_operand_bytes(hw_c, c));
    l.fused = take(c <= 256 ? cov_fused_workspace_bytes(c) : 0);
    l.shifts = take((size_t)2 * n * 256 * sizeof(float));
    l.total = o;
    return l;
}

// Steps 1-2 for n contiguous [c, hw] tensors: channel means mean [n, c] (fp32) and centred covariances cov [n, c, c] (fp64,
// / (hw - 1), + diag_add on the diagonal).  path kCovPathAuto: the fused kernels of cov.cu where the shape allows (cov_fused
// picks the one-launch TMA kernel or the register-staged one), else pack + split-K GEMM + reduce; the other values force
// one path (tests).  *taken (may be null) receives the path that ran.  `shifts` holds n * 256 floats.
int wct_covariances(const float* x, int64_t n, int64_t c, int64_t hw, int passes, double diag_add, int path, double* cov,
                    float* mean, float* shifts, const WctLayout& l, char* w, int* taken, cudaStream_t st) {
    const bool fused_ok = cov_fused_supported(x, c, hw) && (c * hw) % 4 == 0;
    if (path == kCovPathAuto && !(g_knobs.wct_fused_cov && fused_ok)) path = kCovPathPack;
    if (path != kCovPathPack) {
        RPST_CHECK_ARG(fused_ok, "wct covariance: the fused kernels need c <= 256, hw >= 64, hw %% 4 == 0 and 16-byte "
                                 "aligned rows (c %lld, hw %lld)", (long long)c, (long long)hw);
        // 1+2. means and centred covariances from ONE pass over each tensor (cov.cu); the centring shifts of all n tensors
        // in one small launch (inside the covariance launch they cost a grid barrier each)
        int rc = cov_shifts_batched(x, n, c, hw, shifts, st);
        if (rc) return rc;
        const int cp = c <= 128 ? 128 : 256;
        for (int64_t i = 0; i < n; ++i)
            if ((rc = cov_fused(x + i * c * hw, c, hw, passes, diag_add, cov + i * c * c, mean + i * c, w + l.fused, st,
                                shifts + i * cp, path, taken))) return rc;
        return RPST_OK;
    }
    // 1. channel means (network/wct_rp.py:85,92)
    int rc = rpst_stats_nchw(x, n * c, hw, 0.f, mean, nullptr, w + l.stats, l.mean_c - l.stats, st);
    if (rc) return rc;
    // 2. covariances
    void* ct_hi = w + l.cov_tiles_hi;
    void* ct_lo = w + l.cov_tiles_lo;
    float* partial = reinterpret_cast<float*>(w + l.partial);
    const int cc = (int)(c * c);
    const int splits = cov_splits(c, hw);
    for (int64_t i = 0; i < n; ++i) {
        rc = pack_operand_shift(x + i * c * hw, c, hw, hw, 1, nullptr, mean + i * c, ct_hi, passes == 3 ? ct_lo : nullptr, st);
        if (rc) return rc;
        rc = gemm_packed_splitk(ct_hi, ct_lo, ct_hi, ct_lo, partial, c, c, hw, c, passes, 1.f, nullptr, nullptr, splits, c * c, st);
        if (rc) return rc;
        cov_reduce_kernel<<<(cc + 255) / 256, 256, 0, st>>>(partial, splits, (int)c, 1.0 / ((double)hw - 1.0), diag_add,
                                                           cov + i * c * c);
        RPST_CUDA(cudaGetLastError());
    }
    if (taken) *taken = kCovPathPack;
    return RPST_OK;
}

}  // namespace
}  // namespace rpst

using namespace rpst;

extern "C" size_t rpst_wct_workspace_bytes(int64_t n, int64_t c, int64_t hw_c, int64_t hw_s) {
    if (n <= 0 || c <= 0 || hw_c <= 0 || hw_s <= 0 || c > 512) return 256;
    return wct_layout(n, c, hw_c, hw_s).total;
}

extern "C" int rpst_wct_fuse(const float* content, const float* style, float* out, int64_t n, int64_t c, int64_t hw_c,
                             int64_t hw_s, int method, int passes, double* transform_out, void* workspace,
                             size_t workspace_bytes, void* stream) {
    RPST_CHECK_ARG(n >= 0 && c >= 0 && hw_c >= 0 && hw_s >= 0, "wct: negative size");
    if (n == 0 || c == 0 || hw_c == 0) return RPST_OK;
    RPST_CHECK_ARG(content && style && out, "wct: null pointer");
    RPST_CHECK_ARG(hw_c >= 2 && hw_s >= 2, "wct: need at least two positions per feature map");
    RPST_CHECK_ARG(c <= 512, "wct: at most 512 channels (got %lld)", (long long)c);
    RPST_CHECK_ARG(method == 0 || method == 1, "wct: method must be 0 (closed-form) or 1 (original)");
    RPST_CHECK_ARG(passes == 1 || passes == 3, "wct: passes must be 1 (bf16) or 3 (bf16x3, fp32-grade)");
    const WctLayout l = wct_layout(n, c, hw_c, hw_s);
    if (!workspace || workspace_bytes < l.total) {
        set_error("wct: workspace too small (%zu < %zu bytes)", workspace_bytes, l.total);
        return RPST_ERR_WORKSPACE;
    }
    RPST_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, "wct: workspace must be 256-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    char* w = static_cast<char*>(workspace);
    float* mean_c = reinterpret_cast<float*>(w + l.mean_c);
    float* mean_s = reinterpret_cast<float*>(w + l.mean_s);
    int rc;
    double* cov_c = reinterpret_cast<double*>(w + l.cov_c);
    double* cov_s = reinterpret_cast<double*>(w + l.cov_s);
    // 1+2. means and covariances (network/wct_rp.py:85-94, + I on the content side); both tensors take the same path
    const bool fused = g_knobs.wct_fused_cov && cov_fused_supported(content, c, hw_c) && cov_fused_supported(style, c, hw_s) &&
                       (c * hw_c) % 4 == 0 && (c * hw_s) % 4 == 0;
    const int path = fused ? kCovPathAuto : kCovPathPack;
    float* shifts = reinterpret_cast<float*>(w + l.shifts);
    if ((rc = wct_covariances(content, n, c, hw_c, passes, 1.0, path, cov_c, mean_c, shifts, l, w, nullptr, st))) return rc;
    if ((rc = wct_covariances(style, n, c, hw_s, passes, 0.0, path, cov_s, mean_s, shifts + n * 256, l, w, nullptr, st))) return rc;
    // 3. transform matrices, batched over samples (all fp64)
    double* m[6];
    for (int i = 0; i < 6; ++i) m[i] = reinterpret_cast<double*>(w + l.mats[i]);
    double *ew, *el;
    const size_t eig_bytes = l.mats[0] - l.eig;
    double* T = m[5];
    // (A + 1e-4 I)^(+-1/2): Newton-Schulz where the matrix is positive definite as constructed (lmin), the Jacobi
    // eigensolver with the reference's |s| / 1e-5-cut semantics for the matrices that iteration flags (or for all of
    // them with the knob off)
    int* flag = reinterpret_cast<int*>(w + l.flag);
    auto roots = [&](const double* a, double lmin, double* root, double* iroot) -> int {
        const int* only = nullptr;
        if (g_knobs.wct_roots_ns && c > 64) {          // up to 64 channels the Jacobi solve is as fast as the iteration's launches
            if (int r = ns_roots(a, n, (int)c, 1e-4, lmin, root, iroot, flag, w + l.ns, l.eig - l.ns, st)) return r;
            only = flag;
        }
        if (int r = eig_decompose(a, n, (int)c, 1e-4, w + l.eig, eig_bytes, &ew, &el, nullptr, st, kWctEigTol, only)) return r;
        if (root) if (int r = eig_matfn(ew, el, n, (int)c, 0.5, 1e-5, root, st, only)) return r;
        if (iroot) if (int r = eig_matfn(ew, el, n, (int)c, -0.5, 1e-5, iroot, st, only)) return r;
        return RPST_OK;
    };
    double* iroot = m[1];
    if (method == 0) {
        double* root = m[0];
        if ((rc = roots(cov_c, 1.0, root, iroot))) return rc;                       // cov_c carries + I (network/wct_rp.py:87)
        if ((rc = dgemm_batched(root, cov_s, m[2], n, (int)c, st))) return rc;      // C^1/2 S
        if ((rc = dgemm_batched(m[2], root, m[3], n, (int)c, st))) return rc;       // C^1/2 S C^1/2
        if ((rc = roots(m[3], 1e-4, m[4], nullptr))) return rc;                     // middle^(1/2)
        if ((rc = dgemm_batched(iroot, m[4], m[2], n, (int)c, st))) return rc;
        if ((rc = dgemm_batched(m[2], iroot, T, n, (int)c, st))) return rc;
    } else {
        if ((rc = roots(cov_c, 1.0, nullptr, iroot))) return rc;
        if ((rc = roots(cov_s, 1e-4, m[4], nullptr))) return rc;                    // S^(1/2)
        if ((rc = dgemm_batched(m[4], iroot, T, n, (int)c, st))) return rc;
    }
    if (transform_out)
        RPST_CUDA(cudaMemcpyAsync(transform_out, T, (size_t)n * c * c * sizeof(double), cudaMemcpyDeviceToDevice, st));
    // 4. apply: out_i = T_i X_i + (mu_s - T_i mu_c)
    float* t32 = reinterpret_cast<float*>(w + l.t32);
    float* bias = reinterpret_cast<float*>(w + l.bias);
    // all samples at once: fp32 transforms + biases, packed transforms, and (fused path) ONE persistent colouring launch
    // over the batch with per-sample weights (16 launches of each kind before: their tails added up to ~15 us per sample)
    transform_finalize_kernel<<<dim3((unsigned)c, (unsigned)n), 128, 0, st>>>(T, mean_c, mean_s, (int)c, t32, bias);
    RPST_CUDA(cudaGetLastError());
    rc = pack_operand_batched(t32, c, c, c, 1, nullptr, nullptr, w + l.t_hi, w + l.t_lo, (int)n, c * c, (int64_t)l.t_tile, 0, st);
    if (rc) return rc;
    if (g_knobs.wct_fused_apply && wct_apply_fused_supported(c, hw_c))
        return wct_apply_fused(content, mean_c, mean_s, w + l.t_hi, w + l.t_lo, out, n, (int64_t)l.t_tile, c, hw_c, passes, st);
    for (int64_t i = 0; i < n; ++i) {
        rc = pack_operand_shift(content + i * c * hw_c, hw_c, c, 1, hw_c, nullptr, nullptr, w + l.x_hi,
                                passes == 3 ? w + l.x_lo : nullptr, st);
        if (rc) return rc;
        rc = gemm_packed_splitk(w + l.t_hi + i * l.t_tile, w + l.t_lo + i * l.t_tile, w + l.x_hi, w + l.x_lo, out + i * c * hw_c, c, hw_c,
                                c, hw_c, passes, 1.f, bias + i * c, nullptr, 1, 0, st);
        if (rc) return rc;
    }
    return RPST_OK;
}

#ifdef RPST_DEBUG_EXPORTS   // white-box test hooks: only in librpst_debug.so (loaded by tests alone), never in the product library
extern "C" size_t rpst_debug_wct_covariances_workspace_bytes(int64_t n, int64_t c, int64_t hw) {
    return rpst_wct_workspace_bytes(n, c, hw, hw);
}

// Test hook: steps 1-2 of rpst_wct_fuse (the same wct_covariances call) on one batch of n [c, hw] tensors, with the
// covariance path chosen by `path` (0 production dispatch, 1 one-launch TMA kernel at any grid, 2 register-staged kernel +
// finalize launches, 3 pack + split-K GEMM + reduce).  *path_taken (host) receives the path that ran.
extern "C" int rpst_debug_wct_covariances(const float* x, int64_t n, int64_t c, int64_t hw, int passes, double diag_add,
                                          int path, double* cov_out, float* mean_out, int32_t* path_taken, void* workspace,
                                          size_t workspace_bytes, void* stream) {
    RPST_CHECK_ARG(n > 0 && c > 0 && c <= 512 && hw >= 2, "debug_wct_covariances: bad sizes");
    RPST_CHECK_ARG(x && cov_out && mean_out && path_taken && workspace, "debug_wct_covariances: null pointer");
    RPST_CHECK_ARG(passes == 1 || passes == 3, "debug_wct_covariances: passes must be 1 or 3");
    RPST_CHECK_ARG(path >= kCovPathAuto && path <= kCovPathPack, "debug_wct_covariances: path must be 0..3");
    RPST_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, "debug_wct_covariances: workspace must be 256-byte aligned");
    const WctLayout l = wct_layout(n, c, hw, hw);
    if (workspace_bytes < l.total) {
        set_error("debug_wct_covariances: workspace too small (%zu < %zu bytes)", workspace_bytes, l.total);
        return RPST_ERR_WORKSPACE;
    }
    char* w = static_cast<char*>(workspace);
    int taken = -1;
    const int rc = wct_covariances(x, n, c, hw, passes, diag_add, path, cov_out, mean_out, reinterpret_cast<float*>(w + l.shifts),
                                   l, w, &taken, static_cast<cudaStream_t>(stream));
    *path_taken = taken;
    return rc;
}
#endif  // RPST_DEBUG_EXPORTS

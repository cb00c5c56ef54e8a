/* librpst — C ABI of the B200-native stylization transform for RP-Style-Transfer.
 *
 * The reference (LuletterSoul/RP-Style-Transfer) is pure Python/PyTorch and has no FFI of its own
 * (SURVEY.md §2b); each entry point below therefore cites the reference *Python* interface it
 * replaces (file:line relative to the reference root).  INTEGRATION.md shows the ctypes binding a
 * maintainer adds on the reference side.
 *
 * Conventions
 *  - plain pointers + sizes, no torch types; all tensors are contiguous NCHW fp32 device memory
 *    unless stated; labels are uint8; index outputs are int64.
 *  - the caller owns every buffer (inputs const, outputs and workspace pre-allocated); the library
 *    keeps no device allocations between calls.  `*_workspace_bytes` tells how much scratch a call
 *    needs; workspace contents need not be initialised.
 *  - every call only ENQUEUES work on `stream` (a cudaStream_t passed as void*); no host
 *    synchronisation, re-entrant, safe to drive one stream per device from one thread each.
 *  - return value: 0 on success, a negative RPST_ERR_* code otherwise; `rpst_last_error()` returns
 *    a thread-local human-readable message.  Nothing throws or aborts.
 */
#ifndef RPST_H_
#define RPST_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RPST_VERSION 100 /* major*100 + minor */

#if defined(__GNUC__)
#define RPST_API __attribute__((visibility("default")))
#else
#define RPST_API
#endif

#define RPST_OK 0
#define RPST_ERR_INVALID (-1)   /* bad argument / shape mismatch (Python side raises AssertionError) */
#define RPST_ERR_CUDA (-2)      /* a CUDA runtime call failed */
#define RPST_ERR_WORKSPACE (-3) /* workspace too small */
#define RPST_ERR_UNSUPPORTED (-4)

RPST_API int rpst_version(void);
RPST_API const char* rpst_last_error(void);
/* Tuning knobs: process-wide integers that select kernel paths and schedule parameters, for experiments and A/B
 * comparisons; the defaults are the production choice.  rpst_set_tuning returns RPST_ERR_INVALID and leaves the knob
 * as it was for an unknown name or a value outside the knob's range (rpst_last_error() names the range).
 * rpst_get_tuning returns the current value, or -1 for an unknown name ("wct_ns_flagged" also reads -1 when its counter
 * cannot be read).
 *
 *   name                        range         default    meaning
 * AdaIN (rpst_adain_fwd, rpst_adain_fwd_mapped, rpst_stats_nchw, rpst_adain_bwd):
 *   "adain_path"                0..1          0          0: TMA-staged kernel when planes are 16-byte aligned, 1: register-staged
 *                                                        kernel; 1 also turns off the segment AdaIN TMA kernel (rpst_seg_adain_fwd)
 *   "adain_lag_bytes"           0..INT64_MAX  33554432   content bytes kept L2-resident between a plane's statistics and its
 *                                                        apply (32 MiB); also used by the backward pass and by the
 *                                                        register-staged segment AdaIN kernel
 *   "adain_big_lag_bytes"       0..INT64_MAX  134217728  the same for planes of 4 MiB and more (128 MiB)
 *   "adain_mvn_lag_bytes"       0..INT64_MAX  46137344   the same for mean_variance_norm, i.e. style == NULL (44 MiB)
 *   "adain_hints"               0..1          1          L2 eviction-priority hints on the streaming loads / stores (the
 *                                                        register-staged segment AdaIN kernel too)
 *   "adain_twin_apply"          0..1          1          TMA kernel without prev: each apply item carries two content chunks
 *   "adain_group_merge_min_spp" 0..INT64_MAX  512        TMA kernel: planes with at least this many statistics slots are merged
 *                                                        by a whole warp group instead of one warp
 *   "adain_merge_lead"          0..INT64_MAX  0          TMA kernel: planes between a plane's merge and its first apply, clamped
 *                                                        to 1..lag-1; 0: lag / 2
 * Segment AdaIN, TMA kernel (rpst_seg_adain_fwd, rpst_seg_adain_fwd_mapped):
 *   "seg_lag_bytes"             0..INT64_MAX  268435456  content bytes between a plane's statistics and its apply (256 MiB)
 * SANet attention (rpst_sanet_attn_fwd):
 *   "attn_flash"                0..1          1          1: C = 512 attention runs as one flash-style kernel when the shape
 *                                                        allows; 0: GEMM -> rows -> GEMM
 *   "attn_flash_prof"           0..INT64_MAX  0          device pointer to 32 x uint64 cycle counters filled by the flash
 *                                                        kernel's pair 0 (0 = off)
 * WCT (rpst_wct_fuse) and its matrix functions (rpst_spd_roots, rpst_sym_eig_fn):
 *   "wct_fused_cov"             0..1          1          1: covariances by the fused convert+centre+SYRK kernels when the shape
 *                                                        allows (C <= 256); 0: pack + split-K GEMM
 *   "wct_cov_tma"               0..1          1          1: fused covariance as ONE cooperative launch with TMA-staged fp32
 *                                                        boxes; 0: register-staged kernel + separate shift / row-sum / finalize
 *   "wct_cov_prof"              0..INT64_MAX  0          device pointer to 16 x uint64 %globaltimer stamps of the covariance
 *                                                        launch (0 = off)
 *   "wct_roots_ns"              0..2          1          1: matrix roots by Newton-Schulz for C > 64, Jacobi for the matrices it
 *                                                        flags; 0: Jacobi only; 2: Newton-Schulz with every matrix flagged
 *                                                        (exercises the predicated Jacobi path)
 *   "ns_dmma"                   0..1          1          1: Newton-Schulz products on fp64 tensor-core MMAs (even orders);
 *                                                        0: DFMA kernel
 *   "wct_fused_apply"           0..1          1          1: colouring by the fused pointwise-convolution kernel (C <= 512);
 *                                                        0: pack + GEMM per sample
 * Pointwise convolution (rpst_conv1x1, and the WCT colouring):
 *   "pw_x_tma"                  0..1          1          1: fp32 input tiles staged by tensor-map TMA when the shape allows
 *                                                        (C_in % 64 == 0, 16-byte aligned rows); 0: register-staged converters
 * Safety and diagnostics:
 *   "watchdog_ms"               any           4000       every in-kernel spin wait traps after this many ms instead of hanging
 *                                                        the device; <= 0 disables the watchdog (debuggers, MPS time-slicing,
 *                                                        profilers that stretch waits); applies to all devices
 *   "wct_ns_flagged"            read only                matrices handed to the Jacobi path by the Newton-Schulz acceptance
 *                                                        test since load (reading it synchronises the device) */
RPST_API int rpst_set_tuning(const char* name, int64_t value);
RPST_API int64_t rpst_get_tuning(const char* name);

/* ------------------------------------------------------------------------------------------
 * a1  calc_mean_std(feat, eps=1e-5)                                   network/base.py:399-407
 * Per-(n,c) plane mean and sqrt(unbiased variance + eps) over H*W.
 *   x      [planes, hw]  (planes = N*C)
 *   mean, std  [planes]  (either may be NULL)
 * ------------------------------------------------------------------------------------------ */
RPST_API size_t rpst_stats_workspace_bytes(int64_t planes, int64_t hw);
RPST_API int rpst_stats_nchw(const float* x, int64_t planes, int64_t hw, float eps, float* mean, float* std,
                    void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * a2  adaptive_instance_normalization(content_feat, style_feat)       network/base.py:410-418
 * a3  stylized + AdaIN(c_l, s_l)  (multiscale blend)                  network/adain_rp.py:295-301
 *     cat([stylized, AdaIN(c_l, s_l)], 1)  (LD4/LD5 concat-write)     network/adain_rp.py:786-798
 * a8  mean_variance_norm(feat)                                        network/sanet.py:20-24
 *
 *   out[n,ch,:] = (content - mu_c)/sd_c * sd_s + mu_s  (+ prev)
 *   content [n, c, hw]; style [n, c, hw] or NULL (=> sd_s=1, mu_s=0: mean_variance_norm);
 *   prev    [n, c, hw] or NULL (=> plain AdaIN); prev may alias content (LDMS variants);
 *   out     plane (i, ch) is written at out + i*out_batch_stride + ch*hw (elements), so the call can
 *           write into a channel slice of a wider tensor; out_batch_stride = c*hw for a dense result.
 *   saved_stats [n*c, 4] or NULL: (mu_c, sd_c, mu_s, sd_s) per plane, kept for the backward pass.
 * ------------------------------------------------------------------------------------------ */
RPST_API size_t rpst_adain_workspace_bytes(int64_t n, int64_t c, int64_t hw);
RPST_API int rpst_adain_fwd(const float* content, const float* style, const float* prev, float* out,
                   int64_t n, int64_t c, int64_t hw, int64_t out_batch_stride, float eps,
                   float* saved_stats, void* workspace, size_t workspace_bytes, void* stream);

/* f3  channel shuffle / sort-by-SE-weight folded into the loads     network/adain_rp.py:230-249,304-311
 * Same as rpst_adain_fwd, but output plane p = i*c + ch reads its content from plane content_map[p]
 * and its style from plane style_map[p] of the SAME tensors (global plane indices in [0, n*c); either
 * map may be NULL = identity), so `shuffle(feats)` / `sort_by_weights(feats)` never materialise a
 * permuted copy.  prev and out are indexed by the output plane. */
RPST_API int rpst_adain_fwd_mapped(const float* content, const float* style, const float* prev, float* out,
                          int64_t n, int64_t c, int64_t hw, int64_t out_batch_stride, float eps,
                          const int32_t* content_map, const int32_t* style_map, void* workspace,
                          size_t workspace_bytes, void* stream);

/* Backward of rpst_adain_fwd w.r.t. content and style (autograd gives this to the reference for
 * free; gradients reach the shared RP encoder through both arguments, SURVEY.md §7 hard part 7).
 *   grad_out [n,c,hw]; saved_stats from the forward; grad_content / grad_style [n,c,hw]
 *   (grad_style may be NULL; style may then be NULL as well).  d/dprev is grad_out itself. */
RPST_API size_t rpst_adain_bwd_workspace_bytes(int64_t n, int64_t c, int64_t hw);
RPST_API int rpst_adain_bwd(const float* grad_out, const float* content, const float* style,
                   const float* saved_stats, float* grad_content, float* grad_style,
                   int64_t n, int64_t c, int64_t hw, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * a15 SELayer.forward: x * gate[n,c]   (the pooling is rpst_stats_nchw)  network/attention.py:17-22
 *   out[p,:] = x[p,:] * scale[p] + shift[p]   (shift may be NULL)
 * ------------------------------------------------------------------------------------------ */
RPST_API int rpst_plane_affine(const float* x, const float* scale, const float* shift, float* out,
                      int64_t planes, int64_t hw, void* stream);

/* ------------------------------------------------------------------------------------------
 * f1  calc_style_loss(input, target)            network/adain_rp.py:84-88, network/sanet.py:232-236
 *     calc_content_loss(input, target, norm=True)                    network/sanet.py:226-230
 * One streaming pass over the pair (x, y) (2*E*4 bytes) yields per-plane statistics and both losses:
 *   losses[0] = mse(mean_x, mean_y) + mse(std_x, std_y)              (mean over the N*C planes)
 *   losses[1] = mse(mean_variance_norm(x), mean_variance_norm(y))    (mean over N*C*H*W elements)
 *   x, y   [planes, hw];  losses [2] (device);
 *   stats  [planes, 8] or NULL: (mu_x, sd_x, mu_y, sd_y, M2_x, M2_y, C_xy, 0) — what the backward
 *          pass needs (M2 = sum of squared deviations, C_xy = sum of cross deviations).
 * rpst_plane_affine2 is that backward pass: out[p,:] = ax[p]*x[p,:] + ay[p]*y[p,:] + b[p] (b may be NULL).
 * ------------------------------------------------------------------------------------------ */
RPST_API size_t rpst_pair_stats_workspace_bytes(int64_t planes, int64_t hw);
RPST_API int rpst_pair_stats(const float* x, const float* y, int64_t planes, int64_t hw, float eps, float* stats,
                    float* losses, void* workspace, size_t workspace_bytes, void* stream);
RPST_API int rpst_plane_affine2(const float* x, const float* y, const float* ax, const float* ay, const float* b,
                       float* out, int64_t planes, int64_t hw, void* stream);
/* Gradient of losses[which] (0 style, 1 normalised content) w.r.t. x (wrt_second = 0) or y (1), scaled by
 * the upstream gradient *grad (device scalar); per-plane coefficients come from `stats` inside the kernel. */
RPST_API int rpst_pair_loss_bwd(const float* x, const float* y, const float* stats, const float* grad, int which,
                       int wrt_second, float* out, int64_t planes, int64_t hw, void* stream);

/* ------------------------------------------------------------------------------------------
 * a4  adaptive_instance_normalization_with_segment(content_feat, style_feat, c_seg, s_seg)
 *                                                                     network/base.py:494-530
 *     compute_label_info (validity rule)                              network/base.py:421-439
 *     do_mask_stylized (per-sample loop over the batch)               network/adain_rp.py:313-319
 *
 * Whole batch in one call; label maps are uint8 tensors already at feature resolution (the reference
 * loads PNG paths and resizes them with PIL at network/base.py:450-451 — that I/O stays in Python).
 *   content [n,c,hw_c], style [n,c,hw_s] (content and style may differ in H*W);
 *   c_labels [n,hw_c], s_labels [n,hw_s]; prev [n,c,hw_c] or NULL (out = prev + seg-AdaIN);
 *   out [n,c,hw_c].  For every label value present in a sample's CONTENT map that is usable
 *   (cnt_c>10, cnt_s>10, cnt_c/cnt_s<100, cnt_s/cnt_c<100) the content pixels carrying it are
 *   AdaIN'd with the masked statistics (unbiased variance, eps inside sqrt); all other pixels are
 *   copied through bit-exactly.
 *   label_info [n,256,3] int32 or NULL: (cnt_c, cnt_s, usable) per label value.
 * ------------------------------------------------------------------------------------------ */
RPST_API size_t rpst_seg_adain_workspace_bytes(int64_t n, int64_t c, int64_t hw_c, int64_t hw_s);
RPST_API int rpst_seg_adain_fwd(const float* content, const float* style, const uint8_t* c_labels,
                       const uint8_t* s_labels, const float* prev, float* out, int64_t n, int64_t c,
                       int64_t hw_c, int64_t hw_s, float eps, int32_t* label_info, void* workspace,
                       size_t workspace_bytes, void* stream);

/* Same as rpst_seg_adain_fwd, with plane maps and a strided output, as rpst_adain_fwd_mapped adds to
 * rpst_adain_fwd, so the masked decodes neither gather shuffled / sorted features nor concatenate copies:
 *   output plane p = i*c + ch reads its content from plane content_map[p] and its style from plane
 *   style_map[p] of the SAME tensors (global plane indices in [0, n*c); either map may be NULL = identity);
 *   the label maps, the validity rule and label_info belong to the OUTPUT sample i (c_labels[i],
 *   s_labels[i]), as they would for the gathered tensors; prev [n,c,hw_c] is indexed by the output plane;
 *   plane (i, ch) of out is written at out + i*out_batch_stride + ch*hw_c (out_batch_stride >= c*hw_c;
 *   (c_prev + c)*hw_c writes the channel slice of cat([prev_feats, seg-AdaIN], 1)).
 * Workspace: rpst_seg_adain_workspace_bytes.  n*c must be < 2^31. */
RPST_API int rpst_seg_adain_fwd_mapped(const float* content, const float* style, const uint8_t* c_labels,
                              const uint8_t* s_labels, const float* prev, float* out, int64_t n, int64_t c,
                              int64_t hw_c, int64_t hw_s, int64_t out_batch_stride, float eps,
                              const int32_t* content_map, const int32_t* style_map, int32_t* label_info,
                              void* workspace, size_t workspace_bytes, void* stream);

/* Backward of rpst_seg_adain_fwd w.r.t. content and style (the reference differentiates its index_select / var /
 * index_copy_ sequence with autograd; masked training needs the same gradients).  For sample i, channel ch and a
 * usable label with n_c content pixels, x^ = (c - mu_c)/sd_c, a = sd_s/sd_c, G1 = sum g, G2 = sum g*x^ over those
 * pixels (g = grad_out):
 *   content pixel of the label:  dc = a*(g - G1/n_c - x^*G2/(n_c - 1))
 *   style pixel of the label:    ds = G1/n_s + G2*(s - mu_s)/((n_s - 1)*sd_s)
 *   content pixel of an unusable label: dc = g bit-exactly; style pixel without a usable label: ds = 0.
 * d/dprev is grad_out itself.  Shapes and labels as in rpst_seg_adain_fwd (content and style may differ in H*W).
 * The masked statistics are recomputed here, so no forward state is needed; the result is run-to-run bit-identical.
 *   grad_content [n,c,hw_c] or NULL, grad_style [n,c,hw_s] or NULL: a NULL half is skipped (style is still read).
 *   Outputs must not overlap each other or an input.  n*c < 2^31; hw_c, hw_s < 2^31.
 * Workspace: rpst_seg_adain_bwd_workspace_bytes (from the shapes alone; 256-byte aligned). */
RPST_API size_t rpst_seg_adain_bwd_workspace_bytes(int64_t n, int64_t c, int64_t hw_c, int64_t hw_s);
RPST_API int rpst_seg_adain_bwd(const float* grad_out, const float* content, const float* style,
                       const uint8_t* c_labels, const uint8_t* s_labels, float* grad_content,
                       float* grad_style, int64_t n, int64_t c, int64_t hw_c, int64_t hw_s, float eps,
                       void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * a12 cal_dist(A, B)                                                  network/base.py:349-360
 *   a [d,m], b [d,n] (d-dimensional column vectors) -> out [m,n] = |a_i|^2 + |b_j|^2 - 2 a_i.b_j
 *   (tensor cores, bf16x3 = fp32-grade accumulation).
 * ------------------------------------------------------------------------------------------ */
RPST_API size_t rpst_pairwise_sqdist_workspace_bytes(int64_t d, int64_t m, int64_t n);
RPST_API int rpst_pairwise_sqdist(const float* a, const float* b, int64_t d, int64_t m, int64_t n, float* out,
                         void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * a13 cal_affinity_map(content_feat, style_feat, k, reverse)          network/base.py:317-346
 * a14 MRFLoss(k, mean).forward(content_feat, style_feat)              network/mrf_rp.py:12-23
 *
 * content/style [c, l] (one sample, l = H*W).  Channel-L2-normalise (eps 1e-12), l x l cosine map on
 * the tensor cores, top-k along both axes:
 *   idx_dim0 [k,l] int64  topk(map, k, dim=0).indices  (for every style position the best content ones)
 *   idx_dim1 [l,k] int64  topk(map, k, dim=1).indices  (for every content position the best style ones)
 *   affinity [l,l] or NULL: the dense binary map (1 where (i,j) is in either set)
 *   loss     [1]   or NULL: sum(affinity * sqdist) / (l*k)   (loss_mean_over_all != 0: / (l*l))
 * reverse != 0 negates the map first (network/base.py:326-327).  passes: 3 = bf16x3 (index-exact on
 * tie-free inputs), 1 = plain bf16.  1 <= k <= 8.
 * ------------------------------------------------------------------------------------------ */
RPST_API size_t rpst_mrf_workspace_bytes(int64_t c, int64_t l, int k);
RPST_API int rpst_mrf_match(const float* content, const float* style, int64_t c, int64_t l, int k, int reverse,
                   int passes, int64_t* idx_dim0, int64_t* idx_dim1, float* affinity, float* loss,
                   int loss_mean_over_all, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * a5  matrix_sqrt(A) / matrix_inv_sqrt(A)                             network/wct_rp.py:7-40
 * Batched symmetric eigen-decomposition (cluster-resident one-sided Jacobi, fp64, no host sync) and
 * V diag(s^(+-1/2)) V^T, with the reference's conditioning: `diag_add` (1e-4 in the reference) is added
 * to the diagonal first and eigenvalues below 1e-5 are dropped.
 *   a [batch,n,n] fp64 symmetric positive semi-definite, n <= 512;
 *   out_sqrt / out_inv_sqrt [batch,n,n] fp64 (either may be NULL); eigenvalues [batch,n] or NULL
 *   (unsorted); sweeps [batch] int32 or NULL (Jacobi sweeps used).
 * ------------------------------------------------------------------------------------------ */
RPST_API size_t rpst_sym_eig_fn_workspace_bytes(int64_t batch, int64_t n);
RPST_API int rpst_sym_eig_fn(const double* a, int64_t batch, int64_t n, double diag_add, double* out_sqrt,
                    double* out_inv_sqrt, double* eigenvalues, int32_t* sweeps, void* workspace,
                    size_t workspace_bytes, void* stream);

/* The same two functions for matrices that are positive DEFINITE after the shift, by a scaled coupled
 * Newton-Schulz iteration (fp64 products on every SM; what rpst_wct_fuse uses for C > 64): every
 * eigenvalue of a + diag_add I must be >= lmin > 0 (the WCT's covariances + 1e-4 I: lmin = 1e-4), where the
 * reference's 1e-5 cut never fires and V diag(s^(+-1/2)) V^T is the principal root.  No host
 * synchronisation: flags[b] = 1 marks a matrix whose iteration was NOT accepted (||Z Y - I||_F > 1e-7:
 * indefinite input, eigenvalues far below lmin) — its outputs must not be used; run rpst_sym_eig_fn
 * for it.  flags [batch] int32 (required).
 * ------------------------------------------------------------------------------------------ */
RPST_API size_t rpst_spd_roots_workspace_bytes(int64_t batch, int64_t n);
RPST_API int rpst_spd_roots(const double* a, int64_t batch, int64_t n, double diag_add, double lmin, double* out_sqrt,
                   double* out_inv_sqrt, int32_t* flags, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * a6  WCTRPNet.whiten_and_color(cF, sF, method='closed-form')          network/wct_rp.py:82-114
 * a7  WCTRPNet.fuse(content_feats, style_feats)                        network/wct_rp.py:157-166
 * Whole batch, no gradient (the reference detaches): centre, covariances (+I on content), transform
 *   method 0 'closed-form': T = C^-1/2 (C^1/2 S C^1/2)^1/2 C^-1/2      method 1 'original': T = S^1/2 C^-1/2
 * and out = T (X - mu_c) + mu_s.
 *   content [n,c,hw_c], style [n,c,hw_s] fp32 -> out [n,c,hw_c] fp32; c <= 512.
 *   passes 3 = bf16x3 tensor-core products (fp32-grade, default), 1 = plain bf16.
 *   transform_out [n,c,c] fp64 or NULL.
 * ------------------------------------------------------------------------------------------ */
RPST_API size_t rpst_wct_workspace_bytes(int64_t n, int64_t c, int64_t hw_c, int64_t hw_s);
RPST_API int rpst_wct_fuse(const float* content, const float* style, float* out, int64_t n, int64_t c,
                  int64_t hw_c, int64_t hw_s, int method, int passes, double* transform_out,
                  void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * a9  SANet.forward attention core                                    network/sanet.py:85-94
 *   f [b,c,lc] (queries, = f(mean_variance_norm(content))), g [b,c,ls] (keys), h [b,c,ls] (values),
 *   all fp32 outputs of the module's own 1x1 convolutions (which stay in cuDNN).
 *   S = softmax_j(sum_c f[c,i] g[c,j])  (no temperature),  out[b,c,i] = sum_j h[c,j] S[i,j].
 *   attn_out [b,lc,ls] or NULL receives S.  passes: 3 = bf16x3 (fp32-grade, rel-L2 <= 1e-3 contract),
 *   1 = bf16 (<= 1e-2 contract).
 * ------------------------------------------------------------------------------------------ */
 /* The workspace query returns the PER-SAMPLE minimum; a workspace of k times that size makes the call
  * run k samples per kernel launch (batched tcgen05 GEMMs) — worth it when L is small and launches dominate. */
RPST_API size_t rpst_sanet_attn_workspace_bytes(int64_t c, int64_t lc, int64_t ls);
RPST_API int rpst_sanet_attn_fwd(const float* f, const float* g, const float* h, float* out, int64_t b, int64_t c,
                        int64_t lc, int64_t ls, int passes, float* attn_out, void* workspace,
                        size_t workspace_bytes, void* stream);

/* f2  backward of rpst_sanet_attn_fwd (autograd gives it to the reference for free; needed to train
 *     SAModel, network/sanet.py:253-276).  grad_out [b,c,lc] -> grad_f [b,c,lc], grad_g / grad_h [b,c,ls].
 *     The attention matrix is recomputed, not saved. */
RPST_API size_t rpst_sanet_attn_bwd_workspace_bytes(int64_t c, int64_t lc, int64_t ls);
RPST_API int rpst_sanet_attn_bwd(const float* f, const float* g, const float* h, const float* grad_out,
                        float* grad_f, float* grad_g, float* grad_h, int64_t b, int64_t c, int64_t lc,
                        int64_t ls, int passes, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * a11 cal_affinity_matrix(content_feat, style_feat)                   network/sanet.py:12-18
 *   out[b,i,j] = cosine similarity of the channel vectors (F.normalize eps 1e-12) of the RAW features.
 * ------------------------------------------------------------------------------------------ */
RPST_API size_t rpst_cosine_affinity_workspace_bytes(int64_t c, int64_t lc, int64_t ls);
RPST_API int rpst_cosine_affinity(const float* content, const float* style, float* out, int64_t b, int64_t c,
                         int64_t lc, int64_t ls, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * a11 AdaptiveSANet.forward attention core with AEAModule / AEALReluModule
 *                                                                     network/sanet.py:26-71,114-138
 *   f,g,h as above; content_raw/style_raw [b,c_raw,l] raw features for the cosine affinity;
 *   f_psi = Linear(l, lh) -> LeakyReLU(0.2) -> Linear(lh, 1): w0 [lh,l], b0 [lh], w2 [lh], b2 [1];
 *   mode 1 'aea' : clamp = sigmoid(psi)*value_interval + from_value ; S' = sigmoid(scale_value*(S-clamp))
 *   mode 2 'relu': clamp = (tanh(psi)+1)/2 ; S' = softmax_j(relu(S-clamp))
 *   out[b,c,i] = sum_j h[c,j] S'[i,j].  claim_before (S) / claim_after (S') [b,l,l], claim_value [b,l]
 *   are optional outputs (the reference stashes them for visualisation, network/sanet.py:126-137).
 * ------------------------------------------------------------------------------------------ */
RPST_API size_t rpst_sanet_adaptive_workspace_bytes(int64_t c, int64_t lc, int64_t ls, int64_t lh);
RPST_API int rpst_sanet_attn_adaptive_fwd(const float* f, const float* g, const float* h, const float* content_raw,
                                 const float* style_raw, int64_t c_raw, const float* w0, const float* b0,
                                 const float* w2, const float* b2, int mode, float scale_value,
                                 float from_value, float value_interval, float* out, float* claim_before,
                                 float* claim_after, float* claim_value, int64_t b, int64_t c, int64_t lc,
                                 int64_t ls, int64_t lh, int passes, void* workspace, size_t workspace_bytes,
                                 void* stream);

/* a11 training path: clamped attention with the per-row clamp GIVEN (the clamp MLP f_psi and the cosine
 * affinity stay in the caller's autograd graph; the L x L work — softmax, clamp, both products and their
 * backward — is here).  mode 1 'aea': S' = sigmoid(scale (P - clamp_i)); mode 2 'relu': S' = softmax(relu(P -
 * clamp_i)); P = softmax(f^T g); out = h S'^T.  clamp / grad_clamp [b, lc].  network/sanet.py:41-46,66-71,114-138 */
RPST_API size_t rpst_sanet_attn_clamped_workspace_bytes(int64_t c, int64_t lc, int64_t ls);
RPST_API int rpst_sanet_attn_clamped_fwd(const float* f, const float* g, const float* h, const float* clamp, int mode,
                                float scale, float* out, int64_t b, int64_t c, int64_t lc, int64_t ls,
                                int passes, void* workspace, size_t workspace_bytes, void* stream);
RPST_API int rpst_sanet_attn_clamped_bwd(const float* f, const float* g, const float* h, const float* clamp, int mode,
                                float scale, const float* grad_out, float* grad_f, float* grad_g,
                                float* grad_h, float* grad_clamp, int64_t b, int64_t c, int64_t lc,
                                int64_t ls, int passes, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Building blocks shared by the contraction kernels (exposed for tests and for callers that want to
 * keep packed operands around): fp32 matrix -> bf16 hi/lo operand tiles, and D = alpha*A.B^T
 * (+row_add[i] +col_add[j]) on tcgen05 with fp32 accumulation in TMEM.
 *   x element (r, kk) is read at x[r*stride_r + kk*stride_k]; row_scale [rows] or NULL;
 *   hi/lo: rpst_packed_operand_bytes(rows, k) bytes each, 128-byte aligned (lo may be NULL);
 *   passes 1 (bf16) or 3 (bf16x3).
 * ------------------------------------------------------------------------------------------ */
RPST_API size_t rpst_packed_operand_bytes(int64_t rows, int64_t k);
RPST_API int rpst_pack_operand(const float* x, int64_t rows, int64_t k, int64_t stride_r, int64_t stride_k,
                      const float* row_scale, void* hi, void* lo, void* stream);
RPST_API int rpst_gemm_packed(const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo, float* out,
                     int64_t m, int64_t n, int64_t k, int64_t ldo, int passes, float alpha,
                     const float* row_add, const float* col_add, void* stream);

/* ------------------------------------------------------------------------------------------
 * f2 / f4  Pointwise (1x1) convolution with fused prologue / epilogue (csrc/pwconv.cu):
 *     y[b,o,n] = act( sum_c W[o,c] * ((x[b,c,n] - sub[b,c]) * mul[b,c]) + bias[o] ) (+ residual[b,o,n])
 *   - SANet projections with `mean_variance_norm` folded into the operand conversion (sub = mean, mul = 1/std) and
 *     Q / K emitted as packed attention operands                         network/sanet.py:82-99
 *   - RP-encoder 1x1 conv + LeakyReLU with the AdaIN statistics from the epilogue        network/base.py:170-198
 *   x [b,cin,hw] fp32; w_hi / w_lo: the [cout,cin] weight packed with rpst_pack_operand(w, cout, cin, cin, 1, ...);
 *   bias [cout], sub / mul [b,cin], residual [b,cout,hw] may be NULL; act 0 none, 1 LeakyReLU(slope);
 *   out fp32 [b,cout,hw] and / or out_hi, out_lo: packed [hw x cout] operand tiles per sample (rows = positions; sample
 *   stride align_up(rpst_packed_operand_bytes(hw, cout), 256); needs hw % 128 == 0, cout % 64 == 0);
 *   stats_partial (rpst_conv1x1_stats_bytes) receives per-warp (sum, sum of squares) of y; rpst_conv1x1_stats_finalize
 *   turns them into mean / sqrt(unbiased var + eps) [b,cout] — calc_mean_std of y without reading y again.
 * ------------------------------------------------------------------------------------------ */
RPST_API size_t rpst_conv1x1_stats_bytes(int64_t b, int64_t cout, int64_t hw);
RPST_API int rpst_conv1x1(const float* x, const void* w_hi, const void* w_lo, const float* bias, const float* sub,
                 const float* mul, const float* residual, float* out, void* out_hi, void* out_lo,
                 float* stats_partial, int64_t b, int64_t cin, int64_t cout, int64_t hw, int act, float slope,
                 int passes, void* stream);
RPST_API int rpst_conv1x1_stats_finalize(const float* stats_partial, int64_t b, int64_t cout, int64_t hw, float eps,
                                float* mean, float* std, void* stream);
/* Attention core (rpst_sanet_attn_fwd) with Q / K already packed by rpst_conv1x1 (C = 512, Lc % 128 == 0, Ls % 256 == 0). */
RPST_API size_t rpst_sanet_attn_packed_workspace_bytes(int64_t b, int64_t lc, int64_t ls);
RPST_API int rpst_sanet_attn_fwd_packed(const void* q_hi, const void* q_lo, const void* k_hi, const void* k_lo, const float* h,
                               float* out, int64_t b, int64_t c, int64_t lc, int64_t ls, int passes, void* workspace,
                               size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RPST_H_ */

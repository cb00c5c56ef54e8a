/* rpst_debug.h — white-box test hooks of librpst.  NOT part of the product ABI: these entry points exist only in
 * librpst_debug.so (the same sources compiled with -DRPST_DEBUG_EXPORTS; built by rp-style-transfer_b200/build.py
 * next to librpst.so) and are used by tests/test_schedule_gpu.py and tests/test_wct_linalg_gpu.py alone. */
#ifndef RPST_DEBUG_H
#define RPST_DEBUG_H
#include "rpst.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Test hook (no data touched): the ticket schedule the TMA-staged AdaIN kernel walks for a call shape.
 * info[5] (host) = {tickets, statistics items per plane, apply items per plane, lag, merge lead};
 * tickets (device, [max_tickets,3] int32, may be NULL) = (kind, plane, chunk), kind 0 statistics / 1 apply / 2 merge. */
RPST_API int rpst_debug_adain_schedule(int64_t planes, int64_t hw, int has_style, int has_prev, int stats_only,
                              int32_t* tickets, int64_t max_tickets, int64_t* info, void* stream);


/* Test hook: ticket schedule of the segment kernel (see rpst_debug_adain_schedule).  info[5] = {tickets, content
 * statistics items, style statistics items, apply items per plane, lag}; kind 0 content statistics, 1 style
 * statistics, 2 apply, 3 merge. */
RPST_API int rpst_debug_seg_schedule(int64_t n, int64_t c, int64_t hw_c, int64_t hw_s, int has_prev, int32_t* tickets,
                            int64_t max_tickets, int64_t* info, void* stream);


/* Test hook: steps 1-2 of rpst_wct_fuse on n contiguous [c, hw] fp32 tensors x: channel means mean_out [n, c] (fp32) and
 * centred covariances cov_out [n, c, c] (fp64, / (hw - 1), + diag_add on the diagonal), through the same internal function
 * the WCT calls.  path: 0 production dispatch, 1 one-launch cooperative TMA kernel (at any grid size), 2 register-staged
 * kernel + separate rowsum / finalize launches, 3 pack + split-K tcgen05 GEMM + reduce; 1 and 2 need c <= 256, hw >= 64 and
 * hw % 4 == 0.  path_taken (host) receives the path that ran.  passes 1 (bf16) or 3 (bf16x3). */
RPST_API size_t rpst_debug_wct_covariances_workspace_bytes(int64_t n, int64_t c, int64_t hw);
RPST_API int rpst_debug_wct_covariances(const float* x, int64_t n, int64_t c, int64_t hw, int passes, double diag_add, int path,
                                        double* cov_out, float* mean_out, int32_t* path_taken, void* workspace,
                                        size_t workspace_bytes, void* stream);


/* Test hook: c[b] = a[b] b[b] for batch n x n row-major fp64 matrices, through the product kernels of the Newton-Schulz
 * roots and the WCT transform (nsroot.cu dgemm_batched). */
RPST_API int rpst_debug_dgemm_batched(const double* a, const double* b, double* c, int64_t batch, int64_t n, void* stream);


#ifdef __cplusplus
}
#endif
#endif

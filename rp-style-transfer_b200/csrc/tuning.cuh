// Tuning knobs (host side): the integers that select kernel paths and schedule parameters.  The defaults are the
// production choice; rpst_set_tuning / rpst_get_tuning (api.cu) set and read them by name, within the range that
// api.cu's table gives each one.  include/rpst.h documents every knob.
#pragma once
#include <stdint.h>

namespace rpst {

struct Knobs {
    // AdaIN (adain.cu; the register-staged segment AdaIN kernel in seg.cu reads adain_lag_bytes and adain_hints too)
    int64_t adain_lag_bytes = 32ll << 20;       // content bytes kept L2-resident between a plane's statistics and its apply
    int64_t adain_big_lag_bytes = 128ll << 20;  // the same for planes >= 4 MiB: see plan_schedule
    int64_t adain_mvn_lag_bytes = 44ll << 20;   // the same for style == NULL (mean_variance_norm): see plan_schedule
    int64_t adain_hints = 1;                    // L2 eviction-priority hints on the streaming loads / stores
    int64_t adain_ctas_per_sm = 4;              // persistent CTAs per SM of the register-staged pipelined kernel
    int64_t adain_path = 0;      // 0: TMA-staged kernel when alignment allows, 1: register-staged kernel; 1 also turns
                                 // off the segment AdaIN TMA kernel (seg.cu)
    int64_t adain_stages = 6;    // TMA ring depth (32 KiB per stage)
    int64_t adain_twin_apply = 1;               // TMA kernel, no prev: apply items carry two content chunks (32 KiB per stage)
    int64_t adain_group_merge_min_spp = 512;    // see merge_plane_coef_group
    int64_t adain_merge_lead = 0;               // 0: lag / 2
    // segment AdaIN (seg.cu)
    int64_t seg_lag_bytes = 256ll << 20;  // content bytes between statistics and apply
    int64_t seg_groups = 4;               // consumer groups (= stages) of the segment TMA kernel
    int64_t seg_flush = 2;                // final flush: 0 shared atomics per lane, 1 warp-aggregated, 2 staged gather (atomic-free)
    // SANet attention (sanet.cu, flash.cu)
    int64_t attn_flash = 1;       // 1: C = 512 attention takes the single-kernel flash path when the shape allows
    int64_t attn_flash_prof = 0;  // device pointer to 32 x uint64 cycle counters (0 = off); bring-up / tuning only
    // WCT (wct.cu, cov.cu, nsroot.cu, eig.cu, pwconv.cu)
    int64_t wct_fused_cov = 1;    // 1: WCT covariances through the fused convert+centre+SYRK kernel (cov.cu) when the shape allows
    int64_t wct_fused_apply = 1;  // 1: WCT colouring through the fused transpose+convert+GEMM kernel (pwconv.cu) when the shape allows
    int64_t wct_cov_tma = 1;      // 1 = TMA-staged covariance kernel, 0 = register-staged kernel
    int64_t wct_cov_prof = 0;     // device pointer to 16 x uint64 time stamps (0 = off); bring-up / tuning only
    int64_t wct_roots_ns = 1;     // 1 Newton-Schulz roots with Jacobi for flagged matrices, 0 Jacobi only,
                                  // 2 Newton-Schulz but every matrix flagged (exercises the predicated path)
    int64_t ns_dmma = 1;          // 1 = fp64 tensor-core products (mma.sync f64) for even orders, 0 = DFMA kernel
    int64_t eig_wide = -1;        // -1 auto, 0 / 1 force 16- / 32-column blocks, -2 auto + print cluster occupancy,
                                  // 2 16-column blocks padded to one CTA per SM + print cluster occupancy
    // pointwise convolution (pwconv.cu)
    int64_t pw_x_tma = 1;  // 1 = x tiles by tensor-map TMA when the shape allows, 0 = register-staged converters
};

extern Knobs g_knobs;

}  // namespace rpst

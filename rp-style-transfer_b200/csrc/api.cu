// librpst: version, error plumbing, tuning registry, device attributes.
#include "common.cuh"
#include "tuning.cuh"

#include <string.h>

namespace rpst {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
    set_error("CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
    return RPST_ERR_CUDA;
}

int sm_count() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

Knobs g_knobs;

struct KnobSpec {
    const char* name;
    int64_t Knobs::*field;
    int64_t lo, hi;   // accepted values, inclusive
};

// Every settable knob; include/rpst.h documents each one with its range and default (tests/test_abi.py checks both)
static const KnobSpec kKnobs[] = {
    {"adain_lag_bytes", &Knobs::adain_lag_bytes, 0, INT64_MAX},
    {"adain_big_lag_bytes", &Knobs::adain_big_lag_bytes, 0, INT64_MAX},
    {"adain_mvn_lag_bytes", &Knobs::adain_mvn_lag_bytes, 0, INT64_MAX},
    {"adain_hints", &Knobs::adain_hints, 0, 1},
    {"adain_ctas_per_sm", &Knobs::adain_ctas_per_sm, 2, 6},
    {"adain_path", &Knobs::adain_path, 0, 1},
    {"adain_stages", &Knobs::adain_stages, 2, 7},
    {"adain_twin_apply", &Knobs::adain_twin_apply, 0, 1},
    {"adain_group_merge_min_spp", &Knobs::adain_group_merge_min_spp, 0, INT64_MAX},
    {"adain_merge_lead", &Knobs::adain_merge_lead, 0, INT64_MAX},
    {"seg_lag_bytes", &Knobs::seg_lag_bytes, 0, INT64_MAX},
    {"seg_groups", &Knobs::seg_groups, 3, 4},
    {"seg_flush", &Knobs::seg_flush, 0, 2},
    {"attn_flash", &Knobs::attn_flash, 0, 1},
    {"attn_flash_prof", &Knobs::attn_flash_prof, 0, INT64_MAX},
    {"wct_fused_cov", &Knobs::wct_fused_cov, 0, 1},
    {"wct_fused_apply", &Knobs::wct_fused_apply, 0, 1},
    {"wct_cov_tma", &Knobs::wct_cov_tma, 0, 1},
    {"wct_cov_prof", &Knobs::wct_cov_prof, 0, INT64_MAX},
    {"wct_roots_ns", &Knobs::wct_roots_ns, 0, 2},
    {"ns_dmma", &Knobs::ns_dmma, 0, 1},
    {"eig_wide", &Knobs::eig_wide, -2, 2},
    {"pw_x_tma", &Knobs::pw_x_tma, 0, 1},
};

static const KnobSpec* find_knob(const char* name) {
    for (const KnobSpec& k : kKnobs)
        if (!strcmp(name, k.name)) return &k;
    return nullptr;
}

int set_watchdog_adain(unsigned long long ns);
int set_watchdog_cov(unsigned long long ns);
int set_watchdog_flash(unsigned long long ns);
int set_watchdog_gemm(unsigned long long ns);
int set_watchdog_sanet(unsigned long long ns);
int set_watchdog_seg(unsigned long long ns);
int set_watchdog_pwconv(unsigned long long ns);

static int64_t g_watchdog_ms = 4000;

// the limit lives in one device variable per translation unit and per device: write it everywhere
static int apply_watchdog(int64_t ms) {
    const unsigned long long ns = ms <= 0 ? 0ull : (unsigned long long)ms * 1000000ull;
    int count = 0, cur = 0;
    g_watchdog_ms = ms <= 0 ? 0 : ms;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) return RPST_OK;   // no device: nothing to configure
    cudaGetDevice(&cur);
    int rc = 0;
    for (int d = 0; d < count; ++d) {
        if (cudaSetDevice(d) != cudaSuccess) continue;
        rc |= set_watchdog_adain(ns);
        rc |= set_watchdog_cov(ns);
        rc |= set_watchdog_flash(ns);
        rc |= set_watchdog_gemm(ns);
        rc |= set_watchdog_sanet(ns);
        rc |= set_watchdog_seg(ns);
        rc |= set_watchdog_pwconv(ns);
    }
    cudaSetDevice(cur);
    if (rc) {
        set_error("watchdog_ms: cudaMemcpyToSymbol failed");
        return RPST_ERR_CUDA;
    }
    return RPST_OK;
}

}  // namespace rpst

extern "C" int rpst_version(void) { return RPST_VERSION; }

namespace rpst { int64_t ns_flagged_total(); }

extern "C" const char* rpst_last_error(void) { return rpst::g_err; }

extern "C" int rpst_set_tuning(const char* name, int64_t value) {
    RPST_CHECK_ARG(name, "rpst_set_tuning: null knob name");
    if (!strcmp(name, "watchdog_ms")) return rpst::apply_watchdog(value);
    RPST_CHECK_ARG(strcmp(name, "wct_ns_flagged") != 0, "tuning knob 'wct_ns_flagged' is read-only");
    const rpst::KnobSpec* k = rpst::find_knob(name);
    RPST_CHECK_ARG(k, "unknown tuning knob '%s'", name);
    RPST_CHECK_ARG(value >= k->lo && value <= k->hi, "tuning knob '%s' takes %lld..%lld (got %lld)", name,
                   (long long)k->lo, (long long)k->hi, (long long)value);
    rpst::g_knobs.*k->field = value;
    return RPST_OK;
}

extern "C" int64_t rpst_get_tuning(const char* name) {
    if (!name) return -1;
    if (!strcmp(name, "watchdog_ms")) return rpst::g_watchdog_ms;
    if (!strcmp(name, "wct_ns_flagged")) return rpst::ns_flagged_total();   // read-only counter (synchronises)
    const rpst::KnobSpec* k = rpst::find_knob(name);
    return k ? rpst::g_knobs.*k->field : -1;
}

// mbarrier + TMA bulk-copy (cp.async.bulk) PTX wrappers for sm_100a.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace rpst {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
// make barrier initialisation visible to the async proxy / other threads before first use
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ uint64_t global_timer_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// Watchdog: a wait that lasts longer than this is a protocol bug; trap (the launch fails with an error) instead of
// hanging the device.  Opt-out / adjustable: rpst_set_tuning("watchdog_ms", 0) disables it (debuggers, MPS
// time-slicing and compute-sanitizer stretch waits legitimately).  The limit is a per-translation-unit device
// variable (no relocatable device code in this library); RPST_WATCHDOG_SETTER registers the TU's setter with api.cu.
static __device__ unsigned long long g_watchdog_ns = 4000000000ull;
__device__ __forceinline__ bool watchdog_expired(uint64_t t0) {
    const unsigned long long limit = g_watchdog_ns;
    return limit != 0 && global_timer_ns() - t0 > limit;
}
#define RPST_WATCHDOG_SETTER(tag)                                                                            \
    namespace rpst {                                                                                         \
    int set_watchdog_##tag(unsigned long long ns) {                                                          \
        return cudaMemcpyToSymbol(g_watchdog_ns, &ns, sizeof(ns)) == cudaSuccess ? 0 : -2;                   \
    }                                                                                                        \
    }

// Global-memory spin wait on a value the caller has loaded once already: while `ready()` says it is not ready, back off
// `sleep_ns`, `reload()` it and trap once the watchdog expires.  A value that is ready at once costs no timer read, no
// sleep and no load.  A reload that finds the value ready returns at once: the watchdog (a load of its limit and a
// timer read) is looked at only on the way back to sleep.
template <class Reload, class Ready>
__device__ __forceinline__ void spin_wait(unsigned sleep_ns, Reload reload, Ready ready) {
    if (ready()) return;
    const uint64_t t0 = global_timer_ns();
    for (;;) {
        __nanosleep(sleep_ns);
        reload();
        if (ready()) return;
        if (watchdog_expired(t0)) __trap();
    }
}

__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const uint64_t t0 = global_timer_ns();
    while (!mbar_try_wait(bar, parity)) {
        if (watchdog_expired(t0)) __trap();
    }
}

// The same wait for threads that poll next to working warps: optional back-off, and the watchdog (a slow
// %globaltimer read) is looked at every 1024 polls only.
__device__ __forceinline__ void mbar_wait_quiet(uint64_t* bar, uint32_t parity, unsigned sleep_ns = 0) {
    if (mbar_try_wait(bar, parity)) return;
    uint64_t t0 = 0;
    unsigned polls = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (sleep_ns) __nanosleep(sleep_ns);
        if ((++polls & 1023u) == 0) {
            if (t0 == 0) t0 = global_timer_ns();
            else if (watchdog_expired(t0)) __trap();
        }
    }
}

// 1-D bulk copy global -> shared (TMA engine, no tensor map needed for contiguous data).
// dst/src 16-byte aligned, bytes a multiple of 16; completion is signalled on `bar` (complete_tx).
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar,
                                            uint64_t l2_policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
        :: "r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)), "l"(l2_policy) : "memory");
}

// 2-D tiled load through a tensor map (CUtensorMap in kernel parameter space): box at element coordinates {c0 (inner), c1}.
__device__ __forceinline__ void tma_load_box_2d(void* smem_dst, const void* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        :: "r"(smem_u32(smem_dst)), "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar)) : "memory");
}

// 1-D bulk copy shared -> global (bulk async-group completion).
__device__ __forceinline__ void tma_store_1d(void* gmem_dst, const void* smem_src, uint32_t bytes, uint64_t l2_policy) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
                 :: "l"(gmem_dst), "r"(smem_u32(smem_src)), "r"(bytes), "l"(l2_policy) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" :: "n"(N) : "memory");
}
// order generic-proxy smem writes before subsequent async-proxy (TMA) reads of the same memory
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t threads) {
    asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(threads) : "memory");
}

}  // namespace rpst

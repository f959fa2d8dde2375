// Shared declarations of libhgt (B200 / sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <map>
#include <string>

#include "../../include/hgt.h"

// Caching allocator of a context: device (cudaMalloc) and page-locked host (cudaMallocHost) blocks are kept on free
// lists when released and handed out again to later batches, so the steady state of a typing service does no
// driver allocation at all (cudaMalloc / cudaMallocHost / cudaFree cost 0.1-10 ms each and synchronise the device).
struct MemPool {
    std::multimap<size_t, void *> free_dev, free_pin;
    size_t held_dev = 0, held_pin = 0;
    static size_t round_up(size_t n) {
        if (n < 4096) return 4096;
        size_t g = 4096;
        while (g * 16 < n) g <<= 1;  // granularity = 1/16 .. 1/8 of the size: <= 12.5 % slack
        return (n + g - 1) / g * g;
    }
    int get(bool pinned, size_t n, void **out, size_t *cap);
    void put(bool pinned, void *p, size_t cap);
    void drain();
};

struct hgt_ctx {
    int device = 0;
    int sm_count = 0;
    size_t smem_optin = 0;
    int64_t launches = 0;
    cudaStream_t stream = nullptr;  // stream used by the host-pointer entry points
    // accounting read by bench.py through hgt_profile_read()
    MemPool pool;
    int64_t h2d_bytes = 0, d2h_bytes = 0;
    int profile = 0;
    double stage_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // pileup, compat, class, counts, em1, project, em2, -
    int64_t stage_launches[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    double host_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // intake, pileup prep, pileup GPU+wait, walk, pack, upload, finish host, -
};

void hgt_set_error(const char *fmt, ...);

// Small host->device transfers of execute / finish (job descriptors, EM arguments: bytes to a few hundred KB) are done by
// a kernel that reads the PAGE-LOCKED source over PCIe itself.  A cudaMemcpyAsync would queue on the host-to-device copy
// engine behind the bulk text transfer of ANOTHER batch in flight (typing_core.BatchPipeline) and stall this batch's
// kernels for the length of that transfer.  src must come from cudaMallocHost / cudaHostAlloc and stay untouched until
// the stream has passed this point (the rule of cudaMemcpyAsync).
cudaError_t hgt_small_h2d(void *dst_dev, const void *src_pinned, size_t bytes, cudaStream_t st);

// Raises the dynamic shared-memory limit of `kernel` on the current device to at least `bytes`; never lowers it.  The
// limit is a property of the kernel for the whole process, and batches on other host threads (one context each,
// typing_core.BatchPipeline) launch the same kernels with their own sizes: a thread that set the exact size of its own
// launch could lower the limit between another thread's set and launch, and that launch would fail.
cudaError_t hgt_smem_at_least(const void *kernel, size_t bytes);

#include <chrono>
struct HostTimer {  // wall-clock bracket of one host stage, accumulated into ctx->host_ms (bench.py reads it)
    hgt_ctx *ctx;
    int k;
    std::chrono::steady_clock::time_point t0;
    HostTimer(hgt_ctx *c, int stage) : ctx(c), k(stage), t0(std::chrono::steady_clock::now()) {}
    ~HostTimer() {
        if (ctx) ctx->host_ms[k] += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
};

#define HGT_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t e_ = (call);                                                                \
        if (e_ != cudaSuccess) {                                                                \
            hgt_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            return HGT_ERR_CUDA;                                                                \
        }                                                                                       \
    } while (0)

#define HGT_CHECK(expr)               \
    do {                              \
        int rc_ = (expr);             \
        if (rc_ != HGT_OK) return rc_; \
    } while (0)

// ---- device helpers ------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// 1-D bulk copy global -> shared through the TMA unit (SASS: UBLKCP); bytes % 16 == 0, both 16-B aligned.
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// Context, error plumbing and small helpers of libhgt.
#include <stdarg.h>

#include <algorithm>
#include <mutex>
#include <utility>

#include "common.cuh"

static thread_local char g_err[1024] = "";

cudaError_t hgt_smem_at_least(const void *kernel, size_t bytes) {
    static std::mutex mu;
    static std::map<std::pair<int, const void *>, size_t> limit;  // (device, kernel) -> limit set so far
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lock(mu);
    size_t &cur = limit[{dev, kernel}];
    if (cur >= bytes) return cudaSuccess;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) cur = bytes;
    return e;
}

void hgt_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int MemPool::get(bool pinned, size_t n, void **out, size_t *cap) {
    const size_t want = round_up(n);
    std::multimap<size_t, void *> &fl = pinned ? free_pin : free_dev;
    auto it = fl.lower_bound(want);
    if (it != fl.end() && it->first <= want + want / 2) {
        *out = it->second;
        *cap = it->first;
        (pinned ? held_pin : held_dev) -= it->first;
        fl.erase(it);
        return HGT_OK;
    }
    cudaError_t e = pinned ? cudaMallocHost(out, want) : cudaMalloc(out, want);
    if (e != cudaSuccess) {  // give cached blocks back to the driver and retry once
        cudaGetLastError();
        drain();
        e = pinned ? cudaMallocHost(out, want) : cudaMalloc(out, want);
    }
    if (e != cudaSuccess) {
        hgt_set_error("%s(%zu) -> %s", pinned ? "cudaMallocHost" : "cudaMalloc", want, cudaGetErrorString(e));
        *out = nullptr;
        return HGT_ERR_NOMEM;
    }
    *cap = want;
    return HGT_OK;
}
void MemPool::put(bool pinned, void *p, size_t cap) {
    if (!p) return;
    (pinned ? free_pin : free_dev).emplace(cap, p);
    (pinned ? held_pin : held_dev) += cap;
}
void MemPool::drain() {
    for (auto &kv : free_dev) cudaFree(kv.second);
    for (auto &kv : free_pin) cudaFreeHost(kv.second);
    free_dev.clear();
    free_pin.clear();
    held_dev = held_pin = 0;
}

__global__ void small_h2d_kernel(unsigned char *dst, const unsigned char *src, size_t bytes) {
    const size_t tid = blockIdx.x * (size_t)blockDim.x + threadIdx.x, nth = (size_t)gridDim.x * blockDim.x;
    if ((((uintptr_t)dst | (uintptr_t)src) & 15) == 0) {
        const size_t n16 = bytes / 16;
        for (size_t i = tid; i < n16; i += nth) reinterpret_cast<uint4 *>(dst)[i] = reinterpret_cast<const uint4 *>(src)[i];
        for (size_t i = n16 * 16 + tid; i < bytes; i += nth) dst[i] = src[i];
    } else {
        for (size_t i = tid; i < bytes; i += nth) dst[i] = src[i];
    }
}
cudaError_t hgt_small_h2d(void *dst_dev, const void *src_pinned, size_t bytes, cudaStream_t st) {
    if (bytes == 0) return cudaSuccess;
    const unsigned blocks = (unsigned)std::min<size_t>((bytes / 16 + 255) / 256 + 1, 64);
    small_h2d_kernel<<<blocks, 256, 0, st>>>(static_cast<unsigned char *>(dst_dev), static_cast<const unsigned char *>(src_pinned),
                                            bytes);
    return cudaGetLastError();
}

extern "C" const char *hgt_last_error(void) { return g_err; }
extern "C" int hgt_abi_version(void) { return 3; }
extern "C" int hgt_row_pitch(int n_alleles) {
    int w = (n_alleles + 63) / 64;
    if (w < 2) w = 2;
    return (w + 1) & ~1;
}

extern "C" int hgt_init(int device, hgt_ctx **out) {
    if (!out) {
        hgt_set_error("hgt_init: out is null");
        return HGT_ERR_ARG;
    }
    *out = nullptr;
    int n = 0;
    HGT_CUDA(cudaGetDeviceCount(&n));
    if (device < 0 || device >= n) {
        hgt_set_error("hgt_init: device %d out of range (%d visible)", device, n);
        return HGT_ERR_ARG;
    }
    HGT_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    HGT_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        hgt_set_error("hgt_init: device %d is sm_%d%d; this library is built for sm_100a (B200) only", device,
                      prop.major, prop.minor);
        return HGT_ERR_UNSUPPORTED;
    }
    hgt_ctx *c = new hgt_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->smem_optin = prop.sharedMemPerBlockOptin;
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        hgt_set_error("cudaStreamCreate: %s", cudaGetErrorString(e));
        delete c;
        return HGT_ERR_CUDA;
    }
    *out = c;
    return HGT_OK;
}

extern "C" void hgt_free(hgt_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    ctx->pool.drain();
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" int hgt_host_alloc(size_t n_bytes, void **out) {
    if (!out) return HGT_ERR_ARG;
    *out = nullptr;
    HGT_CUDA(cudaHostAlloc(out, n_bytes ? n_bytes : 16, cudaHostAllocPortable));
    return HGT_OK;
}
extern "C" void hgt_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

extern "C" int64_t hgt_launch_count(const hgt_ctx *ctx) { return ctx ? ctx->launches : 0; }
extern "C" int hgt_sm_count(const hgt_ctx *ctx) { return ctx ? ctx->sm_count : 0; }

extern "C" void hgt_profile_enable(hgt_ctx *ctx, int on) {
    if (ctx) ctx->profile = on;
}
extern "C" void hgt_profile_reset(hgt_ctx *ctx) {
    if (!ctx) return;
    ctx->h2d_bytes = ctx->d2h_bytes = 0;
    for (int i = 0; i < 8; i++) {
        ctx->stage_ms[i] = 0;
        ctx->stage_launches[i] = 0;
        ctx->host_ms[i] = 0;
    }
}
extern "C" void hgt_profile_read(const hgt_ctx *ctx, double *stage_ms, int64_t *stage_launches, int64_t *h2d_bytes,
                                 int64_t *d2h_bytes) {
    if (!ctx) return;
    for (int i = 0; i < 8; i++) {
        if (stage_ms) stage_ms[i] = ctx->stage_ms[i];
        if (stage_launches) stage_launches[i] = ctx->stage_launches[i];
    }
    if (h2d_bytes) *h2d_bytes = ctx->h2d_bytes;
    if (d2h_bytes) *d2h_bytes = ctx->d2h_bytes;
}
extern "C" void hgt_profile_host(const hgt_ctx *ctx, double *host_ms) {
    if (!ctx || !host_ms) return;
    for (int i = 0; i < 8; i++) host_ms[i] = ctx->host_ms[i];
}

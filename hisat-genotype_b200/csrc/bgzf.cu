// BGZF inflate (BAM's compression) on the GPU: host walk of the block headers (hgt_bgzf_open), one warp per block on the
// device with CRC32 and ISIZE checked in the same kernel (hgt_bgzf_inflate), and the host emulation of the same decoder
// (hgt_bgzf_inflate_host).  The decoder is csrc/bgzf_dev.cuh.
#include <algorithm>
#include <atomic>
#include <string.h>
#include <thread>
#include <vector>

#include "bgzf_dev.cuh"
#include "common.cuh"

namespace {

constexpr int WARPS = 8;  // blocks per CTA

// the wording of zlib (inflate.c) and of sam_intake.read_bgzf where the rule is the same
const char *rule_text(uint32_t st) {
    static const char *const t[hgtz::N_STATUS] = {
        "ok",
        "invalid block type",
        "invalid stored block lengths",
        "too many length or distance symbols",
        "invalid code lengths set",
        "invalid bit length repeat",
        "invalid code -- missing end-of-block",
        "invalid literal/lengths set",
        "invalid distances set",
        "invalid literal/length code",
        "invalid distance code",
        "invalid distance too far back",
        "deflate stream runs past the end of the block",
        "deflate stream does not end with the block",
        "ISIZE",
        "ISIZE",
        "CRC32 mismatch",
    };
    return st < hgtz::N_STATUS ? t[st] : "unknown status";
}

uint32_t le32(const uint8_t *p) { return p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24; }

}  // namespace

struct hgt_bgzf {
    int32_t n_streams = 0;
    std::vector<const uint8_t *> data;
    std::vector<size_t> n_bytes;
    std::vector<int32_t> has_eof;
    // blocks of all streams in order; in_off / out_off [n_blocks + 1]: block b = input [in_off[b], in_off[b+1]) of the
    // streams laid end to end, output [out_off[b], out_off[b+1])
    std::vector<uint64_t> in_off, out_off;
    std::vector<int64_t> stream_blk;    // [n_streams + 1] first block of each stream
    std::vector<uint64_t> stream_in, stream_out;  // [n_streams + 1]
    int64_t n_blocks() const { return (int64_t)in_off.size() - 1; }
    int32_t stream_of(int64_t b) const {
        return (int32_t)(std::upper_bound(stream_blk.begin(), stream_blk.end(), b) - stream_blk.begin() - 1);
    }
};

// Failure word of a block: (block << 32) | status << 24 | bytes written.  The smallest one is the first failing block.
static __host__ __device__ uint64_t fail_word(int64_t b, uint32_t st, uint32_t n_out) {
    return (uint64_t)b << 32 | (uint64_t)st << 24 | (n_out & 0xffffffu);
}

static int report_failure(const hgt_bgzf *z, uint64_t w) {
    const int64_t b = (int64_t)(w >> 32);
    const uint32_t st = (uint32_t)(w >> 24) & 0xff, n_out = (uint32_t)w & 0xffffff;
    const int32_t s = z->stream_of(b);
    const long long at = (long long)(z->in_off[b] - z->stream_in[s]);
    const uint32_t isize = (uint32_t)(z->out_off[b + 1] - z->out_off[b]);
    if (st == hgtz::ISIZE_OVER)
        hgt_set_error("stream %d: BGZF block at byte %lld: ISIZE %u, inflated more than %u bytes", s, at, isize, n_out);
    else if (st == hgtz::ISIZE_UNDER)
        hgt_set_error("stream %d: BGZF block at byte %lld: ISIZE %u, inflated %u bytes", s, at, isize, n_out);
    else
        hgt_set_error("stream %d: BGZF block at byte %lld: %s", s, at, rule_text(st));
    return HGT_ERR_PARSE;
}

static const uint8_t kEof[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 0x42, 0x43, 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};

// The header rules of sam_intake._bgzf_blocks, byte for byte, plus ISIZE <= 65536.
static int walk_stream(hgt_bgzf *z, int32_t s) {
    const uint8_t *d = z->data[s];
    const size_t n = z->n_bytes[s];
    const uint64_t base = z->stream_in[s];
    size_t o = 0;
    while (o < n) {
        if (n - o < 18) {
            hgt_set_error("stream %d: truncated BGZF block header at byte %zu", s, o);
            return HGT_ERR_PARSE;
        }
        if (!(d[o] == 31 && d[o + 1] == 139 && d[o + 2] == 8 && (d[o + 3] & 4))) {
            hgt_set_error("stream %d: not a BGZF block at byte %zu", s, o);
            return HGT_ERR_PARSE;
        }
        const size_t xlen = d[o + 10] | (size_t)d[o + 11] << 8;
        if (o + 12 + xlen > n) {
            hgt_set_error("stream %d: truncated BGZF block header at byte %zu", s, o);
            return HGT_ERR_PARSE;
        }
        long bsize = -1;
        for (size_t x = o + 12; x + 4 <= o + 12 + xlen;) {
            const size_t slen = d[x + 2] | (size_t)d[x + 3] << 8;
            if (d[x] == 66 && d[x + 1] == 67 && slen == 2) {
                if (x + 6 > n) {  // read_bgzf reads BSIZE even where it leaves the extra field, and fails at the end of data
                    hgt_set_error("stream %d: truncated BGZF block header at byte %zu", s, o);
                    return HGT_ERR_PARSE;
                }
                bsize = d[x + 4] | (long)d[x + 5] << 8;
            }
            x += 4 + slen;
        }
        if (bsize < 0) {
            hgt_set_error("stream %d: gzip member without the BGZF BC field at byte %zu", s, o);
            return HGT_ERR_PARSE;
        }
        const size_t end = o + (size_t)bsize + 1;
        if (!(12 + xlen + 8 <= (size_t)bsize + 1 && end <= n)) {
            hgt_set_error("stream %d: truncated BGZF block at byte %zu", s, o);
            return HGT_ERR_PARSE;
        }
        const uint32_t isize = le32(d + end - 4);
        if (isize > hgtz::MAX_ISIZE) {
            hgt_set_error("stream %d: BGZF block at byte %zu: ISIZE %u > %u", s, o, isize, hgtz::MAX_ISIZE);
            return HGT_ERR_PARSE;
        }
        z->in_off.push_back(base + o);
        z->out_off.push_back(z->out_off.back() + isize);
        o = end;
    }
    return HGT_OK;
}

extern "C" int hgt_bgzf_open(int32_t n_streams, const void *const *data, const size_t *n_bytes, hgt_bgzf **out) {
    if (!out || n_streams < 0 || (n_streams > 0 && (!data || !n_bytes))) {
        hgt_set_error("hgt_bgzf_open: bad arguments");
        return HGT_ERR_ARG;
    }
    *out = nullptr;
    hgt_bgzf *z = new hgt_bgzf();
    z->n_streams = n_streams;
    z->stream_in.push_back(0);
    z->stream_out.push_back(0);
    z->out_off.push_back(0);
    for (int32_t s = 0; s < n_streams; s++) {
        if (!data[s] && n_bytes[s]) {
            delete z;
            hgt_set_error("hgt_bgzf_open: stream %d has no data pointer", s);
            return HGT_ERR_ARG;
        }
        z->data.push_back(static_cast<const uint8_t *>(data[s]));
        z->n_bytes.push_back(n_bytes[s]);
        z->stream_blk.push_back((int64_t)z->in_off.size());
        const int rc = walk_stream(z, s);
        if (rc != HGT_OK) {
            delete z;
            return rc;
        }
        z->stream_in.push_back(z->stream_in.back() + n_bytes[s]);
        z->stream_out.push_back(z->out_off.back());
        z->has_eof.push_back(n_bytes[s] >= 28 && memcmp(z->data[s] + n_bytes[s] - 28, kEof, 28) == 0);
    }
    z->stream_blk.push_back((int64_t)z->in_off.size());
    z->in_off.push_back(z->stream_in.back());
    if (z->n_blocks() >= (1ll << 31)) {
        hgt_set_error("hgt_bgzf_open: %lld blocks in one call (at most 2^31 - 1)", (long long)z->n_blocks());
        delete z;
        return HGT_ERR_UNSUPPORTED;
    }
    *out = z;
    return HGT_OK;
}

extern "C" int hgt_bgzf_sizes(const hgt_bgzf *z, size_t *out_bytes, int64_t *n_blocks, int32_t *has_eof) {
    if (!z) return HGT_ERR_ARG;
    for (int32_t s = 0; s < z->n_streams; s++) {
        if (out_bytes) out_bytes[s] = (size_t)(z->stream_out[s + 1] - z->stream_out[s]);
        if (n_blocks) n_blocks[s] = z->stream_blk[s + 1] - z->stream_blk[s];
        if (has_eof) has_eof[s] = z->has_eof[s];
    }
    return HGT_OK;
}

extern "C" void hgt_bgzf_free(hgt_bgzf *z) { delete z; }

// ---- device ---------------------------------------------------------------------------------------------------------
// One warp per block; the host walk has checked every header, so the block's XLEN, CRC32 and ISIZE are read here as they
// are.  *fail receives the smallest failure word (atomicMin; initialised to all ones).
__global__ void __launch_bounds__(WARPS * 32) bgzf_inflate_kernel(const uint8_t *__restrict__ in, const uint64_t *__restrict__ in_off,
                                                                  const uint64_t *__restrict__ out_off, int64_t n_blocks,
                                                                  uint8_t *__restrict__ out, unsigned long long *fail) {
    __shared__ uint32_t crc_tab[256];
    __shared__ hgtz::Tables tabs[WARPS];
    for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) crc_tab[i] = hgtz::crc_entry(i);
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t b = (int64_t)blockIdx.x * WARPS + warp;
    if (b >= n_blocks) return;
    const uint8_t *blk = in + in_off[b];
    const uint32_t bytes = (uint32_t)(in_off[b + 1] - in_off[b]);
    const uint32_t xlen = blk[10] | (uint32_t)blk[11] << 8;
    const uint32_t crc_want = blk[bytes - 8] | (uint32_t)blk[bytes - 7] << 8 | (uint32_t)blk[bytes - 6] << 16 |
                              (uint32_t)blk[bytes - 5] << 24;
    const uint32_t isize = (uint32_t)(out_off[b + 1] - out_off[b]);
    uint8_t *dst = out + out_off[b];
    uint32_t n_out = 0;
    uint32_t st = hgtz::inflate(blk + 12 + xlen, bytes - 12 - xlen - 8, dst, isize, tabs[warp], hgtz::Warp{lane, 32}, &n_out);
    if (st == hgtz::OK) {
        uint32_t lo, hi;
        hgtz::crc_slice(isize, lane, &lo, &hi);
        const uint32_t mine = hgtz::crc_update(crc_tab, 0, dst + lo, hi - lo);
        uint32_t full_lo, full_hi;
        hgtz::crc_slice(isize, 0, &full_lo, &full_hi);
        const uint32_t shift_full = hgtz::x8nmodp(full_hi - full_lo);
        uint32_t crc = 0;
        for (uint32_t k = 0; k < hgtz::CRC_SLICES; k++) {
            const uint32_t ck = __shfl_sync(0xffffffffu, mine, k);
            uint32_t a, e;
            hgtz::crc_slice(isize, k, &a, &e);
            crc = hgtz::crc_combine(crc, ck, e - a == full_hi - full_lo ? shift_full : hgtz::x8nmodp(e - a));
        }
        if (crc != crc_want) st = hgtz::CRC;
    }
    if (st != hgtz::OK && lane == 0) atomicMin(fail, (unsigned long long)fail_word(b, st, n_out));
}

extern "C" int hgt_bgzf_inflate(hgt_ctx *ctx, const hgt_bgzf *z, void *const *dst) {
    if (!ctx || !z || (z->n_streams > 0 && !dst)) {
        hgt_set_error("hgt_bgzf_inflate: bad arguments");
        return HGT_ERR_ARG;
    }
    for (int32_t s = 0; s < z->n_streams; s++)
        if (!dst[s] && z->stream_out[s + 1] > z->stream_out[s]) {
            hgt_set_error("hgt_bgzf_inflate: stream %d has no destination", s);
            return HGT_ERR_ARG;
        }
    const int64_t nb = z->n_blocks();
    if (nb == 0) return HGT_OK;
    HGT_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const size_t in_bytes = z->stream_in.back(), out_bytes = z->stream_out.back();
    const size_t desc_bytes = 2 * (size_t)(nb + 1) * sizeof(uint64_t);
    // device: input | output | descriptors | failure word; page-locked: descriptors | failure word
    const size_t o_out = (in_bytes + 15) & ~(size_t)15, o_desc = (o_out + out_bytes + 15) & ~(size_t)15,
                 o_fail = o_desc + desc_bytes, dev_bytes = o_fail + 8;
    void *dev = nullptr, *pin = nullptr;
    size_t dev_cap = 0, pin_cap = 0;
    HGT_CHECK(ctx->pool.get(false, dev_bytes, &dev, &dev_cap));
    int rc = ctx->pool.get(true, desc_bytes + 8, &pin, &pin_cap);
    if (rc != HGT_OK) {
        ctx->pool.put(false, dev, dev_cap);
        return rc;
    }
    uint8_t *d = static_cast<uint8_t *>(dev), *h = static_cast<uint8_t *>(pin);
    memcpy(h, z->in_off.data(), (nb + 1) * sizeof(uint64_t));
    memcpy(h + (nb + 1) * sizeof(uint64_t), z->out_off.data(), (nb + 1) * sizeof(uint64_t));
    uint64_t *h_fail = reinterpret_cast<uint64_t *>(h + desc_bytes);
    auto run = [&]() -> int {
        for (int32_t s = 0; s < z->n_streams; s++)
            if (z->n_bytes[s])
                HGT_CUDA(cudaMemcpyAsync(d + z->stream_in[s], z->data[s], z->n_bytes[s], cudaMemcpyHostToDevice, st));
        HGT_CUDA(cudaMemcpyAsync(d + o_desc, h, desc_bytes, cudaMemcpyHostToDevice, st));
        HGT_CUDA(cudaMemsetAsync(d + o_fail, 0xff, 8, st));
        ctx->h2d_bytes += (int64_t)(in_bytes + desc_bytes);
        const uint64_t *d_in_off = reinterpret_cast<const uint64_t *>(d + o_desc);
        bgzf_inflate_kernel<<<(unsigned)((nb + WARPS - 1) / WARPS), WARPS * 32, 0, st>>>(
            d, d_in_off, d_in_off + nb + 1, nb, d + o_out, reinterpret_cast<unsigned long long *>(d + o_fail));
        HGT_CUDA(cudaGetLastError());
        ctx->launches++;
        for (int32_t s = 0; s < z->n_streams; s++) {
            const size_t n = z->stream_out[s + 1] - z->stream_out[s];
            if (n) HGT_CUDA(cudaMemcpyAsync(dst[s], d + o_out + z->stream_out[s], n, cudaMemcpyDeviceToHost, st));
        }
        HGT_CUDA(cudaMemcpyAsync(h_fail, d + o_fail, 8, cudaMemcpyDeviceToHost, st));
        ctx->d2h_bytes += (int64_t)(out_bytes + 8);
        HGT_CUDA(cudaStreamSynchronize(st));
        return HGT_OK;
    };
    rc = run();
    const uint64_t w = *h_fail;
    ctx->pool.put(false, dev, dev_cap);
    ctx->pool.put(true, pin, pin_cap);
    if (rc != HGT_OK) return rc;
    return w == ~0ull ? HGT_OK : report_failure(z, w);
}

// ---- host emulation -------------------------------------------------------------------------------------------------
extern "C" int hgt_bgzf_inflate_host(const hgt_bgzf *z, int32_t n_threads, void *const *dst) {
    if (!z || (z->n_streams > 0 && !dst)) {
        hgt_set_error("hgt_bgzf_inflate_host: bad arguments");
        return HGT_ERR_ARG;
    }
    for (int32_t s = 0; s < z->n_streams; s++)
        if (!dst[s] && z->stream_out[s + 1] > z->stream_out[s]) {
            hgt_set_error("hgt_bgzf_inflate_host: stream %d has no destination", s);
            return HGT_ERR_ARG;
        }
    const int64_t nb = z->n_blocks();
    uint32_t crc_tab[256];
    for (uint32_t i = 0; i < 256; i++) crc_tab[i] = hgtz::crc_entry(i);
    std::atomic<int64_t> next{0};
    std::atomic<uint64_t> fail{~0ull};
    auto worker = [&]() {
        hgtz::Tables *T = new hgtz::Tables();
        for (int64_t b; (b = next.fetch_add(1)) < nb;) {
            const int32_t s = z->stream_of(b);
            const uint8_t *blk = z->data[s] + (z->in_off[b] - z->stream_in[s]);
            const uint32_t bytes = (uint32_t)(z->in_off[b + 1] - z->in_off[b]);
            const uint32_t xlen = blk[10] | (uint32_t)blk[11] << 8;
            const uint32_t isize = (uint32_t)(z->out_off[b + 1] - z->out_off[b]);
            uint8_t *out = static_cast<uint8_t *>(dst[s]) + (z->out_off[b] - z->stream_out[s]);
            uint32_t n_out = 0;
            uint32_t st = hgtz::inflate(blk + 12 + xlen, bytes - 12 - xlen - 8, out, isize, *T, hgtz::Warp{0, 1}, &n_out);
            if (st == hgtz::OK) {  // the kernel's 32 slices, combined in the same order
                uint32_t crc = 0;
                for (uint32_t k = 0; k < hgtz::CRC_SLICES; k++) {
                    uint32_t a, e;
                    hgtz::crc_slice(isize, k, &a, &e);
                    crc = hgtz::crc_combine(crc, hgtz::crc_update(crc_tab, 0, out + a, e - a), hgtz::x8nmodp(e - a));
                }
                if (crc != le32(blk + bytes - 8)) st = hgtz::CRC;
            }
            if (st != hgtz::OK) {
                const uint64_t w = fail_word(b, st, n_out);
                uint64_t cur = fail.load();
                while (w < cur && !fail.compare_exchange_weak(cur, w)) {
                }
            }
        }
        delete T;
    };
    int nt = n_threads > 0 ? n_threads : (int)std::max(1u, std::thread::hardware_concurrency());
    nt = (int)std::min<int64_t>(nt, std::max<int64_t>(nb, 1));
    std::vector<std::thread> pool;
    for (int t = 1; t < nt; t++) pool.emplace_back(worker);
    worker();
    for (auto &t : pool) t.join();
    const uint64_t w = fail.load();
    return w == ~0ull ? HGT_OK : report_failure(z, w);
}

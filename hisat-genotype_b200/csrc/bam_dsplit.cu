// Device split of BGZF-compressed BAM files (hgt_bam_dsplit_*): the work of the host split (bam_split.cpp) on the GPU,
// from the inflated streams kept in HBM.  The compressed bytes and small tables cross PCIe; the inflated bytes do not.
//
//   inflate      bgzf_launch (bgzf.cu) into an arena the handle owns
//   headers      bam_header_kernel walks every header on the device; the first 64 KB of each stream come back with the
//                inflate's failure word (one synchronisation; a longer header one more) and the host parses them with the
//                host split's code (bam_parse_header).  Up go per stream: first record, refID -> bucket, the name table.
//   index        the block_size chain, exact under the host's rule: the stream is cut into chunks; every chunk guesses its
//                first record (bam_plausible) and walks the chain to its end (index_guess_kernel); fix-up passes replace a
//                guess that disagrees with the exit of the chunk before (index_fix_kernel); one thread per stream then
//                checks every chunk in order and re-walks the few still wrong (index_resolve_kernel).  A guess only
//                decides where a walk starts, never the result.  Record counts come back (one synchronisation).
//   validation   bam_check_record per record; the first failing record in input order wins (atomicMin)
//   order        one sort of all records of all streams by (stream, bucket, read name bytewise with a prefix first, POS,
//                input order): merge passes of width 1, 2, 4, ... where every element finds its rank in the other run
//                by binary search (the key is unique, so no stability is needed), records of no bucket last
//   text sizes   bam_text_len_kernel over the ordered records, one scan; bucket sizes come back (one synchronisation)
//
// The host emulation of the index (hgt_bam_index_host) runs the same chunk functions on host threads.
#include <string.h>

#include <algorithm>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "bam_dsplit.h"
#include "bam_rec.cuh"
#include "bgzf_host.h"

namespace {

constexpr uint64_t WINDOW = 1u << 16;  // first read-back of every stream
constexpr uint64_t CHUNK = 4096;       // bytes of stream per index chunk
constexpr int FIX_PASSES = 2;          // fix-up passes launched before the serial resolve
constexpr uint32_t DROP = 0xffffffffu;  // sort key of a record in no bucket
constexpr int T = 256;

struct StreamDev {  // one stream of a call, as the index and validation kernels read it
    uint64_t base;   // of the stream in the inflated arena
    uint64_t n;      // inflated bytes
    uint64_t rec0;   // first record byte (end of the header)
    int64_t chunk0;  // first chunk of the stream (call-wide)
    int32_t n_hdr, pad;
    uint64_t tab;  // byte offset of the stream's tables in the table arena: name_off[n_hdr + 1] | bucket[n_hdr] | names
};
struct Chunk {
    uint64_t s, e;  // walk start, exit
    uint32_t n, brk;
};
struct StreamIdx {  // result of the index of one stream
    int64_t n_rec;
    uint64_t brk_at;  // chain break (byte of the stream), when broke
    int64_t broke;
};
struct HdrDev {
    uint64_t touched, end;
    int32_t n_hdr, code;
    int64_t pad;
};

// ---- the chunk functions of the index (device kernels and host emulation) ----------------------------------------------
HGT_HD void chunk_bounds(const StreamDev &S, int64_t j, uint64_t chunk, uint64_t *c0, uint64_t *c1) {
    *c0 = S.rec0 + (uint64_t)j * chunk;
    *c1 = *c0 + chunk < S.n ? *c0 + chunk : S.n;
}

HGT_HD void chunk_walk(const unsigned char *d, const StreamDev &S, uint64_t s, uint64_t c1, Chunk *c) {
    uint64_t e;
    uint32_t k;
    bool b;
    hgtb::bam_chunk_walk(d, S.n, s, c1, &e, &k, &b);
    *c = Chunk{s, e, k, b ? 1u : 0u};
}

// chunk j of stream S (d = the stream's bytes): a guessed start (the exact one for chunk 0) and its walk
HGT_HD void chunk_first(const unsigned char *d, const StreamDev &S, int64_t j, uint64_t chunk, Chunk *c) {
    uint64_t c0, c1;
    chunk_bounds(S, j, chunk, &c0, &c1);
    const uint64_t s = j == 0 ? c0 : hgtb::bam_chunk_guess(d, S.n, c0, c1, S.n_hdr);
    chunk_walk(d, S, s, c1, c);
}

// chunk j given the chunk before: its walk restarts from the exit of the one before when the two disagree
HGT_HD void chunk_fix(const unsigned char *d, const StreamDev &S, int64_t j, uint64_t chunk, const Chunk &prev,
                      const Chunk &cur, Chunk *out) {
    if (j == 0 || prev.brk || cur.s == prev.e) {
        *out = cur;
        return;
    }
    uint64_t c0, c1;
    chunk_bounds(S, j, chunk, &c0, &c1);
    chunk_walk(d, S, prev.e, c1, out);
}

// every chunk of the stream in order: the ones still wrong are re-walked; cnt[j] = records of chunk j (0 after a break)
HGT_HD void stream_resolve(const unsigned char *d, const StreamDev &S, int64_t nc, uint64_t chunk, Chunk *ch, int64_t *cnt,
                           StreamIdx *res) {
    int64_t total = 0;
    bool broke = false;
    uint64_t at = 0;
    for (int64_t j = 0; j < nc; j++) {
        if (broke) {
            cnt[j] = 0;
            continue;
        }
        if (j > 0 && ch[j].s != ch[j - 1].e) {
            uint64_t c0, c1;
            chunk_bounds(S, j, chunk, &c0, &c1);
            chunk_walk(d, S, ch[j - 1].e, c1, &ch[j]);
        }
        cnt[j] = ch[j].n;
        total += ch[j].n;
        if (ch[j].brk) {
            broke = true;
            at = ch[j].e;
        }
    }
    *res = StreamIdx{total, at, broke ? 1 : 0};
}

int64_t n_chunks_of(uint64_t n, uint64_t rec0, uint64_t chunk) { return n > rec0 ? (int64_t)((n - rec0 + chunk - 1) / chunk) : 0; }

// ---- kernels -------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int stream_of_chunk(const StreamDev *__restrict__ sd, int ns, int64_t k) {
    int lo = 0, hi = ns - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (sd[mid].chunk0 <= k) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

__global__ void bam_header_kernel(const unsigned char *__restrict__ data, const uint64_t *__restrict__ stream_out, int ns,
                                  HdrDev *__restrict__ out) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= ns) return;
    HdrDev h{};
    h.code = hgtb::bam_header_walk(data + stream_out[s], stream_out[s + 1] - stream_out[s], &h.end, &h.n_hdr, &h.touched);
    out[s] = h;
}

__global__ void __launch_bounds__(T) index_guess_kernel(const unsigned char *__restrict__ data, const StreamDev *__restrict__ sd,
                                                        int ns, int64_t n_chunks, Chunk *__restrict__ ch) {
    const int64_t k = (int64_t)blockIdx.x * T + threadIdx.x;
    if (k >= n_chunks) return;
    const StreamDev S = sd[stream_of_chunk(sd, ns, k)];
    chunk_first(data + S.base, S, k - S.chunk0, CHUNK, &ch[k]);
}

__global__ void __launch_bounds__(T) index_fix_kernel(const unsigned char *__restrict__ data, const StreamDev *__restrict__ sd,
                                                      int ns, int64_t n_chunks, const Chunk *__restrict__ in,
                                                      Chunk *__restrict__ out) {
    const int64_t k = (int64_t)blockIdx.x * T + threadIdx.x;
    if (k >= n_chunks) return;
    const StreamDev S = sd[stream_of_chunk(sd, ns, k)];
    const int64_t j = k - S.chunk0;
    chunk_fix(data + S.base, S, j, CHUNK, j > 0 ? in[k - 1] : in[k], in[k], &out[k]);
}

__global__ void index_resolve_kernel(const unsigned char *__restrict__ data, const StreamDev *__restrict__ sd, int ns,
                                     Chunk *__restrict__ ch, int64_t *__restrict__ cnt, StreamIdx *__restrict__ res) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= ns) return;
    const StreamDev S = sd[s];
    stream_resolve(data + S.base, S, sd[s + 1].chunk0 - S.chunk0, CHUNK, ch + S.chunk0, cnt + S.chunk0, &res[s]);
}

// record offsets (call-wide bytes of the arena) of every chunk, at the chunk's scanned record index
__global__ void __launch_bounds__(T) index_emit_kernel(const unsigned char *__restrict__ data, const StreamDev *__restrict__ sd,
                                                       int ns, int64_t n_chunks, const Chunk *__restrict__ ch,
                                                       const int64_t *__restrict__ first, uint64_t *__restrict__ off) {
    const int64_t k = (int64_t)blockIdx.x * T + threadIdx.x;
    if (k >= n_chunks) return;
    const int64_t n = first[k + 1] - first[k];
    if (n == 0) return;
    const StreamDev S = sd[stream_of_chunk(sd, ns, k)];
    const unsigned char *d = data + S.base;
    uint64_t o = ch[k].s;
    for (int64_t i = 0; i < n; i++) {
        off[first[k] + i] = S.base + o;
        o += 4 + (uint64_t)hgtb::ld_u32(d + o);
    }
}

// sort key parts: (stream, bucket) or DROP, and the first 8 name bytes big-endian, zero-padded
__device__ __forceinline__ int stream_of_record(const StreamDev *__restrict__ sd, int ns, const int64_t *__restrict__ first,
                                                int64_t g) {
    int lo = 0, hi = ns - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (first[sd[mid].chunk0] <= g) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

__global__ void __launch_bounds__(T) validate_kernel(const unsigned char *__restrict__ data, const unsigned char *__restrict__ tab,
                                                     const StreamDev *__restrict__ sd, int ns, const int64_t *__restrict__ first,
                                                     const uint64_t *__restrict__ off, int64_t n_rec, int32_t n_refs,
                                                     uint32_t *__restrict__ seg, uint64_t *__restrict__ pref,
                                                     unsigned long long *__restrict__ err) {
    const int64_t g = (int64_t)blockIdx.x * T + threadIdx.x;
    if (g >= n_rec) return;
    const int s = stream_of_record(sd, ns, first, g);
    const StreamDev &S = sd[s];
    const unsigned char *p = data + off[g];
    unsigned char tag[2];
    const int rule = hgtb::bam_check_record(p, hgtb::ld_u32(p) + 4, S.n_hdr, tag);
    uint32_t key = DROP;
    uint64_t pf = 0;
    if (rule != hgtb::RULE_OK) {
        atomicMin(err, (unsigned long long)g);
    } else {
        const int32_t ref = hgtb::ld_i32(p + 4);
        const int32_t *bucket = reinterpret_cast<const int32_t *>(tab + S.tab) + S.n_hdr + 1;
        const int32_t b = ref < 0 ? -1 : bucket[ref];
        if (b >= 0) {
            key = (uint32_t)s * (uint32_t)n_refs + (uint32_t)b;
            const uint32_t ln = p[12] - 1u;
            for (uint32_t i = 0; i < 8; i++) pf = pf << 8 | (i < ln ? p[hgtb::REC_FIXED + i] : 0);
        }
    }
    seg[g] = key;
    pref[g] = pf;
}

struct SortView {
    const unsigned char *data;
    const uint64_t *off;
    const uint32_t *seg;
    const uint64_t *pref;
    // the order rule of split_order.hpp within a bucket; buckets by (stream, bucket); records of no bucket last, in input order
    __device__ __forceinline__ bool less(uint32_t a, uint32_t b) const {
        if (seg[a] != seg[b]) return seg[a] < seg[b];
        if (seg[a] == DROP) return a < b;
        if (pref[a] != pref[b]) return pref[a] < pref[b];
        const unsigned char *pa = data + off[a], *pb = data + off[b];
        const uint32_t la = pa[12] - 1u, lb = pb[12] - 1u, m = la < lb ? la : lb;
        for (uint32_t i = 8; i < m; i++) {
            const unsigned char x = pa[hgtb::REC_FIXED + i], y = pb[hgtb::REC_FIXED + i];
            if (x != y) return x < y;
        }
        if (la != lb) return la < lb;
        const int32_t xa = hgtb::ld_i32(pa + 8), xb = hgtb::ld_i32(pb + 8);
        if (xa != xb) return xa < xb;
        return a < b;
    }
};

// one merge pass: runs of width w are merged pairwise; element i of a run lands at its rank in the merged pair
__global__ void __launch_bounds__(T) merge_rank_kernel(SortView v, const uint32_t *__restrict__ in, uint32_t *__restrict__ out,
                                                       int64_t n, int64_t w) {
    const int64_t i = (int64_t)blockIdx.x * T + threadIdx.x;
    if (i >= n) return;
    const uint32_t x = in[i];
    const int64_t run = i / w, base = (run & ~1ll) * w;
    int64_t lo, hi;
    if (run & 1) {
        lo = base;
        hi = base + w;
    } else {
        lo = base + w < n ? base + w : n;
        hi = base + 2 * w < n ? base + 2 * w : n;
    }
    const int64_t o0 = lo;
    while (lo < hi) {  // first element of the other run not less than x
        const int64_t mid = (lo + hi) >> 1;
        if (v.less(in[mid], x)) lo = mid + 1;
        else hi = mid;
    }
    out[base + (i - run * w) + (lo - o0)] = x;
}

__global__ void __launch_bounds__(T) iota_kernel(uint32_t *__restrict__ p, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * T + threadIdx.x;
    if (i < n) p[i] = (uint32_t)i;
}

// ordered offsets, and the bucket sizes (records of every (stream, bucket))
__global__ void __launch_bounds__(T) gather_kernel(const uint32_t *__restrict__ perm, const uint64_t *__restrict__ off,
                                                   const uint32_t *__restrict__ seg, int64_t n, uint64_t *__restrict__ ord,
                                                   uint32_t *__restrict__ oseg, unsigned long long *__restrict__ count) {
    const int64_t j = (int64_t)blockIdx.x * T + threadIdx.x;
    if (j >= n) return;
    const uint32_t i = perm[j];
    ord[j] = off[i];
    oseg[j] = seg[i];
    if (seg[i] != DROP) atomicAdd(&count[seg[i]], 1ull);
}

// the ordered records as a render source: record j of bucket oseg[j] (records of no bucket are measured and never used)
struct SortedSrc {
    const unsigned char *data;
    const uint64_t *ord;
    const uint32_t *oseg;
    const StreamDev *sd;
    const unsigned char *tab;
    const int32_t *own;  // [n_streams * n_refs]
    int32_t n_refs;
    bool hide_qual;
    __device__ __forceinline__ void view(int64_t j, hgtb::BamRec *r, hgtb::BamNames *nm, int64_t *) const {
        const unsigned char *p = data + ord[j];
        hgtb::bam_decode(p, (uint64_t)hgtb::ld_u32(p) + 4, false, r, hide_qual);
        const uint32_t k = oseg[j];
        const StreamDev &S = sd[k == DROP ? 0 : k / (uint32_t)n_refs];
        r->ref = k == DROP ? -1 : own[k];
        nm->off = reinterpret_cast<const uint32_t *>(tab + S.tab);
        nm->bytes = tab + S.tab + 8ull * S.n_hdr + 4;
        nm->n = k == DROP ? 0 : (uint32_t)S.n_hdr;
    }
};

// text offset at the first record of every bucket, and the failing record's head on the error path
__global__ void seg_text_kernel(const int64_t *__restrict__ seg0, const int64_t *__restrict__ toff, int64_t n_seg,
                                int64_t *__restrict__ out) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k <= n_seg) out[k] = toff[seg0[k]];
}

constexpr uint32_t FETCH = 296;  // fixed fields + the longest read name
struct Fetched {
    uint32_t size, rule;
    int32_t stream;
    unsigned char tag[2], pad[2];
    unsigned char head[FETCH];
};
__global__ void fetch_kernel(const unsigned char *__restrict__ data, const StreamDev *__restrict__ sd, int ns,
                             const int64_t *__restrict__ first, const uint64_t *__restrict__ off,
                             const unsigned long long *__restrict__ err, Fetched *__restrict__ out) {
    const int64_t g = (int64_t)*err;
    const unsigned char *p = data + off[g];
    const uint32_t size = hgtb::ld_u32(p) + 4;
    const int s = stream_of_record(sd, ns, first, g);
    if (threadIdx.x == 0) {
        out->size = size;
        out->stream = s;
        out->tag[0] = out->tag[1] = 0;
        out->rule = (uint32_t)hgtb::bam_check_record(p, size, sd[s].n_hdr, out->tag);
    }
    for (uint32_t i = threadIdx.x; i < FETCH; i += blockDim.x) out->head[i] = i < size ? p[i] : 0;
}

inline size_t a16(size_t x) { return (x + 15) & ~(size_t)15; }
inline size_t a8(size_t x) { return (x + 7) & ~(size_t)7; }
unsigned grid(int64_t n) { return (unsigned)((n + T - 1) / T); }

std::string chain_message(uint64_t at, int64_t n_rec) {
    char buf[160];
    snprintf(buf, sizeof buf, "truncated or malformed record at byte %llu of the BAM stream (after %lld records)",
             (unsigned long long)at, (long long)n_rec);
    return buf;
}

// temporaries of one create, from the context's pool
struct Temp {
    hgt_ctx *ctx;
    std::vector<std::pair<void *, size_t>> dev, pin;
    int get(bool pinned, size_t n, void **p) {
        size_t cap = 0;
        HGT_CHECK(ctx->pool.get(pinned, n ? n : 16, p, &cap));
        (pinned ? pin : dev).push_back({*p, cap});
        return HGT_OK;
    }
    ~Temp() {
        cudaStreamSynchronize(ctx->stream);  // nothing may still use a block that goes back to the pool
        for (auto &x : dev) ctx->pool.put(false, x.first, x.second);
        for (auto &x : pin) ctx->pool.put(true, x.first, x.second);
    }
};

}  // namespace

struct hgt_bam_dsplit {
    int device = 0;
    int32_t n_streams = 0, n_refs = 0;
    bool drop_qual = false;
    void *arena = nullptr;  // inflate arena: the streams at data (end to end)
    void *tab_mem = nullptr;  // per stream: name_off[n_hdr + 1] | bucket[n_hdr] | names (StreamDev::tab)
    void *hold = nullptr;     // ordered offsets | text offsets
    const unsigned char *data = nullptr, *tab = nullptr;
    const uint64_t *ord = nullptr;
    const int64_t *toff = nullptr;
    std::vector<StreamDev> sd;
    std::vector<int64_t> seg0, seg_text;  // [n_streams * n_refs + 1]: first ordered record, its text offset
    std::vector<int32_t> own;             // [n_streams * n_refs]
    ~hgt_bam_dsplit() {
        cudaSetDevice(device);
        if (arena) cudaFree(arena);
        if (tab_mem) cudaFree(tab_mem);
        if (hold) cudaFree(hold);
    }
};

int bam_dsplit_unit(const hgt_bam_dsplit *s, int32_t stream, int32_t ref, hgtk::DsplitUnitDev *u, int64_t *n_records,
                    size_t *text_bytes, int *device) {
    if (!s || stream < 0 || stream >= s->n_streams || ref < 0 || ref >= s->n_refs) return HGT_ERR_ARG;
    const size_t k = (size_t)stream * s->n_refs + ref;
    const StreamDev &S = s->sd[(size_t)stream];
    *u = hgtk::DsplitUnitDev{};
    u->data = s->data;
    u->rec = s->ord + s->seg0[k];
    u->toff = s->toff + s->seg0[k];
    u->name_off = reinterpret_cast<const uint32_t *>(s->tab + S.tab);
    u->name_bytes = s->tab + S.tab + 8ull * S.n_hdr + 4;
    u->n_names = (uint32_t)S.n_hdr;
    u->own = s->own[k];
    u->hide_qual = s->drop_qual ? 1u : 0u;
    *n_records = s->seg0[k + 1] - s->seg0[k];
    *text_bytes = (size_t)(s->seg_text[k + 1] - s->seg_text[k]);
    *device = s->device;
    return HGT_OK;
}

static int dsplit_run(hgt_ctx *ctx, const hgt_bgzf *z, int32_t n_refs, const char *const *ref_names, hgt_bam_dsplit *s) {
    using namespace hgtb;
    cudaStream_t st = ctx->stream;
    const int32_t ns = z->n_streams;
    Temp tmp{ctx, {}, {}};
    // ---- inflate into the handle's arena, header walk, first read-back
    const BgzfLayout L = bgzf_layout(z);
    HGT_CUDA(cudaMalloc(&s->arena, L.bytes));
    uint8_t *d = static_cast<uint8_t *>(s->arena);
    s->data = d + L.o_out;
    std::vector<uint64_t> win(ns + 1, 0);  // window offsets in the page-locked read-back
    for (int32_t i = 0; i < ns; i++) win[i + 1] = win[i] + a16(std::min<uint64_t>(z->stream_out[i + 1] - z->stream_out[i], WINDOW));
    const size_t o_hdr = a16(L.desc_bytes), o_so = o_hdr + 32ull * ns, o_fail = a16(o_so + 8ull * (ns + 1)),
                 o_win = o_fail + 16, pin1 = o_win + win[ns];
    uint8_t *h = nullptr, *dt = nullptr;
    HGT_CHECK(tmp.get(true, pin1, (void **)&h));
    HGT_CHECK(tmp.get(false, 32ull * ns + 8ull * (ns + 1), (void **)&dt));
    bgzf_descriptors(z, h);
    HGT_CHECK(bgzf_launch(ctx, z, L, d, h));
    memcpy(h + o_so, z->stream_out.data(), 8ull * (ns + 1));
    HdrDev *d_hdr = reinterpret_cast<HdrDev *>(dt);
    uint64_t *d_so = reinterpret_cast<uint64_t *>(dt + 32ull * ns);
    HGT_CUDA(cudaMemcpyAsync(d_so, h + o_so, 8ull * (ns + 1), cudaMemcpyHostToDevice, st));
    ctx->h2d_bytes += 8ll * (ns + 1);
    bam_header_kernel<<<(ns + 127) / 128, 128, 0, st>>>(s->data, d_so, ns, d_hdr);
    HGT_CUDA(cudaGetLastError());
    ctx->launches++;
    HGT_CUDA(cudaMemcpyAsync(h + o_hdr, d_hdr, 32ull * ns, cudaMemcpyDeviceToHost, st));
    HGT_CUDA(cudaMemcpyAsync(h + o_fail, d + L.o_fail, 8, cudaMemcpyDeviceToHost, st));
    ctx->d2h_bytes += 32ll * ns + 8;
    for (int32_t i = 0; i < ns; i++) {
        const uint64_t n = std::min<uint64_t>(z->stream_out[i + 1] - z->stream_out[i], WINDOW);
        if (n) HGT_CUDA(cudaMemcpyAsync(h + o_win + win[i], s->data + z->stream_out[i], n, cudaMemcpyDeviceToHost, st));
        ctx->d2h_bytes += (int64_t)n;
    }
    HGT_CUDA(cudaStreamSynchronize(st));
    const uint64_t fail = *reinterpret_cast<const uint64_t *>(h + o_fail);
    if (fail != ~0ull) return bgzf_report_failure(z, fail);
    const HdrDev *hh = reinterpret_cast<const HdrDev *>(h + o_hdr);
    // ---- headers longer than the window: one more read-back of exactly the bytes the walk read
    std::vector<uint64_t> big(ns + 1, 0);
    for (int32_t i = 0; i < ns; i++) big[i + 1] = big[i] + (hh[i].touched > WINDOW ? a16(hh[i].touched) : 0);
    uint8_t *hb = nullptr;
    if (big[ns]) {
        HGT_CHECK(tmp.get(true, big[ns], (void **)&hb));
        for (int32_t i = 0; i < ns; i++)
            if (big[i + 1] > big[i]) {
                HGT_CUDA(cudaMemcpyAsync(hb + big[i], s->data + z->stream_out[i], hh[i].touched, cudaMemcpyDeviceToHost, st));
                ctx->d2h_bytes += (int64_t)hh[i].touched;
            }
        HGT_CUDA(cudaStreamSynchronize(st));
    }
    // ---- parse on the host; n_ok = streams before the first bad header
    std::unordered_map<std::string, int> ref_index;
    for (int r = 0; r < n_refs; r++) ref_index[ref_names[r]] = r;  // the last of equal names, as the host split
    int32_t n_ok = ns, hdr_code = HDR_OK;
    std::vector<std::vector<std::string>> names((size_t)ns);
    s->sd.assign((size_t)ns + 1, StreamDev{});
    s->own.assign((size_t)ns * n_refs, -1);
    std::vector<uint8_t> tab_img;
    int64_t n_chunks = 0;
    for (int32_t i = 0; i < ns; i++) {
        const uint8_t *b = big[i + 1] > big[i] ? hb + big[i] : h + o_win + win[i];
        uint64_t end = 0;
        const int rc = bam_parse_header(b, z->stream_out[i + 1] - z->stream_out[i], &end, &names[(size_t)i]);
        if (rc != HDR_OK) {
            n_ok = i;
            hdr_code = rc;
            break;
        }
        StreamDev &S = s->sd[(size_t)i];
        S.base = z->stream_out[i];
        S.n = z->stream_out[i + 1] - z->stream_out[i];
        S.rec0 = end;
        S.chunk0 = n_chunks;
        S.n_hdr = (int32_t)names[(size_t)i].size();
        S.tab = tab_img.size();
        n_chunks += n_chunks_of(S.n, S.rec0, CHUNK);
        // name_off[n_hdr + 1] | bucket[n_hdr] | names, padded to 8 bytes
        std::vector<uint32_t> no(1, 0);
        std::vector<int32_t> bk;
        std::string bytes;
        for (int32_t k = 0; k < S.n_hdr; k++) {
            const std::string &nm = names[(size_t)i][(size_t)k];
            bytes += nm;
            no.push_back((uint32_t)bytes.size());
            auto it = ref_index.find(nm);
            bk.push_back(it == ref_index.end() ? -1 : it->second);
            if (it != ref_index.end() && s->own[(size_t)i * n_refs + it->second] < 0) s->own[(size_t)i * n_refs + it->second] = k;
        }
        const size_t at = tab_img.size();
        tab_img.resize(at + a8(8ull * S.n_hdr + 4 + bytes.size()), 0);
        memcpy(tab_img.data() + at, no.data(), 4 * no.size());
        if (S.n_hdr) memcpy(tab_img.data() + at + 4 * no.size(), bk.data(), 4 * bk.size());
        memcpy(tab_img.data() + at + 8ull * S.n_hdr + 4, bytes.data(), bytes.size());
    }
    s->sd[(size_t)n_ok].chunk0 = n_chunks;
    for (int32_t i = n_ok + 1; i <= ns; i++) s->sd[(size_t)i].chunk0 = n_chunks;
    // ---- index of the streams before the first bad header
    const size_t sd_bytes = sizeof(StreamDev) * ((size_t)n_ok + 1);
    const size_t o_tab = a16(sd_bytes);
    uint8_t *hu = nullptr, *du = nullptr;
    HGT_CHECK(tmp.get(true, o_tab + tab_img.size() + 32ull * (n_ok + 1) + 16, (void **)&hu));
    memcpy(hu, s->sd.data(), sd_bytes);
    if (!tab_img.empty()) memcpy(hu + o_tab, tab_img.data(), tab_img.size());
    HGT_CHECK(tmp.get(false, o_tab, (void **)&du));
    HGT_CUDA(cudaMemcpyAsync(du, hu, sd_bytes, cudaMemcpyHostToDevice, st));
    const StreamDev *d_sd = reinterpret_cast<const StreamDev *>(du);
    ctx->h2d_bytes += (int64_t)(sd_bytes + tab_img.size());
    HGT_CUDA(cudaMalloc(&s->tab_mem, std::max<size_t>(tab_img.size(), 16)));
    s->tab = static_cast<const unsigned char *>(s->tab_mem);
    if (!tab_img.empty()) HGT_CUDA(cudaMemcpyAsync(s->tab_mem, hu + o_tab, tab_img.size(), cudaMemcpyHostToDevice, st));
    Chunk *ch[2] = {nullptr, nullptr};
    int64_t *cnt = nullptr, *part = nullptr;
    StreamIdx *d_res = nullptr;
    HGT_CHECK(tmp.get(false, sizeof(Chunk) * (size_t)std::max<int64_t>(n_chunks, 1), (void **)&ch[0]));
    HGT_CHECK(tmp.get(false, sizeof(Chunk) * (size_t)std::max<int64_t>(n_chunks, 1), (void **)&ch[1]));
    HGT_CHECK(tmp.get(false, 8 * (size_t)(n_chunks + 1), (void **)&cnt));
    HGT_CHECK(tmp.get(false, 8 * (size_t)hgt_dev_scan_partials(std::max<int64_t>(n_chunks, 1)), (void **)&part));
    HGT_CHECK(tmp.get(false, sizeof(StreamIdx) * (size_t)std::max(n_ok, 1), (void **)&d_res));
    int cur = 0;
    if (n_chunks > 0) {
        index_guess_kernel<<<grid(n_chunks), T, 0, st>>>(s->data, d_sd, n_ok, n_chunks, ch[0]);
        ctx->launches++;
        for (int p = 0; p < FIX_PASSES; p++, cur ^= 1) {
            index_fix_kernel<<<grid(n_chunks), T, 0, st>>>(s->data, d_sd, n_ok, n_chunks, ch[cur], ch[cur ^ 1]);
            ctx->launches++;
        }
    }
    if (n_ok > 0) {
        index_resolve_kernel<<<(n_ok + 63) / 64, 64, 0, st>>>(s->data, d_sd, n_ok, ch[cur], cnt, d_res);
        ctx->launches++;
    }
    HGT_CUDA(cudaGetLastError());
    HGT_CHECK(hgt_dev_scan(ctx, st, cnt, n_chunks, cnt, part));
    StreamIdx *h_res = reinterpret_cast<StreamIdx *>(hu + o_tab + a16(tab_img.size()));
    if (n_ok > 0) HGT_CUDA(cudaMemcpyAsync(h_res, d_res, sizeof(StreamIdx) * n_ok, cudaMemcpyDeviceToHost, st));
    ctx->d2h_bytes += (int64_t)(sizeof(StreamIdx) * n_ok);
    HGT_CUDA(cudaStreamSynchronize(st));
    // ---- streams before the first broken chain: their records are checked and ordered
    int32_t n_val = n_ok;
    for (int32_t i = 0; i < n_ok; i++)
        if (h_res[i].broke) {
            n_val = i;
            break;
        }
    int64_t N = 0;
    for (int32_t i = 0; i < n_val; i++) N += h_res[i].n_rec;
    if (N > 0x7fffffffll) {
        hgt_set_error("hgt_bam_dsplit_create: %lld records in one call (at most 2^31 - 1)", (long long)N);
        return HGT_ERR_UNSUPPORTED;
    }
    const int64_t n_seg = (int64_t)ns * n_refs;
    const size_t o_toff = a16(8 * (size_t)N);
    HGT_CUDA(cudaMalloc(&s->hold, o_toff + 8 * (size_t)(N + 1)));
    uint8_t *hold = static_cast<uint8_t *>(s->hold);
    s->ord = reinterpret_cast<const uint64_t *>(hold);
    s->toff = reinterpret_cast<const int64_t *>(hold + o_toff);
    uint64_t *off = nullptr, *pref = nullptr;
    uint32_t *seg = nullptr, *perm[2] = {nullptr, nullptr}, *oseg = nullptr;
    int64_t *segn = nullptr, *len = nullptr, *part2 = nullptr;
    int32_t *d_own = nullptr;
    unsigned long long *d_err = nullptr;
    Fetched *d_fetch = nullptr;
    const size_t NN = (size_t)std::max<int64_t>(N, 1);
    HGT_CHECK(tmp.get(false, 8 * NN, (void **)&off));
    HGT_CHECK(tmp.get(false, 8 * NN, (void **)&pref));
    HGT_CHECK(tmp.get(false, 4 * NN, (void **)&seg));
    HGT_CHECK(tmp.get(false, 4 * NN, (void **)&perm[0]));
    HGT_CHECK(tmp.get(false, 4 * NN, (void **)&perm[1]));
    HGT_CHECK(tmp.get(false, 4 * NN, (void **)&oseg));
    HGT_CHECK(tmp.get(false, 8 * (size_t)(n_seg + 1) * 2, (void **)&segn));
    HGT_CHECK(tmp.get(false, 8 * (NN + 1), (void **)&len));
    HGT_CHECK(tmp.get(false, 8 * (size_t)hgt_dev_scan_partials(std::max<int64_t>(std::max<int64_t>(N, n_seg), 1)), (void **)&part2));
    HGT_CHECK(tmp.get(false, a16(4 * (size_t)n_seg) + 16 + sizeof(Fetched), (void **)&d_own));
    d_err = reinterpret_cast<unsigned long long *>(reinterpret_cast<uint8_t *>(d_own) + a16(4 * (size_t)n_seg));
    d_fetch = reinterpret_cast<Fetched *>(reinterpret_cast<uint8_t *>(d_err) + 16);
    // the own table rides in the page-locked block after the stream results
    uint8_t *hx = nullptr;
    const size_t o_hown = 0, o_hsz = a16(4 * (size_t)n_seg), o_herr = o_hsz + 16 * (size_t)(n_seg + 1);
    HGT_CHECK(tmp.get(true, o_herr + 16 + sizeof(Fetched), (void **)&hx));
    memcpy(hx + o_hown, s->own.data(), 4 * (size_t)n_seg);
    HGT_CUDA(cudaMemcpyAsync(d_own, hx + o_hown, 4 * (size_t)n_seg, cudaMemcpyHostToDevice, st));
    ctx->h2d_bytes += 4 * n_seg;
    HGT_CUDA(cudaMemsetAsync(d_err, 0xff, 8, st));
    HGT_CUDA(cudaMemsetAsync(segn, 0, 8 * (size_t)(n_seg + 1), st));
    const unsigned char *dtab = s->tab;
    const int64_t n_chunks_val = s->sd[(size_t)n_val].chunk0;
    if (N > 0) {
        index_emit_kernel<<<grid(n_chunks_val), T, 0, st>>>(s->data, d_sd, n_val, n_chunks_val, ch[cur], cnt, off);
        validate_kernel<<<grid(N), T, 0, st>>>(s->data, dtab, d_sd, n_val, cnt, off, N, n_refs, seg, pref, d_err);
        iota_kernel<<<grid(N), T, 0, st>>>(perm[0], N);
        ctx->launches += 3;
        const SortView v{s->data, off, seg, pref};
        int pc = 0;
        for (int64_t w = 1; w < N; w *= 2, pc ^= 1) {
            merge_rank_kernel<<<grid(N), T, 0, st>>>(v, perm[pc], perm[pc ^ 1], N, w);
            ctx->launches++;
        }
        gather_kernel<<<grid(N), T, 0, st>>>(perm[pc], off, seg, N, const_cast<uint64_t *>(s->ord), oseg,
                                              reinterpret_cast<unsigned long long *>(segn));
        const SortedSrc src{s->data, s->ord, oseg, d_sd, dtab, d_own, n_refs, s->drop_qual};
        hgtk::bam_text_len_kernel<<<grid(N), T, 0, st>>>(src, N, len);
        ctx->launches += 2;
        HGT_CUDA(cudaGetLastError());
    }
    HGT_CHECK(hgt_dev_scan(ctx, st, len, N, const_cast<int64_t *>(s->toff), part2));
    HGT_CHECK(hgt_dev_scan(ctx, st, segn, n_seg, segn, part2));
    int64_t *d_st = segn + (n_seg + 1);
    seg_text_kernel<<<grid(n_seg + 1), T, 0, st>>>(segn, s->toff, n_seg, d_st);
    ctx->launches++;
    HGT_CUDA(cudaGetLastError());
    HGT_CUDA(cudaMemcpyAsync(hx + o_hsz, segn, 16 * (size_t)(n_seg + 1), cudaMemcpyDeviceToHost, st));
    HGT_CUDA(cudaMemcpyAsync(hx + o_herr, d_err, 8, cudaMemcpyDeviceToHost, st));
    ctx->d2h_bytes += 16 * (n_seg + 1) + 8;
    HGT_CUDA(cudaStreamSynchronize(st));
    const uint64_t err = *reinterpret_cast<const uint64_t *>(hx + o_herr);
    if (err != ~0ull) {  // the first bad record: its head and rule back, the host split's message
        Fetched *hf = reinterpret_cast<Fetched *>(hx + o_herr + 16);
        fetch_kernel<<<1, 128, 0, st>>>(s->data, d_sd, n_val, cnt, off, d_err, d_fetch);
        ctx->launches++;
        HGT_CUDA(cudaGetLastError());
        HGT_CUDA(cudaMemcpyAsync(hf, d_fetch, sizeof(Fetched), cudaMemcpyDeviceToHost, st));
        ctx->d2h_bytes += sizeof(Fetched);
        HGT_CUDA(cudaStreamSynchronize(st));
        const std::string msg = bam_record_message(hf->head, hf->size, (int)hf->rule, hf->tag);
        hgt_set_error("stream %d: %s", hf->stream, msg.c_str());
        return rule_unsupported((int)hf->rule) ? HGT_ERR_UNSUPPORTED : HGT_ERR_PARSE;
    }
    if (n_val < n_ok) {
        hgt_set_error("stream %d: %s", n_val, chain_message(h_res[n_val].brk_at, h_res[n_val].n_rec).c_str());
        return HGT_ERR_PARSE;
    }
    if (n_ok < ns) {
        hgt_set_error("stream %d: %s", n_ok, bam_header_why(hdr_code));
        return HGT_ERR_PARSE;
    }
    const int64_t *hsz = reinterpret_cast<const int64_t *>(hx + o_hsz);
    s->seg0.assign(hsz, hsz + n_seg + 1);
    s->seg_text.assign(hsz + n_seg + 1, hsz + 2 * (n_seg + 1));
    return HGT_OK;
}

extern "C" int hgt_bam_dsplit_create(hgt_ctx *ctx, const hgt_bgzf *z, int32_t n_refs, const char *const *ref_names,
                                     int32_t flags, hgt_bam_dsplit **out) {
    if (!ctx || !z || !out || n_refs < 1 || !ref_names || (flags & ~HGT_SPLIT_DROP_QUAL)) {
        hgt_set_error("hgt_bam_dsplit_create: bad argument");
        return HGT_ERR_ARG;
    }
    *out = nullptr;
    for (int32_t r = 0; r < n_refs; r++)
        if (!ref_names[r]) {
            hgt_set_error("hgt_bam_dsplit_create: bad argument");
            return HGT_ERR_ARG;
        }
    if (z->n_streams < 1 || (int64_t)z->n_streams * n_refs >= (1ll << 31)) {
        hgt_set_error("hgt_bam_dsplit_create: %d streams x %d references (1 .. 2^31 - 1 buckets)", z->n_streams, n_refs);
        return HGT_ERR_UNSUPPORTED;
    }
    HGT_CUDA(cudaSetDevice(ctx->device));
    hgt_bam_dsplit *s = new hgt_bam_dsplit();
    s->device = ctx->device;
    s->n_streams = z->n_streams;
    s->n_refs = n_refs;
    s->drop_qual = (flags & HGT_SPLIT_DROP_QUAL) != 0;
    const int rc = dsplit_run(ctx, z, n_refs, ref_names, s);
    if (rc != HGT_OK) {
        cudaStreamSynchronize(ctx->stream);
        delete s;
        return rc;
    }
    *out = s;
    return HGT_OK;
}

extern "C" int hgt_bam_dsplit_sizes(const hgt_bam_dsplit *s, int64_t *records, size_t *text_bytes) {
    if (!s) return HGT_ERR_ARG;
    for (size_t k = 0; k + 1 < s->seg0.size(); k++) {
        if (records) records[k] = s->seg0[k + 1] - s->seg0[k];
        if (text_bytes) text_bytes[k] = (size_t)(s->seg_text[k + 1] - s->seg_text[k]);
    }
    return HGT_OK;
}

extern "C" void hgt_bam_dsplit_free(hgt_bam_dsplit *s) { delete s; }

// ---- host emulation of the index ----------------------------------------------------------------------------------------
extern "C" int hgt_bam_index_host(const void *bam, size_t n_bytes, int64_t chunk_bytes, int32_t n_threads, int64_t cap,
                                  uint64_t *offsets, int64_t *n_records) {
    if ((!bam && n_bytes) || chunk_bytes < 1 || cap < 0 || (cap > 0 && !offsets) || !n_records) {
        hgt_set_error("hgt_bam_index_host: bad argument");
        return HGT_ERR_ARG;
    }
    const unsigned char *d = static_cast<const unsigned char *>(bam);
    std::vector<std::string> names;
    StreamDev S{};
    S.n = n_bytes;
    const int hrc = hgtb::bam_parse_header(d, n_bytes, &S.rec0, &names);
    if (hrc != hgtb::HDR_OK) {
        hgt_set_error("hgt_bam_index_host: %s", hgtb::bam_header_why(hrc));
        return HGT_ERR_PARSE;
    }
    S.n_hdr = (int32_t)names.size();
    const uint64_t chunk = (uint64_t)chunk_bytes;
    const int64_t nc = n_chunks_of(S.n, S.rec0, chunk);
    std::vector<Chunk> a((size_t)nc), b((size_t)nc);
    const int nt = std::max(1, std::min<int>(n_threads > 0 ? n_threads : (int)std::max(1u, std::thread::hardware_concurrency()),
                                             (int)std::min<int64_t>(nc, 1 << 20) + 1));
    auto par = [&](auto f) {  // f(j) for every chunk, in slices over nt threads
        std::vector<std::thread> th;
        for (int t = 0; t < nt; t++)
            th.emplace_back([&, t]() {
                for (int64_t j = nc * t / nt; j < nc * (t + 1) / nt; j++) f(j);
            });
        for (auto &x : th) x.join();
    };
    par([&](int64_t j) { chunk_first(d, S, j, chunk, &a[(size_t)j]); });
    for (int p = 0; p < FIX_PASSES; p++) {
        par([&](int64_t j) { chunk_fix(d, S, j, chunk, j > 0 ? a[(size_t)j - 1] : a[(size_t)j], a[(size_t)j], &b[(size_t)j]); });
        std::swap(a, b);
    }
    std::vector<int64_t> cnt((size_t)nc + 1, 0);
    StreamIdx res{};
    stream_resolve(d, S, nc, chunk, a.data(), cnt.data(), &res);
    if (res.broke) {
        hgt_set_error("hgt_bam_index_host: %s", chain_message(res.brk_at, res.n_rec).c_str());
        return HGT_ERR_PARSE;
    }
    *n_records = res.n_rec;
    int64_t g = 0;
    for (int64_t j = 0; j < nc; j++) {
        uint64_t o = a[(size_t)j].s;
        for (int64_t i = 0; i < cnt[(size_t)j]; i++, g++) {
            if (g < cap) offsets[g] = o;
            o += 4 + (uint64_t)hgtb::ld_u32(d + o);
        }
    }
    return HGT_OK;
}

// Kernels around walk_dev.cuh: line index of the text arena, record parse, pileup straight from the CIGAR text, run
// heads / mate de-dup, the walk (common case + ambiguity pass), the pair stage (count pass, scans, fill pass), plus the
// host emulation of the same sequence (hgt_host_walk, no GPU).  Included by typing.cu.
//
// Everything here is byte / integer work bound by HBM and L2 bandwidth (SURVEY.md 8d): thread per line for the serial
// state machines (a line is ~350 B, a warp's 32 lines ~11 KB: L1-resident while the warp scans them), warp per line
// where lanes can share a record (pileup), 16-byte loads for the newline scan.
#pragma once
#include <vector>

#include "common.cuh"
#include "walk_dev.cuh"

namespace hgtk {
using namespace hgtd;

constexpr int LINE_THREADS = 256;
constexpr int CHUNK_BYTES = LINE_THREADS * 64;  // bytes of text per CTA of the newline kernels
constexpr int SCAN_THREADS = 256, SCAN_ITEMS = 16, SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

// '\n' bytes of a 32-bit word, exact (no borrow artefacts): 0x80 in every byte that equals 0x0A
__device__ __forceinline__ uint32_t nl_mask(uint32_t w) {
    const uint32_t x = w ^ 0x0A0A0A0Au;
    const uint32_t t = (x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu;
    return ~(t | x | 0x7F7F7F7Fu);
}

// exclusive prefix sum of `v` over the CTA (blockDim.x = 256); *total receives the CTA sum
__device__ __forceinline__ int block_exclusive_scan(int v, int *total) {
    __shared__ int s_warp[LINE_THREADS / 32];
    __shared__ int s_total;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    if (warp == 0) {
        int w = lane < LINE_THREADS / 32 ? s_warp[lane] : 0;
#pragma unroll
        for (int o = 1; o < LINE_THREADS / 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += y;
        }
        if (lane < LINE_THREADS / 32) s_warp[lane] = w;
        if (lane == LINE_THREADS / 32 - 1) s_total = w;
    }
    __syncthreads();
    const int base = warp ? s_warp[warp - 1] : 0;
    *total = s_total;
    __syncthreads();
    return base + x - v;
}

// pass 1 of the line index: newlines per 16 KB chunk (text is 16-byte aligned and padded with '\n' to a multiple of 16)
__global__ void __launch_bounds__(LINE_THREADS) count_newlines_kernel(const char *__restrict__ text, int64_t n_bytes,
                                                                     int64_t *__restrict__ chunk_count) {
    const int64_t base = (int64_t)blockIdx.x * CHUNK_BYTES + (int64_t)threadIdx.x * 64;
    int c = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int64_t o = base + k * 16;
        if (o < n_bytes) {
            const uint4 v = *reinterpret_cast<const uint4 *>(text + o);
            c += __popc(nl_mask(v.x)) + __popc(nl_mask(v.y)) + __popc(nl_mask(v.z)) + __popc(nl_mask(v.w));
        }
    }
    int total;
    block_exclusive_scan(c, &total);
    if (threadIdx.x == 0) chunk_count[blockIdx.x] = total;
}

// pass 2: line_off[k + 1] = offset of the byte after the k-th newline (chunk_base = exclusive scan of the chunk counts)
__global__ void __launch_bounds__(LINE_THREADS) index_lines_kernel(const char *__restrict__ text, int64_t n_bytes,
                                                                  const int64_t *__restrict__ chunk_base,
                                                                  int64_t *__restrict__ line_off) {
    const int64_t base = (int64_t)blockIdx.x * CHUNK_BYTES + (int64_t)threadIdx.x * 64;
    uint32_t m[16];
    int c = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int64_t o = base + k * 16;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (o < n_bytes) v = *reinterpret_cast<const uint4 *>(text + o);
        m[4 * k] = nl_mask(v.x); m[4 * k + 1] = nl_mask(v.y); m[4 * k + 2] = nl_mask(v.z); m[4 * k + 3] = nl_mask(v.w);
        if (o >= n_bytes) m[4 * k] = m[4 * k + 1] = m[4 * k + 2] = m[4 * k + 3] = 0;
        c += __popc(m[4 * k]) + __popc(m[4 * k + 1]) + __popc(m[4 * k + 2]) + __popc(m[4 * k + 3]);
    }
    int total;
    int64_t at = chunk_base[blockIdx.x] + block_exclusive_scan(c, &total);
    if (blockIdx.x == 0 && threadIdx.x == 0) line_off[0] = 0;
#pragma unroll
    for (int w = 0; w < 16; w++) {
        uint32_t x = m[w];
        while (x) {
            const int bit = __ffs((int)x) - 1;  // 7, 15, 23 or 31
            x &= x - 1;
            line_off[++at] = base + w * 4 + (bit >> 3) + 1;
        }
    }
}

// ---- exclusive scan of int64 arrays: out[0..n] (n + 1 entries, out[n] = total); in place allowed ----------------------------
__global__ void __launch_bounds__(SCAN_THREADS) scan_partials_kernel(const int64_t *__restrict__ in, int64_t n,
                                                                    int64_t *__restrict__ partial) {
    __shared__ int64_t s[SCAN_THREADS / 32];
    const int64_t t0 = (int64_t)blockIdx.x * SCAN_TILE;
    int64_t v = 0;
    for (int k = 0; k < SCAN_ITEMS; k++) {
        const int64_t i = t0 + (int64_t)k * SCAN_THREADS + threadIdx.x;
        if (i < n) v += in[i];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        int64_t t = 0;
        for (int w = 0; w < SCAN_THREADS / 32; w++) t += s[w];
        partial[blockIdx.x] = t;
    }
}
// one CTA: exclusive scan of the partials in place, total to partial[n_part]
__global__ void __launch_bounds__(1024) scan_single_kernel(int64_t *__restrict__ partial, int64_t n_part) {
    __shared__ int64_t s_warp[32];
    __shared__ int64_t s_carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int64_t b = 0; b < n_part; b += 1024) {
        const int64_t i = b + threadIdx.x;
        const int64_t v = i < n_part ? partial[i] : 0;
        int64_t x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) s_warp[warp] = x;
        __syncthreads();
        if (warp == 0) {
            int64_t w = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int64_t y = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += y;
            }
            s_warp[lane] = w;
        }
        __syncthreads();
        const int64_t base = s_carry + (warp ? s_warp[warp - 1] : 0);
        if (i < n_part) partial[i] = base + x - v;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = base + x;
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[n_part] = s_carry;
}
__global__ void __launch_bounds__(SCAN_THREADS) scan_apply_kernel(const int64_t *in, int64_t n,
                                                                 const int64_t *__restrict__ partial, int64_t n_part,
                                                                 int64_t *out) {  // in == out allowed
    __shared__ int64_t s_warp[SCAN_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t t0 = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;  // thread owns 16 adjacent items
    int64_t v[SCAN_ITEMS];
    int64_t sum = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) {
        v[k] = t0 + k < n ? in[t0 + k] : 0;
        sum += v[k];
    }
    int64_t x = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int64_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    int64_t base = partial[blockIdx.x];
    for (int w = 0; w < warp; w++) base += s_warp[w];
    int64_t run = base + x - sum;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) {
        if (t0 + k < n) out[t0 + k] = run;
        run += v[k];
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) out[n] = partial[n_part];
}

// ---- thread per line ---------------------------------------------------------------------------------------------------------
__global__ void unit_lines_kernel(ReadsView R) {  // first line of every unit: lower_bound(line_off, unit_off[u])
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u > R.n_units) return;
    const int64_t key = R.unit_off[u];
    int64_t lo = 0, hi = R.n_lines;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (R.line_off[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    R.unit_line0[u] = lo;
}
// The CTA's 128 consecutive lines are one contiguous piece of the arena (~45 KB at 100 bp reads): ONE bulk copy through
// the TMA unit (cp.async.bulk, SASS UBLKCP) brings it to shared memory behind an mbarrier, and the byte-serial state
// machines of the threads (one line each) then read shared memory instead of issuing 32 different L1 lines per load.
// A block of lines that does not fit (very long lines) is read from the arena directly.
constexpr int STAGE_LINES = 128;
struct Stage {
    uint64_t *mbar;
    uint32_t phase;
    char *smem;
    int smem_bytes;
};
__device__ __forceinline__ void stage_init(Stage &s, uint64_t *mbar, char *smem, int smem_bytes) {
    s.mbar = mbar; s.phase = 0; s.smem = smem; s.smem_bytes = smem_bytes;
    if (threadIdx.x == 0) {
        mbar_init(mbar, 1);
        fence_barrier_init();
    }
    __syncthreads();
}
// base pointer such that base + line_off[i] addresses line i for i in [i0, i1)
__device__ __forceinline__ const char *stage_lines(Stage &s, const ReadsView &R, int64_t i0, int64_t i1) {
    const int64_t b = R.line_off[i0] & ~(int64_t)15, e = (R.line_off[i1] + 15) & ~(int64_t)15;
    if (e - b > s.smem_bytes) return R.text;
    __syncthreads();  // every thread is done with the previous image
    if (threadIdx.x == 0) {
        mbar_expect_tx(s.mbar, (uint32_t)(e - b));
        bulk_g2s(s.smem, R.text + b, (uint32_t)(e - b), s.mbar);
    }
    mbar_wait(s.mbar, s.phase);
    s.phase ^= 1u;
    return s.smem - b;
}

// ---- pileup (common:1100-1121) straight from the CIGAR text: warp per line, lanes over the bases of each M / D op ------------
__device__ __forceinline__ void pileup_line(const ReadsView &R, int64_t r, const char *line, uint32_t *__restrict__ counts_all, int lane) {
    const RecFields f = R.rec[r];
    const char *cig = line + f.cig_off, *seq = line + f.seq_off;
    const int u = R.unit[r];
    const int L = R.loci[R.unit_locus[u]].L;
    uint32_t *counts = counts_all + (size_t)R.unit_pos0[u] * 6;
    int gpos = f.pos, rpos = 0, len = 0;
    for (int k = 0; k < f.cig_len; k++) {
        const char c = cig[k];  // same address in every lane: one broadcast load
        if (c >= '0' && c <= '9') {
            len = len * 10 + (c - '0');
            continue;
        }
        if (c == 'M' || c == 'D') {
            for (int j = lane; j < len; j += 32) {
                const int g = gpos + j;
                if (g < L) {
                    int code = 5;
                    if (c == 'M') {
                        const char ch = rpos + j < f.seq_len ? seq[rpos + j] : 'N';
                        code = ch == 'A' ? 0 : ch == 'C' ? 1 : ch == 'G' ? 2 : ch == 'T' ? 3 : 4;
                    }
                    atomicAdd(&counts[(size_t)g * 6 + code], 1u);
                }
            }
        }
        if (c == 'M' || c == 'D' || c == 'N') gpos += len;
        if (c == 'M' || c == 'I' || c == 'S') rpos += len;
        len = 0;
    }
}
__global__ void __launch_bounds__(256) pileup_text_kernel(ReadsView R, uint32_t *__restrict__ counts_all) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp0; r < R.n_lines; r += nwarps)
        if (R.st[r] & ST_PU) pileup_line(R, r, R.text + R.line_off[r], counts_all, lane);
}

__global__ void __launch_bounds__(STAGE_LINES) parse_kernel(ReadsView R, WalkParams P, int smem_bytes) {
    extern __shared__ __align__(128) char s_text[];
    __shared__ uint64_t mbar;
    Stage sg;
    stage_init(sg, &mbar, s_text, smem_bytes);
    const int64_t n_blk = (R.n_lines + STAGE_LINES - 1) / STAGE_LINES;
    for (int64_t blk = blockIdx.x; blk < n_blk; blk += gridDim.x) {
        const int64_t i0 = blk * STAGE_LINES, i1 = min(i0 + (int64_t)STAGE_LINES, R.n_lines);
        const char *base = stage_lines(sg, R, i0, i1);
        const int64_t i = i0 + threadIdx.x;
        if (i < i1) parse_line(R, P, base, i);
    }
}
__global__ void __launch_bounds__(256) head_kernel(ReadsView R) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < R.n_lines; i += (int64_t)gridDim.x * blockDim.x)
        mark_head(R, i);
}
__global__ void __launch_bounds__(256) candidate_kernel(ReadsView R) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < R.n_lines; i += (int64_t)gridDim.x * blockDim.x)
        mark_candidate(R, i);
}
// Error-correction bits of the warp's 32 records (EcMask, walk_dev.cuh).
//   1. every lane parses the CIGAR of ITS record into at most three M segments (read range, backbone shift) - 32 records in
//      parallel, the (short, divergent) byte loads all in flight together - and parks them in shared memory;
//   2. record by record the whole warp covers a segment in one step: lane l takes the four read bases 4l .. 4l+3 of the
//      segment (two aligned 32-bit loads + funnel shift each for SEQ and for the representative-base sets, coalesced over the
//      warp), tests them, and three shuffle steps gather the 32 nibbles into four words, which the owner lane ORs into its
//      mask at the segment's read offset.
// Reads longer than 128 bases, more than three M segments, or a malformed CIGAR leave valid = false: the walk then tests the
// bases itself (and reports the CIGAR error).
struct EcParams {
    const char *seq;
    const uint8_t *ntm;
    int32_t L, nseg;
    struct Seg {
        uint16_t r0, r1;  // read bases [r0, r1)
        int32_t shift;    // backbone position = read index + shift
    } seg[3];
    int32_t pad[2];
};
static_assert(sizeof(EcParams) == 56, "EcParams layout");
__device__ __forceinline__ uint32_t load4_unaligned(const void *p) {  // bytes p[0..3] as a little-endian word
    const uintptr_t a = (uintptr_t)p;
    const uint32_t *w = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3);
    const uint32_t lo = w[0], hi = w[1];
    return __funnelshift_r(lo, hi, (uint32_t)(a & 3) * 8u);
}
__device__ __forceinline__ EcMask warp_ec_masks(const ReadsView &R, const WalkParams &P, const char *text, int64_t i, bool cand,
                                                EcParams *s_warp /* [32], this warp's */) {
    const int lane = threadIdx.x & 31;
    EcMask mine;
    mine.w0 = mine.w1 = mine.w2 = mine.w3 = 0;
    mine.valid = false;
    if (cand && P.error_correction) {
        const RecFields f = R.rec[i];
        const int u = R.unit[i];
        const char *line = text + R.line_off[i];
        EcParams p;
        p.seq = line + f.seq_off;
        p.ntm = R.nt_mask + R.unit_pos0[u];
        p.L = R.loci[R.unit_locus[u]].L;
        p.nseg = 0;
        p.pad[0] = p.pad[1] = 0;
        bool ok = f.seq_len <= ECM_MAX_SEQ;
        const char *cig = line + f.cig_off;
        const int cn = f.cig_len, sl = f.seq_len;
        int32_t right_pos = f.pos, read_pos = 0;
        int cp = 0;
        while (ok && cp < cn) {
            int32_t length = 0;
            char c = cig[cp];
            bool have = false;
            while (is_dig(c)) {
                have = true;
                if (length < (1 << 24)) length = length * 10 + (c - '0');
                cp++;
                if (cp >= cn) break;
                c = cig[cp];
            }
            if (!have || cp >= cn) {
                ok = false;  // malformed: the walk reports it
                break;
            }
            cp++;
            if (c == 'M') {
                // read bases of the segment that exist and lie on the backbone
                const int32_t shift = right_pos - read_pos;
                const int32_t lo = max(read_pos, -shift), hi = min(min(read_pos + length, sl), p.L - shift);
                if (hi > lo) {
                    if (p.nseg >= 3) ok = false;
                    else {
                        p.seg[p.nseg].r0 = (uint16_t)lo;
                        p.seg[p.nseg].r1 = (uint16_t)hi;
                        p.seg[p.nseg].shift = shift;
                        p.nseg++;
                    }
                }
            }
            if (c == 'M' || c == 'N' || c == 'D') right_pos += length;
            if (c == 'M' || c == 'I' || c == 'S') read_pos += length;
        }
        if (ok) s_warp[lane] = p;
        mine.valid = ok;
    }
    unsigned todo = __ballot_sync(0xffffffffu, mine.valid);  // (also orders the shared-memory writes before the reads)
    while (todo) {
        const int r = __ffs((int)todo) - 1;
        todo &= todo - 1;
        const EcParams *p = s_warp + r;
        const char *seq = p->seq;
        const uint8_t *ntm = p->ntm;
        const int nseg = p->nseg;
        uint32_t a0 = 0, a1 = 0, a2 = 0, a3 = 0;
        for (int sg = 0; sg < nseg; sg++) {
            const int r0 = p->seg[sg].r0, r1 = p->seg[sg].r1, shift = p->seg[sg].shift;
            const int rp = r0 + 4 * lane;  // this lane's four read bases
            uint32_t f = 0;
            if (rp < r1) {
                const uint32_t sv = load4_unaligned(seq + rp), mv = load4_unaligned(ntm + rp + shift);
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const uint32_t ch = (sv >> (8 * k)) & 0xffu, m = (mv >> (8 * k)) & 0xffu;
                    // A 0x41, C 0x43, G 0x47, T 0x54: bits 1-2 give 0, 1, 3, 2 -> x ^ (x >> 1) = 0, 1, 2, 3; the letters
                    // themselves are bits 1, 3, 7, 20 of a 32-bit table indexed by the low five bits
                    const uint32_t x = (ch >> 1) & 3u, code = x ^ (x >> 1);
                    const bool acgt = (ch >> 5) == 2u && ((0x0010008Au >> (ch & 31u)) & 1u);
                    const bool flag = m != 0 && !(acgt && ((m >> code) & 1u));
                    f |= (flag ? 1u : 0u) << k;
                }
                const int nv = r1 - rp;  // bases of this lane inside the segment
                if (nv < 4) f &= (1u << nv) - 1u;
            }
            // nibbles of 8 consecutive lanes -> one word (at lanes 0, 8, 16, 24)
            uint32_t x = f | (__shfl_down_sync(0xffffffffu, f, 1) << 4);
            x |= __shfl_down_sync(0xffffffffu, x, 2) << 8;
            x |= __shfl_down_sync(0xffffffffu, x, 4) << 16;
            const uint32_t v0 = __shfl_sync(0xffffffffu, x, 0), v1 = __shfl_sync(0xffffffffu, x, 8),
                           v2 = __shfl_sync(0xffffffffu, x, 16), v3 = __shfl_sync(0xffffffffu, x, 24);
            // segment-relative bits -> read index: shift the 128-bit vector left by r0 (bits past 127 belong to no base)
            const int ws = r0 >> 5, bs = r0 & 31;
            uint32_t t0 = v0, t1 = v1, t2 = v2, t3 = v3;
            if (bs) {
                t3 = (v3 << bs) | (v2 >> (32 - bs));
                t2 = (v2 << bs) | (v1 >> (32 - bs));
                t1 = (v1 << bs) | (v0 >> (32 - bs));
                t0 = v0 << bs;
            }
            if (ws == 0) { a0 |= t0; a1 |= t1; a2 |= t2; a3 |= t3; }
            else if (ws == 1) { a1 |= t0; a2 |= t1; a3 |= t2; }
            else if (ws == 2) { a2 |= t0; a3 |= t1; }
            else a3 |= t0;
        }
        if (lane == r) {
            mine.w0 = a0; mine.w1 = a1; mine.w2 = a2; mine.w3 = a3;
        }
    }
    __syncwarp();
    return mine;
}

// The walk reads its lines from the arena, not from a staged image like parse_kernel: with the ambiguity work split off
// into two list passes, L1-cached global loads measured faster for it (DESIGN.md 7).  Compiled for 6 CTAs per SM
// (80 registers): without the bound ptxas picks 72 registers and more spill loads, and the walk measured 1 % slower.
__global__ void __launch_bounds__(STAGE_LINES, 6) walk_kernel(ReadsView R, WalkParams P) {
    __shared__ __align__(16) EcParams s_ecp[STAGE_LINES];
    const int64_t n_blk = (R.n_lines + STAGE_LINES - 1) / STAGE_LINES;
    for (int64_t blk = blockIdx.x; blk < n_blk; blk += gridDim.x) {
        const int64_t i0 = blk * STAGE_LINES, i1 = min(i0 + (int64_t)STAGE_LINES, R.n_lines);
        const int64_t i = i0 + threadIdx.x;
        const bool cand = i < i1 && (R.st[i] & ST_CAND);
        const EcMask M = warp_ec_masks(R, P, R.text, i, cand, s_ecp + (threadIdx.x & ~31));
        if (cand) walk_record<0>(R, P, R.text, i, -1, M);
    }
}
// ---- list passes by position ---------------------------------------------------------------------------------------------------
// walk_kernel queues records in arrival order; the reads of a unit are name-grouped, i.e. at random positions, so the 32
// records of a warp of the second / third pass would walk 32 different stretches of the Alts tables - different trip
// counts (2 of 32 lanes active in those loops) and no sharing of the table lines.  A counting sort by (locus, position / 32)
// puts neighbours on the backbone into the same warp.  Three small kernels, list length read on the device.
constexpr int SORT_BUCKETS = 16384;
__device__ __forceinline__ int list_sort_key(const ReadsView &R, int32_t i) {
    const int locus = R.unit_locus[R.unit[i]] & 31;
    int p = R.rec[i].pos >> 5;
    p = p < 0 ? 0 : (p > 511 ? 511 : p);
    return (locus << 9) | p;
}
__global__ void __launch_bounds__(256) list_hist_kernel(ReadsView R, const int32_t *__restrict__ list, const int32_t *__restrict__ n_ptr,
                                                        int32_t *__restrict__ hist) {
    const int n = *n_ptr;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x)
        atomicAdd(&hist[list_sort_key(R, list[k])], 1);
}
__global__ void __launch_bounds__(1024) list_scan_kernel(int32_t *__restrict__ hist) {  // counts -> exclusive offsets, one CTA
    __shared__ int32_t s_warp[32];
    constexpr int PER = SORT_BUCKETS / 1024;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    int32_t v[PER], sum = 0;
#pragma unroll
    for (int k = 0; k < PER; k++) {
        v[k] = hist[t * PER + k];
        sum += v[k];
    }
    int32_t x = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    if (warp == 0) {
        int32_t w = s_warp[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int32_t y = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += y;
        }
        s_warp[lane] = w;
    }
    __syncthreads();
    int32_t run = (warp ? s_warp[warp - 1] : 0) + x - sum;
#pragma unroll
    for (int k = 0; k < PER; k++) {
        hist[t * PER + k] = run;
        run += v[k];
    }
}
__global__ void __launch_bounds__(256) list_scatter_kernel(ReadsView R, const int32_t *__restrict__ list, const int32_t *__restrict__ n_ptr,
                                                           int32_t *__restrict__ cursor, int32_t *__restrict__ out) {
    const int n = *n_ptr;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        const int32_t i = list[k];
        out[atomicAdd(&cursor[list_sort_key(R, i)], 1)] = i;
    }
}

// second pass: records with an Alts anchor in reach (amb_list, filled by walk_kernel; its length stays on the device),
// `list` = amb_list in backbone order
__global__ void __launch_bounds__(128) walk_amb_kernel(ReadsView R, WalkParams P, const int32_t *__restrict__ list) {
    __shared__ __align__(16) EcParams s_ecp[128];
    const int n = *R.n_amb, n_round = (n + 31) & ~31;  // whole warps: the lanes compute the masks together
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n_round; k += gridDim.x * blockDim.x) {
        const bool on = k < n;
        const int64_t i = on ? list[k] : 0;
        const EcMask M = warp_ec_masks(R, P, R.text, i, on, s_ecp + (threadIdx.x & ~31));
        if (on) walk_record<1>(R, P, R.text, i, -1, M);
    }
}
// third pass: records with several haplotypes, `list` = slow_list in backbone order
__global__ void __launch_bounds__(128) walk_slow_kernel(ReadsView R, WalkParams P, const int32_t *__restrict__ list, int n_slow) {
    __shared__ __align__(16) EcParams s_ecp[128];
    const int n_round = (n_slow + 31) & ~31;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n_round; k += gridDim.x * blockDim.x) {
        const bool on = k < n_slow;
        const int64_t i = on ? list[k] : 0;
        const EcMask M = warp_ec_masks(R, P, R.text, i, on, s_ecp + (threadIdx.x & ~31));
        if (on) walk_record<2>(R, P, R.text, i, k, M);
    }
}
__global__ void __launch_bounds__(128) pair_count_kernel(ReadsView R) {  // thread per run (head_list)
    const int n = *R.n_heads;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) pair_jobs<false>(R, R.head_list[k], k);
}
__global__ void __launch_bounds__(128) pair_fill_kernel(ReadsView R) {
    const int n = *R.n_heads;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) pair_jobs<true>(R, R.head_list[k], k);
}

// per-locus totals of the pair stage from the scanned arrays: out[l][6] = pairs, haplotypes, rows, small jobs, big jobs,
// first line of the locus
__global__ void locus_totals_kernel(ReadsView R, int n_loci, const int32_t *__restrict__ locus_unit0, int64_t *__restrict__ out) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= n_loci) return;
    const int64_t a = R.unit_line0[locus_unit0[l]], b = R.unit_line0[locus_unit0[l + 1]];
    out[l * 6 + 0] = R.s_pairs[b] - R.s_pairs[a];
    out[l * 6 + 1] = R.s_haps[b] - R.s_haps[a];
    out[l * 6 + 2] = R.s_rows[b] - R.s_rows[a];
    out[l * 6 + 3] = R.s_small[b] - R.s_small[a];
    out[l * 6 + 4] = R.s_big[b] - R.s_big[a];
    out[l * 6 + 5] = a;
}


}  // namespace hgtk

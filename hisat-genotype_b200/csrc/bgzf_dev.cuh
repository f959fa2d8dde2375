// BGZF block inflate (RFC 1951 DEFLATE plus the CRC32 / ISIZE trailer of the gzip member) as __host__ __device__
// functions: the kernel (bgzf.cu: bgzf_inflate_kernel, one warp per block) and the host emulation (hgt_bgzf_inflate_host)
// run the same code, so the CPU tests pin what the device decides.
//
// Accept / reject is zlib's raw inflate as sam_intake.read_bgzf runs it (zlib.decompressobj(-15), then eof, no unused
// data, ISIZE, CRC32): the rules and their wording are zlib's inflate.c / inftrees.c (inflate_table: an over-subscribed
// set is refused, an incomplete one too except a literal/length or distance set whose only code has length 1; a distance
// set without codes is legal until a distance is decoded).  Two zlib behaviours are folded into plain rules: a stream
// that runs past the block's bytes (zlib waits for more input, read_bgzf then refuses it as not ended) is OVERRUN, and a
// code-length code without any code (zlib decodes every length as 0 and then finds no end-of-block code) is CL_SET.
//
// Termination: every loop below consumes at least one input bit or produces at least one output byte per iteration and
// checks the bit count against the block's extent (Bits::overrun) or the output against ISIZE, so any input ends with a
// status.  The bit reader never loads outside [in, in + n); bits past the end read as zeros.
//
// Warp form: all lanes of a warp run the same serial symbol decode in lockstep (table reads are shared-memory broadcasts),
// lane 0 writes literals, and the lanes copy a match together: byte j of a match of distance d is out[o - d + j % d], so
// every lane reads bytes written before the match and an overlapping match needs one pass.  The host runs it as one lane.
#pragma once
#include <stdint.h>

#ifndef HGT_HD
#define HGT_HD __host__ __device__ __forceinline__
#endif

namespace hgtz {

enum Status : uint32_t {
    OK = 0,
    BTYPE,        // BTYPE 3
    STORED_LEN,   // stored block LEN != ~NLEN
    COUNTS,       // HLIT > 286 or HDIST > 30 (as counts: 257 + HLIT > 286, 1 + HDIST > 30)
    CL_SET,       // code-length code over-subscribed, incomplete or empty
    REPEAT,       // code 16 without a previous length, or a repeat past HLIT + HDIST
    NO_EOB,       // no code for symbol 256
    LIT_SET,      // literal/length set over-subscribed or incomplete
    DIST_SET,     // distance set over-subscribed or incomplete
    LIT_CODE,     // bit pattern without a literal/length code, or symbol 286 / 287
    DIST_CODE,    // bit pattern without a distance code, or distance code 30 / 31
    FAR,          // distance before the block's first output byte
    OVERRUN,      // the stream reads past the block's compressed bytes
    TRAILING,     // bytes left after the final DEFLATE block
    ISIZE_OVER,   // more output than ISIZE
    ISIZE_UNDER,  // the final block ends with less output than ISIZE
    CRC,          // CRC32 of the output differs from the trailer's
    N_STATUS
};

constexpr int LIT_FAST = 10, DIST_FAST = 8, CL_FAST = 7;  // first-level lookup bits; longer codes take the canonical walk
constexpr uint32_t MAX_ISIZE = 65536;                      // BGZF: one block inflates to at most 64 KiB
constexpr uint32_t CRC_POLY = 0xEDB88320u;
constexpr uint32_t CRC_SLICES = 32;                        // a block's CRC32 is hashed in 32 slices and combined

// Decode tables of one warp (shared memory in the kernel): canonical code counts per length, the symbols sorted by
// (length, value), and a first-level table indexed by the next FAST input bits: symbol | length << 9, or 0 when no code
// of at most FAST bits matches (then decode() walks the canonical code).  The code-length code lives in the distance
// arrays while the literal/length lengths are read.
struct Tables {
    uint16_t lcnt[16], dcnt[16], offs[16];
    uint16_t lsym[288], dsym[32];
    uint16_t lfast[1 << LIT_FAST], dfast[1 << DIST_FAST];
    uint8_t lens[320];
};

struct Warp {
    uint32_t lane, n;  // n = 32 in the kernel, 1 on the host
};

HGT_HD void wsync() {
#ifdef __CUDA_ARCH__
    __syncwarp();
#endif
}

// LSB-first bit reader clamped to [p, p + n).
struct Bits {
    const uint8_t *p;
    uint32_t n, next, cnt;  // bytes, next byte to load, bits held in buf
    uint64_t buf, used;     // used = bits consumed
    HGT_HD void init(const uint8_t *q, uint32_t nb) {
        p = q;
        n = nb;
        next = cnt = 0;
        buf = used = 0;
    }
    HGT_HD void refill() {  // at least 57 bits held afterwards
        while (cnt <= 56) {
            const uint64_t b = next < n ? p[next] : 0;
            buf |= b << cnt;
            next++;
            cnt += 8;
        }
    }
    HGT_HD uint32_t peek(int k) const { return (uint32_t)(buf & ((1ull << k) - 1)); }
    HGT_HD void drop(int k) {
        buf >>= k;
        cnt -= k;
        used += k;
    }
    HGT_HD uint32_t get(int k) {  // k <= 16
        refill();
        const uint32_t v = peek(k);
        drop(k);
        return v;
    }
    HGT_HD bool overrun() const { return used > 8ull * n; }
    HGT_HD void align() { drop(cnt & 7); }  // loads are whole bytes, so cnt % 8 = bits to the next byte boundary
};

// Canonical decode of the first `fbits` (the fast table) or 15 bits (the walk) of `bits`: symbol | length << 9, 0 if none.
HGT_HD uint32_t canonical(uint32_t bits, int max_len, const uint16_t *cnt, const uint16_t *sym) {
    int code = 0, first = 0, index = 0;
    for (int len = 1; len <= max_len; len++) {
        code |= (bits >> (len - 1)) & 1;
        const int count = cnt[len];
        if (code - first < count) return sym[index + code - first] | (uint32_t)len << 9;
        index += count;
        first += count;
        first <<= 1;
        code <<= 1;
    }
    return 0;
}

// One symbol; the caller has refilled.  -1: no code matches.
HGT_HD int decode(Bits &br, const uint16_t *fast, int fbits, const uint16_t *cnt, const uint16_t *sym) {
    uint32_t e = fast[br.peek(fbits)];
    if (!e) e = canonical(br.peek(15), 15, cnt, sym);
    if (!e) return -1;
    br.drop(e >> 9);
    return (int)(e & 511);
}

enum { KIND_CODES = 0, KIND_LENS = 1, KIND_DISTS = 2 };

// Tables of a code from its lengths (lens[0, n) readable by every lane).  Nonzero: the set is refused.
HGT_HD int build(const uint8_t *lens, int n, uint16_t *cnt, uint16_t *sym, uint16_t *fast, int fbits, int kind, uint16_t *offs,
                 Warp w) {
    if (w.lane == 0) {
        for (int l = 0; l < 16; l++) cnt[l] = 0;
        for (int s = 0; s < n; s++) cnt[lens[s]]++;
    }
    wsync();
    int left = 1, max = 0;
    for (int l = 1; l < 16; l++) {
        left = (left << 1) - cnt[l];
        if (left < 0) return 1;  // over-subscribed
        if (cnt[l]) max = l;
    }
    if (max == 0) {
        if (kind == KIND_CODES) return 1;
    } else if (left > 0 && (kind == KIND_CODES || max != 1)) {
        return 1;  // incomplete
    }
    if (w.lane == 0) {
        offs[1] = 0;
        for (int l = 1; l < 15; l++) offs[l + 1] = offs[l] + cnt[l];
        for (int s = 0; s < n; s++)
            if (lens[s]) sym[offs[lens[s]]++] = (uint16_t)s;
    }
    wsync();
    for (uint32_t i = w.lane; i < (1u << fbits); i += w.n) fast[i] = (uint16_t)canonical(i, fbits, cnt, sym);
    wsync();
    return 0;
}

HGT_HD uint32_t cl_order(uint32_t i) {  // 16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15
    if (i < 3) return 16 + i;
    if (i == 3) return 0;
    const uint32_t j = i - 4;
    return j & 1 ? 7 - j / 2 : 8 + j / 2;
}

HGT_HD uint32_t fixed_tables(Tables &T, Warp w) {
    for (uint32_t i = w.lane; i < 320; i += w.n)
        T.lens[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : i < 288 ? 8 : 5;
    wsync();
    build(T.lens, 288, T.lcnt, T.lsym, T.lfast, LIT_FAST, KIND_LENS, T.offs, w);
    build(T.lens + 288, 32, T.dcnt, T.dsym, T.dfast, DIST_FAST, KIND_DISTS, T.offs, w);
    return OK;
}

HGT_HD uint32_t dynamic_tables(Bits &br, Tables &T, Warp w) {
    const uint32_t nlen = br.get(5) + 257, ndist = br.get(5) + 1, ncode = br.get(4) + 4;
    if (br.overrun()) return OVERRUN;
    if (nlen > 286 || ndist > 30) return COUNTS;
    if (w.lane == 0)
        for (uint32_t i = 0; i < 19; i++) T.lens[i] = 0;
    for (uint32_t i = 0; i < ncode; i++) {
        const uint32_t v = br.get(3);
        if (w.lane == 0) T.lens[cl_order(i)] = (uint8_t)v;
    }
    if (br.overrun()) return OVERRUN;
    wsync();
    if (build(T.lens, 19, T.dcnt, T.dsym, T.dfast, CL_FAST, KIND_CODES, T.offs, w)) return CL_SET;
    const uint32_t total = nlen + ndist;
    uint32_t i = 0, prev = 0;
    while (i < total) {
        br.refill();
        const int sym = decode(br, T.dfast, CL_FAST, T.dcnt, T.dsym);  // the code is complete: always a symbol
        if (br.overrun()) return OVERRUN;
        uint32_t val, rep;
        if (sym < 16) {
            val = (uint32_t)sym;
            rep = 1;
        } else if (sym == 16) {
            if (i == 0) return REPEAT;
            val = prev;
            rep = 3 + br.get(2);
        } else if (sym == 17) {
            val = 0;
            rep = 3 + br.get(3);
        } else {
            val = 0;
            rep = 11 + br.get(7);
        }
        if (br.overrun()) return OVERRUN;
        if (rep > total - i) return REPEAT;
        // the lens bytes being written here are read only after the wsync below (the code-length tables live elsewhere)
        for (uint32_t k = w.lane; k < rep; k += w.n) T.lens[i + k] = (uint8_t)val;
        i += rep;
        prev = val;
    }
    wsync();
    if (T.lens[256] == 0) return NO_EOB;
    if (build(T.lens, (int)nlen, T.lcnt, T.lsym, T.lfast, LIT_FAST, KIND_LENS, T.offs, w)) return LIT_SET;
    if (build(T.lens + nlen, (int)ndist, T.dcnt, T.dsym, T.dfast, DIST_FAST, KIND_DISTS, T.offs, w)) return DIST_SET;
    return OK;
}

// Length symbol 257 + s (s < 29) and distance code d (d < 30): base and extra bits of RFC 1951 3.2.5, computed.
HGT_HD uint32_t len_extra(uint32_t s) { return s < 8 || s == 28 ? 0 : (s >> 2) - 1; }
HGT_HD uint32_t len_base(uint32_t s) { return s < 8 ? 3 + s : s == 28 ? 258 : ((4 + (s & 3)) << len_extra(s)) + 3; }
HGT_HD uint32_t dist_extra(uint32_t d) { return d < 4 ? 0 : (d >> 1) - 1; }
HGT_HD uint32_t dist_base(uint32_t d) { return d < 4 ? d + 1 : ((2 + (d & 1)) << dist_extra(d)) + 1; }

HGT_HD uint32_t codes(Bits &br, Tables &T, uint8_t *out, uint32_t &o, uint32_t isize, Warp w) {
    for (;;) {
        br.refill();
        int sym = decode(br, T.lfast, LIT_FAST, T.lcnt, T.lsym);
        if (br.overrun()) return OVERRUN;
        if (sym < 0) return LIT_CODE;
        if (sym < 256) {
            if (o >= isize) return ISIZE_OVER;
            if (w.lane == 0) out[o] = (uint8_t)sym;
            o++;
            continue;
        }
        if (sym == 256) return OK;
        sym -= 257;
        if (sym >= 29) return LIT_CODE;
        const uint32_t len = len_base(sym) + br.get(len_extra(sym));
        br.refill();
        const int ds = decode(br, T.dfast, DIST_FAST, T.dcnt, T.dsym);
        if (br.overrun()) return OVERRUN;
        if (ds < 0 || ds >= 30) return DIST_CODE;
        const uint32_t dist = dist_base(ds) + br.get(dist_extra(ds));
        if (br.overrun()) return OVERRUN;
        if (dist > o) return FAR;
        if (len > isize - o) return ISIZE_OVER;
        wsync();  // literals and earlier copies are visible to every lane
        const uint8_t *src = out + o - dist;
        for (uint32_t j = w.lane; j < len; j += w.n) out[o + j] = src[dist >= len ? j : j % dist];
        o += len;
    }
}

// Inflates one block's DEFLATE data in[0, n_in) into out[0, isize).  Returns a Status; *n_out = bytes written.  The
// caller checks the CRC32 of a block that returns OK (crc_slice / crc_combine).
HGT_HD uint32_t inflate(const uint8_t *in, uint32_t n_in, uint8_t *out, uint32_t isize, Tables &T, Warp w, uint32_t *n_out) {
    Bits br;
    br.init(in, n_in);
    uint32_t o = 0, st = OK, last = 0;
    while (!last) {
        last = br.get(1);
        const uint32_t type = br.get(2);
        if (br.overrun()) {
            st = OVERRUN;
            break;
        }
        if (type == 0) {
            br.align();
            const uint32_t len = br.get(16), nlen = br.get(16);
            if (br.overrun()) {
                st = OVERRUN;
                break;
            }
            if (len != (~nlen & 0xffffu)) {
                st = STORED_LEN;
                break;
            }
            const uint32_t at = (uint32_t)(br.used >> 3);
            if (len > n_in - at) {
                st = OVERRUN;
                break;
            }
            if (len > isize - o) {
                st = ISIZE_OVER;
                break;
            }
            for (uint32_t j = w.lane; j < len; j += w.n) out[o + j] = in[at + j];
            o += len;
            br.buf = 0;
            br.cnt = 0;
            br.next = at + len;
            br.used = 8ull * (at + len);
            continue;
        }
        if (type == 3) {
            st = BTYPE;
            break;
        }
        st = type == 1 ? fixed_tables(T, w) : dynamic_tables(br, T, w);
        if (st == OK) st = codes(br, T, out, o, isize, w);
        if (st != OK) break;
    }
    if (st == OK) {
        if (br.overrun())
            st = OVERRUN;
        else if ((br.used + 7) / 8 < n_in)
            st = TRAILING;
        else if (o != isize)
            st = ISIZE_UNDER;
    }
    wsync();
    *n_out = o;
    return st;
}

// ---- CRC32 (zlib's: reflected 0xEDB88320, pre- and post-inverted) -----------------------------------------------------
HGT_HD uint32_t crc_entry(uint32_t i) {
    uint32_t c = i;
    for (int k = 0; k < 8; k++) c = c & 1 ? (c >> 1) ^ CRC_POLY : c >> 1;
    return c;
}
HGT_HD uint32_t crc_update(const uint32_t *tab, uint32_t crc, const uint8_t *p, uint32_t n) {
    crc = ~crc;
    for (uint32_t i = 0; i < n; i++) crc = tab[(crc ^ p[i]) & 255] ^ (crc >> 8);
    return ~crc;
}
// a * b modulo P in the reflected representation (zlib's multmodp, with a fixed 32-step loop)
HGT_HD uint32_t multmodp(uint32_t a, uint32_t b) {
    uint32_t p = 0;
    for (int k = 31; k >= 0; k--) {
        if ((a >> k) & 1) p ^= b;
        b = b & 1 ? (b >> 1) ^ CRC_POLY : b >> 1;
    }
    return p;
}
// x^(8n) modulo P: the operator that shifts a CRC over n zero bytes (zlib's x2nmodp(n, 3))
HGT_HD uint32_t x8nmodp(uint32_t n) {
    uint32_t p = 1u << 31, sq = 1u << 23;  // x^0, x^8
    while (n) {
        if (n & 1) p = multmodp(sq, p);
        sq = multmodp(sq, sq);
        n >>= 1;
    }
    return p;
}
// crc32(A || B) from crc32(A), crc32(B) and x8nmodp(|B|) (zlib's crc32_combine)
HGT_HD uint32_t crc_combine(uint32_t crc_a, uint32_t crc_b, uint32_t shift_b) { return multmodp(shift_b, crc_a) ^ crc_b; }
// slice k of CRC_SLICES over isize bytes: [*b, *e)
HGT_HD void crc_slice(uint32_t isize, uint32_t k, uint32_t *b, uint32_t *e) {
    const uint32_t sl = (isize + CRC_SLICES - 1) / CRC_SLICES;
    *b = k * sl < isize ? k * sl : isize;
    *e = (k + 1) * sl < isize ? (k + 1) * sl : isize;
}

}  // namespace hgtz

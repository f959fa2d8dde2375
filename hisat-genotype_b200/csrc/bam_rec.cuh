// The rules of a decompressed BAM stream as __host__ __device__ functions, shared by the host split (bam_split.cpp) and
// the device split (bam_dsplit.cu): the header walk, the complete check of one record, and the pieces of the record
// index (the block_size chain walk of one chunk, and the cheap plausibility test that guesses a chunk's first record).
#pragma once
#include <stdint.h>

#include <string>
#include <vector>

#include "bam_dev.cuh"

namespace hgtb {

// ---- header: magic, l_text, text, n_ref, (l_name, name, l_ref) * n_ref ---------------------------------------------------
enum { HDR_OK = 0, HDR_MAGIC, HDR_TRUNC, HDR_NEG_NREF, HDR_REFLIST };

// Walks the header of the n-byte stream b.  *end = first record byte (HDR_OK), *n_hdr = reference count, *touched = one past
// the last byte read: a copy of the first *touched bytes is all a second walk needs to reach the same result.
HGT_HD int bam_header_walk(const unsigned char *b, uint64_t n, uint64_t *end, int32_t *n_hdr, uint64_t *touched) {
    *touched = 0;
    *n_hdr = 0;
    if (n < 12) return HDR_MAGIC;
    *touched = 4;
    if (!(b[0] == 'B' && b[1] == 'A' && b[2] == 'M' && b[3] == 1)) return HDR_MAGIC;
    *touched = 8;
    const int32_t l_text = ld_i32(b + 4);
    if (l_text < 0 || 8ull + (uint64_t)l_text + 4 > n) return HDR_TRUNC;
    uint64_t o = 8 + (uint64_t)l_text;
    const int32_t nh = ld_i32(b + o);
    o += 4;
    *touched = o;
    if (nh < 0) return HDR_NEG_NREF;
    *n_hdr = nh;
    for (int32_t k = 0; k < nh; k++) {
        const int32_t l_name = o + 4 <= n ? ld_i32(b + o) : -1;
        if (o + 4 <= n) *touched = o + 4;
        if (l_name < 1 || o + 4 + (uint64_t)l_name + 4 > n) return HDR_REFLIST;
        *touched = o + 4 + (uint64_t)l_name;
        if (b[o + 4 + (uint64_t)l_name - 1] != 0) return HDR_REFLIST;
        o += 4 + (uint64_t)l_name + 4;
    }
    *end = o;
    return HDR_OK;
}

// ---- one record ------------------------------------------------------------------------------------------------------------
enum {
    RULE_OK = 0, RULE_SHORT, RULE_NAME, RULE_LSEQ, RULE_SIZE, RULE_REF, RULE_CIGAR, RULE_AUX_END, RULE_CG, RULE_FLOAT,
    RULE_TAG_END, RULE_B_FLOAT, RULE_B_SUBTYPE, RULE_TYPE
};
// rules that give HGT_ERR_UNSUPPORTED (the others give HGT_ERR_PARSE)
HGT_HD bool rule_unsupported(int rule) { return rule == RULE_CG || rule == RULE_FLOAT || rule == RULE_B_FLOAT; }

// Complete check of the record at p (size = block_size + 4 bytes, all inside the stream).  Returns RULE_OK or the first rule
// the record breaks; tag[0..1] = the aux tag the rule names.
HGT_HD int bam_check_record(const unsigned char *p, uint32_t size, int32_t n_hdr, unsigned char tag[2]) {
    if (size < REC_FIXED) return RULE_SHORT;
    const uint32_t l_name = p[12], n_cigar = ld_u16(p + 16);
    const int32_t l_seq = ld_i32(p + 20), ref = ld_i32(p + 4), next_ref = ld_i32(p + 24);
    if (l_name < 1 || REC_FIXED + l_name > size || p[REC_FIXED + l_name - 1] != 0) return RULE_NAME;
    if (l_seq < 0) return RULE_LSEQ;
    const uint64_t aux = (uint64_t)REC_FIXED + l_name + 4ull * n_cigar + ((uint64_t)l_seq + 1) / 2 + (uint64_t)l_seq;
    if (aux > size) return RULE_SIZE;
    if (ref < -1 || ref >= n_hdr || next_ref < -1 || next_ref >= n_hdr) return RULE_REF;
    for (uint32_t k = 0; k < n_cigar; k++)
        if ((ld_u32(p + REC_FIXED + l_name + 4 * k) & 15) > 8) return RULE_CIGAR;
    uint64_t o = aux;
    while (o < size) {
        if (o + 3 > size) return RULE_AUX_END;
        const unsigned char *t = p + o;
        tag[0] = t[0];
        tag[1] = t[1];
        if (t[0] == 'C' && t[1] == 'G') return RULE_CG;
        const unsigned char ty = t[2];
        uint64_t n = 0;
        if (ty == 'f' || ty == 'd') {
            return RULE_FLOAT;
        } else if (ty == 'Z' || ty == 'H') {
            uint64_t e = o + 3;
            while (e < size && p[e]) e++;
            if (e >= size) return RULE_TAG_END;
            n = e - o + 1;
        } else if (ty == 'B') {
            if (o + 8 > size) return RULE_TAG_END;
            if (t[3] == 'f') return RULE_B_FLOAT;
            const uint32_t w = t[3] == 'A' ? 0 : aux_int_size(t[3]);
            if (!w) return RULE_B_SUBTYPE;
            n = 8 + (uint64_t)ld_u32(t + 4) * w;
        } else {
            const uint32_t w = aux_int_size(ty);
            if (!w) return RULE_TYPE;
            n = 3 + w;
        }
        if (o + n > size) return RULE_TAG_END;
        o += n;
    }
    return RULE_OK;
}

// ---- record index: the block_size chain --------------------------------------------------------------------------------
// The chain rule of the host split: at o (< n) a record starts when 4 bytes remain, block_size >= 32 and the record fits.
// The stream past the header is cut into chunks [c0, c1); a chunk's walk starts at s (its first record start, or >= c1
// when a record of an earlier chunk covers it) and leaves at the first chain offset >= c1 (*e), after *cnt records; *brk
// when the chain breaks at *e < c1 instead.
HGT_HD void bam_chunk_walk(const unsigned char *d, uint64_t n, uint64_t s, uint64_t c1, uint64_t *e, uint32_t *cnt,
                           bool *brk) {
    uint64_t o = s;
    uint32_t k = 0;
    bool b = false;
    while (o < c1) {
        if (n - o < 4) {
            b = true;
            break;
        }
        const int32_t bs = ld_i32(d + o);
        if (bs < 32 || (uint64_t)bs > n - o - 4) {
            b = true;
            break;
        }
        k++;
        o += 4 + (uint64_t)bs;
    }
    *e = o;
    *cnt = k;
    *brk = b;
}

// The O(1) part of bam_check_record at o, as a guess that a record starts there: block_size by the chain rule, a read name
// with its NUL inside the record, l_seq >= 0, the fixed + name + CIGAR + SEQ + QUAL bytes inside the record, refIDs in
// range.  A guess only decides where a chunk's walk starts; the fix-up passes replace every wrong one.
HGT_HD bool bam_plausible(const unsigned char *d, uint64_t n, uint64_t o, int32_t n_hdr) {
    if (n - o < REC_FIXED) return false;
    const unsigned char *p = d + o;
    const int32_t bs = ld_i32(p);
    if (bs < 32 || (uint64_t)bs > n - o - 4) return false;
    const uint32_t size = (uint32_t)bs + 4, l_name = p[12];
    if (l_name < 1 || REC_FIXED + l_name > size || p[REC_FIXED + l_name - 1] != 0) return false;
    const int32_t l_seq = ld_i32(p + 20), ref = ld_i32(p + 4), next_ref = ld_i32(p + 24);
    if (l_seq < 0) return false;
    if ((uint64_t)REC_FIXED + l_name + 4ull * ld_u16(p + 16) + ((uint64_t)l_seq + 1) / 2 + (uint64_t)l_seq > size) return false;
    return ref >= -1 && ref < n_hdr && next_ref >= -1 && next_ref < n_hdr;
}

// first plausible offset in [c0, c1), or c1
HGT_HD uint64_t bam_chunk_guess(const unsigned char *d, uint64_t n, uint64_t c0, uint64_t c1, int32_t n_hdr) {
    for (uint64_t o = c0; o < c1; o++)
        if (bam_plausible(d, n, o, n_hdr)) return o;
    return c1;
}

// ---- host: the messages of the rules, the header's reference names ------------------------------------------------------
inline const char *bam_header_why(int code) {
    switch (code) {
        case HDR_MAGIC: return "not a BAM stream (bad magic)";
        case HDR_TRUNC: return "truncated BAM header";
        case HDR_NEG_NREF: return "negative reference count in the BAM header";
        default: return "truncated or malformed reference list in the BAM header";
    }
}

// what is wrong with a record, naming the tag where the rule has one (the tag's two bytes as they are)
inline std::string bam_rule_why(int rule, const unsigned char tag[2]) {
    const std::string t((const char *)tag, 2);
    switch (rule) {
        case RULE_SHORT: return "block_size shorter than the fixed fields";
        case RULE_NAME: return "read name is not NUL-terminated inside the record";
        case RULE_LSEQ: return "negative l_seq";
        case RULE_SIZE: return "block_size inconsistent with l_read_name, n_cigar_op and l_seq";
        case RULE_REF: return "refID or next_refID outside the reference list";
        case RULE_CIGAR: return "unknown CIGAR operation";
        case RULE_AUX_END: return "aux tag runs past the record end";
        case RULE_CG: return "tag CG (long CIGAR placeholder) is not supported";
        case RULE_FLOAT: return "tag " + t + " of float type is not supported";
        case RULE_TAG_END: return "aux tag " + t + " runs past the record end";
        case RULE_B_FLOAT: return "tag " + t + " (B array of floats) is not supported";
        case RULE_B_SUBTYPE: return "aux tag " + t + " has an unknown B subtype";
        default: return "aux tag " + t + " has an unknown type";
    }
}

// "read '<name>': <why>" for the record at p (size bytes) that breaks `rule`
inline std::string bam_record_message(const unsigned char *p, uint32_t size, int rule, const unsigned char tag[2]) {
    uint32_t ln = 0;
    if (p[12] && REC_FIXED + p[12] <= size)
        while (ln < p[12] && p[REC_FIXED + ln]) ln++;
    return "read '" + std::string((const char *)p + REC_FIXED, ln) + "': " + bam_rule_why(rule, tag);
}

// Header walk plus the reference names (refID order).  b must hold the first `touched` bytes bam_header_walk reports for
// the n-byte stream.
inline int bam_parse_header(const unsigned char *b, uint64_t n, uint64_t *end, std::vector<std::string> *names) {
    int32_t n_hdr = 0;
    uint64_t touched = 0;
    const int rc = bam_header_walk(b, n, end, &n_hdr, &touched);
    if (rc != HDR_OK) return rc;
    names->clear();
    uint64_t o = 8 + (uint64_t)ld_i32(b + 4) + 4;
    for (int32_t k = 0; k < n_hdr; k++) {
        const int32_t l_name = ld_i32(b + o);
        names->emplace_back((const char *)b + o + 4, (size_t)l_name - 1);
        o += 4 + (uint64_t)l_name + 4;
    }
    return HDR_OK;
}

}  // namespace hgtb

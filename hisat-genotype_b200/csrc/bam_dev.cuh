// BAM records -> SAM text lines, the rules of htslib's sam_format1 (what `samtools view` prints), as __host__ __device__
// functions: the device render of a batch (typing.cu: bam_text_len_kernel, bam_render_kernel) and the host render of the
// BAM split (bam_split.cpp: hgt_bam_split_write_text) call the same code, so the host render pins the device's output.
//
// Packed unit (hgt_bam_split_write_records, hgt_batch_add_unit_bam), little-endian, offsets from the blob's first byte:
//   BamUnitHeader                  magic "HGB1", flags (HGT_SPLIT_DROP_QUAL: records carry no QUAL bytes), n_records,
//                                  n_names, names_bytes
//   uint32 name_off[n_names + 1]   into the name bytes that follow (names without terminator; name 0 = the backbone)
//   names, zero padding to 8 bytes
//   uint64 rec_off[n_records + 1]  record i = [rec_off[i], rec_off[i+1]), 4-byte aligned, >= 36 bytes each
//   records                        BAM records (block_size first) in output order; refID / next_refID index the names
//
// The host validates every record of a BAM split completely (bam_split.cpp).  hgt_batch_add_unit_bam accepts any blob whose
// header, name table and offset table pass bam_unit_check(); the decoder below clamps every field to the record's extent,
// so whatever a record holds, the device reads only inside [rec_off[i], rec_off[i+1]) and the name table.
#pragma once
#include <stdint.h>
#include <string.h>

#ifndef HGT_HD
#define HGT_HD __host__ __device__ __forceinline__
#endif

namespace hgtb {

constexpr uint32_t UNIT_MAGIC = 0x31424748u;  // "HGB1"
constexpr uint32_t UNIT_DROP_QUAL = 1;
constexpr uint32_t REC_FIXED = 36;            // block_size .. tlen

struct BamUnitHeader {
    uint32_t magic, flags;
    int64_t n_records;
    uint32_t n_names, names_bytes;
};
static_assert(sizeof(BamUnitHeader) == 24, "packed unit header");

// byte offsets inside a blob (n_names, names_bytes from the header)
HGT_HD uint64_t unit_name_off_at() { return sizeof(BamUnitHeader); }
HGT_HD uint64_t unit_names_at(uint32_t n_names) { return sizeof(BamUnitHeader) + 4ull * (n_names + 1ull); }
HGT_HD uint64_t unit_rec_off_at(uint32_t n_names, uint32_t names_bytes) {
    return (unit_names_at(n_names) + names_bytes + 7) & ~7ull;
}

HGT_HD int32_t ld_i32(const unsigned char *p) {
    return (int32_t)((uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24);
}
HGT_HD uint32_t ld_u32(const unsigned char *p) { return (uint32_t)ld_i32(p); }
HGT_HD uint16_t ld_u16(const unsigned char *p) { return (uint16_t)(p[0] | p[1] << 8); }

// the name table of one unit
struct BamNames {
    const uint32_t *off;
    const unsigned char *bytes;
    uint32_t n;
};

// one record, every extent clamped to the record's bytes
struct BamRec {
    const unsigned char *p;
    int32_t ref, pos, next_ref, next_pos, tlen;
    uint32_t flag, mapq;
    uint32_t l_name, n_cigar, l_seq;
    uint32_t o_cigar, o_seq, o_qual, o_aux, end;
    bool has_qual;  // QUAL bytes are present and not 0xff-marked as absent
};

// p: 4-byte aligned, extent >= REC_FIXED (bam_unit_check guarantees both)
HGT_HD void bam_decode(const unsigned char *p, uint64_t extent, bool qual_dropped, BamRec *r) {
    r->p = p;
    const int64_t bs = (int64_t)ld_i32(p) + 4;
    const uint32_t end = (uint32_t)(bs < (int64_t)REC_FIXED ? REC_FIXED : (uint64_t)bs > extent ? extent : (uint64_t)bs);
    r->end = end;
    r->ref = ld_i32(p + 4);
    r->pos = ld_i32(p + 8);
    r->mapq = p[13];
    r->flag = ld_u16(p + 18);
    r->next_ref = ld_i32(p + 24);
    r->next_pos = ld_i32(p + 28);
    r->tlen = ld_i32(p + 32);
    uint32_t o = REC_FIXED;
    r->l_name = p[12] < end - o ? p[12] : end - o;
    o += r->l_name;
    r->o_cigar = o;
    const uint32_t nc = ld_u16(p + 16);
    r->n_cigar = nc < (end - o) / 4 ? nc : (end - o) / 4;
    o += 4 * r->n_cigar;
    const int32_t ls = ld_i32(p + 20);
    uint64_t l_seq = ls > 0 ? (uint64_t)ls : 0;
    if ((l_seq + 1) / 2 > end - o) l_seq = 2ull * (end - o);
    r->l_seq = (uint32_t)l_seq;
    r->o_seq = o;
    o += (r->l_seq + 1) / 2;
    r->o_qual = o;
    r->has_qual = false;
    if (!qual_dropped) {
        if (r->l_seq <= end - o) {
            r->has_qual = r->l_seq > 0 && p[o] != 0xff;
            o += r->l_seq;
        } else {
            o = end;
        }
    }
    r->o_aux = o;
}

struct CountSink {
    int64_t n = 0;
    HGT_HD void put(char) { n++; }
    HGT_HD void put(const unsigned char *, uint32_t k) { n += k; }
};
struct WriteSink {
    char *o;
    HGT_HD void put(char c) { *o++ = c; }
    HGT_HD void put(const unsigned char *s, uint32_t k) {
        for (uint32_t i = 0; i < k; i++) o[i] = (char)s[i];
        o += k;
    }
};

template <class S>
HGT_HD void put_u64(S &s, uint64_t v) {
    char d[20];
    int k = 0;
    do {
        d[k++] = (char)('0' + v % 10);
        v /= 10;
    } while (v);
    while (k) s.put(d[--k]);
}
template <class S>
HGT_HD void put_i64(S &s, int64_t v) {
    if (v < 0) {
        s.put('-');
        put_u64(s, (uint64_t)0 - (uint64_t)v);
    } else {
        put_u64(s, (uint64_t)v);
    }
}
template <class S>
HGT_HD void put_name(S &s, const BamNames &nm, int32_t id) {
    if (id < 0 || (uint32_t)id >= nm.n) {
        s.put('*');
        return;
    }
    s.put(nm.bytes + nm.off[id], nm.off[id + 1] - nm.off[id]);
}

// QNAME without its NUL
HGT_HD uint32_t qname_len(const BamRec &r) {
    if (r.l_name == 0) return 0;
    return r.p[REC_FIXED + r.l_name - 1] == 0 ? r.l_name - 1 : r.l_name;
}

// "\tFLAG\tRNAME\tPOS\tMAPQ\tCIGAR\tRNEXT\tPNEXT\tTLEN\t": the columns between QNAME and SEQ
template <class S>
HGT_HD void bam_head(const BamRec &r, const BamNames &nm, S &s) {
    s.put('\t');
    put_u64(s, r.flag);
    s.put('\t');
    put_name(s, nm, r.ref < 0 ? -1 : r.ref);
    s.put('\t');
    put_i64(s, (int64_t)r.pos + 1);
    s.put('\t');
    put_u64(s, r.mapq);
    s.put('\t');
    if (r.n_cigar == 0) s.put('*');
    for (uint32_t k = 0; k < r.n_cigar; k++) {
        const uint32_t c = ld_u32(r.p + r.o_cigar + 4 * k);
        put_u64(s, c >> 4);
        s.put("MIDNSHP=XB??????"[c & 15]);
    }
    s.put('\t');
    if (r.next_ref < 0) s.put('*');
    else if (r.next_ref == r.ref) s.put('=');
    else put_name(s, nm, r.next_ref);
    s.put('\t');
    put_i64(s, (int64_t)r.next_pos + 1);
    s.put('\t');
    put_i64(s, r.tlen);
    s.put('\t');
}

HGT_HD char seq_base(const BamRec &r, uint32_t i) {
    const unsigned char b = r.p[r.o_seq + (i >> 1)];
    return "=ACMGRSVTWYHKDBN"[(i & 1) ? (b & 15) : (b >> 4)];
}

HGT_HD uint32_t aux_int_size(unsigned char t) {
    switch (t) {
        case 'c': case 'C': case 'A': return 1;
        case 's': case 'S': return 2;
        case 'i': case 'I': return 4;
        default: return 0;
    }
}
template <class S>
HGT_HD void put_aux_int(S &s, unsigned char t, const unsigned char *v) {
    switch (t) {
        case 'c': put_i64(s, (int8_t)v[0]); break;
        case 'C': put_u64(s, v[0]); break;
        case 's': put_i64(s, (int16_t)ld_u16(v)); break;
        case 'S': put_u64(s, ld_u16(v)); break;
        case 'i': put_i64(s, ld_i32(v)); break;
        default: put_u64(s, ld_u32(v)); break;  // 'I'
    }
}

// "\tXX:T:value" for every tag; stops at the first tag that does not fit the record or has a type outside A, c C s S i I,
// Z, H and B of an integer subtype (the host split refuses such records, so it never stops early on its own output)
template <class S>
HGT_HD void bam_tags(const BamRec &r, S &s) {
    uint32_t o = r.o_aux;
    const uint32_t end = r.end;
    while (o + 3 <= end) {
        const unsigned char *t = r.p + o;
        const unsigned char ty = t[2];
        if (ty == 'Z' || ty == 'H') {
            uint32_t e = o + 3;
            while (e < end && r.p[e]) e++;
            if (e >= end) return;
            s.put('\t'); s.put((char)t[0]); s.put((char)t[1]); s.put(':'); s.put((char)ty); s.put(':');
            s.put(t + 3, e - o - 3);
            o = e + 1;
        } else if (ty == 'B') {
            if (o + 8 > end) return;
            const unsigned char sub = t[3];
            const uint32_t w = sub == 'A' ? 0 : aux_int_size(sub);
            const uint32_t n = ld_u32(t + 4);
            if (w == 0 || (uint64_t)n * w > end - o - 8) return;
            s.put('\t'); s.put((char)t[0]); s.put((char)t[1]); s.put(':'); s.put('B'); s.put(':'); s.put((char)sub);
            for (uint32_t k = 0; k < n; k++) {
                s.put(',');
                put_aux_int(s, sub, t + 8 + k * w);
            }
            o += 8 + n * w;
        } else {
            const uint32_t w = aux_int_size(ty);
            if (w == 0 || o + 3 + w > end) return;
            s.put('\t'); s.put((char)t[0]); s.put((char)t[1]); s.put(':');
            if (ty == 'A') {
                s.put('A'); s.put(':'); s.put((char)t[3]);
            } else {
                s.put('i'); s.put(':');
                put_aux_int(s, ty, t + 3);
            }
            o += 3 + w;
        }
    }
}

// one whole line, serially (host render, text length)
template <class S>
HGT_HD void bam_line(const BamRec &r, const BamNames &nm, S &s) {
    s.put(r.p + REC_FIXED, qname_len(r));
    bam_head(r, nm, s);
    if (r.l_seq == 0) s.put('*');
    for (uint32_t i = 0; i < r.l_seq; i++) s.put(seq_base(r, i));
    s.put('\t');
    if (!r.has_qual) s.put('*');
    else
        for (uint32_t i = 0; i < r.l_seq; i++) s.put((char)(r.p[r.o_qual + i] + 33));
    bam_tags(r, s);
    s.put('\n');
}

HGT_HD int64_t bam_line_len(const BamRec &r, const BamNames &nm) {
    CountSink c;
    bam_line(r, nm, c);
    return c.n;
}

// Host-side check of a blob before it may reach the device: header, name table and offset table stay inside the blob,
// offsets are monotone, records 4-byte aligned and at least the fixed part long.  Returns nullptr or what is wrong.
inline const char *bam_unit_check(const void *blob, uint64_t n_bytes, BamUnitHeader *hdr) {
    const unsigned char *b = static_cast<const unsigned char *>(blob);
    if (!blob || n_bytes < sizeof(BamUnitHeader) || ((uintptr_t)b & 7)) return "blob missing, shorter than its header or not 8-byte aligned";
    memcpy(hdr, b, sizeof(BamUnitHeader));
    if (hdr->magic != UNIT_MAGIC) return "bad magic";
    if (hdr->flags & ~UNIT_DROP_QUAL) return "unknown flags";
    if (hdr->n_records < 0 || hdr->n_names > (1u << 24) || hdr->names_bytes > n_bytes) return "bad header counts";
    const uint64_t o_recs = unit_rec_off_at(hdr->n_names, hdr->names_bytes);
    if (o_recs > n_bytes || (uint64_t)hdr->n_records + 1 > (n_bytes - o_recs) / 8) return "tables run past the blob";
    const uint32_t *no = reinterpret_cast<const uint32_t *>(b + unit_name_off_at());
    if (no[0] != 0) return "name table does not start at 0";
    for (uint32_t k = 0; k < hdr->n_names; k++)
        if (no[k + 1] < no[k]) return "name offsets not monotone";
    if (no[hdr->n_names] > hdr->names_bytes) return "names run past their table";
    const uint64_t *ro = reinterpret_cast<const uint64_t *>(b + o_recs);
    const uint64_t data0 = o_recs + 8 * ((uint64_t)hdr->n_records + 1);
    if (ro[0] < data0) return "records overlap the offset table";
    for (int64_t i = 0; i < hdr->n_records; i++) {
        if (ro[i] & 3) return "record not 4-byte aligned";
        if (ro[i + 1] < ro[i] + REC_FIXED) return "record offsets not monotone or record shorter than 36 bytes";
    }
    if (ro[hdr->n_records] > n_bytes) return "records run past the blob";
    return nullptr;
}

}  // namespace hgtb

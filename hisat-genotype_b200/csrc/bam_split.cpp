// Native intake of a BAM file (host C++, threads): the BAM counterpart of sam_split.cpp.  The caller passes the
// DECOMPRESSED stream (sam_intake.read_bgzf inflates BGZF with Python's zlib, so the library gains no zlib dependency).
// Records are validated completely, bucketed by refID into the given backbones (the SAM split's RNAME rule, so
// split_bam(bam) == split_sam(samtools view bam)) and ordered by the shared order rule (split_order.hpp).  A bucket leaves
// as a packed unit (layout in bam_dev.cuh) that the GPU renders into alignment text (hgt_batch_add_unit_bam), or as the
// same text rendered here by the same formatting functions.
#include <string.h>

#include <string>
#include <unordered_map>
#include <vector>

#include "bam_dev.cuh"
#include "common.cuh"
#include "split_order.hpp"

struct hgt_bam_split {
    const unsigned char *bam = nullptr;
    bool drop_qual = false;
    std::vector<std::string> ref_names;  // the backbones asked for
    std::vector<std::string> hdr_names;  // the file's reference list (refID order)
    struct Rec {
        uint64_t off;  // of block_size in the stream
        uint32_t name_len;
        int32_t pos;
        uint32_t size;  // block_size + 4
        int32_t next_ref;
        uint32_t qual_bytes;  // l_seq (the QUAL bytes a drop_qual unit leaves out)
    };
    std::vector<std::vector<Rec>> bucket;
    std::vector<std::vector<int32_t>> names;  // per bucket: header refIDs of its name table, its own first
    std::vector<size_t> blob_bytes;
};

namespace {

using hgt_split::run_threads;

struct RecError {
    uint64_t index = UINT64_MAX;  // first failing record (input order): the same message for any thread count
    int code = HGT_OK;
    std::string msg;
};

uint32_t a4(uint64_t x) { return (uint32_t)((x + 3) & ~3ull); }

// Complete check of the record at p (size = block_size + 4 bytes, inside the stream).  Returns HGT_OK, HGT_ERR_PARSE or
// HGT_ERR_UNSUPPORTED with *why set.
int check_record(const unsigned char *p, uint32_t size, int32_t n_hdr, std::string *why) {
    using namespace hgtb;
    if (size < REC_FIXED) {
        *why = "block_size shorter than the fixed fields";
        return HGT_ERR_PARSE;
    }
    const uint32_t l_name = p[12], n_cigar = ld_u16(p + 16);
    const int32_t l_seq = ld_i32(p + 20), ref = ld_i32(p + 4), next_ref = ld_i32(p + 24);
    if (l_name < 1 || REC_FIXED + l_name > size || p[REC_FIXED + l_name - 1] != 0) {
        *why = "read name is not NUL-terminated inside the record";
        return HGT_ERR_PARSE;
    }
    if (l_seq < 0) {
        *why = "negative l_seq";
        return HGT_ERR_PARSE;
    }
    const uint64_t aux = (uint64_t)REC_FIXED + l_name + 4ull * n_cigar + ((uint64_t)l_seq + 1) / 2 + (uint64_t)l_seq;
    if (aux > size) {
        *why = "block_size inconsistent with l_read_name, n_cigar_op and l_seq";
        return HGT_ERR_PARSE;
    }
    if (ref < -1 || ref >= n_hdr || next_ref < -1 || next_ref >= n_hdr) {
        *why = "refID or next_refID outside the reference list";
        return HGT_ERR_PARSE;
    }
    for (uint32_t k = 0; k < n_cigar; k++)
        if ((ld_u32(p + REC_FIXED + l_name + 4 * k) & 15) > 8) {
            *why = "unknown CIGAR operation";
            return HGT_ERR_PARSE;
        }
    uint64_t o = aux;
    while (o < size) {
        if (o + 3 > size) {
            *why = "aux tag runs past the record end";
            return HGT_ERR_PARSE;
        }
        const unsigned char *t = p + o;
        const std::string tag((const char *)t, 2);
        if (tag == "CG") {
            *why = "tag CG (long CIGAR placeholder) is not supported";
            return HGT_ERR_UNSUPPORTED;
        }
        const unsigned char ty = t[2];
        uint64_t n = 0;
        if (ty == 'f' || ty == 'd') {
            *why = "tag " + tag + " of float type is not supported";
            return HGT_ERR_UNSUPPORTED;
        } else if (ty == 'Z' || ty == 'H') {
            const void *z = memchr(t + 3, 0, size - o - 3);
            if (!z) {
                *why = "aux tag " + tag + " runs past the record end";
                return HGT_ERR_PARSE;
            }
            n = 3 + (uint64_t)((const unsigned char *)z - (t + 3)) + 1;
        } else if (ty == 'B') {
            if (o + 8 > size) {
                *why = "aux tag " + tag + " runs past the record end";
                return HGT_ERR_PARSE;
            }
            if (t[3] == 'f') {
                *why = "tag " + tag + " (B array of floats) is not supported";
                return HGT_ERR_UNSUPPORTED;
            }
            const uint32_t w = t[3] == 'A' ? 0 : aux_int_size(t[3]);
            if (!w) {
                *why = "aux tag " + tag + " has an unknown B subtype";
                return HGT_ERR_PARSE;
            }
            n = 8 + (uint64_t)ld_u32(t + 4) * w;
        } else {
            const uint32_t w = aux_int_size(ty);
            if (!w) {
                *why = "aux tag " + tag + " has an unknown type";
                return HGT_ERR_PARSE;
            }
            n = 3 + w;
        }
        if (o + n > size) {
            *why = "aux tag " + tag + " runs past the record end";
            return HGT_ERR_PARSE;
        }
        o += n;
    }
    return HGT_OK;
}

void pack(const hgt_bam_split *s, size_t r, unsigned char *dst) {
    using namespace hgtb;
    const auto &b = s->bucket[r];
    const auto &nm = s->names[r];
    BamUnitHeader h{};
    h.magic = UNIT_MAGIC;
    h.flags = s->drop_qual ? UNIT_DROP_QUAL : 0;
    h.n_records = (int64_t)b.size();
    h.n_names = (uint32_t)nm.size();
    std::unordered_map<int32_t, int32_t> local;
    uint32_t nb = 0;
    uint32_t *no = reinterpret_cast<uint32_t *>(dst + unit_name_off_at());
    no[0] = 0;
    for (size_t k = 0; k < nm.size(); k++) {
        local[nm[k]] = (int32_t)k;
        nb += (uint32_t)s->hdr_names[(size_t)nm[k]].size();
        no[k + 1] = nb;
    }
    h.names_bytes = nb;
    memcpy(dst, &h, sizeof(h));
    unsigned char *names = dst + unit_names_at(h.n_names);
    for (size_t k = 0; k < nm.size(); k++) memcpy(names + no[k], s->hdr_names[(size_t)nm[k]].data(), no[k + 1] - no[k]);
    const uint64_t o_recs = unit_rec_off_at(h.n_names, nb);
    memset(names + nb, 0, o_recs - unit_names_at(h.n_names) - nb);
    uint64_t *ro = reinterpret_cast<uint64_t *>(dst + o_recs);
    uint64_t o = o_recs + 8 * (b.size() + 1);
    for (size_t i = 0; i < b.size(); i++) {
        const hgt_bam_split::Rec &rec = b[i];
        const unsigned char *p = s->bam + rec.off;
        ro[i] = o;
        unsigned char *d = dst + o;
        uint32_t n = rec.size;
        if (s->drop_qual) {
            const uint32_t q = REC_FIXED + p[12] + 4u * ld_u16(p + 16) + (rec.qual_bytes + 1) / 2;
            memcpy(d, p, q);
            memcpy(d + q, p + q + rec.qual_bytes, rec.size - q - rec.qual_bytes);
            n -= rec.qual_bytes;
            const int32_t bs = (int32_t)(n - 4);
            memcpy(d, &bs, 4);
        } else {
            memcpy(d, p, n);
        }
        const int32_t own = 0, next = rec.next_ref < 0 ? -1 : local[rec.next_ref];
        memcpy(d + 4, &own, 4);
        memcpy(d + 24, &next, 4);
        memset(d + n, 0, a4(n) - n);
        o += a4(n);
    }
    ro[b.size()] = o;
}

// text of a packed unit (dst == nullptr: length only) through the functions the device render uses
int64_t render(const unsigned char *blob, char *dst) {
    using namespace hgtb;
    BamUnitHeader h;
    memcpy(&h, blob, sizeof(h));
    const BamNames nm{reinterpret_cast<const uint32_t *>(blob + unit_name_off_at()), blob + unit_names_at(h.n_names), h.n_names};
    const uint64_t *ro = reinterpret_cast<const uint64_t *>(blob + unit_rec_off_at(h.n_names, h.names_bytes));
    int64_t n = 0;
    for (int64_t i = 0; i < h.n_records; i++) {
        BamRec r;
        bam_decode(blob + ro[i], ro[i + 1] - ro[i], (h.flags & UNIT_DROP_QUAL) != 0, &r);
        if (dst) {
            WriteSink w{dst + n};
            bam_line(r, nm, w);
            n = w.o - dst;
        } else {
            n += bam_line_len(r, nm);
        }
    }
    return n;
}

}  // namespace

extern "C" int hgt_bam_split_create(const void *bam, size_t n_bytes, int32_t n_refs, const char *const *ref_names,
                                    int32_t n_threads, int32_t flags, hgt_bam_split **out) {
    using namespace hgtb;
    if (!out || (!bam && n_bytes) || n_refs < 1 || !ref_names || (flags & ~HGT_SPLIT_DROP_QUAL)) {
        hgt_set_error("hgt_bam_split_create: bad argument");
        return HGT_ERR_ARG;
    }
    *out = nullptr;
    n_threads = hgt_split::default_threads(n_threads);
    const unsigned char *b = static_cast<const unsigned char *>(bam);
    // header: magic, l_text, text, n_ref, (l_name, name, l_ref) * n_ref
    if (n_bytes < 12 || memcmp(b, "BAM\1", 4) != 0) {
        hgt_set_error("hgt_bam_split_create: not a BAM stream (bad magic)");
        return HGT_ERR_PARSE;
    }
    const int32_t l_text = ld_i32(b + 4);
    if (l_text < 0 || 8ull + (uint64_t)l_text + 4 > n_bytes) {
        hgt_set_error("hgt_bam_split_create: truncated BAM header");
        return HGT_ERR_PARSE;
    }
    uint64_t o = 8 + (uint64_t)l_text;
    const int32_t n_hdr = ld_i32(b + o);
    o += 4;
    if (n_hdr < 0) {
        hgt_set_error("hgt_bam_split_create: negative reference count in the BAM header");
        return HGT_ERR_PARSE;
    }
    hgt_bam_split *s = new hgt_bam_split();
    s->bam = b;
    s->drop_qual = (flags & HGT_SPLIT_DROP_QUAL) != 0;
    for (int32_t r = 0; r < n_refs; r++) s->ref_names.emplace_back(ref_names[r]);
    std::unordered_map<std::string, int> ref_index;
    for (int r = 0; r < n_refs; r++) ref_index[ref_names[r]] = r;
    std::vector<int> ref_of_hdr;
    for (int32_t k = 0; k < n_hdr; k++) {
        const int32_t l_name = o + 4 <= n_bytes ? ld_i32(b + o) : -1;
        if (l_name < 1 || o + 4 + (uint64_t)l_name + 4 > n_bytes || b[o + 4 + (uint64_t)l_name - 1] != 0) {
            delete s;
            hgt_set_error("hgt_bam_split_create: truncated or malformed reference list in the BAM header");
            return HGT_ERR_PARSE;
        }
        s->hdr_names.emplace_back((const char *)b + o + 4, (size_t)l_name - 1);
        auto it = ref_index.find(s->hdr_names.back());
        ref_of_hdr.push_back(it == ref_index.end() ? -1 : it->second);
        o += 4 + (uint64_t)l_name + 4;
    }
    // record boundaries: one sequential pass over the block_size chain
    std::vector<uint64_t> rec_at;
    while (o < n_bytes) {
        if (n_bytes - o < 4) break;
        const int32_t bs = ld_i32(b + o);
        if (bs < 32 || (uint64_t)bs > n_bytes - o - 4) break;
        rec_at.push_back(o);
        o += 4 + (uint64_t)bs;
    }
    if (o != n_bytes) {
        delete s;
        hgt_set_error("hgt_bam_split_create: truncated or malformed record at byte %llu of the BAM stream (after %zu records)",
                      (unsigned long long)o, rec_at.size());
        return HGT_ERR_PARSE;
    }
    // slices of records: validate completely and bucket
    const size_t n_rec = rec_at.size();
    const size_t n_slices = std::max<size_t>(1, std::min<size_t>((size_t)n_threads * 4, n_rec / 4096 + 1));
    std::vector<std::vector<std::vector<hgt_bam_split::Rec>>> part(n_slices, std::vector<std::vector<hgt_bam_split::Rec>>((size_t)n_refs));
    std::vector<RecError> err(n_slices);
    run_threads(n_threads, n_slices, [&](size_t k) {
        const size_t i0 = n_rec * k / n_slices, i1 = n_rec * (k + 1) / n_slices;
        for (size_t i = i0; i < i1; i++) {
            const unsigned char *p = b + rec_at[i];
            const uint32_t size = (uint32_t)ld_i32(p) + 4;
            std::string why;
            const int rc = check_record(p, size, n_hdr, &why);
            if (rc != HGT_OK) {
                err[k].index = i;
                err[k].code = rc;
                const size_t ln = p[12] && REC_FIXED + p[12] <= size ? strnlen((const char *)p + REC_FIXED, p[12]) : 0;
                err[k].msg = "read '" + std::string((const char *)p + REC_FIXED, ln) + "': " + why;
                return;
            }
            const int32_t ref = ld_i32(p + 4);
            const int bucket = ref < 0 ? -1 : ref_of_hdr[(size_t)ref];
            if (bucket < 0) continue;
            part[k][(size_t)bucket].push_back({rec_at[i], (uint32_t)p[12] - 1, ld_i32(p + 8), size, ld_i32(p + 24),
                                               (uint32_t)ld_i32(p + 20)});
        }
    });
    const RecError *first = nullptr;
    for (const RecError &e : err)
        if (e.code != HGT_OK && (!first || e.index < first->index)) first = &e;
    if (first) {
        const int code = first->code;
        hgt_set_error("hgt_bam_split_create: %s", first->msg.c_str());
        delete s;
        return code;
    }
    // per reference: input order, stable sort by (name, pos); then the unit's name table and size
    s->bucket.resize((size_t)n_refs);
    s->names.resize((size_t)n_refs);
    s->blob_bytes.assign((size_t)n_refs, 0);
    hgt_split::bucket_and_order(n_threads, part, s->bucket, [b](const hgt_bam_split::Rec &x) { return b + x.off + REC_FIXED; },
                                [s, &ref_of_hdr, n_hdr](size_t r) {
                                    std::vector<int32_t> &nm = s->names[r];
                                    for (int32_t k = 0; k < n_hdr; k++)
                                        if (ref_of_hdr[(size_t)k] == (int)r) {
                                            nm.push_back(k);
                                            break;
                                        }
                                    uint64_t rec_bytes = 0, names_bytes = nm.empty() ? 0 : s->hdr_names[(size_t)nm[0]].size();
                                    for (const auto &rec : s->bucket[r]) {
                                        rec_bytes += a4(rec.size - (s->drop_qual ? rec.qual_bytes : 0));
                                        if (rec.next_ref >= 0 && std::find(nm.begin(), nm.end(), rec.next_ref) == nm.end()) {
                                            nm.push_back(rec.next_ref);
                                            names_bytes += s->hdr_names[(size_t)rec.next_ref].size();
                                        }
                                    }
                                    s->blob_bytes[r] = unit_rec_off_at((uint32_t)nm.size(), (uint32_t)names_bytes) +
                                                       8 * (s->bucket[r].size() + 1) + rec_bytes;
                                });
    *out = s;
    return HGT_OK;
}

extern "C" int hgt_bam_split_sizes(const hgt_bam_split *s, size_t *blob_bytes, size_t *text_bytes, int64_t *records) {
    if (!s) return HGT_ERR_ARG;
    for (size_t r = 0; r < s->bucket.size(); r++) {
        if (blob_bytes) blob_bytes[r] = s->blob_bytes[r];
        if (records) records[r] = (int64_t)s->bucket[r].size();
        if (text_bytes) {
            std::vector<uint64_t> blob((s->blob_bytes[r] + 7) / 8);
            pack(s, r, reinterpret_cast<unsigned char *>(blob.data()));
            text_bytes[r] = (size_t)render(reinterpret_cast<const unsigned char *>(blob.data()), nullptr);
        }
    }
    return HGT_OK;
}

extern "C" int hgt_bam_split_write_records(const hgt_bam_split *s, int32_t ref, void *dst) {
    if (!s || ref < 0 || (size_t)ref >= s->bucket.size() || !dst || ((uintptr_t)dst & 7)) {
        hgt_set_error("hgt_bam_split_write_records: bad argument (dst must be 8-byte aligned)");
        return HGT_ERR_ARG;
    }
    pack(s, (size_t)ref, static_cast<unsigned char *>(dst));
    return HGT_OK;
}

extern "C" int hgt_bam_split_write_text(const hgt_bam_split *s, int32_t ref, char *dst) {
    if (!s || ref < 0 || (size_t)ref >= s->bucket.size()) {
        hgt_set_error("hgt_bam_split_write_text: bad argument");
        return HGT_ERR_ARG;
    }
    std::vector<uint64_t> blob((s->blob_bytes[(size_t)ref] + 7) / 8);
    pack(s, (size_t)ref, reinterpret_cast<unsigned char *>(blob.data()));
    if (!dst && render(reinterpret_cast<const unsigned char *>(blob.data()), nullptr) > 0) {
        hgt_set_error("hgt_bam_split_write_text: bad argument");
        return HGT_ERR_ARG;
    }
    if (dst) render(reinterpret_cast<const unsigned char *>(blob.data()), dst);
    return HGT_OK;
}

extern "C" void hgt_bam_split_free(hgt_bam_split *s) { delete s; }

// Native intake of an aligner's SAM stream (host C++, threads): what the reference does with external processes per locus,
//   samtools view <bam> <backbone> | sort -k1,1 -s            (hisatgenotype_typing_core.py:436-468)
// on a coordinate-sorted BAM (samtools sort, hisatgenotype_typing_common.py:1038-1054), for ALL loci of a sample in one pass
// over the text: records are bucketed by RNAME and each bucket is ordered by (read name bytewise, position, input order) -
// the order the two stable sorts of the reference produce under LC_ALL=C.  The output of a bucket is the alignment text
// hgt_batch_add_unit() takes (name-grouped); it can be written straight into page-locked memory.
#include <string.h>

#include <algorithm>
#include <atomic>
#include <string>
#include <unordered_map>
#include <vector>

#include "common.cuh"
#include "split_order.hpp"

using hgt_split::run_threads;

struct hgt_sam_split {
    const char *text = nullptr;
    struct Rec {
        uint64_t off;
        uint32_t len;       // including the newline (one is added for a last line without)
        uint32_t name_len;
        int32_t pos;
        uint32_t q_off, q_len;  // QUAL column (11th) inside the line; q_len = 0: absent or kept as it is
    };
    std::vector<std::vector<Rec>> bucket;  // per reference, ordered
    std::vector<size_t> bytes;
    bool last_needs_newline = false;
    uint64_t last_off = 0;
    bool drop_qual = false;  // write '*' for the QUAL column (the typing path never reads it: 27 % of a 2x100 bp record)
};

extern "C" int hgt_sam_split_create(const char *sam_text, size_t n_bytes, int32_t n_refs, const char *const *ref_names,
                                    int32_t n_threads, hgt_sam_split **out) {
    return hgt_sam_split_create_opts(sam_text, n_bytes, n_refs, ref_names, n_threads, 0, out);
}

extern "C" int hgt_sam_split_create_opts(const char *sam_text, size_t n_bytes, int32_t n_refs, const char *const *ref_names,
                                         int32_t n_threads, int32_t flags, hgt_sam_split **out) {
    if (!out || (!sam_text && n_bytes) || n_refs < 1 || !ref_names) {
        hgt_set_error("hgt_sam_split_create: bad argument");
        return HGT_ERR_ARG;
    }
    *out = nullptr;
    n_threads = hgt_split::default_threads(n_threads);
    std::unordered_map<std::string, int> ref_index;
    for (int r = 0; r < n_refs; r++) ref_index[ref_names[r]] = r;
    hgt_sam_split *s = new hgt_sam_split();
    s->text = sam_text;
    s->drop_qual = (flags & HGT_SPLIT_DROP_QUAL) != 0;
    const bool drop_qual = s->drop_qual;
    s->bucket.resize((size_t)n_refs);
    s->bytes.assign((size_t)n_refs, 0);
    // pass 1: slices of the text (cut at newlines) -> records per slice and reference
    const size_t n_slices = (size_t)std::max<int64_t>(1, std::min<int64_t>((int64_t)n_threads * 4, (int64_t)(n_bytes >> 16) + 1));
    std::vector<size_t> cut(n_slices + 1, n_bytes);
    cut[0] = 0;
    for (size_t k = 1; k < n_slices; k++) {
        size_t p = n_bytes / n_slices * k;
        const void *nl = p < n_bytes ? memchr(sam_text + p, '\n', n_bytes - p) : nullptr;
        cut[k] = nl ? (size_t)((const char *)nl - sam_text) + 1 : n_bytes;
    }
    for (size_t k = 1; k <= n_slices; k++) cut[k] = std::max(cut[k], cut[k - 1]);
    std::vector<std::vector<std::vector<hgt_sam_split::Rec>>> part(n_slices, std::vector<std::vector<hgt_sam_split::Rec>>((size_t)n_refs));
    std::atomic<int> bad{0};
    run_threads(n_threads, n_slices, [&](size_t k) {
        size_t p = cut[k];
        const size_t end = cut[k + 1];
        while (p < end) {
            const void *nl = memchr(sam_text + p, '\n', end - p);
            const size_t e = nl ? (size_t)((const char *)nl - sam_text) : end;  // line = [p, e)
            const char *ln = sam_text + p;
            const size_t n = e - p;
            if (n > 0 && ln[0] != '@') {
                // QNAME \t FLAG \t RNAME \t POS
                const char *t1 = (const char *)memchr(ln, '\t', n);
                const char *t2 = t1 ? (const char *)memchr(t1 + 1, '\t', (size_t)(ln + n - t1 - 1)) : nullptr;
                const char *t3 = t2 ? (const char *)memchr(t2 + 1, '\t', (size_t)(ln + n - t2 - 1)) : nullptr;
                const char *t4 = t3 ? (const char *)memchr(t3 + 1, '\t', (size_t)(ln + n - t3 - 1)) : nullptr;
                if (!t4) {
                    bad.store(1);
                } else {
                    auto it = ref_index.find(std::string(t2 + 1, (size_t)(t3 - t2 - 1)));
                    if (it != ref_index.end()) {
                        int64_t pos = 0;
                        bool ok = t4 > t3 + 1;
                        for (const char *c = t3 + 1; c < t4 && ok; c++) {
                            ok = *c >= '0' && *c <= '9';
                            pos = pos * 10 + (*c - '0');
                            if (pos > 2000000000) ok = false;
                        }
                        uint32_t q_off = 0, q_len = 0;
                        if (ok && drop_qual) {  // columns 5 .. 10 follow POS; QUAL is the 11th
                            const char *t = t4;
                            for (int col = 5; col <= 10 && t; col++) t = (const char *)memchr(t + 1, '\t', (size_t)(ln + n - t - 1));
                            if (t) {
                                const char *qe = (const char *)memchr(t + 1, '\t', (size_t)(ln + n - t - 1));
                                if (!qe) qe = ln + n;
                                q_off = (uint32_t)(t + 1 - ln);
                                q_len = (uint32_t)(qe - (t + 1));
                                if (q_len <= 1) q_len = 0;  // already '*' (or empty): nothing to save
                            }
                        }
                        if (!ok) bad.store(1);
                        else
                            part[k][(size_t)it->second].push_back({(uint64_t)p, (uint32_t)(n + 1), (uint32_t)(t1 - ln), (int32_t)pos, q_off, q_len});
                    }
                }
            }
            p = e + 1;
        }
    });
    if (bad.load()) {
        delete s;
        hgt_set_error("hgt_sam_split_create: malformed alignment record (fewer than 4 columns or bad POS)");
        return HGT_ERR_PARSE;
    }
    s->last_needs_newline = n_bytes > 0 && sam_text[n_bytes - 1] != '\n';
    // pass 2: per reference - concatenate the slices (input order), stable sort by (name, pos)
    hgt_split::bucket_and_order(n_threads, part, s->bucket, [sam_text](const hgt_sam_split::Rec &x) { return sam_text + x.off; },
                                [s](size_t r) {
                                    size_t bytes = 0;
                                    for (const auto &rec : s->bucket[r]) bytes += rec.len - (rec.q_len ? rec.q_len - 1 : 0);
                                    s->bytes[r] = bytes;
                                });
    *out = s;
    return HGT_OK;
}

extern "C" int hgt_sam_split_sizes(const hgt_sam_split *s, size_t *bytes_per_ref, int64_t *lines_per_ref) {
    if (!s) return HGT_ERR_ARG;
    for (size_t r = 0; r < s->bucket.size(); r++) {
        if (bytes_per_ref) bytes_per_ref[r] = s->bytes[r];
        if (lines_per_ref) lines_per_ref[r] = (int64_t)s->bucket[r].size();
    }
    return HGT_OK;
}

extern "C" int hgt_sam_split_write(const hgt_sam_split *s, int32_t ref, char *dst) {
    if (!s || ref < 0 || (size_t)ref >= s->bucket.size() || (!dst && s->bytes[(size_t)ref])) {
        hgt_set_error("hgt_sam_split_write: bad argument");
        return HGT_ERR_ARG;
    }
    char *o = dst;
    for (const auto &rec : s->bucket[(size_t)ref]) {
        const char *ln = s->text + rec.off;
        if (rec.q_len) {  // QUAL column replaced by '*'
            memcpy(o, ln, rec.q_off);
            o += rec.q_off;
            *o++ = '*';
            const size_t rest = rec.len - 1 - rec.q_off - rec.q_len;
            memcpy(o, ln + rec.q_off + rec.q_len, rest);
            o += rest;
            *o++ = '\n';
        } else {
            memcpy(o, ln, rec.len - 1);
            o[rec.len - 1] = '\n';
            o += rec.len;
        }
    }
    return HGT_OK;
}

extern "C" void hgt_sam_split_free(hgt_sam_split *s) { delete s; }

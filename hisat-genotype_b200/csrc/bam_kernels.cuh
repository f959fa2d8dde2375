// BAM records -> alignment text on the device (bam_dev.cuh is the formatter), over two record sources:
//   BlobSrc   packed units of a batch (hgt_batch_add_unit_bam): blobs in the blob arena, their offset tables;
//   DsplitSrc buckets of a device split (hgt_bam_dsplit_*): the inflated stream in HBM and the bucket's ordered offsets.
// typing.cu renders both kinds of unit with these kernels; bam_dsplit.cu measures its buckets with bam_text_len_kernel.
#pragma once
#include <stdint.h>

#include "bam_dev.cuh"

namespace hgtk {

constexpr int BAM_THREADS = 256;

struct BamUnitDev {  // one BAM unit of a batch: blob in the blob arena, first record (batch-wide), slice of the text arena
    int64_t blob_off, rec0, text_off, pad;
};

// One bucket of a device split as a unit: records rec[0 .. n) (offsets into data, not 4-byte aligned) with text offsets
// toff[0 .. n] relative to any base; the stream's header name table; own = the header refID whose name the bucket's
// packed unit would carry as its name 0 (RNAME and the '=' of RNEXT follow it, as for a packed unit).
struct DsplitUnitDev {
    const unsigned char *data;
    const uint64_t *rec;
    const int64_t *toff;
    const uint32_t *name_off;
    const unsigned char *name_bytes;
    uint32_t n_names;
    int32_t own;
    int64_t rec0, text_off;  // first record (batch-wide), slice of the text arena
    uint32_t hide_qual;      // HGT_SPLIT_DROP_QUAL: the QUAL bytes are in the stream and left out of the text
    uint32_t pad;
};

// unit of batch-wide record g: the last unit whose first record is <= g (units without records are skipped that way)
template <class U>
__device__ __forceinline__ int bam_unit_of(const U *__restrict__ u, int nb, int64_t g) {
    int lo = 0, hi = nb - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (u[mid].rec0 <= g) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

// record g decoded, its unit's name table, and where its line goes in the text arena
struct BlobSrc {
    const unsigned char *blobs;
    const BamUnitDev *u;
    int nb;
    const int64_t *off;  // text offset of every record (scan of the length pass)
    __device__ __forceinline__ void view(int64_t g, hgtb::BamRec *r, hgtb::BamNames *nm, int64_t *at) const {
        using namespace hgtb;
        const int k = bam_unit_of(u, nb, g);
        const BamUnitDev &U = u[k];
        const unsigned char *blob = blobs + U.blob_off;
        const BamUnitHeader h = *reinterpret_cast<const BamUnitHeader *>(blob);
        nm->off = reinterpret_cast<const uint32_t *>(blob + unit_name_off_at());
        nm->bytes = blob + unit_names_at(h.n_names);
        nm->n = h.n_names;
        const uint64_t *ro = reinterpret_cast<const uint64_t *>(blob + unit_rec_off_at(h.n_names, h.names_bytes));
        const int64_t i = g - U.rec0;
        const uint64_t a = ro[i], e = ro[i + 1];
        bam_decode(blob + a, e - a, (h.flags & UNIT_DROP_QUAL) != 0, r);
        if (off) *at = U.text_off + (off[g] - off[U.rec0]);
    }
};

struct DsplitSrc {
    const DsplitUnitDev *u;
    int nb;
    __device__ __forceinline__ void view(int64_t g, hgtb::BamRec *r, hgtb::BamNames *nm, int64_t *at) const {
        const int k = bam_unit_of(u, nb, g);
        const DsplitUnitDev &U = u[k];
        const int64_t i = g - U.rec0;
        const unsigned char *p = U.data + U.rec[i];
        // the index checked the block_size chain: the record's extent is its block_size
        hgtb::bam_decode(p, (uint64_t)hgtb::ld_u32(p) + 4, false, r, U.hide_qual != 0);
        r->ref = U.own;
        nm->off = U.name_off;
        nm->bytes = U.name_bytes;
        nm->n = U.n_names;
        if (U.toff) *at = U.text_off + (U.toff[i] - U.toff[0]);
    }
};

// text length of every record (one thread per record)
template <class Src>
__global__ void __launch_bounds__(BAM_THREADS) bam_text_len_kernel(Src src, int64_t n_rec, int64_t *__restrict__ len) {
    const int64_t g = (int64_t)blockIdx.x * BAM_THREADS + threadIdx.x;
    if (g >= n_rec) return;
    hgtb::BamRec r;
    hgtb::BamNames nm;
    int64_t at;
    src.view(g, &r, &nm, &at);
    len[g] = hgtb::bam_line_len(r, nm);
}

// one warp per record: QNAME, SEQ and QUAL lane-parallel, the other columns and the tags by lane 0 (bam_dev.cuh)
template <class Src>
__global__ void __launch_bounds__(BAM_THREADS) bam_render_kernel(Src src, int64_t n_rec, char *__restrict__ text) {
    const int64_t g = ((int64_t)blockIdx.x * BAM_THREADS + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (g >= n_rec) return;
    hgtb::BamRec r;
    hgtb::BamNames nm;
    int64_t at = 0;
    src.view(g, &r, &nm, &at);
    char *dst = text + at;
    const uint32_t qn = hgtb::qname_len(r);
    for (uint32_t i = lane; i < qn; i += 32) dst[i] = (char)r.p[hgtb::REC_FIXED + i];
    dst += qn;
    int64_t hl = 0;
    if (lane == 0) {
        hgtb::WriteSink w{dst};
        hgtb::bam_head(r, nm, w);
        hl = w.o - dst;
    }
    dst += __shfl_sync(0xffffffffu, hl, 0);
    if (r.l_seq == 0) {
        if (lane == 0) dst[0] = '*';
        dst += 1;
    } else {
        for (uint32_t i = lane; i < r.l_seq; i += 32) dst[i] = hgtb::seq_base(r, i);
        dst += r.l_seq;
    }
    if (lane == 0) dst[0] = '\t';
    dst += 1;
    if (!r.has_qual) {
        if (lane == 0) dst[0] = '*';
        dst += 1;
    } else {
        for (uint32_t i = lane; i < r.l_seq; i += 32) dst[i] = (char)(r.p[r.o_qual + i] + 33);
        dst += r.l_seq;
    }
    if (lane == 0) {
        hgtb::WriteSink w{dst};
        hgtb::bam_tags(r, w);
        *w.o = '\n';
    }
}

}  // namespace hgtk

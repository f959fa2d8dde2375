// The BGZF handle (hgt_bgzf_open's host walk) and the launch of the device inflate, shared by hgt_bgzf_inflate (bgzf.cu:
// output copied back to the caller) and the device split (bam_dsplit.cu: output kept in HBM).
#pragma once
#include <stdint.h>

#include <algorithm>
#include <vector>

#include "common.cuh"

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

// Device arena of one inflate: input at 0 | output at o_out | block offsets at o_desc (desc_bytes) | failure word at o_fail.
struct BgzfLayout {
    size_t o_out = 0, o_desc = 0, o_fail = 0, bytes = 0, desc_bytes = 0;
};
BgzfLayout bgzf_layout(const hgt_bgzf *z);
// the block offsets as the kernel reads them (desc_bytes), into page-locked h
void bgzf_descriptors(const hgt_bgzf *z, uint8_t *h);
// On ctx->stream: compressed bytes and the descriptors h_desc (page-locked, bgzf_descriptors) to the arena d, failure word
// set to all ones, bgzf_inflate_kernel when there is a block.  h2d_bytes grows by the input plus desc_bytes.
int bgzf_launch(hgt_ctx *ctx, const hgt_bgzf *z, const BgzfLayout &L, uint8_t *d, const uint8_t *h_desc);
// HGT_ERR_PARSE with the message of the first failing block (failure word w != all ones)
int bgzf_report_failure(const hgt_bgzf *z, uint64_t w);

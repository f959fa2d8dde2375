// Internal interface of the device split (bam_dsplit.cu) for the batch (typing.cu): a bucket as a render source.
#pragma once
#include <stddef.h>
#include <stdint.h>

#include "bam_kernels.cuh"
#include "common.cuh"

// Bucket `ref` of stream `stream`: its records, text bytes and device; *u filled except rec0 and text_off.
// HGT_ERR_ARG for a stream or ref out of range.
int bam_dsplit_unit(const hgt_bam_dsplit *s, int32_t stream, int32_t ref, hgtk::DsplitUnitDev *u, int64_t *n_records,
                    size_t *text_bytes, int *device);

// Batched diploid pair model (pair_batch.cu) as the batch entry point of typing.cu calls it.
#pragma once
#include <vector>

#include "common.cuh"

// One (unit, table) problem: the class rows of the region as the batch holds them (insertion order, not moved), and the
// name-containment relation of its locus in HBM (sub(a) = alleles whose name occurs inside a's name, sup = the inverse).
struct PairUnit {
    const uint64_t *bits = nullptr;             // [C][wp]
    const unsigned long long *count = nullptr;  // [C]
    const int32_t *first = nullptr;             // [C] dict order key (unique inside a region)
    const int64_t *sub_off = nullptr, *sup_off = nullptr;  // [A + 1]
    const int32_t *sub_idx = nullptr, *sup_idx = nullptr;
    int32_t C = 0, A = 0, wp = 0;
};

// The complete result of one call, on the host: unit u's pairs in (-p, lo, hi) order are [off[u], off[u + 1]) of lo / hi / p.
struct PairResult {
    std::vector<int64_t> off, n_pairs;  // n_pairs[u]: pairs after the first pruning (0 for an empty table)
    std::vector<int32_t> lo, hi, n_total, iters, status;
    std::vector<double> p;
};

// units[u] for every unit of the batch (C = 0: empty table).  cap = result rows per unit read back with the results; a unit
// with more is read back on its own (one more synchronisation, only then).
int hgt_pair_batch_run(hgt_ctx *ctx, cudaStream_t st, const std::vector<PairUnit> &units, int64_t max_pairs, int32_t cap,
                       PairResult *res);

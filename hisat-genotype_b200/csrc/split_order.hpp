// The order rule of the native intake, shared by the SAM split (sam_split.cpp) and the BAM split (bam_split.cpp): records
// found per input slice and reference are concatenated in input order and every reference's bucket is stably sorted by
// (read name bytewise, position).  That is the order `samtools view <aln> <backbone> | sort -k1,1 -s` produces on a
// coordinate-sorted file under LC_ALL=C (hisatgenotype_typing_core.py:436-468): both sorts of the reference are stable.
#pragma once
#include <string.h>

#include <algorithm>
#include <atomic>
#include <thread>
#include <vector>

namespace hgt_split {

inline int default_threads(int n_threads) {
    if (n_threads > 0) return n_threads;
    const unsigned hc = std::thread::hardware_concurrency();
    return hc ? (int)hc : 1;
}

template <class F>
void run_threads(int n_threads, size_t n, F f) {
    if (n_threads <= 1 || n <= 1) {
        for (size_t i = 0; i < n; i++) f(i);
        return;
    }
    std::atomic<size_t> next{0};
    std::vector<std::thread> th;
    const int nt = (int)std::min<size_t>((size_t)n_threads, n);
    for (int t = 0; t < nt; t++)
        th.emplace_back([&]() {
            while (true) {
                const size_t i = next.fetch_add(1);
                if (i >= n) break;
                f(i);
            }
        });
    for (auto &x : th) x.join();
}

// part[slice][ref] -> bucket[ref] in the order rule.  Rec needs `name_len` and `pos`; name_of(rec) gives the name's first
// byte.  done(ref) runs on the same thread once the bucket is ordered.
template <class Rec, class NameOf, class Done>
void bucket_and_order(int n_threads, std::vector<std::vector<std::vector<Rec>>> &part, std::vector<std::vector<Rec>> &bucket,
                      NameOf name_of, Done done) {
    const size_t n_slices = part.size();
    run_threads(n_threads, bucket.size(), [&](size_t r) {
        std::vector<Rec> &b = bucket[r];
        size_t total = 0;
        for (size_t k = 0; k < n_slices; k++) total += part[k][r].size();
        b.reserve(total);
        for (size_t k = 0; k < n_slices; k++) b.insert(b.end(), part[k][r].begin(), part[k][r].end());
        std::stable_sort(b.begin(), b.end(), [&name_of](const Rec &x, const Rec &y) {
            const uint32_t m = std::min(x.name_len, y.name_len);
            const int c = memcmp(name_of(x), name_of(y), m);
            if (c != 0) return c < 0;
            if (x.name_len != y.name_len) return x.name_len < y.name_len;
            return x.pos < y.pos;
        });
        done(r);
    });
}

}  // namespace hgt_split

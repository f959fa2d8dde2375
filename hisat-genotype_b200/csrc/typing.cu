// Stage (a): per-read allele compatibility -> Gene_cmpt / Gene_counts, on the GPU.
//
// Replaces the per-read loop of typing() (reference hisatgenotype_typing_core.py:598-1596) and get_mpileup
// (hisatgenotype_typing_common.py:1059-1184).  Everything runs on the GPU once the alignment text has been copied:
//   record stage (reads.cuh / walk_dev.cuh)  line index, parse, pileup histogram + nt_set, run heads / mate de-dup, CIGAR x
//                      MD x Zs walk, error correction, ambiguity expansion, exon clipping  ->  per pair and table a list of
//                      haplotypes (left, right, sorted variant rows)
//   set stage (this file)  haplotype -> allele bitset (add_count, core:626-677); per-pair arg-max class (add_stat,
//                      core:1171-1236); class de-duplication into (bitset, count, first-seen) tables; Gene_counts.
// walk.hpp only holds the host-side description of a locus (hgt_locus_create -> build_walk_tables).
//
// HBM layout per locus (built once by hgt_locus_create):
//   var_pos[V] int32 (Var_list order), delr_{right,row}[D] deletions sorted by right end,
//   st[levels][V][wp] uint64: level 0 = Links as a bit matrix (one row per variant, one bit per allele),
//   level j = OR of 2^j consecutive rows (sparse table: OR is idempotent, so any contiguous range of
//   variant rows is the OR of two rows) -> a haplotype with k known variants touches 3k+2 rows instead of
//   every row its span covers.  mask[3][wp] = table masks (all alleles / exon reps / primary-exon reps).
#include <math.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <deque>
#include <memory>
#include <mutex>
#include <numeric>
#include <thread>
#include <string>
#include <string_view>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include "common.cuh"
#include "em_internal.h"
#include "walk.hpp"
#include "walk_dev.cuh"
#include "reads.cuh"
#include "bam_dev.cuh"
#include "bam_dsplit.h"
#include "bam_kernels.cuh"
#include "pair_batch.h"

using namespace hgt;

// ================================================================================================================
// Locus
// ================================================================================================================
struct hgt_locus {
    LocusHost host;
    int A = 0, V = 0, L = 0, wp = 0, levels = 0, n_delr = 0;
    bool is_hla = false;
    std::vector<uint64_t> mask;  // [3][wp]
    std::vector<int32_t> gn_rank;
    std::vector<int32_t> delr_right, delr_row;
    std::vector<int64_t> group_off;      // [A+1] members of the exon group represented by allele a (allele_rep_groups)
    std::vector<int32_t> group_member;
    std::vector<double> allele_len;      // [A] Gene_lengths
    hgt_ctx *ctx = nullptr;
    int32_t *d_var_pos = nullptr, *d_delr_right = nullptr, *d_delr_row = nullptr, *d_gn_rank = nullptr;
    int32_t *d_lb = nullptr;  // [2][L + 2] lower-bound tables by position (variants, deletion right ends)
    uint64_t *d_st = nullptr, *d_mask = nullptr;
    double *d_allele_len = nullptr;
    // tables of the record walk (walk_dev.cuh): one blob, viewed through host pointers (emulation, tests) and device pointers
    std::vector<unsigned char> wt_blob;
    std::vector<size_t> wt_off;
    uint32_t wt_hash_mask = 0;
    int32_t wt_num_lo = 0, wt_num_n = 0, wt_tok_regular = 0;
    int wt_n_alt[2] = {0, 0};
    unsigned char *d_wt = nullptr;
    hgtd::LocusWalk wt_host, wt_dev;
    // containment relation of the allele names (hgt_locus_set_names), for the pair model.  Loci are shared by batches on
    // several host threads (one context each): the relation is replaced as a whole under names_mu, never changed in
    // place except for its lazily made device copy (also under names_mu), and a pair call holds a reference until it
    // has synchronised, so a replaced relation's device arrays outlive every kernel that reads them.
    std::mutex names_mu;
    std::shared_ptr<struct NameRel> names;
};

// sub(a) = alleles whose name occurs inside a's name (a included), sup(x) = alleles whose name contains x's; CSR in
// sorted-name index space.  The device copy is made at the first pair call and freed with the relation.
struct NameRel {
    std::vector<int64_t> sub_off, sup_off;
    std::vector<int32_t> sub_idx, sup_idx;
    int device = -1;
    int64_t *d_sub_off = nullptr, *d_sup_off = nullptr;
    int32_t *d_sub_idx = nullptr, *d_sup_idx = nullptr;
    ~NameRel() {
        if (device < 0) return;
        cudaSetDevice(device);
        cudaFree(d_sub_off); cudaFree(d_sub_idx); cudaFree(d_sup_off); cudaFree(d_sup_idx);
    }
};

struct LocusDev {
    const int32_t *var_pos, *delr_right, *delr_row;
    const int32_t *lb_var, *lb_del;  // [L + 2] each: number of variants / of deletion right ends below position x
    const uint64_t *st, *mask;
    int V, wp, n_delr, levels, L;
};

static LocusDev locus_dev(const hgt_locus *l) {
    LocusDev d;
    d.var_pos = l->d_var_pos; d.delr_right = l->d_delr_right; d.delr_row = l->d_delr_row;
    d.st = l->d_st; d.mask = l->d_mask; d.V = l->V; d.wp = l->wp; d.n_delr = l->n_delr; d.levels = l->levels;
    d.lb_var = l->d_lb; d.lb_del = l->d_lb + (l->L + 2); d.L = l->L;
    return d;
}

__global__ void st_build_kernel(uint64_t *st, int V, int wp, int level) {
    const size_t n = (size_t)V * wp;
    const uint64_t *src = st + (size_t)(level - 1) * n;
    uint64_t *dst = st + (size_t)level * n;
    const int half = 1 << (level - 1);
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int row = (int)(i / wp), j = (int)(i % wp);
        const int r2 = row + half;
        uint64_t v = src[i];
        if (r2 < V) v |= src[(size_t)r2 * wp + j];
        dst[i] = v;
    }
}

static bool split_tokens(const std::string &s, char sep, std::vector<std::string> *out) {
    out->clear();
    size_t p = 0;
    while (true) {
        size_t q = s.find(sep, p);
        if (q == std::string::npos) {
            out->push_back(s.substr(p));
            break;
        }
        out->push_back(s.substr(p, q - p));
        p = q + 1;
    }
    return true;
}

static int parse_alts(hgt_locus *loc, const char *text) {
    if (!text) return HGT_OK;
    const char *p = text;
    std::vector<std::string> toks;
    while (*p) {
        const char *e = strchr(p, '\n');
        if (!e) e = p + strlen(p);
        std::string line(p, e - p);
        p = *e ? e + 1 : e;
        if (line.empty()) continue;
        std::vector<std::string> cols;
        split_tokens(line, '\t', &cols);
        if (cols.size() != 3 || (cols[0] != "L" && cols[0] != "R")) {
            hgt_set_error("alts_text: malformed line '%s'", line.c_str());
            return HGT_ERR_ARG;
        }
        AltEntry ent;
        ent.key = cols[1];
        split_tokens(ent.key, '-', &ent.toks);
        if (ent.toks.size() < 2) {
            hgt_set_error("alts_text: malformed key '%s'", ent.key.c_str());
            return HGT_ERR_ARG;
        }
        ent.anchor = atoi(cols[0] == "L" ? ent.toks.back().c_str() : ent.toks.front().c_str());
        std::vector<std::string> alts;
        split_tokens(cols[2], ',', &alts);
        for (const std::string &a : alts) {
            split_tokens(a, '-', &toks);
            if (toks.size() < 2) {
                hgt_set_error("alts_text: malformed alternative '%s'", a.c_str());
                return HGT_ERR_ARG;
            }
            AltHap h;
            h.left = atoi(toks.front().c_str());
            h.right = atoi(toks.back().c_str());
            for (size_t i = 1; i + 1 < toks.size(); i++) {
                auto f = loc->host.row_of.find(toks[i]);
                if (f == loc->host.row_of.end()) {
                    hgt_set_error("alts_text: unknown variant id '%s'", toks[i].c_str());
                    return HGT_ERR_ARG;
                }
                if (loc->host.vars[f->second].type == T_INSERTION) {
                    hgt_set_error("alts_text: insertion '%s' inside an alternative haplotype", toks[i].c_str());
                    return HGT_ERR_ARG;
                }
                h.rows.push_back(f->second);
            }
            ent.alts.push_back(std::move(h));
        }
        (cols[0] == "L" ? loc->host.alts_left : loc->host.alts_right).push_back(std::move(ent));
    }
    auto by_anchor = [](const AltEntry &a, const AltEntry &b) { return a.anchor < b.anchor; };
    std::stable_sort(loc->host.alts_left.begin(), loc->host.alts_left.end(), by_anchor);
    std::stable_sort(loc->host.alts_right.begin(), loc->host.alts_right.end(), by_anchor);
    return HGT_OK;
}

extern "C" void hgt_locus_free(hgt_locus *l) {
    if (!l) return;
    if (l->ctx) {
        cudaSetDevice(l->ctx->device);
        cudaFree(l->d_var_pos); cudaFree(l->d_delr_right); cudaFree(l->d_delr_row); cudaFree(l->d_gn_rank); cudaFree(l->d_lb);
        cudaFree(l->d_st); cudaFree(l->d_mask); cudaFree(l->d_allele_len); cudaFree(l->d_wt);
    }
    delete l;
}

// ---- allele names: the name-containment relation of the pair model --------------------------------------------------------
// The legacy pair model tests `allele in allele_pair` on the key string "a-b"; names hold no '-', so x matches the pair
// exactly when x's name is a substring of a's or of b's.  That relation is a property of the locus: every substring of
// every name is looked up in a hash set of the names, O(A len^2) lookups instead of O(A^2) string tests.
extern "C" int hgt_locus_set_names(hgt_locus *loc, int32_t n, const char *const *names) {
    if (!loc || !names || n != loc->A) {
        hgt_set_error("hgt_locus_set_names: need the locus and its %d allele names", loc ? loc->A : 0);
        return HGT_ERR_ARG;
    }
    std::vector<std::string_view> nm((size_t)n);
    for (int32_t a = 0; a < n; a++) {
        if (!names[a] || !names[a][0] || strchr(names[a], '-')) {
            hgt_set_error("hgt_locus_set_names: name %d is empty or contains '-'", a);
            return HGT_ERR_ARG;
        }
        nm[a] = names[a];
        if (a > 0 && !(nm[a - 1] < nm[a])) {
            hgt_set_error("hgt_locus_set_names: names must be distinct and in sorted order (name %d)", a);
            return HGT_ERR_ARG;
        }
    }
    std::unordered_map<std::string_view, int32_t> index;
    index.reserve((size_t)n * 2);
    size_t max_len = 0;
    for (int32_t a = 0; a < n; a++) {
        index.emplace(nm[a], a);
        max_len = std::max(max_len, nm[a].size());
    }
    auto rel = std::make_shared<NameRel>();
    std::vector<int64_t> &sub_off = rel->sub_off, &sup_off = rel->sup_off;
    std::vector<int32_t> &sub_idx = rel->sub_idx, found;
    sub_off.assign((size_t)n + 1, 0);
    sup_off.assign((size_t)n + 1, 0);
    for (int32_t a = 0; a < n; a++) {
        const std::string_view s = nm[a];
        found.clear();
        for (size_t i = 0; i < s.size(); i++)
            for (size_t len = 1; i + len <= s.size(); len++) {
                auto it = index.find(s.substr(i, len));
                if (it != index.end()) found.push_back(it->second);
            }
        std::sort(found.begin(), found.end());
        found.erase(std::unique(found.begin(), found.end()), found.end());
        sub_idx.insert(sub_idx.end(), found.begin(), found.end());
        sub_off[a + 1] = (int64_t)sub_idx.size();
    }
    std::vector<int32_t> &sup_idx = rel->sup_idx;
    sup_idx.resize(sub_idx.size());
    for (int32_t x : sub_idx) sup_off[x + 1]++;
    for (int32_t a = 0; a < n; a++) sup_off[a + 1] += sup_off[a];
    std::vector<int64_t> fill(sup_off.begin(), sup_off.end() - 1);
    for (int32_t a = 0; a < n; a++)  // a ascending: every sup list comes out ascending
        for (int64_t s = sub_off[a]; s < sub_off[a + 1]; s++) sup_idx[fill[sub_idx[s]]++] = a;
    std::shared_ptr<NameRel> old;
    {
        std::lock_guard<std::mutex> g(loc->names_mu);
        old.swap(loc->names);
        loc->names = std::move(rel);
    }
    return HGT_OK;  // (old is released here, or by the last pair call still holding it)
}

static std::shared_ptr<NameRel> locus_names(const hgt_locus *loc) {
    std::lock_guard<std::mutex> g(const_cast<hgt_locus *>(loc)->names_mu);
    return loc->names;
}

extern "C" int hgt_locus_name_subsets(const hgt_locus *loc, int64_t *off, int32_t *idx, int64_t *n_idx) {
    const std::shared_ptr<NameRel> rel = loc ? locus_names(loc) : nullptr;
    if (!rel) {
        hgt_set_error("hgt_locus_name_subsets: no names set on this locus");
        return HGT_ERR_ARG;
    }
    // one relation for the whole read: another thread may replace it between a size query and this call, so idx comes
    // with its capacity in *n_idx
    const int64_t n = (int64_t)rel->sub_idx.size();
    if (idx && (!n_idx || *n_idx < n)) {
        if (n_idx) *n_idx = n;
        hgt_set_error("hgt_locus_name_subsets: idx holds fewer than the %lld entries of the relation", (long long)n);
        return HGT_ERR_ARG;
    }
    if (n_idx) *n_idx = n;
    if (off) memcpy(off, rel->sub_off.data(), rel->sub_off.size() * sizeof(int64_t));
    if (idx) memcpy(idx, rel->sub_idx.data(), (size_t)n * sizeof(int32_t));
    return HGT_OK;
}

// The locus's current relation with its device copy made (on `device`); the caller keeps the reference until its kernels
// have finished.  The copy is complete before any thread can see it: it is built and published under names_mu.
static int locus_names_dev(hgt_locus *l, int device, std::shared_ptr<NameRel> *out) {
    std::lock_guard<std::mutex> g(l->names_mu);
    std::shared_ptr<NameRel> rel = l->names;
    if (!rel) {
        hgt_set_error("hgt_batch_pairs: no allele names set on a locus of the batch (hgt_locus_set_names)");
        return HGT_ERR_ARG;
    }
    if (!rel->d_sub_off) {
        void *p[4] = {nullptr, nullptr, nullptr, nullptr};
        const void *src[4] = {rel->sub_off.data(), rel->sub_idx.data(), rel->sup_off.data(), rel->sup_idx.data()};
        const size_t n[4] = {rel->sub_off.size() * 8, rel->sub_idx.size() * 4, rel->sup_off.size() * 8, rel->sup_idx.size() * 4};
        cudaError_t e = cudaSuccess;
        for (int i = 0; i < 4 && e == cudaSuccess; i++) {
            e = cudaMalloc(&p[i], std::max<size_t>(n[i], 8));
            if (e == cudaSuccess && n[i]) e = cudaMemcpy(p[i], src[i], n[i], cudaMemcpyHostToDevice);
        }
        if (e != cudaSuccess) {
            for (void *x : p) cudaFree(x);
            hgt_set_error("hgt_batch_pairs: device copy of the allele names: %s", cudaGetErrorString(e));
            return HGT_ERR_CUDA;
        }
        rel->device = device;
        rel->d_sub_off = static_cast<int64_t *>(p[0]); rel->d_sub_idx = static_cast<int32_t *>(p[1]);
        rel->d_sup_off = static_cast<int64_t *>(p[2]); rel->d_sup_idx = static_cast<int32_t *>(p[3]);
    }
    *out = std::move(rel);
    return HGT_OK;
}

// ---- tables of the record walk as one blob ----------------------------------------------------------------------------------
namespace {
struct Blob {
    std::vector<unsigned char> data;
    std::vector<size_t> off;
    template <class T>
    void add(const std::vector<T> &v) {
        const size_t o = (data.size() + 15) & ~(size_t)15;
        data.resize(o + std::max<size_t>(v.size() * sizeof(T), 16), 0);
        if (!v.empty()) memcpy(data.data() + o, v.data(), v.size() * sizeof(T));
        off.push_back(o);
    }
};
struct AltFlat {
    std::vector<int32_t> anchor, key_off{0}, tok_off{0}, tok_row, tok_num, alt_off{0}, alt_left, alt_right, altrow_off{0}, altrow;
    std::vector<char> key_pool;
    void build(const std::vector<AltEntry> &tab) {
        for (const AltEntry &e : tab) {
            anchor.push_back(e.anchor);
            key_pool.insert(key_pool.end(), e.key.begin(), e.key.end());
            key_off.push_back((int32_t)key_pool.size());
            for (size_t t = 0; t < e.toks.size(); t++) {
                tok_row.push_back(e.tok_rows[t]);
                tok_num.push_back(atoi(e.toks[t].c_str()));
            }
            tok_off.push_back((int32_t)tok_row.size());
            for (const AltHap &a : e.alts) {
                alt_left.push_back(a.left);
                alt_right.push_back(a.right);
                altrow.insert(altrow.end(), a.rows.begin(), a.rows.end());
                altrow_off.push_back((int32_t)altrow.size());
            }
            alt_off.push_back((int32_t)alt_left.size());
        }
    }
};
}  // namespace

static void build_walk_tables(hgt_locus *l) {
    const LocusHost &h = l->host;
    const int V = l->V;
    std::vector<int32_t> vpos(V), vlen(V), id_off{0};
    std::vector<uint8_t> vtype(V), vflags(V);
    std::vector<char> vbase(V), id_pool;
    for (int i = 0; i < V; i++) {
        vpos[i] = h.vars[i].pos; vlen[i] = h.vars[i].len; vtype[i] = h.vars[i].type; vbase[i] = h.vars[i].base;
        vflags[i] = (uint8_t)((h.vars[i].in_links ? 1 : 0) | (h.vars[i].is_hv ? 2 : 0));
        id_pool.insert(id_pool.end(), h.vars[i].id.begin(), h.vars[i].id.end());
        id_off.push_back((int32_t)id_pool.size());
    }
    uint32_t cap = 16;
    while (cap < 2u * (uint32_t)std::max(V, 1)) cap <<= 1;
    std::vector<int32_t> id_hash(cap, -1);
    for (int i = 0; i < V; i++) {  // a later duplicate id replaces the earlier one, like row_of[id] = i
        const std::string &id = h.vars[i].id;
        uint32_t slot = hgtd::id_slot(id.data(), (int)id.size(), cap - 1);
        while (id_hash[slot] >= 0 && h.vars[id_hash[slot]].id != id) slot = (slot + 1) & (cap - 1);
        id_hash[slot] = i;
    }
    AltFlat fl, fr;
    fl.build(h.alts_left);
    fr.build(h.alts_right);
    std::vector<int32_t> ex, pex;
    for (auto &e : h.exons) { ex.push_back(e.first); ex.push_back(e.second); }
    for (auto &e : h.primary_exons) { pex.push_back(e.first); pex.push_back(e.second); }
    std::vector<char> ref(h.ref.begin(), h.ref.end());
    Blob b;
    b.add(ref);                                                              // 0
    b.add(vpos); b.add(vlen); b.add(vtype); b.add(vbase); b.add(vflags);     // 1..5
    b.add(id_off); b.add(id_pool); b.add(id_hash);                           // 6..8
    for (const AltFlat *f : {&fl, &fr}) {                                    // 9..20, 21..32
        b.add(f->anchor); b.add(f == &fl ? h.altl_below : h.altr_below); b.add(f->key_off); b.add(f->key_pool);
        b.add(f->tok_off); b.add(f->tok_row); b.add(f->tok_num); b.add(f->alt_off); b.add(f->alt_left); b.add(f->alt_right);
        b.add(f->altrow_off); b.add(f->altrow);
    }
    b.add(ex); b.add(pex);                                                   // 33, 34
    std::vector<int32_t> lbv((size_t)l->L + 2);
    {
        size_t k = 0;
        for (size_t x = 0; x < lbv.size(); x++) {
            while (k < (size_t)V && h.var_pos[k] < (int32_t)x) k++;
            lbv[x] = (int32_t)k;
        }
    }
    b.add(lbv);                                                              // 35
    // regular ids: direct table number -> row
    std::vector<int32_t> num_row;
    l->wt_num_lo = 0;
    {
        int64_t lo = INT64_MAX, hi = -1;
        bool regular = V > 0;
        std::vector<int64_t> num((size_t)V);
        for (int i = 0; i < V && regular; i++) {
            num[i] = hgtd::regular_id_number(h.vars[i].id.data(), (int)h.vars[i].id.size());
            regular = num[i] >= 0;
            lo = std::min(lo, num[i]); hi = std::max(hi, num[i]);
        }
        if (regular && hi - lo + 1 <= 8 * (int64_t)V + 1024 && hi < (1ll << 31)) {
            num_row.assign((size_t)(hi - lo + 1), -1);
            for (int i = 0; i < V && regular; i++) {
                regular = num_row[(size_t)(num[i] - lo)] < 0;  // unique
                num_row[(size_t)(num[i] - lo)] = i;
            }
            if (regular) l->wt_num_lo = (int32_t)lo;
            else num_row.clear();
        }
    }
    if (getenv("HGT_IRREGULAR_IDS")) num_row.clear();  // tests: the general paths (id hash table, character substring rule)
    l->wt_num_n = (int32_t)num_row.size();
    l->wt_tok_regular = l->wt_num_n > 0;
    for (const std::vector<AltEntry> *tab : {&h.alts_left, &h.alts_right})
        for (const AltEntry &e : *tab)
            for (size_t t = 0; t < e.toks.size(); t++) {
                bool digits = !e.toks[t].empty();
                for (char ch : e.toks[t]) digits &= ch >= '0' && ch <= '9';
                if (e.tok_rows[t] < 0 && !digits) l->wt_tok_regular = 0;
            }
    b.add(num_row);                                                          // 36
    std::vector<int32_t> id_num((size_t)V, 0);
    if (l->wt_num_n > 0)
        for (int i = 0; i < V; i++) id_num[i] = (int32_t)hgtd::regular_id_number(h.vars[i].id.data(), (int)h.vars[i].id.size());
    b.add(id_num);                                                           // 37
    // read ends identify_ambigious_diffs can act on (AltTab::end_flag)
    {
        auto vright = [&](int32_t r) { return h.vars[r].type == hgtd::T_DELETION ? h.vars[r].pos + h.vars[r].len - 1 : h.vars[r].pos; };
        std::vector<uint8_t> fl_left((size_t)l->L + 2, 0), fl_right((size_t)l->L + 2, 0);
        for (const AltEntry &e : h.alts_left) {
            const int ntok = (int)e.toks.size() - 1;  // key.split('-')[:-1]
            if (ntok < 1) continue;
            int64_t bound = atoi(e.toks[0].c_str());
            for (int k = 1; k < ntok; k++) bound = e.tok_rows[k] < 0 ? 0 : std::min<int64_t>(bound, (int64_t)vright(e.tok_rows[k]) + 1);
            for (int64_t x = std::max<int64_t>(bound, 0); x <= std::min<int64_t>(e.anchor, l->L + 1); x++) fl_left[(size_t)x] = 1;
        }
        for (const AltEntry &e : h.alts_right) {
            const int ntok = (int)e.toks.size() - 1;  // key.split('-')[1:]
            if (ntok < 1) continue;
            int64_t bound = atoi(e.toks[ntok].c_str());
            for (int k = 1; k < ntok; k++) bound = e.tok_rows[k] < 0 ? l->L + 1 : std::max<int64_t>(bound, (int64_t)h.vars[e.tok_rows[k]].pos - 1);
            for (int64_t x = std::max<int64_t>(e.anchor, 0); x <= std::min<int64_t>(bound, l->L + 1); x++) fl_right[(size_t)x] = 1;
        }
        b.add(fl_left); b.add(fl_right);                                     // 38, 39
    }
    l->wt_blob.swap(b.data);
    l->wt_off.swap(b.off);
    l->wt_hash_mask = cap - 1;
    l->wt_n_alt[0] = (int)fl.anchor.size();
    l->wt_n_alt[1] = (int)fr.anchor.size();
}

// view of the blob through `base` (host copy or device copy)
static hgtd::LocusWalk walk_view(const hgt_locus *l, const unsigned char *base) {
    hgtd::LocusWalk w;
    auto at = [&](int k) { return base + l->wt_off[k]; };
    w.ref = reinterpret_cast<const char *>(at(0));
    w.L = l->L;
    w.is_hla = l->is_hla ? 1 : 0;
    w.v.V = l->V;
    w.v.pos = reinterpret_cast<const int32_t *>(at(1)); w.v.len = reinterpret_cast<const int32_t *>(at(2));
    w.v.lb = reinterpret_cast<const int32_t *>(at(35)); w.v.L = l->L;
    w.v.type = at(3); w.v.base = reinterpret_cast<const char *>(at(4)); w.v.flags = at(5);
    w.v.id_off = reinterpret_cast<const int32_t *>(at(6)); w.v.id_pool = reinterpret_cast<const char *>(at(7));
    w.v.id_hash = reinterpret_cast<const int32_t *>(at(8)); w.v.id_hash_mask = l->wt_hash_mask;
    w.v.num_row = reinterpret_cast<const int32_t *>(at(36)); w.v.id_num = reinterpret_cast<const int32_t *>(at(37)); w.v.num_lo = l->wt_num_lo; w.v.num_n = l->wt_num_n;
    w.v.tok_regular = l->wt_tok_regular;
    for (int side = 0; side < 2; side++) {
        hgtd::AltTab &t = side ? w.ar : w.al;
        const int k = 9 + 12 * side;
        t.n = l->wt_n_alt[side];
        t.anchor = reinterpret_cast<const int32_t *>(at(k)); t.below = reinterpret_cast<const int32_t *>(at(k + 1));
        t.key_off = reinterpret_cast<const int32_t *>(at(k + 2)); t.key_pool = reinterpret_cast<const char *>(at(k + 3));
        t.tok_off = reinterpret_cast<const int32_t *>(at(k + 4)); t.tok_row = reinterpret_cast<const int32_t *>(at(k + 5));
        t.tok_num = reinterpret_cast<const int32_t *>(at(k + 6)); t.alt_off = reinterpret_cast<const int32_t *>(at(k + 7));
        t.alt_left = reinterpret_cast<const int32_t *>(at(k + 8)); t.alt_right = reinterpret_cast<const int32_t *>(at(k + 9));
        t.altrow_off = reinterpret_cast<const int32_t *>(at(k + 10)); t.altrow = reinterpret_cast<const int32_t *>(at(k + 11));
        t.end_flag = at(38 + side);
    }
    w.n_exons = (int)l->host.exons.size(); w.n_pexons = (int)l->host.primary_exons.size();
    w.exons = reinterpret_cast<const int32_t *>(at(33)); w.pexons = reinterpret_cast<const int32_t *>(at(34));
    return w;
}

extern "C" int hgt_locus_create(hgt_ctx *ctx, const hgt_locus_desc *d, hgt_locus **out) {
    if (!d || !out) {
        hgt_set_error("hgt_locus_create: null argument");
        return HGT_ERR_ARG;
    }
    *out = nullptr;
    if (d->n_alleles < 1 || d->n_vars < 0 || d->ref_len < 1 || !d->ref_seq) {
        hgt_set_error("hgt_locus_create: need n_alleles >= 1, ref_len >= 1");
        return HGT_ERR_ARG;
    }
    hgt_locus *l = new hgt_locus();
    l->ctx = ctx;
    l->A = d->n_alleles; l->V = d->n_vars; l->L = d->ref_len; l->wp = hgt_row_pitch(d->n_alleles);
    l->is_hla = d->is_hla != 0;
    LocusHost &h = l->host;
    h.is_hla = l->is_hla;
    h.ref.assign(d->ref_seq, d->ref_len);
    h.vars.resize(l->V);
    h.var_pos.resize(l->V);
    const char *ids = d->var_ids;
    for (int i = 0; i < l->V; i++) {
        VarInfo &v = h.vars[i];
        v.pos = d->var_pos[i]; v.len = d->var_len[i]; v.type = d->var_type[i]; v.base = d->var_base[i];
        v.in_links = d->var_flags[i] & 1; v.is_hv = (d->var_flags[i] >> 1) & 1;
        v.id = ids;
        ids += v.id.size() + 1;
        h.var_pos[i] = v.pos;
        h.row_of[v.id] = i;
        if (i > 0 && h.var_pos[i] < h.var_pos[i - 1]) {
            hgt_set_error("hgt_locus_create: variants must be sorted by position (Var_list order)");
            delete l;
            return HGT_ERR_ARG;
        }
    }
    for (int i = 0; i < d->n_exons; i++) h.exons.push_back({d->exons[2 * i], d->exons[2 * i + 1]});
    for (int i = 0; i < d->n_primary_exons; i++)
        h.primary_exons.push_back({d->primary_exons[2 * i], d->primary_exons[2 * i + 1]});
    int rc = parse_alts(l, d->alts_text);
    if (rc != HGT_OK) {
        delete l;
        return rc;
    }
    h.finalize();
    const int wp = l->wp;
    l->mask.assign((size_t)3 * wp, 0);
    for (int a = 0; a < l->A; a++) l->mask[a >> 6] |= 1ull << (a & 63);
    if (l->is_hla) {
        if (!d->exon_rep_mask || !d->primary_rep_mask) {
            hgt_set_error("hgt_locus_create: is_hla needs exon_rep_mask and primary_rep_mask");
            delete l;
            return HGT_ERR_ARG;
        }
        for (int j = 0; j < wp; j++) {
            l->mask[wp + j] = d->exon_rep_mask[j] & l->mask[j];
            l->mask[2 * wp + j] = d->primary_rep_mask[j] & l->mask[j];
        }
    }
    l->gn_rank.assign(l->A, 0);
    for (int a = 0; a < l->A; a++) l->gn_rank[a] = d->gene_names_rank ? d->gene_names_rank[a] : a;
    // deletions sorted by right end: a deletion starting left of a haplotype but ending inside it is negative
    // evidence too (core:663-669)
    std::vector<int32_t> order;
    for (int i = 0; i < l->V; i++)
        if (h.vars[i].type == T_DELETION && h.vars[i].in_links && h.vars[i].len > 1) order.push_back(i);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return h.vars[a].right() < h.vars[b].right(); });
    for (int r : order) {
        l->delr_right.push_back(h.vars[r].right());
        l->delr_row.push_back(r);
    }
    l->n_delr = (int)order.size();
    l->group_off.assign(l->A + 1, 0);
    if (d->group_off && d->group_member) {
        l->group_off.assign(d->group_off, d->group_off + l->A + 1);
        l->group_member.assign(d->group_member, d->group_member + d->group_off[l->A]);
    }
    l->allele_len.assign(l->A, 1.0);
    if (d->allele_len) l->allele_len.assign(d->allele_len, d->allele_len + l->A);
    if (!ctx) {
        build_walk_tables(l);
        l->wt_host = walk_view(l, l->wt_blob.data());
        *out = l;
        return HGT_OK;
    }
    // ---- device tables -----------------------------------------------------------------------------------
    cudaError_t e = cudaSetDevice(ctx->device);
    const int V = l->V;
    int levels = 1;
    while ((1 << levels) <= V) levels++;
    l->levels = levels;
    std::vector<uint64_t> lbits((size_t)std::max(V, 1) * wp, 0);
    for (int i = 0; i < V; i++) {
        if (!h.vars[i].in_links) continue;
        for (int64_t k = d->link_off[i]; k < d->link_off[i + 1]; k++) {
            const int a = d->link_allele[k];
            if (a < 0 || a >= l->A) {
                hgt_set_error("hgt_locus_create: link allele index %d out of range", a);
                delete l;
                return HGT_ERR_ARG;
            }
            lbits[(size_t)i * wp + (a >> 6)] |= 1ull << (a & 63);
        }
    }
    const size_t lvl_words = (size_t)std::max(V, 1) * wp;
#define LTRY(call)                                                                                 \
    if (e == cudaSuccess) {                                                                        \
        e = (call);                                                                                \
        if (e != cudaSuccess) hgt_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e)); \
    }
    // lower_bound by position as a table: lb[x] = number of entries < x for x in [0, L + 1] (the kernels clamp x)
    std::vector<int32_t> lb(2 * (size_t)(l->L + 2));
    {
        const size_t n = (size_t)l->L + 2;
        size_t k = 0;
        for (size_t x = 0; x < n; x++) {
            while (k < (size_t)V && h.var_pos[k] < (int32_t)x) k++;
            lb[x] = (int32_t)k;
        }
        k = 0;
        for (size_t x = 0; x < n; x++) {
            while (k < (size_t)l->n_delr && l->delr_right[k] < (int32_t)x) k++;
            lb[n + x] = (int32_t)k;
        }
    }
    LTRY(cudaMalloc(&l->d_lb, sizeof(int32_t) * lb.size()));
    LTRY(cudaMalloc(&l->d_var_pos, sizeof(int32_t) * std::max(V, 1)));
    LTRY(cudaMalloc(&l->d_delr_right, sizeof(int32_t) * std::max(l->n_delr, 1)));
    LTRY(cudaMalloc(&l->d_delr_row, sizeof(int32_t) * std::max(l->n_delr, 1)));
    LTRY(cudaMalloc(&l->d_gn_rank, sizeof(int32_t) * l->A));
    LTRY(cudaMalloc(&l->d_mask, sizeof(uint64_t) * 3 * wp));
    LTRY(cudaMalloc(&l->d_st, sizeof(uint64_t) * lvl_words * levels));
    LTRY(cudaMalloc(&l->d_allele_len, sizeof(double) * l->A));
    cudaStream_t st = ctx->stream;
    LTRY(cudaMemcpyAsync(l->d_lb, lb.data(), sizeof(int32_t) * lb.size(), cudaMemcpyHostToDevice, st));
    if (V > 0) LTRY(cudaMemcpyAsync(l->d_var_pos, h.var_pos.data(), sizeof(int32_t) * V, cudaMemcpyHostToDevice, st));
    if (l->n_delr > 0) {
        LTRY(cudaMemcpyAsync(l->d_delr_right, l->delr_right.data(), sizeof(int32_t) * l->n_delr, cudaMemcpyHostToDevice, st));
        LTRY(cudaMemcpyAsync(l->d_delr_row, l->delr_row.data(), sizeof(int32_t) * l->n_delr, cudaMemcpyHostToDevice, st));
    }
    LTRY(cudaMemcpyAsync(l->d_gn_rank, l->gn_rank.data(), sizeof(int32_t) * l->A, cudaMemcpyHostToDevice, st));
    LTRY(cudaMemcpyAsync(l->d_allele_len, l->allele_len.data(), sizeof(double) * l->A, cudaMemcpyHostToDevice, st));
    LTRY(cudaMemcpyAsync(l->d_mask, l->mask.data(), sizeof(uint64_t) * 3 * wp, cudaMemcpyHostToDevice, st));
    LTRY(cudaMemcpyAsync(l->d_st, lbits.data(), sizeof(uint64_t) * lvl_words, cudaMemcpyHostToDevice, st));
    if (e == cudaSuccess) {
        for (int lv = 1; lv < levels; lv++) {
            st_build_kernel<<<ctx->sm_count * 4, 256, 0, st>>>(l->d_st, V, wp, lv);
            ctx->launches++;
        }
        LTRY(cudaGetLastError());
    }
    build_walk_tables(l);
    LTRY(cudaMalloc(&l->d_wt, l->wt_blob.size()));
    LTRY(cudaMemcpyAsync(l->d_wt, l->wt_blob.data(), l->wt_blob.size(), cudaMemcpyHostToDevice, st));
    l->wt_host = walk_view(l, l->wt_blob.data());
    if (e == cudaSuccess) l->wt_dev = walk_view(l, l->d_wt);
    LTRY(cudaStreamSynchronize(st));
#undef LTRY
    if (e != cudaSuccess) {
        hgt_locus_free(l);
        return HGT_ERR_CUDA;
    }
    *out = l;
    return HGT_OK;
}

// ================================================================================================================
// Kernels
// ================================================================================================================
namespace {

constexpr int WARPS_PER_CTA = 8;

__device__ __forceinline__ int lower_bound_dev(const int32_t *a, int n, int key) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (a[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// ---- haplotype -> allele bitset (add_count, core:626-677; set form in SURVEY.md appendix A.5) ----------------
// warp per haplotype; lane l owns words l, l+32, ... of the row (WPL words per lane).
// Allele set of one haplotype (left, right, sorted variant rows rw[0..k1)) under table mask `mask` (already offset by the
// lane): lane l holds words l, l+32, ... in set[].
// Bounds of a haplotype by position: variant rows [lo, hi) lie inside [left, right], deletions [dlo, dhi) of the
// right-end order end inside it.  Two table look-ups each (lb_var / lb_del, L + 2 entries, L1/L2-resident) instead of
// binary searches.
struct HapBounds {
    int lo, hi, dlo, dhi;
};
__device__ __forceinline__ HapBounds hap_bounds(const LocusDev &loc, int left, int right) {
    const int xmax = loc.L + 1;
    const int xl = min(max(left, 0), xmax), xr = min(max(right + 1, 0), xmax);
    HapBounds b;
    b.lo = loc.lb_var[xl];
    b.hi = loc.lb_var[xr];
    b.dlo = b.dhi = 0;
    if (loc.n_delr > 0) {
        b.dlo = loc.lb_del[xl];
        b.dhi = loc.lb_del[xr];
    }
    return b;
}

// Lane l tests deletion d0 + l of the right-end order ([d0, dhi) end inside the haplotype): does it start left of the
// haplotype without being one of its own rows?  Returns the ballot; `row` = the lane's candidate.
template <class RowFn>
__device__ __forceinline__ unsigned del_rows_left_of(const LocusDev &loc, int d0, int dhi, int left, RowFn ROW, int k1, int lane,
                                                     int &row) {
    const int dd = d0 + lane;
    bool q = false;
    row = 0;
    if (dd < dhi) {
        row = loc.delr_row[dd];
        q = loc.var_pos[row] < left;
    }
    if (__any_sync(0xffffffffu, q))
        for (int k = 0; k < k1; k++) q &= ROW(k) != row;
    return __ballot_sync(0xffffffffu, q);
}

// Set algebra of one haplotype.  ROW(k) yields its k-th sorted variant row (k < k1).
template <int WPL, class RowFn>
__device__ __forceinline__ void hap_allele_set_core(const LocusDev &loc, int left, const HapBounds &hb, RowFn ROW, int k1,
                                                    const uint64_t *__restrict__ mask, int lane, uint64_t (&set)[WPL]) {
    const int wp = loc.wp;
    const size_t lvl = (size_t)max(loc.V, 1) * wp;
    const int lo = hb.lo, hi = hb.hi;
    uint64_t neg[WPL];
#pragma unroll
    for (int i = 0; i < WPL; i++) {
        set[i] = lane + 32 * i < wp ? mask[32 * i] : 0ull;
        neg[i] = 0ull;
    }
    // positives, and the negatives with the left end inside [left, right]: rows [lo, hi) minus the haplotype's own
    // rows, every gap as the OR of two sparse-table rows
    int prev = lo;
    for (int k = 0; k <= k1; k++) {
        int endr = hi;
        if (k < k1) {
            endr = ROW(k);
            const uint64_t *row = loc.st + (size_t)endr * wp + lane;
#pragma unroll
            for (int i = 0; i < WPL; i++)
                if (lane + 32 * i < wp) set[i] &= row[32 * i];
            if (endr < lo) continue;
            if (endr > hi) endr = hi;
        }
        if (endr > prev && prev < hi) {
            const int n = endr - prev;
            const int lv = 31 - __clz(n);
            const uint64_t *ra = loc.st + lv * lvl + (size_t)prev * wp + lane;
            const uint64_t *rb = loc.st + lv * lvl + (size_t)(endr - (1 << lv)) * wp + lane;
#pragma unroll
            for (int i = 0; i < WPL; i++)
                if (lane + 32 * i < wp) neg[i] |= ra[32 * i] | rb[32 * i];
        }
        prev = max(prev, endr + 1);
    }
    // deletions that start left of the haplotype and end inside it: the candidates (right end inside) are tested 32 at a
    // time, one per lane - a read spans a dozen of them and hardly any qualifies
    for (int d0 = hb.dlo; d0 < hb.dhi; d0 += 32) {
        int row = 0;
        unsigned qm = del_rows_left_of(loc, d0, hb.dhi, left, ROW, k1, lane, row);
        while (qm) {
            const int src = __ffs((int)qm) - 1;
            qm &= qm - 1;
            const uint64_t *rp = loc.st + (size_t)__shfl_sync(0xffffffffu, row, src) * wp + lane;
#pragma unroll
            for (int i = 0; i < WPL; i++)
                if (lane + 32 * i < wp) neg[i] |= rp[32 * i];
        }
    }
#pragma unroll
    for (int i = 0; i < WPL; i++) set[i] &= ~neg[i];
}

template <int WPL>
__device__ __forceinline__ void hap_allele_set(const LocusDev &loc, int left, int right, const int32_t *__restrict__ rw, int k1,
                                               const uint64_t *__restrict__ mask, int lane, uint64_t (&set)[WPL]) {
    const HapBounds hb = hap_bounds(loc, left, right);
    hap_allele_set_core<WPL>(loc, left, hb, [rw](int k) { return rw[k]; }, k1, mask, lane, set);
}

// warp per haplotype -> hapbits (read by class_kernel)
template <int WPL>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32)
    compat_kernel(LocusDev loc, const int32_t *__restrict__ hap_table, const int32_t *__restrict__ hap_left,
                  const int32_t *__restrict__ hap_right,
                  const int64_t *__restrict__ row_off, const int32_t *__restrict__ rows, int64_t n_haps,
                  uint64_t *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int wp = loc.wp;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t h = warp0; h < n_haps; h += nwarps) {
        uint64_t set[WPL];
        hap_allele_set<WPL>(loc, hap_left[h], hap_right[h], rows + row_off[h], (int)(row_off[h + 1] - row_off[h]),
                            loc.mask + (size_t)hap_table[h] * wp + lane, lane, set);
        uint64_t *o = out + (size_t)h * wp + lane;
#pragma unroll
        for (int i = 0; i < WPL; i++)
            if (lane + 32 * i < wp) o[32 * i] = set[i];
    }
}

// ---- per-pair class (add_stat, core:1171-1236) + de-duplication --------------------------------------------
// Classes of every (unit, table) are de-duplicated through one open-addressing hash table per locus batch; the
// rows of table `ut` are allocated contiguously inside a region reserved for it (its number of pairs bounds the
// number of classes), so the EM kernel can stream them without a gather.
struct ClassPool {
    unsigned long long *keys;  // open-addressing table, 0 = empty; else tag (high 36 bits) | id field (POOL_ID_BITS)
    uint32_t cap_mask;
    uint64_t *bits;            // [rows][wp]
    unsigned long long *count; // [rows]
    int32_t *first;            // [rows] first pair index
    const int64_t *ut_base;    // [n_ut] first row of each (unit, table) region
    int32_t *ut_ncls;          // [n_ut] classes created so far
};
// A slot word carries the hash tag of its class AND the class row (absolute row + 1), so a hit costs the CAS round trip
// plus the row compare and nothing in between.  PENDING = the owner has not published the row yet (readers spin on the
// slot word); OVERFLOW = the owner's region was full (readers move on, so an overflow can never hang a kernel).
constexpr int POOL_ID_BITS = 28;
constexpr unsigned long long POOL_ID_MASK = (1ull << POOL_ID_BITS) - 1, POOL_PENDING = POOL_ID_MASK,
                             POOL_OVERFLOW = POOL_ID_MASK - 1;
constexpr int64_t POOL_MAX_ROWS = (int64_t)POOL_ID_MASK - 2;

__device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
    return x;
}

// Insert in two halves: the CAS on the home slot, then the probe that resolves it (pool_insert runs both back to back).
struct PoolProbe {
    unsigned long long tag, prev;  // prev: what lane 0's CAS found in the first slot
    uint32_t slot;
};
template <int WPL>
__device__ __forceinline__ void pool_probe_issue(const ClassPool &pool, int wp, int ut, const uint64_t (&best)[WPL], int lane,
                                                 PoolProbe &pp) {
    // multilinear hash of the row: per 32-bit half an odd key derived from its position, 32 x 32 -> 64-bit multiply-adds
    // (two IMAD.WIDE per word instead of a 64-bit mixer); the warp sum is mixed once below.  Equal tags are always
    // confirmed by comparing the rows, so the hash only has to spread.
    uint64_t hsh = 0;
#pragma unroll
    for (int i = 0; i < WPL; i++) {
        const uint32_t j = (uint32_t)(lane + 32 * i);
        if ((int)j < wp) {
            const uint32_t k1 = (2u * j + 1u) * 0x9E3779B1u | 1u, k2 = (2u * j + 2u) * 0x85EBCA77u | 1u;
            hsh += (uint64_t)(uint32_t)best[i] * k1 + (uint64_t)(uint32_t)(best[i] >> 32) * k2;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) hsh += __shfl_xor_sync(0xffffffffu, hsh, o);
    const unsigned long long h = mix64(hsh + 0x632be59bd9b4e019ULL * (uint64_t)(ut + 1));
    pp.tag = (h | (1ull << POOL_ID_BITS)) & ~POOL_ID_MASK;
    pp.slot = (uint32_t)(h >> 31) & pool.cap_mask;
    pp.prev = 0;
    if (lane == 0) pp.prev = atomicCAS(&pool.keys[pp.slot], 0ull, pp.tag | POOL_PENDING);
}
// Second half: adds `add` to the class's count and lowers its first index.  [base, limit) = rows of table `ut`.
template <int WPL>
__device__ __forceinline__ void pool_probe_resolve(const ClassPool &pool, int wp, int ut, int64_t base, int64_t limit,
                                                   const uint64_t (&best)[WPL], unsigned long long add, int first, int lane,
                                                   const PoolProbe &pp) {
    uint32_t slot = pp.slot;
    unsigned long long prev = __shfl_sync(0xffffffffu, pp.prev, 0);
    int64_t cid = -1;
    while (true) {
        if (prev == 0ull) {  // we own the slot: publish a new class row
            int c = 0;
            if (lane == 0) c = atomicAdd(&pool.ut_ncls[ut], 1);
            c = __shfl_sync(0xffffffffu, c, 0);
            cid = base + c;
            if (cid < limit) {
#pragma unroll
                for (int i = 0; i < WPL; i++) {
                    const int j = lane + 32 * i;
                    if (j < wp) pool.bits[(size_t)cid * wp + j] = best[i];
                }
                __threadfence();
                __syncwarp();
                if (lane == 0) atomicExch(&pool.keys[slot], pp.tag | (unsigned long long)(cid + 1));
            } else {  // region full (cannot happen while regions are sized by the pair bound): readers see it and move on
                if (lane == 0) atomicExch(&pool.keys[slot], pp.tag | POOL_OVERFLOW);
                cid = -1;
            }
            break;
        }
        if ((prev & ~POOL_ID_MASK) == pp.tag) {
            unsigned long long idf = prev & POOL_ID_MASK;
            if (idf == POOL_PENDING) {
                if (lane == 0) {
                    while (((prev = *((volatile unsigned long long *)&pool.keys[slot])) & POOL_ID_MASK) == POOL_PENDING) {
                    }
                    __threadfence();
                }
                idf = __shfl_sync(0xffffffffu, prev, 0) & POOL_ID_MASK;
            }
            // the slot holds a published (fully written) row; it is ours iff it lies in our table's region and carries
            // the same bits
            const int64_t c = (int64_t)idf - 1;
            bool same = idf != POOL_OVERFLOW && c >= base && c < limit;
            if (same) {
#pragma unroll
                for (int i = 0; i < WPL; i++) {
                    const int j = lane + 32 * i;
                    if (j < wp) same &= (__ldcg(&pool.bits[(size_t)c * wp + j]) == best[i]);
                }
            }
            if (__all_sync(0xffffffffu, same)) {
                cid = c;
                break;
            }
        }
        slot = (slot + 1) & pool.cap_mask;
        prev = 0;
        if (lane == 0) prev = atomicCAS(&pool.keys[slot], 0ull, pp.tag | POOL_PENDING);
        prev = __shfl_sync(0xffffffffu, prev, 0);
    }
    if (lane == 0 && cid >= 0) {
        atomicAdd(&pool.count[cid], add);
        atomicMin(&pool.first[cid], first);
    }
}

// Insert bitset `best` (WPL words per lane) into table `ut`; adds `add` to its count and lowers its first index.
template <int WPL>
__device__ __forceinline__ void pool_insert(const ClassPool &pool, int wp, int ut, const uint64_t (&best)[WPL],
                                            unsigned long long add, int first, int lane) {
    PoolProbe pp;
    pool_probe_issue<WPL>(pool, wp, ut, best, lane, pp);
    pool_probe_resolve<WPL>(pool, wp, ut, pool.ut_base[ut], pool.ut_base[ut + 1], best, add, first, lane, pp);
}

// ---- class rows in the reference's dict order ------------------------------------------------------------------------
// pool_insert hands out the rows of a (unit, table) region in warp-scheduling order.  The EM accumulates per allele over
// the class rows in row order, so that order decides the floating-point association - and with it the outcome of EXACT ties
// (two alleles at 0.5 / 0.5 in the reference).  The reference walks its Gene_cmpt dict in insertion order = order of the
// first pair of each class, which is `first`: one CTA per region ranks the rows by `first` (unique inside a region) and
// moves bits / count / first accordingly, through a scratch copy of ONE table's rows (two parallel passes, warp per row,
// 16-byte words).  Only the tables an EM runs on are ordered.  Regions above CLASS_SORT_MAX classes (one oversized locus;
// its EM shards the rows over CTAs anyway) keep the insertion order.
constexpr int CLASS_SORT_MAX = 8192, CLASS_SORT_THREADS = 512;
struct SortScratch {
    uint64_t *bits;            // [rows of one table][wp]
    unsigned long long *count;
    int32_t *first;
    int n_active;              // regions per unit with room (4 on the hla path, 1 otherwise): scratch row = ut_base[unit * 4] / n_active
};
__global__ void __launch_bounds__(CLASS_SORT_THREADS) class_sort_kernel(ClassPool pool, SortScratch scr, int wp, int table) {
    extern __shared__ int32_t s_sort[];  // first[C], rank[C]
    __shared__ int s_flag;
    const int ut = blockIdx.x * 4 + table, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = CLASS_SORT_THREADS / 32;
    const int64_t base = pool.ut_base[ut], cap = pool.ut_base[ut + 1] - base;
    const int C = (int)min((int64_t)pool.ut_ncls[ut], cap);
    if (C <= 1 || C > CLASS_SORT_MAX) return;
    int32_t *fs = s_sort, *rk = s_sort + C;
    for (int r = tid; r < C; r += CLASS_SORT_THREADS) fs[r] = pool.first[base + r];
    if (tid == 0) s_flag = 0;
    __syncthreads();
    bool moved = false;
    for (int r = tid; r < C; r += CLASS_SORT_THREADS) {
        const int32_t f = fs[r];
        int n = 0;
        for (int q = 0; q < C; q++) n += fs[q] < f;
        rk[r] = n;
        moved |= n != r;
    }
    if (moved) s_flag = 1;
    __syncthreads();
    if (!s_flag) return;
    uint64_t *bits = pool.bits + (size_t)base * wp;
    unsigned long long *cnt = pool.count + base;
    int32_t *first = pool.first + base;
    const int64_t s0 = pool.ut_base[blockIdx.x * 4] / scr.n_active;
    uint64_t *sb = scr.bits + (size_t)s0 * wp;
    unsigned long long *sc = scr.count + s0;
    int32_t *sf = scr.first + s0;
    for (int r = warp; r < C; r += NW) {
        const ulonglong2 *src = reinterpret_cast<const ulonglong2 *>(bits + (size_t)r * wp);
        ulonglong2 *dst = reinterpret_cast<ulonglong2 *>(sb + (size_t)rk[r] * wp);
        for (int j = lane; j < wp / 2; j += 32) dst[j] = src[j];
    }
    for (int r = tid; r < C; r += CLASS_SORT_THREADS) {
        sc[rk[r]] = cnt[r];
        sf[rk[r]] = first[r];
    }
    __syncthreads();
    {
        const ulonglong2 *src = reinterpret_cast<const ulonglong2 *>(sb);
        ulonglong2 *dst = reinterpret_cast<ulonglong2 *>(bits);
        const int64_t n2 = (int64_t)C * wp / 2;
        for (int64_t i = tid; i < n2; i += CLASS_SORT_THREADS) dst[i] = src[i];
    }
    for (int r = tid; r < C; r += CLASS_SORT_THREADS) {
        cnt[r] = sc[r];
        first[r] = sf[r];
    }
}

// warp per job; a job = (unit, table, pair) with a list of haplotype bitsets; P bit-planes count up to 2^P-1
template <int WPL, int P>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, (WPL <= 4 && P <= 3) ? 5 : 1)
    class_kernel(int wp, const uint64_t *__restrict__ masks, const int64_t *__restrict__ job_off,
                 const int32_t *__restrict__ job_ut, const int32_t *__restrict__ job_pair,
                 const int32_t *__restrict__ job_list, int64_t n_jobs, const uint64_t *__restrict__ hapbits,
                 ClassPool pool) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t q = warp0; q < n_jobs; q += nwarps) {
        const int job = job_list[q];
        const int64_t h0 = job_off[job], h1 = job_off[job + 1];
        const int ut = job_ut[job];
        const uint64_t *mask = masks + (size_t)(ut & 3) * wp;
        uint64_t plane[P][WPL], best[WPL];
#pragma unroll
        for (int p = 0; p < P; p++)
#pragma unroll
            for (int i = 0; i < WPL; i++) plane[p][i] = 0ull;
        for (int64_t h = h0; h < h1; h++) {
#pragma unroll
            for (int i = 0; i < WPL; i++) {
                const int j = lane + 32 * i;
                uint64_t carry = j < wp ? hapbits[(size_t)h * wp + j] : 0ull;
#pragma unroll
                for (int p = 0; p < P; p++) {
                    const uint64_t t = plane[p][i] & carry;
                    plane[p][i] ^= carry;
                    carry = t;
                }
            }
        }
#pragma unroll
        for (int i = 0; i < WPL; i++) {
            const int j = lane + 32 * i;
            best[i] = j < wp ? mask[j] : 0ull;
        }
#pragma unroll
        for (int p = P - 1; p >= 0; p--) {
            uint64_t any = 0;
#pragma unroll
            for (int i = 0; i < WPL; i++) any |= best[i] & plane[p][i];
            if (__any_sync(0xffffffffu, any != 0ull)) {
#pragma unroll
                for (int i = 0; i < WPL; i++) best[i] &= plane[p][i];
            }
        }
        pool_insert<WPL>(pool, wp, ut, best, 1ull, job_pair[job], lane);
    }
}

// Projection of the Gene table onto a kept allele set (core:1753-1766): every class of table src_ut is ANDed with
// the unit's keep mask and inserted (count added, first index lowered) into table dst_ut; empty results vanish.
template <int WPL>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32)
    project_kernel(int wp, int n_units, const int32_t *__restrict__ unit_list, const uint64_t *__restrict__ keep,
                   ClassPool pool) {
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    for (int ui = blockIdx.y; ui < n_units; ui += gridDim.y) {
        const int u = unit_list[ui];
        const int src = u * 4 + 0, dst = u * 4 + 3;
        const int n = min(__ldcg(&pool.ut_ncls[src]), (int)(pool.ut_base[src + 1] - pool.ut_base[src]));
        const int64_t base = pool.ut_base[src];
        for (int k = blockIdx.x * WARPS_PER_CTA + warp; k < n; k += gridDim.x * WARPS_PER_CTA) {
            uint64_t row[WPL];
            uint64_t any = 0;
#pragma unroll
            for (int i = 0; i < WPL; i++) {
                const int j = lane + 32 * i;
                row[i] = j < wp ? (pool.bits[(size_t)(base + k) * wp + j] & keep[(size_t)ui * wp + j]) : 0ull;
                any |= row[i];
            }
            if (!__any_sync(0xffffffffu, any != 0ull)) continue;
            pool_insert<WPL>(pool, wp, dst, row, pool.count[base + k], pool.first[base + k], lane);
        }
    }
}

// Read-sharded locus: adopt the gathered class rows this rank owns (owner = row hash mod world) into a fresh one-region
// pool; equal rows of different shards merge (counts add, first index = the smallest).  Warp per input row.
template <int WPL>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32)
    class_merge_kernel(int wp, const uint64_t *__restrict__ rows_in, const unsigned long long *__restrict__ count_in,
                       const int32_t *__restrict__ first_in, int64_t n_in, int rank, int world, ClassPool pool) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t k = warp0; k < n_in; k += nwarps) {
        uint64_t row[WPL];
#pragma unroll
        for (int i = 0; i < WPL; i++) {
            const int j = lane + 32 * i;
            row[i] = j < wp ? rows_in[(size_t)k * wp + j] : 0ull;
        }
        PoolProbe pp;
        // (the owner is taken from the tag, not from the slot: the slot depends on the table size)
        uint64_t hsh = 0;
#pragma unroll
        for (int i = 0; i < WPL; i++) {
            const uint32_t j = (uint32_t)(lane + 32 * i);
            if ((int)j < wp) hsh += mix64(row[i] ^ (0x9e3779b97f4a7c15ULL * (uint64_t)(j + 1)));
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) hsh += __shfl_xor_sync(0xffffffffu, hsh, o);
        if ((int)(mix64(hsh) % (uint64_t)world) != rank) continue;
        pool_probe_issue<WPL>(pool, wp, 0, row, lane, pp);
        pool_probe_resolve<WPL>(pool, wp, 0, pool.ut_base[0], pool.ut_base[1], row, count_in[k], first_in[k], lane, pp);
    }
}

// Gene_counts (core:1187-1190) of table (unit, 0): counts[a] = sum of class counts over classes holding a;
// first[a] = first pair whose class holds a.  grid = (allele tiles, units, class chunks): a CTA folds one chunk of
// `chunk` classes into the totals with integer atomics (order-independent, so still exact).
constexpr int COUNT_CHUNK_MIN = 128, COUNT_CHUNK_MAX = 512;  // classes per CTA: chosen per launch from the pair bound
constexpr int COUNT_THREADS = 256;  // alleles per CTA = 4 words of every class row
constexpr int COUNT_TILE = 64;      // class rows staged in shared memory at a time
__global__ void __launch_bounds__(COUNT_THREADS)
    table_counts_kernel(int A, int wp, int table, int chunk, ClassPool pool, unsigned long long *__restrict__ a_count,
                        int32_t *__restrict__ a_first) {
    // The 32-byte segment [4 words] of COUNT_TILE rows goes to shared memory with one load per thread (a full sector per
    // row); every thread then scans the tile for its own allele out of shared memory, so the serial chain per thread is
    // chunk / COUNT_TILE global round trips instead of chunk.
    __shared__ uint64_t s_bits[COUNT_TILE][COUNT_THREADS / 64];
    __shared__ unsigned long long s_cnt[COUNT_TILE];
    __shared__ unsigned long long s_nz[COUNT_THREADS / 64];  // per word column: the tile rows whose word is non-zero
    __shared__ int32_t s_first[COUNT_TILE];
    const int u = blockIdx.y;
    const int ut = u * 4 + table;
    const int t = threadIdx.x;
    const int a = blockIdx.x * COUNT_THREADS + t;
    const int word0 = blockIdx.x * (COUNT_THREADS / 64);
    const int64_t base = pool.ut_base[ut];
    const int n = min(pool.ut_ncls[ut], (int)(pool.ut_base[ut + 1] - base));
    const int k0 = blockIdx.z * chunk, k1 = min(n, k0 + chunk);
    if (k0 >= k1) return;
    unsigned long long c = 0;
    int32_t f = 0x7fffffff;
    const int lr = t >> 2, lw = t & 3;  // this thread's (row, word) of a tile load
    const int my_word = t >> 6, my_bit = t & 63;
    for (int kt = k0; kt < k1; kt += COUNT_TILE) {
        const int nr = min(COUNT_TILE, k1 - kt);
        uint64_t v = 0ull;
        if (lr < nr && word0 + lw < wp) v = pool.bits[(size_t)(base + kt + lr) * wp + word0 + lw];
        __syncthreads();  // the previous tile has been consumed
        if (t < COUNT_THREADS / 64) s_nz[t] = 0ull;
        __syncthreads();
        s_bits[lr][lw] = v;
        if (v != 0ull) atomicOr(&s_nz[lw], 1ull << lr);
        if (t < nr) {
            s_cnt[t] = pool.count[base + kt + t];
            s_first[t] = pool.first[base + kt + t];
        }
        __syncthreads();
        // only the rows whose word of this thread's column is non-zero (the same rows for the 64 threads of a column)
        unsigned long long m = s_nz[my_word];
        while (m) {
            const int r = __ffsll((long long)m) - 1;
            m &= m - 1;
            if ((s_bits[r][my_word] >> my_bit) & 1ull) {
                c += s_cnt[r];
                f = min(f, s_first[r]);
            }
        }
    }
    if (c && a < A) {
        atomicAdd(&a_count[(size_t)u * A + a], c);
        atomicMin(&a_first[(size_t)u * A + a], f);
    }
}

// ---- EM result as a key list ------------------------------------------------------------------------------------------
// After select_alleles a result has a handful of keys out of thousands of alleles, so finish() fetches (allele, first
// key, probability) triples instead of three dense arrays: one CTA per unit compacts in_result in ascending allele order
// (ballot + running base, no atomics, so the list order is fixed).  n_out receives the true count; a unit with more than
// `cap` keys makes the host fall back to the dense copies.
struct KeyOut {
    int32_t allele, fk;
    double prob;
};
constexpr int KEY_CAP = 256;
constexpr int KEY_THREADS = 256;
__global__ void __launch_bounds__(KEY_THREADS)
    result_keys_kernel(int A, const double *__restrict__ prob, const uint8_t *__restrict__ inres,
                       const int32_t *__restrict__ fk, const int32_t *__restrict__ iters_status, int cap,
                       KeyOut *__restrict__ out, int32_t *__restrict__ n_out) {
    __shared__ int s_warp[KEY_THREADS / 32];
    __shared__ int s_base;
    const int u = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (iters_status[(size_t)u * 3 + 1] != HGT_OK) {  // EM failed or did not run: nothing to list
        if (t == 0) n_out[u] = 0;
        return;
    }
    if (t == 0) s_base = 0;
    __syncthreads();
    const size_t o = (size_t)u * A;
    for (int a0 = 0; a0 < A; a0 += KEY_THREADS) {
        const int a = a0 + t;
        const bool k = a < A && inres[o + a];
        const unsigned m = __ballot_sync(0xffffffffu, k);
        if (lane == 0) s_warp[warp] = __popc(m);
        __syncthreads();
        int before = s_base;
        for (int w = 0; w < warp; w++) before += s_warp[w];
        const int pos = before + __popc(m & ((1u << lane) - 1u));
        if (k && pos < cap) {
            KeyOut e;
            e.allele = a; e.fk = fk[o + a]; e.prob = prob[o + a];
            out[(size_t)u * cap + pos] = e;
        }
        __syncthreads();
        if (t == 0) {
            int n = 0;
            for (int w = 0; w < KEY_THREADS / 32; w++) n += s_warp[w];
            s_base += n;
        }
        __syncthreads();
    }
    if (t == 0) n_out[u] = s_base;
}

// pileup-derived per-position flags the host walk needs: nt_set mask and the hla deletion-artefact flag
// (core:1064-1077: del_count * 6 < nt_count)
__global__ void pileup_flags_kernel(const uint32_t *__restrict__ counts, int64_t n_pos, uint8_t *__restrict__ mask,
                                    uint8_t *__restrict__ del_artefact) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n_pos) return;
    const uint32_t *c = counts + (size_t)i * 6;
    const uint32_t depth = c[0] + c[1] + c[2] + c[3] + c[4] + c[5];
    uint8_t m = 0;
    if (depth >= 20) {
        const double thr = (double)depth * 0.2;  // same IEEE product as Python's num_nt * 0.2
        for (int k = 0; k < 4; k++)
            if ((double)c[k] >= thr || c[k] >= 7) m |= (uint8_t)(1u << k);
    }
    mask[i] = m;
    const uint64_t dels = c[5], nts = (uint64_t)c[0] + c[1] + c[2] + c[3] + c[4];
    del_artefact[i] = dels * 6 < nts ? 1 : 0;
}

}  // namespace

// ================================================================================================================
// Device buffers
// ================================================================================================================
static thread_local hgt_ctx *g_acct = nullptr;  // context of the running entry point: owns the pool and the byte counters

// Device / page-locked host buffers drawn from the context's caching allocator (MemPool, common.cuh).
template <bool PINNED>
struct PoolBuf {
    void *p = nullptr;
    size_t bytes = 0, cap = 0;
    hgt_ctx *owner = nullptr;
    int alloc(size_t n) {
        if (p && cap >= n) {
            bytes = n;
            return HGT_OK;
        }
        release();
        owner = g_acct;
        if (!owner) {
            hgt_set_error("internal: buffer allocation outside an entry point");
            return HGT_ERR_ARG;
        }
        HGT_CHECK(owner->pool.get(PINNED, n ? n : 16, &p, &cap));
        bytes = n;
        return HGT_OK;
    }
    void release() {
        if (p && owner) owner->pool.put(PINNED, p, cap);
        p = nullptr;
        bytes = cap = 0;
    }
    template <class T>
    T *as() const { return static_cast<T *>(p); }
};
using DevBuf = PoolBuf<false>;
using PinBuf = PoolBuf<true>;

  // context whose byte counters the copies below feed

template <class T>
static int upload(DevBuf *b, const std::vector<T> &v, cudaStream_t st) {
    HGT_CHECK(b->alloc(v.size() * sizeof(T)));
    if (g_acct) g_acct->h2d_bytes += (int64_t)(v.size() * sizeof(T));
    if (!v.empty()) HGT_CUDA(cudaMemcpyAsync(b->p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, st));
    return HGT_OK;
}

static inline cudaError_t d2h(void *dst, const void *src, size_t n, cudaStream_t st) {
    if (g_acct) g_acct->d2h_bytes += (int64_t)n;
    return cudaMemcpyAsync(dst, src, n, cudaMemcpyDeviceToHost, st);
}

struct StageTimer {  // CUDA-event bracket of one GPU stage, accumulated into ctx->stage_ms at resolve()
    struct Span { int stage; cudaEvent_t a, b; };
    std::vector<Span> spans;
    hgt_ctx *ctx = nullptr;
    cudaStream_t st = nullptr;
    cudaEvent_t open_ev = nullptr;
    int open_stage = -1;
    void begin(hgt_ctx *c, cudaStream_t s, int stage) {
        if (!c->profile) return;
        ctx = c; st = s; open_stage = stage;
        cudaEventCreate(&open_ev);
        cudaEventRecord(open_ev, st);
    }
    void end(int n_launches) {
        if (open_stage < 0) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, st);
        spans.push_back({open_stage, open_ev, e});
        ctx->stage_launches[open_stage] += n_launches;
        open_stage = -1;
    }
    void resolve() {  // call after the stream has been synchronised
        for (Span &s : spans) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, s.a, s.b) == cudaSuccess) ctx->stage_ms[s.stage] += ms;
            cudaEventDestroy(s.a);
            cudaEventDestroy(s.b);
        }
        spans.clear();
    }
};

static int wpl_of(int wp) {
    const int w = (wp + 31) / 32;
    return w <= 1 ? 1 : w <= 2 ? 2 : w <= 4 ? 4 : 8;
}

// ================================================================================================================
// Batch of (sample, locus) units
// ================================================================================================================
// A unit is one (sample, locus).  Its alignment text goes to the device as it is (one arena per batch, units of one
// locus adjacent); everything from the line index to the ranked alleles happens there.
struct UnitHost {
    int locus = 0;
    const char *sam = nullptr;
    size_t n_bytes = 0;             // text bytes (a BAM unit: its rendered text, known after the length pass of prepare)
    const void *blob = nullptr;     // BAM unit: packed records (bam_dev.cuh), rendered into the arena by prepare
    size_t blob_bytes = 0;
    const hgt_bam_dsplit *ds = nullptr;  // device-split unit: a bucket in HBM (n_bytes known), rendered by prepare
    hgtk::DsplitUnitDev dsu{};
    int64_t n_records = 0;
    int local = 0;  // index inside its locus batch
    int arena = 0;  // index in arena order (loci-major, add order inside a locus)
    int64_t num_reads = 0, num_pairs = 0;
    std::vector<uint32_t> counts;  // kept only when requested (single-unit API / tests)
    std::vector<uint8_t> nt_mask;
    int64_t pos0 = 0;              // first position of the unit in the batch-wide pileup arrays
};

// Device state of the record stage (reads.cuh / walk_dev.cuh): text arena, line index, per-line records, haplotypes.
struct ReadsDev {
    int64_t text_bytes = 0, n_chunks = 0, n_lines = 0, POS = 0;
    int32_t n_slow = 0, max_job_haps = 0;
    std::vector<int> unit_of_arena;
    std::vector<int32_t> locus_unit0;  // [n_loci + 1] first arena index of every locus
    std::vector<int64_t> unit_off;     // [nu + 1] byte offsets in the arena (arena order)
    DevBuf d_text, d_chunk, d_line_off, d_unit, d_rec, d_st, d_hdr, d_hids, d_slow, d_slow_list, d_units, d_loci, d_small,
        d_scan, d_partial, d_jobs_desc, d_cnt, d_mf;
    PinBuf h_units, h_small, h_stage, h_loci, h_jobs_desc;
    DevBuf d_blob, d_blen, d_bunits;  // BAM units: blob arena, per-record text offsets, unit descriptors (prepare only)
    PinBuf h_bstage, h_bunits;
    DevBuf d_dunits;  // device-split units: descriptors (prepare only)
    PinBuf h_dunits;
    size_t o_uoff = 0, o_uline0 = 0, o_upos0 = 0, o_ulocus = 0, o_ulocal = 0, o_lu0 = 0, units_bytes = 0;
    size_t s_reads = 0, s_pairs = 0, s_totals = 0, small_bytes = 0;  // offsets inside the small result block
    void release() {
        DevBuf *all[] = {&d_text, &d_chunk, &d_line_off, &d_unit, &d_rec, &d_st, &d_hdr, &d_hids, &d_slow, &d_slow_list,
                         &d_units, &d_loci, &d_small, &d_scan, &d_partial, &d_jobs_desc, &d_cnt, &d_mf};
        for (DevBuf *x : all) x->release();
        PinBuf *pins[] = {&h_units, &h_small, &h_stage, &h_loci, &h_jobs_desc};
        for (PinBuf *x : pins) x->release();
        release_bam();
    }
    void release_bam() {
        d_blob.release(); d_blen.release(); d_bunits.release(); d_dunits.release();
        h_bstage.release(); h_bunits.release(); h_dunits.release();
    }
};

struct LocusBatch {
    hgt_locus *loc = nullptr;
    std::vector<int> units;  // global unit ids
    // jobs of all units and tables of this locus: one arena, identical layout in page-locked host memory (filled by
    // the host threads in parallel) and on the device (one copy): job_off | row_off | ut_base | job_ut | job_pair |
    // job_list (<= 7 haplotypes first, then the rest) | hap_left | hap_right | hap_table | rows
    struct JobArena {
        size_t o_job_off = 0, o_row_off = 0, o_ut_base = 0, o_job_ut = 0, o_job_pair = 0, o_job_list = 0, o_hl = 0, o_hr = 0,
               o_ht = 0, o_rows = 0, bytes = 0;
    } ja;
    int64_t n_jobs = 0, n_small = 0, n_big = 0, n_haps = 0, n_rows = 0, max_job_haps = 0;
    std::vector<int64_t> ut_base;  // [n_units*4 + 1]
    int64_t n_rows_pool = 0;
    PinBuf h_jobs;
    DevBuf d_jobs, d_hapbits;
    template <class T>
    T *dj(size_t off) const { return reinterpret_cast<T *>(static_cast<unsigned char *>(d_jobs.p) + off); }
    template <class T>
    T *hj(size_t off) const { return reinterpret_cast<T *>(static_cast<unsigned char *>(h_jobs.p) + off); }
    DevBuf d_keys, d_bits, d_count, d_first, d_ut_ncls, d_sortbits, d_sortcnt, d_sortfirst;
    DevBuf d_prob, d_inres, d_fk, d_is, d_emws;      // EM over exon (hla) / gene (other) tables
    DevBuf d_prob2, d_inres2, d_fk2, d_is2, d_keep, d_ulist;  // second-level EM (hla)
    DevBuf d_acount, d_afirst;
    DevBuf d_ck[2], d_cn[2];  // EM results as key lists (result_keys_kernel), first / second level
    PinBuf h_ck[2], h_cn[2];
    bool dense[2] = {true, true};  // the dense host arrays prob/inres/fk (prob2/...) hold this level's result
    std::deque<DevBuf> d_coopws;  // whole-GPU EM workspaces of oversized problems (allocated when class counts are known)
    uint32_t cap = 0;
    int n_live[4] = {0, 0, 0, 0};  // alleles that can be members of a class of table t (popcount of its mask)
    // results on the host (page-locked)
    PinBuf h_ncls, h_prob, h_inres, h_fk, h_is, h_prob2, h_inres2, h_fk2, h_is2, h_keep, h_ulist;
    int32_t *ut_ncls = nullptr;
    double *prob = nullptr, *prob2 = nullptr;
    uint8_t *inres = nullptr, *inres2 = nullptr;
    int32_t *fk = nullptr, *fk2 = nullptr, *is = nullptr, *is2 = nullptr;
    std::vector<uint8_t> has2;  // unit ran the second-level EM
    std::vector<int32_t> slot2;      // its slot in the keep-mask / unit list of the second level
    std::vector<double> exon_prob_sum;  // core:1739-1749
    int n_level2 = 0;
    void release() {
        DevBuf *all[] = {&d_jobs, &d_hapbits,
                         &d_keys, &d_bits, &d_count, &d_first, &d_ut_ncls, &d_sortbits, &d_sortcnt, &d_sortfirst, &d_prob, &d_inres, &d_fk,
                         &d_is, &d_emws, &d_prob2, &d_inres2, &d_fk2, &d_is2, &d_keep, &d_ulist,
                         &d_acount, &d_afirst, &d_ck[0], &d_ck[1], &d_cn[0], &d_cn[1]};
        for (DevBuf *b : all) b->release();
        for (DevBuf &b : d_coopws) b.release();
        d_coopws.clear();
        PinBuf *pins[] = {&h_jobs, &h_ncls, &h_prob, &h_inres, &h_fk, &h_is, &h_prob2, &h_inres2, &h_fk2, &h_is2, &h_keep, &h_ulist,
                          &h_ck[0], &h_ck[1], &h_cn[0], &h_cn[1]};
        for (PinBuf *b : pins) b->release();
    }
    ClassPool pool() const {
        ClassPool p;
        p.keys = d_keys.as<unsigned long long>(); p.cap_mask = cap - 1;
        p.bits = d_bits.as<uint64_t>(); p.count = d_count.as<unsigned long long>(); p.first = d_first.as<int32_t>();
        p.ut_base = dj<int64_t>(ja.o_ut_base); p.ut_ncls = d_ut_ncls.as<int32_t>();
        return p;
    }
};

struct hgt_batch {
    hgt_ctx *ctx = nullptr;
    hgt_params params;
    std::vector<hgt_locus *> loci;
    std::vector<UnitHost> units;
    std::vector<LocusBatch> lb;
    ReadsDev rd;
    bool keep_counts = false;
    bool skip_em = false;
    int (*pileup_hook)(void *arg, void *dev_counts, size_t n_u32, void *stream) = nullptr;
    void *pileup_hook_arg = nullptr;
    bool prepared = false, executed = false, finished = false;
    StageTimer timer;
    int remove_low = 1;
    PinBuf h_em_args[2];   // kernel-argument staging of the two EM levels
    DevBuf d_em_args[2];
    // the last hgt_batch_pairs result, complete, for a repeated call (e.g. with a larger cap) on the same tables and names
    struct {
        bool valid = false;
        int32_t table = -1;
        int64_t max_pairs = -1;
        std::vector<std::shared_ptr<NameRel>> names;  // per locus of the batch (held: their device copies stay valid)
        PairResult r;
    } pairs;
    ~hgt_batch() {
        if (ctx) {
            cudaSetDevice(ctx->device);
            cudaDeviceSynchronize();  // pooled blocks go back to the allocator: nothing may still be using them
        }
        for (LocusBatch &b : lb) b.release();
        rd.release();
        for (int i = 0; i < 2; i++) {
            h_em_args[i].release();
            d_em_args[i].release();
        }
    }
};

// Parallel-for over units on host threads (intake and walk are independent per unit).
template <class F>
static void parallel_units(int n_threads, size_t n, F f) {
    if (n_threads <= 1 || n <= 1) {
        for (size_t i = 0; i < n; i++) f(i);
        return;
    }
    std::atomic<size_t> next{0};
    std::vector<std::thread> th;
    const int nt = (int)std::min<size_t>(n_threads, n);
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

static int batch_threads(const hgt_params &p) {
    if (p.n_threads > 0) return p.n_threads;
    const unsigned hc = std::thread::hardware_concurrency();
    return hc ? (int)hc : 1;
}

// ---- stage 1: text to the device, line count ----------------------------------------------------------------------------------
static inline size_t a16(size_t x) { return (x + 15) & ~(size_t)15; }

static int tune_env(const char *name, int dflt) {  // grid-size experiments without a rebuild
    const char *e = getenv(name);
    const int v = e ? atoi(e) : dflt;
    return v > 0 ? v : dflt;
}

int64_t hgt_dev_scan_partials(int64_t n) { return (n + hgtk::SCAN_TILE - 1) / hgtk::SCAN_TILE + 1; }

int hgt_dev_scan(hgt_ctx *ctx, cudaStream_t st, const int64_t *in, int64_t n, int64_t *out, int64_t *partial) {
    if (n <= 0) {
        HGT_CUDA(cudaMemsetAsync(out, 0, 8, st));
        return HGT_OK;
    }
    const int64_t n_part = (n + hgtk::SCAN_TILE - 1) / hgtk::SCAN_TILE;
    hgtk::scan_partials_kernel<<<(unsigned)n_part, hgtk::SCAN_THREADS, 0, st>>>(in, n, partial);
    hgtk::scan_single_kernel<<<1, 1024, 0, st>>>(partial, n_part);
    hgtk::scan_apply_kernel<<<(unsigned)n_part, hgtk::SCAN_THREADS, 0, st>>>(in, n, partial, n_part, out);
    ctx->launches += 3;
    HGT_CUDA(cudaGetLastError());
    return HGT_OK;
}

static int dev_scan(hgt_ctx *ctx, cudaStream_t st, const int64_t *in, int64_t n, int64_t *out, DevBuf *partial) {
    if (n > 0) HGT_CHECK(partial->alloc((size_t)hgt_dev_scan_partials(n) * 8));
    return hgt_dev_scan(ctx, st, in, n, out, partial->as<int64_t>());
}

static bool is_pinned_host(const void *p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeHost;
}


namespace hgtk {
// text offset of every unit's first record (k = 0 .. nb; u[nb].rec0 = n_rec): the per-unit sizes the host lays out with
__global__ void bam_unit_text_kernel(const int64_t *__restrict__ off, const BamUnitDev *__restrict__ u, int nb,
                                     int64_t *__restrict__ out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k <= nb) out[k] = off[u[k].rec0];
}
}  // namespace hgtk

// Length pass of the BAM units (prepare, only when the batch holds one): blobs to the device, text length per record,
// scan, per-unit sizes back to the host (one synchronisation).  Sets n_bytes of every BAM unit.
static int bam_units_measure(hgt_batch *b, std::vector<int> &bam_arena, int64_t *n_rec) {
    hgt_ctx *ctx = b->ctx;
    cudaStream_t st = ctx->stream;
    ReadsDev &rd = b->rd;
    const int nb = (int)bam_arena.size();
    std::vector<int64_t> blob_off((size_t)nb + 1, 0);
    HGT_CHECK(rd.h_bunits.alloc((size_t)(nb + 1) * sizeof(hgtk::BamUnitDev) + (size_t)(nb + 1) * 8));
    hgtk::BamUnitDev *hu = rd.h_bunits.as<hgtk::BamUnitDev>();
    int64_t R = 0;
    bool all_pinned = true;
    for (int k = 0; k < nb; k++) {
        const UnitHost &U = b->units[rd.unit_of_arena[bam_arena[k]]];
        hu[k] = {blob_off[k], R, 0, 0};
        blob_off[k + 1] = blob_off[k] + (int64_t)a16(U.blob_bytes);
        R += U.n_records;
        all_pinned &= is_pinned_host(U.blob);
    }
    hu[nb] = {blob_off[nb], R, 0, 0};
    *n_rec = R;
    HGT_CHECK(rd.d_blob.alloc((size_t)std::max<int64_t>(blob_off[nb], 16)));
    unsigned char *db = rd.d_blob.as<unsigned char>();
    if (all_pinned) {
        for (int k = 0; k < nb; k++) {
            const UnitHost &U = b->units[rd.unit_of_arena[bam_arena[k]]];
            HGT_CUDA(cudaMemcpyAsync(db + blob_off[k], U.blob, U.blob_bytes, cudaMemcpyHostToDevice, st));
            ctx->h2d_bytes += (int64_t)U.blob_bytes;
        }
    } else {  // pageable blobs: host threads assemble the blob arena in page-locked memory, one copy
        HGT_CHECK(rd.h_bstage.alloc((size_t)std::max<int64_t>(blob_off[nb], 16)));
        unsigned char *hs = rd.h_bstage.as<unsigned char>();
        parallel_units(batch_threads(b->params), (size_t)nb, [&](size_t k) {
            const UnitHost &U = b->units[rd.unit_of_arena[bam_arena[k]]];
            memcpy(hs + blob_off[k], U.blob, U.blob_bytes);
        });
        HGT_CUDA(cudaMemcpyAsync(db, hs, (size_t)blob_off[nb], cudaMemcpyHostToDevice, st));
        ctx->h2d_bytes += blob_off[nb];
    }
    const size_t desc = (size_t)(nb + 1) * sizeof(hgtk::BamUnitDev);
    HGT_CHECK(rd.d_bunits.alloc(desc + (size_t)(nb + 1) * 8));
    HGT_CUDA(cudaMemcpyAsync(rd.d_bunits.p, hu, desc, cudaMemcpyHostToDevice, st));
    ctx->h2d_bytes += (int64_t)desc;
    HGT_CHECK(rd.d_blen.alloc((size_t)(R + 1) * 8));
    if (R > 0) {
        hgtk::bam_text_len_kernel<<<(unsigned)((R + hgtk::BAM_THREADS - 1) / hgtk::BAM_THREADS), hgtk::BAM_THREADS, 0, st>>>(
            hgtk::BlobSrc{db, rd.d_bunits.as<hgtk::BamUnitDev>(), nb, nullptr}, R, rd.d_blen.as<int64_t>());
        ctx->launches++;
        HGT_CUDA(cudaGetLastError());
    }
    HGT_CHECK(dev_scan(ctx, st, rd.d_blen.as<int64_t>(), R, rd.d_blen.as<int64_t>(), &rd.d_partial));
    int64_t *d_sz = reinterpret_cast<int64_t *>(static_cast<unsigned char *>(rd.d_bunits.p) + desc);
    hgtk::bam_unit_text_kernel<<<(unsigned)((nb + 1 + 255) / 256), 256, 0, st>>>(rd.d_blen.as<int64_t>(),
                                                                                rd.d_bunits.as<hgtk::BamUnitDev>(), nb, d_sz);
    ctx->launches++;
    HGT_CUDA(cudaGetLastError());
    int64_t *h_sz = reinterpret_cast<int64_t *>(reinterpret_cast<unsigned char *>(hu) + desc);
    HGT_CUDA(d2h(h_sz, d_sz, (size_t)(nb + 1) * 8, st));
    HGT_CUDA(cudaStreamSynchronize(st));
    for (int k = 0; k < nb; k++) b->units[rd.unit_of_arena[bam_arena[k]]].n_bytes = (size_t)(h_sz[k + 1] - h_sz[k]);
    return HGT_OK;
}

// Text arena of a batch with BAM units: '\n' everywhere, text units copied (page-locked directly, pageable staged), BAM
// units rendered into their slices.
static int bam_units_fill(hgt_batch *b, const std::vector<int> &bam_arena, int64_t R) {
    hgt_ctx *ctx = b->ctx;
    cudaStream_t st = ctx->stream;
    ReadsDev &rd = b->rd;
    const size_t nu = b->units.size();
    char *dt = rd.d_text.as<char>();
    HGT_CUDA(cudaMemsetAsync(dt, '\n', (size_t)rd.text_bytes, st));
    std::vector<size_t> stage_off(nu + 1, 0);
    for (size_t a = 0; a < nu; a++) {
        const UnitHost &U = b->units[rd.unit_of_arena[a]];
        const bool text = !U.blob && !U.ds && U.n_bytes;
        const bool staged = text && !is_pinned_host(U.sam);
        stage_off[a + 1] = stage_off[a] + (staged ? a16(U.n_bytes) : 0);
        if (text && !staged) {
            HGT_CUDA(cudaMemcpyAsync(dt + rd.unit_off[a], U.sam, U.n_bytes, cudaMemcpyHostToDevice, st));
            ctx->h2d_bytes += (int64_t)U.n_bytes;
        }
    }
    if (stage_off[nu]) {
        HGT_CHECK(rd.h_stage.alloc(stage_off[nu]));
        char *hs = rd.h_stage.as<char>();
        parallel_units(batch_threads(b->params), nu, [&](size_t a) {
            const UnitHost &U = b->units[rd.unit_of_arena[a]];
            if (stage_off[a + 1] > stage_off[a]) memcpy(hs + stage_off[a], U.sam, U.n_bytes);
        });
        for (size_t a = 0; a < nu; a++) {
            const UnitHost &U = b->units[rd.unit_of_arena[a]];
            if (stage_off[a + 1] == stage_off[a]) continue;
            HGT_CUDA(cudaMemcpyAsync(dt + rd.unit_off[a], hs + stage_off[a], U.n_bytes, cudaMemcpyHostToDevice, st));
            ctx->h2d_bytes += (int64_t)U.n_bytes;
        }
    }
    if (R == 0) return HGT_OK;
    // the descriptors again, now with the arena slices (the length pass synchronised: the staging copy is idle)
    const int nb = (int)bam_arena.size();
    hgtk::BamUnitDev *hu = rd.h_bunits.as<hgtk::BamUnitDev>();
    for (int k = 0; k < nb; k++) hu[k].text_off = rd.unit_off[bam_arena[k]];
    const size_t desc = (size_t)(nb + 1) * sizeof(hgtk::BamUnitDev);
    HGT_CUDA(cudaMemcpyAsync(rd.d_bunits.p, hu, desc, cudaMemcpyHostToDevice, st));
    ctx->h2d_bytes += (int64_t)desc;
    const int64_t warps_per_cta = hgtk::BAM_THREADS / 32;
    hgtk::bam_render_kernel<<<(unsigned)((R + warps_per_cta - 1) / warps_per_cta), hgtk::BAM_THREADS, 0, st>>>(
        hgtk::BlobSrc{rd.d_blob.as<unsigned char>(), rd.d_bunits.as<hgtk::BamUnitDev>(), nb, rd.d_blen.as<int64_t>()}, R, dt);
    ctx->launches++;
    HGT_CUDA(cudaGetLastError());
    return HGT_OK;
}

// Device-split units: every bucket rendered into its arena slice straight from the split's device memory (one launch; the
// sizes were known when the units were added, so there is no length pass and no synchronisation).
static int dsplit_units_render(hgt_batch *b) {
    hgt_ctx *ctx = b->ctx;
    cudaStream_t st = ctx->stream;
    ReadsDev &rd = b->rd;
    std::vector<hgtk::DsplitUnitDev> du;
    int64_t R = 0;
    for (size_t a = 0; a < b->units.size(); a++) {
        const UnitHost &U = b->units[rd.unit_of_arena[a]];
        if (!U.ds) continue;
        hgtk::DsplitUnitDev d = U.dsu;
        d.rec0 = R;
        d.text_off = rd.unit_off[a];
        du.push_back(d);
        R += U.n_records;
    }
    if (R == 0) return HGT_OK;
    const int nd = (int)du.size();
    const size_t bytes = du.size() * sizeof(hgtk::DsplitUnitDev);
    HGT_CHECK(rd.h_dunits.alloc(bytes));
    HGT_CHECK(rd.d_dunits.alloc(bytes));
    memcpy(rd.h_dunits.p, du.data(), bytes);
    HGT_CUDA(cudaMemcpyAsync(rd.d_dunits.p, rd.h_dunits.p, bytes, cudaMemcpyHostToDevice, st));
    ctx->h2d_bytes += (int64_t)bytes;
    const int64_t warps_per_cta = hgtk::BAM_THREADS / 32;
    hgtk::bam_render_kernel<<<(unsigned)((R + warps_per_cta - 1) / warps_per_cta), hgtk::BAM_THREADS, 0, st>>>(
        hgtk::DsplitSrc{rd.d_dunits.as<hgtk::DsplitUnitDev>(), nd}, R, rd.d_text.as<char>());
    ctx->launches++;
    HGT_CUDA(cudaGetLastError());
    return HGT_OK;
}

static int batch_prepare(hgt_batch *b) {
    hgt_ctx *ctx = b->ctx;
    cudaStream_t st = ctx->stream;
    ReadsDev &rd = b->rd;
    const size_t nu = b->units.size();
    b->lb.assign(b->loci.size(), LocusBatch());
    for (size_t l = 0; l < b->loci.size(); l++) b->lb[l].loc = b->loci[l];
    for (size_t u = 0; u < nu; u++) {
        LocusBatch &lb = b->lb[b->units[u].locus];
        b->units[u].local = (int)lb.units.size();
        lb.units.push_back((int)u);
    }
    // arena order: the units of one locus are adjacent, so every per-locus quantity of the pair stage is a difference of
    // two entries of a scan over lines
    rd.unit_of_arena.clear();
    rd.locus_unit0.assign(b->loci.size() + 1, 0);
    for (size_t l = 0; l < b->loci.size(); l++) {
        rd.locus_unit0[l] = (int32_t)rd.unit_of_arena.size();
        for (int u : b->lb[l].units) {
            b->units[u].arena = (int)rd.unit_of_arena.size();
            rd.unit_of_arena.push_back(u);
        }
    }
    rd.locus_unit0[b->loci.size()] = (int32_t)nu;
    std::vector<int> bam_arena;  // arena indices of the BAM units
    for (size_t a = 0; a < nu; a++)
        if (b->units[rd.unit_of_arena[a]].blob) bam_arena.push_back((int)a);
    int64_t n_bam_rec = 0;
    if (!bam_arena.empty()) {
        HostTimer ht(ctx, 0);
        HGT_CHECK(bam_units_measure(b, bam_arena, &n_bam_rec));
    }
    rd.unit_off.assign(nu + 1, 0);
    rd.POS = 0;
    for (size_t a = 0; a < nu; a++) {
        UnitHost &U = b->units[rd.unit_of_arena[a]];
        rd.unit_off[a + 1] = rd.unit_off[a] + (int64_t)a16(U.n_bytes + 1);  // at least one '\n' closes every unit
        U.pos0 = rd.POS;
        rd.POS += b->loci[U.locus]->L;
    }
    rd.text_bytes = rd.unit_off[nu];
    rd.n_lines = 0;
    if (nu == 0) {
        b->prepared = true;
        return HGT_OK;
    }
    {
        HostTimer ht(ctx, 0);
        HGT_CHECK(rd.d_text.alloc((size_t)rd.text_bytes));
        char *dt = rd.d_text.as<char>();
        bool all_pinned = true;
        for (const UnitHost &U : b->units) all_pinned &= U.blob || U.ds || U.n_bytes == 0 || is_pinned_host(U.sam);
        if (!bam_arena.empty()) {  // text units copied, BAM units rendered (h2d_bytes: the bytes actually copied)
            HGT_CHECK(bam_units_fill(b, bam_arena, n_bam_rec));
        } else if (all_pinned) {  // page-locked input: the DMA engine reads the caller's buffers directly
            ctx->h2d_bytes += rd.text_bytes;
            for (size_t a = 0; a < nu; a++)  // device-split units are rendered, not copied
                if (b->units[rd.unit_of_arena[a]].ds) ctx->h2d_bytes -= rd.unit_off[a + 1] - rd.unit_off[a];
            HGT_CUDA(cudaMemsetAsync(dt, '\n', (size_t)rd.text_bytes, st));
            for (size_t a = 0; a < nu; a++) {
                const UnitHost &U = b->units[rd.unit_of_arena[a]];
                if (U.n_bytes && !U.ds) HGT_CUDA(cudaMemcpyAsync(dt + rd.unit_off[a], U.sam, U.n_bytes, cudaMemcpyHostToDevice, st));
            }
        } else {  // pageable input: host threads assemble the arena image in page-locked memory, one copy
            ctx->h2d_bytes += rd.text_bytes;
            HGT_CHECK(rd.h_stage.alloc((size_t)rd.text_bytes));
            char *hs = rd.h_stage.as<char>();
            parallel_units(batch_threads(b->params), nu, [&](size_t a) {
                const UnitHost &U = b->units[rd.unit_of_arena[a]];
                const size_t n = U.ds ? 0 : U.n_bytes;  // a device-split unit is rendered over its slice below
                if (n) memcpy(hs + rd.unit_off[a], U.sam, n);
                memset(hs + rd.unit_off[a] + n, '\n', (size_t)(rd.unit_off[a + 1] - rd.unit_off[a]) - n);
            });
            HGT_CUDA(cudaMemcpyAsync(dt, hs, (size_t)rd.text_bytes, cudaMemcpyHostToDevice, st));
        }
        HGT_CHECK(dsplit_units_render(b));
    }
    {
        HostTimer ht(ctx, 1);
        // unit tables and the loci's walk tables
        rd.o_uoff = 0;
        rd.o_uline0 = a16(rd.o_uoff + (nu + 1) * 8);
        rd.o_upos0 = a16(rd.o_uline0 + (nu + 1) * 8);
        rd.o_ulocus = a16(rd.o_upos0 + (nu + 1) * 8);
        rd.o_ulocal = a16(rd.o_ulocus + nu * 4);
        rd.o_lu0 = a16(rd.o_ulocal + nu * 4);
        rd.units_bytes = a16(rd.o_lu0 + (b->loci.size() + 1) * 4);
        HGT_CHECK(rd.h_units.alloc(rd.units_bytes));
        HGT_CHECK(rd.d_units.alloc(rd.units_bytes));
        unsigned char *hu = static_cast<unsigned char *>(rd.h_units.p);
        memset(hu, 0, rd.units_bytes);
        memcpy(hu + rd.o_uoff, rd.unit_off.data(), (nu + 1) * 8);
        for (size_t a = 0; a < nu; a++) {
            const UnitHost &U = b->units[rd.unit_of_arena[a]];
            reinterpret_cast<int64_t *>(hu + rd.o_upos0)[a] = U.pos0;
            reinterpret_cast<int32_t *>(hu + rd.o_ulocus)[a] = U.locus;
            reinterpret_cast<int32_t *>(hu + rd.o_ulocal)[a] = U.local;
        }
        memcpy(hu + rd.o_lu0, rd.locus_unit0.data(), (b->loci.size() + 1) * 4);
        ctx->h2d_bytes += (int64_t)rd.units_bytes;
        HGT_CUDA(cudaMemcpyAsync(rd.d_units.p, hu, rd.units_bytes, cudaMemcpyHostToDevice, st));
        const size_t lw = b->loci.size() * sizeof(hgtd::LocusWalk);
        HGT_CHECK(rd.h_loci.alloc(lw));
        HGT_CHECK(rd.d_loci.alloc(lw));
        for (size_t l = 0; l < b->loci.size(); l++) rd.h_loci.as<hgtd::LocusWalk>()[l] = b->loci[l]->wt_dev;
        HGT_CUDA(cudaMemcpyAsync(rd.d_loci.p, rd.h_loci.p, lw, cudaMemcpyHostToDevice, st));
        // line count: newlines per 16 KB chunk, scanned (the chunk bases feed the line index of execute)
        rd.n_chunks = (rd.text_bytes + hgtk::CHUNK_BYTES - 1) / hgtk::CHUNK_BYTES;
        HGT_CHECK(rd.d_chunk.alloc((size_t)(rd.n_chunks + 1) * 8));
        hgtk::count_newlines_kernel<<<(unsigned)rd.n_chunks, hgtk::LINE_THREADS, 0, st>>>(rd.d_text.as<char>(), rd.text_bytes,
                                                                                      rd.d_chunk.as<int64_t>());
        ctx->launches++;
        HGT_CUDA(cudaGetLastError());
        HGT_CHECK(dev_scan(ctx, st, rd.d_chunk.as<int64_t>(), rd.n_chunks, rd.d_chunk.as<int64_t>(), &rd.d_partial));
        HGT_CHECK(rd.h_small.alloc(64));
        HGT_CUDA(d2h(rd.h_small.p, rd.d_chunk.as<int64_t>() + rd.n_chunks, 8, st));
        HGT_CUDA(cudaStreamSynchronize(st));
        rd.n_lines = *rd.h_small.as<int64_t>();
        rd.release_bam();  // the blob arena goes back to the pool: the render has run
    }
    if (rd.n_lines > 0x7fffffff) {
        hgt_set_error("more than 2^31 alignment lines in one batch: split the batch");
        return HGT_ERR_UNSUPPORTED;
    }
    b->prepared = true;
    return HGT_OK;
}

// ---- record stage of execute: line index -> parse -> pileup -> walk -> pair jobs -------------------------------------------------
static const char *walk_error_text(int code, int *status) {
    using namespace hgtd;
    *status = HGT_ERR_PARSE;
    switch (code) {
        case E_RECORD: return "malformed alignment record (fewer than 11 columns or bad integer)";
        case E_NO_NM_NH: return "alignment lacks the NM or NH tag";
        case E_MATE_KIND: return "read is neither first nor second mate and --discordant is off";
        case E_NO_MD: return "MD tag missing";
        case E_CIGAR: return "malformed CIGAR";
        case E_ZS_ITEM: return "malformed Zs item";
        case E_ZS_OFFSET: return "malformed Zs offset";
        case E_MD_SHORT: return "MD shorter than CIGAR";
        case E_MD_PAST_READ: return "MD runs past the read";
        case E_MD_BASE: return "MD reference base is not ACGT";
        case E_ZS_NOT_S: return "Zs item is not a substitution";
        case E_ZS_ID: return "Zs id is not a variant of this locus";
        case E_ZS_NOT_I: return "Zs item is not an insertion";
        case E_MD_CARET: return "MD lacks ^ for a deletion";
        case E_CLIP_MIDDLE: return "soft clip in the middle of a CIGAR";
        case E_CIGAR_OP: return "unsupported CIGAR operation";
        case E_EMPTY: return "read has an empty alignment";
        case E_ALT_INDEX: return "alt haplotype index out of range";
        case E_ALT_TOKEN: return "alt haplotype token is not a variant";
        case E_AMBIGUITY: *status = HGT_ERR_AMBIGUITY; return "ambiguous alternative haplotype sets (check_amb_uniqueness)";
        case E_CAP_CMP: *status = HGT_ERR_UNSUPPORTED; return "more than 96 differences in one alignment";
        case E_CAP_ENDS: *status = HGT_ERR_UNSUPPORTED; return "more than 16 alternative ends (or 16 variants in one) around a read";
        case E_CAP_IDS: *status = HGT_ERR_UNSUPPORTED; return "more than 32 variants inside one read";
        case E_LINE_LONG: *status = HGT_ERR_UNSUPPORTED; return "alignment line longer than 65535 bytes";
        case E_NOVEL_RANGE: *status = HGT_ERR_UNSUPPORTED; return "novel indel outside the supported range (position < 2^19, length < 2^10)";
        case E_PAIR_HTS: *status = HGT_ERR_UNSUPPORTED; return "a read pair expands to more than 255 haplotypes";
        default: return "record stage failed";
    }
}

// first token of a text line (the read name), for error messages
static std::string line_name(const char *p, size_t n) {
    size_t a = 0;
    while (a < n && hgtd::is_ws(p[a])) a++;
    size_t e = a;
    while (e < n && !hgtd::is_ws(p[e])) e++;
    return std::string(p + a, e - a);
}

static int report_walk_error(hgt_batch *b, unsigned long long err, cudaStream_t st) {
    if (err == ~0ull) return HGT_OK;
    const int64_t line = (int64_t)(err >> 8);
    int status = HGT_ERR_PARSE;
    const char *msg = walk_error_text((int)(err & 0xff), &status);
    int64_t off[2] = {0, 0};
    char buf[97];
    memset(buf, 0, sizeof(buf));
    if (cudaMemcpyAsync(off, b->rd.d_line_off.as<int64_t>() + line, 16, cudaMemcpyDeviceToHost, st) == cudaSuccess &&
        cudaStreamSynchronize(st) == cudaSuccess) {
        const size_t n = (size_t)std::min<int64_t>(96, off[1] - off[0]);
        cudaMemcpyAsync(buf, b->rd.d_text.as<char>() + off[0], n, cudaMemcpyDeviceToHost, st);
        cudaStreamSynchronize(st);
    }
    hgt_set_error("%s (read %s)", msg, line_name(buf, strlen(buf)).c_str());
    return status;
}

static hgtd::ReadsView reads_view(hgt_batch *b) {
    ReadsDev &rd = b->rd;
    hgtd::ReadsView R;
    memset(&R, 0, sizeof(R));
    const size_t N = (size_t)rd.n_lines, nu = b->units.size();
    R.text = rd.d_text.as<char>();
    R.n_lines = rd.n_lines;
    R.line_off = rd.d_line_off.as<int64_t>();
    R.unit = rd.d_unit.as<int32_t>();
    R.rec = rd.d_rec.as<hgtd::RecFields>();
    R.st = rd.d_st.as<uint16_t>();
    R.h_left = rd.d_hdr.as<int32_t>();
    R.h_right = R.h_left + N;
    R.h_n = R.h_right + N;
    R.slow_slot = R.h_n + N;
    R.h_ids = rd.d_hids.as<int32_t>();
    R.slow = rd.d_slow.as<hgtd::SlowRec>();
    R.amb_list = rd.d_slow_list.as<int32_t>();
    R.slow_list = R.amb_list + std::max<size_t>(N, 1);
    unsigned char *sm = static_cast<unsigned char *>(rd.d_small.p);
    R.err = reinterpret_cast<unsigned long long *>(sm);
    R.n_slow = reinterpret_cast<int32_t *>(sm + 8);
    R.n_amb = reinterpret_cast<int32_t *>(sm + 16);
    R.n_heads = reinterpret_cast<int32_t *>(sm + 20);
    R.head_list = R.slow_list + std::max<size_t>(N, 1);
    R.pair_cnt = R.amb_list + 4 * std::max<size_t>(N, 1) + hgtk::SORT_BUCKETS;
    R.max_job_haps = reinterpret_cast<int32_t *>(sm + 12);
    R.unit_reads = reinterpret_cast<unsigned long long *>(sm + rd.s_reads);
    R.unit_pairs = reinterpret_cast<unsigned long long *>(sm + rd.s_pairs);
    unsigned char *du = static_cast<unsigned char *>(rd.d_units.p);
    R.n_units = (int)nu;
    R.unit_off = reinterpret_cast<int64_t *>(du + rd.o_uoff);
    R.unit_line0 = reinterpret_cast<int64_t *>(du + rd.o_uline0);
    R.unit_pos0 = reinterpret_cast<int64_t *>(du + rd.o_upos0);
    R.unit_locus = reinterpret_cast<int32_t *>(du + rd.o_ulocus);
    R.unit_local = reinterpret_cast<int32_t *>(du + rd.o_ulocal);
    R.nt_mask = rd.d_mf.as<uint8_t>();
    R.del_flag = rd.d_mf.as<uint8_t>() + rd.POS;
    R.loci = rd.d_loci.as<hgtd::LocusWalk>();
    int64_t *sc = rd.d_scan.as<int64_t>();
    R.s_pairs = sc;
    R.s_haps = sc + (N + 1);
    R.s_rows = sc + 2 * (N + 1);
    R.s_small = sc + 3 * (N + 1);
    R.s_big = sc + 4 * (N + 1);
    R.jobs = rd.d_jobs_desc.as<hgtd::LocusJobs>();
    return R;
}

static int line_grid(hgt_ctx *ctx, int64_t n, int threads, int per_sm) {
    return (int)std::max<int64_t>(1, std::min<int64_t>((n + threads - 1) / threads, (int64_t)ctx->sm_count * per_sm));
}

static int reads_execute(hgt_batch *b, cudaStream_t st) {
    hgt_ctx *ctx = b->ctx;
    ReadsDev &rd = b->rd;
    const size_t nu = b->units.size(), nl = b->loci.size();
    const int64_t N = rd.n_lines;
    hgtd::WalkParams P;
    P.num_editdist = b->params.num_editdist; P.error_correction = b->params.error_correction;
    P.allow_discordant = b->params.allow_discordant; P.simulation = b->params.simulation; P.base_locus = b->params.base_locus;
    // ---- buffers (from the context's pool: a second execute of the same batch re-uses all of them) --------------------------
    HGT_CHECK(rd.d_line_off.alloc((size_t)(N + 1) * 8));
    HGT_CHECK(rd.d_unit.alloc((size_t)std::max<int64_t>(N, 1) * 4));
    HGT_CHECK(rd.d_rec.alloc((size_t)std::max<int64_t>(N, 1) * sizeof(hgtd::RecFields)));
    HGT_CHECK(rd.d_st.alloc((size_t)std::max<int64_t>(N, 1) * 2));
    HGT_CHECK(rd.d_hdr.alloc((size_t)std::max<int64_t>(N, 1) * 16));
    HGT_CHECK(rd.d_hids.alloc((size_t)std::max<int64_t>(N, 1) * hgtd::MAXI * 4));
    // amb_list, slow_list, head_list, the sorted copy of the running list pass, bucket counters
    // (+ the per-run table totals the count pass leaves for the fill pass)
    HGT_CHECK(rd.d_slow_list.alloc((size_t)std::max<int64_t>(N, 1) * 28 + (size_t)hgtk::SORT_BUCKETS * 4));
    HGT_CHECK(rd.d_scan.alloc((size_t)(N + 1) * 8 * 5));
    HGT_CHECK(rd.d_cnt.alloc((size_t)std::max<int64_t>(rd.POS, 1) * 24));
    HGT_CHECK(rd.d_mf.alloc((size_t)std::max<int64_t>(rd.POS, 1) * 2));
    rd.s_reads = 32;
    rd.s_pairs = rd.s_reads + nu * 8;
    rd.s_totals = rd.s_pairs + nu * 8;
    rd.small_bytes = rd.s_totals + nl * 6 * 8;
    HGT_CHECK(rd.d_small.alloc(rd.small_bytes));
    HGT_CHECK(rd.h_small.alloc(rd.small_bytes));
    HGT_CHECK(rd.d_jobs_desc.alloc(nl * sizeof(hgtd::LocusJobs)));
    HGT_CHECK(rd.h_jobs_desc.alloc(nl * sizeof(hgtd::LocusJobs)));
    if (rd.d_slow.p == nullptr) HGT_CHECK(rd.d_slow.alloc(sizeof(hgtd::SlowRec)));
    hgtd::ReadsView R = reads_view(b);
    HGT_CUDA(cudaMemsetAsync(rd.d_small.p, 0, rd.small_bytes, st));
    HGT_CUDA(cudaMemsetAsync(rd.d_small.p, 0xff, 8, st));
    HGT_CUDA(cudaMemsetAsync(rd.d_cnt.p, 0, (size_t)std::max<int64_t>(rd.POS, 1) * 24, st));
    // ---- line index, records, pileup --------------------------------------------------------------------------------------
    b->timer.begin(ctx, st, 0);
    int launches = 4;  // index_lines, unit_lines, parse, pileup_text (pileup_flags below)
    ctx->launches += 5;
    hgtk::index_lines_kernel<<<(unsigned)rd.n_chunks, hgtk::LINE_THREADS, 0, st>>>(rd.d_text.as<char>(), rd.text_bytes,
                                                                               rd.d_chunk.as<int64_t>(), rd.d_line_off.as<int64_t>());
    hgtk::unit_lines_kernel<<<(unsigned)((nu + 1 + 127) / 128), 128, 0, st>>>(R);
    // shared-memory image of a CTA's 128 lines: 15 % above the average, at least 16 KB (HGT_STAGE_KB overrides)
    static const int stage_kb_env = tune_env("HGT_STAGE_KB", 0), stage_ctas = tune_env("HGT_STAGE_CTAS_PER_SM", 4);
    int stage_bytes = (int)std::min<int64_t>(
        160 << 10, std::max<int64_t>(16 << 10, (rd.text_bytes / std::max<int64_t>(N, 1) * 147 + 1023) / 1024 * 1024 + 1024));
    if (stage_kb_env > 0) stage_bytes = stage_kb_env << 10;
    HGT_CUDA(hgt_smem_at_least((const void *)hgtk::parse_kernel, stage_bytes));
    const int stage_grid = (int)std::max<int64_t>(1, std::min<int64_t>((N + hgtk::STAGE_LINES - 1) / hgtk::STAGE_LINES,
                                                                     (int64_t)ctx->sm_count * stage_ctas));
    hgtk::parse_kernel<<<stage_grid, hgtk::STAGE_LINES, stage_bytes, st>>>(R, P, stage_bytes);
    // the pileup is its own pass (warp per line, 8 CTAs of 256 threads per SM): the histogram atomics need more warps in
    // flight than the staged parse kernel holds
    hgtk::pileup_text_kernel<<<line_grid(ctx, N * 32, 256, 8), 256, 0, st>>>(R, rd.d_cnt.as<uint32_t>());
    HGT_CUDA(cudaGetLastError());
    if (b->pileup_hook) {  // read-sharded locus: the caller sums the raw counts over ranks (SURVEY.md 8e)
        HGT_CUDA(cudaStreamSynchronize(st));
        const int rc = b->pileup_hook(b->pileup_hook_arg, rd.d_cnt.p, (size_t)rd.POS * 6, st);
        if (rc != 0) {
            hgt_set_error("pileup hook failed with status %d", rc);
            return HGT_ERR_ARG;
        }
    }
    if (rd.POS > 0) {
        pileup_flags_kernel<<<(unsigned)((rd.POS + 255) / 256), 256, 0, st>>>(rd.d_cnt.as<uint32_t>(), rd.POS, rd.d_mf.as<uint8_t>(),
                                                                             rd.d_mf.as<uint8_t>() + rd.POS);
        launches++;
    }
    b->timer.end(launches);
    if (b->keep_counts) {
        for (UnitHost &U : b->units) {
            const size_t L = (size_t)b->loci[U.locus]->L;
            U.counts.resize(L * 6);
            U.nt_mask.resize(L);
            HGT_CUDA(d2h(U.counts.data(), rd.d_cnt.as<uint32_t>() + (size_t)U.pos0 * 6, L * 24, st));
            HGT_CUDA(d2h(U.nt_mask.data(), rd.d_mf.as<uint8_t>() + U.pos0, L, st));
        }
    }
    // ---- runs, mate de-dup, the walk ------------------------------------------------------------------------------------------
    b->timer.begin(ctx, st, 7);
    hgtk::head_kernel<<<line_grid(ctx, N, 256, 8), 256, 0, st>>>(R);
    hgtk::candidate_kernel<<<line_grid(ctx, N, 256, 8), 256, 0, st>>>(R);
    hgtk::walk_kernel<<<line_grid(ctx, N, 128, 16), hgtk::STAGE_LINES, 0, st>>>(R, P);
    // second pass in backbone order (its length is read on the device)
    int32_t *sorted = rd.d_slow_list.as<int32_t>() + 3 * std::max<size_t>(N, 1), *buckets = sorted + std::max<size_t>(N, 1);
    HGT_CUDA(cudaMemsetAsync(buckets, 0, (size_t)hgtk::SORT_BUCKETS * 4, st));
    hgtk::list_hist_kernel<<<line_grid(ctx, N / 8 + 1, 256, 4), 256, 0, st>>>(R, R.amb_list, R.n_amb, buckets);
    hgtk::list_scan_kernel<<<1, 1024, 0, st>>>(buckets);
    hgtk::list_scatter_kernel<<<line_grid(ctx, N / 8 + 1, 256, 4), 256, 0, st>>>(R, R.amb_list, R.n_amb, buckets, sorted);
    hgtk::walk_amb_kernel<<<line_grid(ctx, N, 128, 16), 128, 0, st>>>(R, P, sorted);
    launches = 7;  // head, candidate, walk, the three list-sort kernels, walk_amb
    ctx->launches += launches;
    HGT_CUDA(cudaGetLastError());
    HGT_CUDA(d2h(rd.h_small.p, rd.d_small.p, 16, st));
    HGT_CUDA(cudaStreamSynchronize(st));  // number of records that need the ambiguity pass
    {
        const unsigned char *hs = static_cast<const unsigned char *>(rd.h_small.p);
        HGT_CHECK(report_walk_error(b, *reinterpret_cast<const unsigned long long *>(hs), st));
        rd.n_slow = *reinterpret_cast<const int32_t *>(hs + 8);
    }
    if (rd.n_slow > 0) {
        HGT_CHECK(rd.d_slow.alloc((size_t)rd.n_slow * sizeof(hgtd::SlowRec)));
        R = reads_view(b);
        HGT_CUDA(cudaMemsetAsync(buckets, 0, (size_t)hgtk::SORT_BUCKETS * 4, st));
        hgtk::list_hist_kernel<<<line_grid(ctx, rd.n_slow, 256, 4), 256, 0, st>>>(R, R.slow_list, R.n_slow, buckets);
        hgtk::list_scan_kernel<<<1, 1024, 0, st>>>(buckets);
        hgtk::list_scatter_kernel<<<line_grid(ctx, rd.n_slow, 256, 4), 256, 0, st>>>(R, R.slow_list, R.n_slow, buckets, sorted);
        hgtk::walk_slow_kernel<<<line_grid(ctx, rd.n_slow, 128, 16), 128, 0, st>>>(R, P, sorted, rd.n_slow);
        launches += 4;
        ctx->launches += 4;
    }
    HGT_CUDA(cudaMemsetAsync(rd.d_scan.p, 0, (size_t)(N + 1) * 8 * 5, st));
    hgtk::pair_count_kernel<<<line_grid(ctx, N, 128, 16), 128, 0, st>>>(R);
    launches += 1 + 15 + 1 + 1;  // + five scans, locus totals, fill
    ctx->launches += 3;         // (the scans count themselves)
    HGT_CUDA(cudaGetLastError());
    for (int k = 0; k < 5; k++) {
        int64_t *a = rd.d_scan.as<int64_t>() + (size_t)k * (N + 1);
        HGT_CHECK(dev_scan(ctx, st, a, N, a, &rd.d_partial));
    }
    hgtk::locus_totals_kernel<<<(unsigned)((nl + 63) / 64), 64, 0, st>>>(
        R, (int)nl, reinterpret_cast<int32_t *>(static_cast<unsigned char *>(rd.d_units.p) + rd.o_lu0),
        reinterpret_cast<int64_t *>(static_cast<unsigned char *>(rd.d_small.p) + rd.s_totals));
    HGT_CUDA(cudaGetLastError());
    HGT_CUDA(d2h(rd.h_small.p, rd.d_small.p, rd.small_bytes, st));
    HGT_CUDA(cudaStreamSynchronize(st));  // sizes of the job arrays and class pools
    const unsigned char *hs = static_cast<const unsigned char *>(rd.h_small.p);
    HGT_CHECK(report_walk_error(b, *reinterpret_cast<const unsigned long long *>(hs), st));
    rd.max_job_haps = *reinterpret_cast<const int32_t *>(hs + 12);
    for (size_t a = 0; a < nu; a++) {
        UnitHost &U = b->units[rd.unit_of_arena[a]];
        U.num_reads = (int64_t) reinterpret_cast<const unsigned long long *>(hs + rd.s_reads)[a];
        U.num_pairs = (int64_t) reinterpret_cast<const unsigned long long *>(hs + rd.s_pairs)[a];
    }
    // ---- job arrays per locus (device only), class pools, EM buffers ---------------------------------------------------------
    hgtd::LocusJobs *hj = rd.h_jobs_desc.as<hgtd::LocusJobs>();
    memset(hj, 0, nl * sizeof(hgtd::LocusJobs));
    for (size_t l = 0; l < nl; l++) {
        LocusBatch &lb = b->lb[l];
        if (lb.units.empty()) continue;
        const hgt_locus *loc = lb.loc;
        const int n_tables = loc->is_hla ? 3 : 1;
        const size_t n_units = lb.units.size();
        const int64_t *tot = reinterpret_cast<const int64_t *>(hs + rd.s_totals) + l * 6;
        const int64_t J = tot[0] * n_tables, H = tot[1], RW = tot[2];
        if (J > 0x7fffffff || H > 0x7fffffff || RW > 0x7fffffff) {
            hgt_set_error("more than 2^31 jobs or haplotypes in one locus batch: split the batch");
            return HGT_ERR_UNSUPPORTED;
        }
        lb.n_jobs = J; lb.n_haps = H; lb.n_rows = RW; lb.n_small = tot[3]; lb.n_big = tot[4];
        lb.max_job_haps = rd.max_job_haps;
        lb.ut_base.assign(n_units * 4 + 1, 0);
        for (size_t i = 0; i < n_units; i++) {
            const UnitHost &U = b->units[lb.units[i]];
            if (U.num_pairs > 0x7fffffff) {
                hgt_set_error("a unit holds more than 2^31 read pairs");
                return HGT_ERR_UNSUPPORTED;
            }
            for (int tb = 0; tb < 4; tb++) {
                const bool active = tb < n_tables || (tb == 3 && loc->is_hla);
                lb.ut_base[i * 4 + tb + 1] = lb.ut_base[i * 4 + tb] + (active ? U.num_pairs : 0);
            }
        }
        lb.n_rows_pool = lb.ut_base.back();
        if (lb.n_rows_pool > POOL_MAX_ROWS) {
            hgt_set_error("more than 2^28 class rows in one locus batch: split the batch");
            return HGT_ERR_UNSUPPORTED;
        }
        LocusBatch::JobArena &ja = lb.ja;
        ja.o_job_off = 0;
        ja.o_row_off = a16(ja.o_job_off + (size_t)(J + 1) * 8);
        ja.o_ut_base = a16(ja.o_row_off + (size_t)(H + 1) * 8);
        ja.o_job_ut = a16(ja.o_ut_base + (n_units * 4 + 1) * 8);
        ja.o_job_pair = a16(ja.o_job_ut + (size_t)J * 4);
        ja.o_job_list = a16(ja.o_job_pair + (size_t)J * 4);
        ja.o_hl = a16(ja.o_job_list + (size_t)J * 4);
        ja.o_hr = a16(ja.o_hl + (size_t)H * 4);
        ja.o_ht = a16(ja.o_hr + (size_t)H * 4);
        ja.o_rows = a16(ja.o_ht + (size_t)H * 4);
        ja.bytes = a16(ja.o_rows + (size_t)RW * 4);
        HGT_CHECK(lb.d_jobs.alloc(ja.bytes));
        HGT_CHECK(lb.h_jobs.alloc((n_units * 4 + 1) * 8));
        memcpy(lb.h_jobs.p, lb.ut_base.data(), (n_units * 4 + 1) * 8);
        ctx->h2d_bytes += (int64_t)((n_units * 4 + 1) * 8);
        HGT_CUDA(hgt_small_h2d(lb.dj<int64_t>(ja.o_ut_base), lb.h_jobs.p, (n_units * 4 + 1) * 8, st));
        HGT_CUDA(cudaMemsetAsync(lb.dj<int64_t>(ja.o_job_off), 0, 8, st));
        HGT_CUDA(cudaMemsetAsync(lb.dj<int64_t>(ja.o_row_off), 0, 8, st));
        hgtd::LocusJobs &d = hj[l];
        d.job_off = lb.dj<int64_t>(ja.o_job_off); d.row_off = lb.dj<int64_t>(ja.o_row_off);
        d.job_ut = lb.dj<int32_t>(ja.o_job_ut); d.job_pair = lb.dj<int32_t>(ja.o_job_pair); d.job_list = lb.dj<int32_t>(ja.o_job_list);
        d.hap_left = lb.dj<int32_t>(ja.o_hl); d.hap_right = lb.dj<int32_t>(ja.o_hr); d.hap_table = lb.dj<int32_t>(ja.o_ht);
        d.rows = lb.dj<int32_t>(ja.o_rows);
        d.n_small = lb.n_small;
        d.n_tables = n_tables;
        d.line0 = tot[5];
    }
    HGT_CUDA(hgt_small_h2d(rd.d_jobs_desc.p, hj, nl * sizeof(hgtd::LocusJobs), st));
    hgtk::pair_fill_kernel<<<line_grid(ctx, N, 128, 16), 128, 0, st>>>(R);
    b->timer.end(launches);
    HGT_CUDA(cudaGetLastError());
    return HGT_OK;
}

static int batch_alloc_tables(hgt_batch *b, cudaStream_t st) {
    hgt_ctx *ctx = b->ctx;
    const size_t nu = b->units.size();
    {
        HostTimer ht(ctx, 5);
        for (LocusBatch &lb : b->lb) {
            if (lb.units.empty()) continue;
            const hgt_locus *loc = lb.loc;
            const int wp = loc->wp;
            const size_t n_units = lb.units.size();
            lb.cap = 64;
            while ((int64_t)lb.cap < 2 * std::max<int64_t>(lb.n_rows_pool, 1)) lb.cap <<= 1;
            HGT_CHECK(lb.d_hapbits.alloc((size_t)std::max<int64_t>(lb.n_haps, 1) * wp * 8));
            HGT_CHECK(lb.d_keys.alloc((size_t)lb.cap * 8));
            const size_t pr = (size_t)std::max<int64_t>(lb.n_rows_pool, 1);
            HGT_CHECK(lb.d_bits.alloc(pr * wp * 8));
            HGT_CHECK(lb.d_count.alloc(pr * 8));
            HGT_CHECK(lb.d_first.alloc(pr * 4));
            HGT_CHECK(lb.d_ut_ncls.alloc(n_units * 4 * 4));
            {  // scratch of class_sort_kernel: the rows of ONE table
                const size_t one = std::max<size_t>(pr / (loc->is_hla ? 4 : 1) + 1, 1);
                HGT_CHECK(lb.d_sortbits.alloc(one * wp * 8));
                HGT_CHECK(lb.d_sortcnt.alloc(one * 8));
                HGT_CHECK(lb.d_sortfirst.alloc(one * 4));
            }
            // EM buffers (both levels; nothing is allocated after prepare)
            const size_t A = (size_t)loc->A;
            HGT_CHECK(lb.d_prob.alloc(n_units * A * 8));
            HGT_CHECK(lb.d_inres.alloc(n_units * A));
            HGT_CHECK(lb.d_fk.alloc(n_units * A * 4));
            HGT_CHECK(lb.d_is.alloc(n_units * 12));
            HGT_CHECK(lb.d_emws.alloc(n_units * hgt_em_problem_ws_bytes(wp)));
            HGT_CHECK(lb.d_acount.alloc(n_units * A * 8));
            HGT_CHECK(lb.d_afirst.alloc(n_units * A * 4));
            HGT_CHECK(lb.h_ncls.alloc(n_units * 16));
            HGT_CHECK(lb.h_prob.alloc(n_units * A * 8));
            HGT_CHECK(lb.h_inres.alloc(n_units * A));
            HGT_CHECK(lb.h_fk.alloc(n_units * A * 4));
            HGT_CHECK(lb.h_is.alloc(n_units * 12));
            for (int lv = 0; lv < (loc->is_hla ? 2 : 1); lv++) {
                HGT_CHECK(lb.d_ck[lv].alloc(n_units * KEY_CAP * sizeof(KeyOut)));
                HGT_CHECK(lb.d_cn[lv].alloc(n_units * 4));
                HGT_CHECK(lb.h_ck[lv].alloc(n_units * KEY_CAP * sizeof(KeyOut)));
                HGT_CHECK(lb.h_cn[lv].alloc(n_units * 4));
            }
            lb.ut_ncls = lb.h_ncls.as<int32_t>(); lb.prob = lb.h_prob.as<double>(); lb.inres = lb.h_inres.as<uint8_t>();
            lb.fk = lb.h_fk.as<int32_t>(); lb.is = lb.h_is.as<int32_t>();
            memset(lb.ut_ncls, 0, n_units * 16);
            for (int tb = 0; tb < 3; tb++) {
                int n = 0;
                for (int j = 0; j < wp; j++) n += __builtin_popcountll(loc->mask[(size_t)tb * wp + j]);
                lb.n_live[tb] = n;
            }
            lb.n_live[3] = loc->A;
            if (loc->is_hla) {
                HGT_CHECK(lb.d_prob2.alloc(n_units * A * 8));
                HGT_CHECK(lb.d_inres2.alloc(n_units * A));
                HGT_CHECK(lb.d_fk2.alloc(n_units * A * 4));
                HGT_CHECK(lb.d_is2.alloc(n_units * 12));
                HGT_CHECK(lb.d_keep.alloc(n_units * (size_t)wp * 8));
                HGT_CHECK(lb.d_ulist.alloc(n_units * 4));
                HGT_CHECK(lb.h_prob2.alloc(n_units * A * 8));
                HGT_CHECK(lb.h_inres2.alloc(n_units * A));
                HGT_CHECK(lb.h_fk2.alloc(n_units * A * 4));
                HGT_CHECK(lb.h_is2.alloc(n_units * 12));
                HGT_CHECK(lb.h_keep.alloc(n_units * (size_t)wp * 8));
                HGT_CHECK(lb.h_ulist.alloc(n_units * 4));
                lb.prob2 = lb.h_prob2.as<double>(); lb.inres2 = lb.h_inres2.as<uint8_t>();
                lb.fk2 = lb.h_fk2.as<int32_t>(); lb.is2 = lb.h_is2.as<int32_t>();
            }
        }
        for (int i = 0; i < 2; i++) {
            HGT_CHECK(b->h_em_args[i].alloc(hgt_em_args_bytes((int)nu)));
            HGT_CHECK(b->d_em_args[i].alloc(hgt_em_args_bytes((int)nu)));
        }
    }
    (void)st;
    return HGT_OK;
}

// ---- EM results: key lists when select_alleles ran (a handful of keys), dense arrays otherwise ---------------------------
struct Ent {
    int32_t a;
    double p;
    int32_t fk;
};
// list capacity per unit: KEY_CAP, or less when HGT_KEY_CAP is set (tests force the dense fall-back with it)
static int key_cap() {
    static const int cap = [] {
        const char *e = getenv("HGT_KEY_CAP");
        const int v = e ? atoi(e) : KEY_CAP;
        return v < 1 ? 1 : (v > KEY_CAP ? KEY_CAP : v);
    }();
    return cap;
}

// keys of one unit's result of `level` (0 first, 1 second) in ascending allele order
static void unit_keys(const LocusBatch &lb, int level, size_t local, std::vector<Ent> *out) {
    out->clear();
    const size_t A = (size_t)lb.loc->A;
    if (lb.dense[level]) {
        const double *p = (level ? lb.prob2 : lb.prob) + local * A;
        const uint8_t *in = (level ? lb.inres2 : lb.inres) + local * A;
        const int32_t *fk = (level ? lb.fk2 : lb.fk) + local * A;
        for (int a = 0; a < (int)A; a++)
            if (in[a]) out->push_back({a, p[a], fk[a]});
        return;
    }
    const KeyOut *k = lb.h_ck[level].as<KeyOut>() + local * key_cap();
    const int n = lb.h_cn[level].as<int32_t>()[local];
    for (int i = 0; i < n; i++) out->push_back({k[i].allele, k[i].prob, k[i].fk});
}
static void sort_ranked(std::vector<Ent> *v) {  // probability descending; ties in dict order (common:1408-1409)
    std::sort(v->begin(), v->end(), [](const Ent &x, const Ent &y) {
        if (x.p != y.p) return x.p > y.p;
        if (x.fk != y.fk) return x.fk < y.fk;
        return x.a < y.a;
    });
}

// Brings the results of one EM level to the host and synchronises the stream.
static int fetch_results(hgt_batch *b, cudaStream_t st, int level) {
    hgt_ctx *ctx = b->ctx;
    const int cap = key_cap();
    auto dense_copies = [&](LocusBatch &lb) -> int {
        const size_t n_units = lb.units.size(), A = (size_t)lb.loc->A;
        HGT_CUDA(d2h(level ? lb.prob2 : lb.prob, (level ? lb.d_prob2 : lb.d_prob).p, n_units * A * 8, st));
        HGT_CUDA(d2h(level ? lb.inres2 : lb.inres, (level ? lb.d_inres2 : lb.d_inres).p, n_units * A, st));
        HGT_CUDA(d2h(level ? lb.fk2 : lb.fk, (level ? lb.d_fk2 : lb.d_fk).p, n_units * A * 4, st));
        lb.dense[level] = true;
        return HGT_OK;
    };
    for (LocusBatch &lb : b->lb) {
        if (lb.units.empty() || (level == 1 && lb.n_level2 == 0)) continue;
        const size_t n_units = lb.units.size();
        // without select_alleles nearly every allele stays a key (first level off the hla path): dense copies
        const bool lists = level == 1 || (lb.loc->is_hla && b->remove_low);
        if (lists) {
            result_keys_kernel<<<(unsigned)n_units, KEY_THREADS, 0, st>>>(
                lb.loc->A, (level ? lb.d_prob2 : lb.d_prob).as<double>(), (level ? lb.d_inres2 : lb.d_inres).as<uint8_t>(),
                (level ? lb.d_fk2 : lb.d_fk).as<int32_t>(), (level ? lb.d_is2 : lb.d_is).as<int32_t>(), cap,
                lb.d_ck[level].as<KeyOut>(), lb.d_cn[level].as<int32_t>());
            HGT_CUDA(cudaGetLastError());
            ctx->launches++;
            HGT_CUDA(d2h(lb.h_cn[level].p, lb.d_cn[level].p, n_units * 4, st));
            HGT_CUDA(d2h(lb.h_ck[level].p, lb.d_ck[level].p, n_units * KEY_CAP * sizeof(KeyOut), st));
            lb.dense[level] = false;
        } else {
            HGT_CHECK(dense_copies(lb));
        }
        HGT_CUDA(d2h(level ? lb.is2 : lb.is, (level ? lb.d_is2 : lb.d_is).p, n_units * 12, st));
        if (level == 1) HGT_CUDA(d2h(lb.ut_ncls, lb.d_ut_ncls.p, n_units * 16, st));
    }
    HGT_CUDA(cudaStreamSynchronize(st));
    bool again = false;
    for (LocusBatch &lb : b->lb) {
        if (lb.units.empty() || (level == 1 && lb.n_level2 == 0) || lb.dense[level]) continue;
        const int32_t *cn = lb.h_cn[level].as<int32_t>();
        bool over = false;
        for (size_t i = 0; i < lb.units.size(); i++) over |= cn[i] > cap;
        if (over) {  // a unit kept more keys than a list holds: this locus goes the dense way
            HGT_CHECK(dense_copies(lb));
            again = true;
        }
    }
    if (again) HGT_CUDA(cudaStreamSynchronize(st));
    return HGT_OK;
}

// ---- stage 2: GPU only, no host synchronisation -----------------------------------------------------------------

template <int WPL>
static void launch_stage_a(hgt_batch *b, cudaStream_t st, LocusBatch &lb) {
    static const int class_per_sm = tune_env("HGT_CLASS_CTAS_PER_SM", 32), compat_per_sm = tune_env("HGT_COMPAT_CTAS_PER_SM", 16);
    hgt_ctx *ctx = b->ctx;
    const hgt_locus *loc = lb.loc;
    const LocusDev ld = locus_dev(loc);
    const int wp = loc->wp;
    const int64_t H = lb.n_haps;
    b->timer.begin(ctx, st, 1);
    if (H > 0) {
        const int ctas = (int)std::min<int64_t>((H + WARPS_PER_CTA - 1) / WARPS_PER_CTA, (int64_t)ctx->sm_count * compat_per_sm);
        compat_kernel<WPL><<<ctas, WARPS_PER_CTA * 32, 0, st>>>(ld, lb.dj<int32_t>(lb.ja.o_ht), lb.dj<int32_t>(lb.ja.o_hl),
                                                                   lb.dj<int32_t>(lb.ja.o_hr), lb.dj<int64_t>(lb.ja.o_row_off),
                                                                   lb.dj<int32_t>(lb.ja.o_rows), H, lb.d_hapbits.as<uint64_t>());
        ctx->launches++;
    }
    b->timer.end(H > 0 ? 1 : 0);
    const ClassPool pool = lb.pool();
    const int64_t ns = lb.n_small, nb = lb.n_big;
    b->timer.begin(ctx, st, 2);
    if (ns > 0) {
        const int ctas = (int)std::min<int64_t>((ns + WARPS_PER_CTA - 1) / WARPS_PER_CTA, (int64_t)ctx->sm_count * class_per_sm);
        class_kernel<WPL, 3><<<ctas, WARPS_PER_CTA * 32, 0, st>>>(wp, loc->d_mask, lb.dj<int64_t>(lb.ja.o_job_off),
                                                                  lb.dj<int32_t>(lb.ja.o_job_ut), lb.dj<int32_t>(lb.ja.o_job_pair),
                                                                  lb.dj<int32_t>(lb.ja.o_job_list), ns, lb.d_hapbits.as<uint64_t>(), pool);
        ctx->launches++;
    }
    if (nb > 0) {
        const int ctas = (int)std::min<int64_t>((nb + WARPS_PER_CTA - 1) / WARPS_PER_CTA, (int64_t)ctx->sm_count * 8);
        class_kernel<WPL, 8><<<ctas, WARPS_PER_CTA * 32, 0, st>>>(wp, loc->d_mask, lb.dj<int64_t>(lb.ja.o_job_off),
                                                                  lb.dj<int32_t>(lb.ja.o_job_ut), lb.dj<int32_t>(lb.ja.o_job_pair),
                                                                  lb.dj<int32_t>(lb.ja.o_job_list) + ns, nb, lb.d_hapbits.as<uint64_t>(), pool);
        ctx->launches++;
    }
    b->timer.end((ns > 0) + (nb > 0));
}

// EM problems of one locus batch on table `table` for the listed local units, appended to `out`.
static void em_problems(hgt_ctx *ctx, int n_launch, LocusBatch &lb, int table, const std::vector<int> &local_units, const int *c_max,
                        const int *a_live, const double *d_len, int remove_low, DevBuf &prob, DevBuf &inres, DevBuf &fk,
                        DevBuf &is, std::vector<EmDevProblem> *out) {
    const hgt_locus *loc = lb.loc;
    const size_t A = (size_t)loc->A;
    const size_t wsb = hgt_em_problem_ws_bytes(loc->wp);
    for (size_t k = 0; k < local_units.size(); k++) {
        const int i = local_units[k];
        const int ut = i * 4 + table;
        EmDevProblem p;
        p.bits = lb.d_bits.as<uint64_t>() + (size_t)lb.ut_base[ut] * loc->wp;
        p.cnt = lb.d_count.as<unsigned long long>() + lb.ut_base[ut];
        p.class_first = lb.d_first.as<int32_t>() + lb.ut_base[ut];
        p.C_ptr = lb.d_ut_ncls.as<int32_t>() + ut;
        p.C_max = std::min<int>(c_max[k], (int)(lb.ut_base[ut + 1] - lb.ut_base[ut]));
        p.A = loc->A;
        p.wp = loc->wp;
        p.A_live_max = a_live[k];
        p.len = d_len;
        p.remove_low = remove_low;
        p.prob = prob.as<double>() + (size_t)i * A;
        p.in_result = inres.as<uint8_t>() + (size_t)i * A;
        p.first_class = fk.as<int32_t>() + (size_t)i * A;
        p.iters_status = is.as<int32_t>() + (size_t)i * 3;
        p.ws = static_cast<unsigned char *>(lb.d_emws.p) + (size_t)i * wsb;
        p.coop_ws = nullptr;
        if (hgt_em_wants_coop(ctx, p.C_max, p.A, p.wp, p.A_live_max, n_launch)) {
            lb.d_coopws.emplace_back();
            if (lb.d_coopws.back().alloc(hgt_em_coop_ws_bytes(ctx, p.A)) == HGT_OK) p.coop_ws = lb.d_coopws.back().p;
        }
        out->push_back(p);
    }
}

static int launch_class_sort(hgt_ctx *ctx, cudaStream_t st, LocusBatch &lb, int table) {
    HGT_CUDA(hgt_smem_at_least((const void *)class_sort_kernel, 2 * CLASS_SORT_MAX * 4));
    int64_t max_pairs = 1;
    for (size_t ut = 0; ut + 1 < lb.ut_base.size(); ut++) max_pairs = std::max<int64_t>(max_pairs, lb.ut_base[ut + 1] - lb.ut_base[ut]);
    const int need = 2 * 4 * (int)std::min<int64_t>(max_pairs, CLASS_SORT_MAX);  // classes of a region <= its pairs
    SortScratch scr;
    scr.bits = lb.d_sortbits.as<uint64_t>(); scr.count = lb.d_sortcnt.as<unsigned long long>(); scr.first = lb.d_sortfirst.as<int32_t>();
    scr.n_active = lb.loc->is_hla ? 4 : 1;
    class_sort_kernel<<<(unsigned)lb.units.size(), CLASS_SORT_THREADS, need, st>>>(lb.pool(), scr, lb.loc->wp, table);
    ctx->launches++;
    HGT_CUDA(cudaGetLastError());
    return HGT_OK;
}

static int batch_execute(hgt_batch *b, cudaStream_t st) {
    hgt_ctx *ctx = b->ctx;
    b->executed = false;
    b->finished = false;
    b->pairs.valid = false;
    if (!b->units.empty()) {
        HGT_CHECK(reads_execute(b, st));
        HGT_CHECK(batch_alloc_tables(b, st));
    }
    for (LocusBatch &lb : b->lb) {
        if (lb.units.empty()) continue;
        const hgt_locus *loc = lb.loc;
        const size_t n_units = lb.units.size();
        const size_t pr = (size_t)std::max<int64_t>(lb.n_rows_pool, 1);
        for (DevBuf &x : lb.d_coopws) x.release();  // (a repeated execute: the previous finish has synchronised)
        lb.d_coopws.clear();
        HGT_CUDA(cudaMemsetAsync(lb.d_keys.p, 0, (size_t)lb.cap * 8, st));
        HGT_CUDA(cudaMemsetAsync(lb.d_count.p, 0, pr * 8, st));
        HGT_CUDA(cudaMemsetAsync(lb.d_first.p, 0x7f, pr * 4, st));
        HGT_CUDA(cudaMemsetAsync(lb.d_ut_ncls.p, 0, n_units * 16, st));
        HGT_CUDA(cudaMemsetAsync(lb.d_is.p, 0, n_units * 12, st));
        switch (wpl_of(loc->wp)) {
            case 1: launch_stage_a<1>(b, st, lb); break;
            case 2: launch_stage_a<2>(b, st, lb); break;
            case 4: launch_stage_a<4>(b, st, lb); break;
            default: launch_stage_a<8>(b, st, lb); break;
        }
        HGT_CUDA(cudaGetLastError());
        b->timer.begin(ctx, st, 2);  // (accounted to the class stage)
        // (the tables an EM runs on: the exon table on the hla path, core:1732; the Gene table otherwise, core:1789; the
        // projected table is ordered after project_kernel)
        HGT_CHECK(launch_class_sort(ctx, st, lb, loc->is_hla ? 1 : 0));
        b->timer.end(1);
        // Gene_counts of the Gene table
        {
            b->timer.begin(ctx, st, 3);
            int64_t max_pairs = 1;
            for (int u : lb.units) max_pairs = std::max<int64_t>(max_pairs, b->units[u].num_pairs);
            // classes per CTA: the serial chain of a CTA is chunk / COUNT_TILE dependent global round trips, so small
            // chunks win as long as the grid (sized from the PAIR bound: class counts are known on the device only) does
            // not drown in empty CTAs
            int chunk = (int)std::min<int64_t>(COUNT_CHUNK_MAX, std::max<int64_t>(COUNT_CHUNK_MIN, (max_pairs / 256 + 63) / 64 * 64));
            while ((max_pairs + chunk - 1) / chunk > 65535) chunk *= 2;
            dim3 grid((loc->A + COUNT_THREADS - 1) / COUNT_THREADS, (unsigned)n_units, (unsigned)((max_pairs + chunk - 1) / chunk));
            HGT_CUDA(cudaMemsetAsync(lb.d_acount.p, 0, n_units * (size_t)loc->A * 8, st));
            HGT_CUDA(cudaMemsetAsync(lb.d_afirst.p, 0x7f, n_units * (size_t)loc->A * 4, st));
            table_counts_kernel<<<grid, COUNT_THREADS, 0, st>>>(loc->A, loc->wp, 0, chunk, lb.pool(), lb.d_acount.as<unsigned long long>(),
                                                      lb.d_afirst.as<int32_t>());
            ctx->launches++;
            b->timer.end(1);
            HGT_CUDA(cudaGetLastError());
        }
        HGT_CUDA(d2h(lb.ut_ncls, lb.d_ut_ncls.p, n_units * 16, st));
    }
    // class counts of every (unit, table) are now known: the one host synchronisation of the GPU stage, it lets the
    // EM launch size each problem's shared memory exactly
    HGT_CUDA(cudaStreamSynchronize(st));
    // first-level EM of every unit of every locus in one go: exon table on the hla path (core:1732-1737), Gene table
    // otherwise (core:1789)
    std::vector<EmDevProblem> probs;
    std::vector<int> all, cmax, alive;
    for (LocusBatch &lb : b->lb) {
        if (lb.units.empty()) continue;
        const hgt_locus *loc = lb.loc;
        const size_t n_units = lb.units.size();
        const int table = loc->is_hla ? 1 : 0;
        all.resize(n_units); cmax.resize(n_units); alive.assign(n_units, lb.n_live[table]);
        std::iota(all.begin(), all.end(), 0);
        for (size_t i = 0; i < n_units; i++) cmax[i] = lb.ut_ncls[i * 4 + table];
        em_problems(ctx, (int)b->units.size(), lb, table, all, cmax.data(), alive.data(), nullptr, loc->is_hla ? b->remove_low : 0, lb.d_prob, lb.d_inres,
                    lb.d_fk, lb.d_is, &probs);
    }
    if (!b->skip_em) {
        b->timer.begin(ctx, st, 4);
        const int64_t l0 = ctx->launches;
        HGT_CHECK(hgt_em_batch_dev(ctx, st, (int)probs.size(), probs.data(), b->h_em_args[0].p, b->d_em_args[0].p));
        b->timer.end((int)(ctx->launches - l0));
    }
    b->executed = true;
    return HGT_OK;
}

// ---- stage 3: results back; on the hla path the second-level EM over full-length alleles (core:1739-1782) -------
static int batch_finish(hgt_batch *b, cudaStream_t st) {
    hgt_ctx *ctx = b->ctx;
    b->pairs.valid = false;
    if (b->skip_em) {
        HGT_CUDA(cudaStreamSynchronize(st));
        b->timer.resolve();
        for (LocusBatch &lb : b->lb) {
            if (lb.units.empty()) continue;
            lb.has2.assign(lb.units.size(), 0);
            for (size_t i = 0; i < lb.units.size() * 3; i++) lb.is[i] = i % 3 == 1 ? 1 : 0;  // status 1 = EM not run
        }
        b->finished = true;
        return HGT_OK;
    }
    for (LocusBatch &lb : b->lb) lb.n_level2 = 0;
    HGT_CHECK(fetch_results(b, st, 0));
    b->timer.resolve();
    HostTimer ht_finish(ctx, 6);
    std::vector<EmDevProblem> probs;
    for (LocusBatch &lb : b->lb) {
        lb.n_level2 = 0;
        if (lb.units.empty() || !lb.loc->is_hla) continue;
        const hgt_locus *loc = lb.loc;
        const size_t n_units = lb.units.size(), A = (size_t)loc->A;
        const int wp = loc->wp;
        // choose exon_alleles per unit (core:1739-1749) from the ranked exon EM result
        int32_t *ulist = lb.h_ulist.as<int32_t>();
        uint64_t *keep = lb.h_keep.as<uint64_t>();
        lb.has2.assign(n_units, 0);
        lb.slot2.assign(n_units, -1);
        lb.exon_prob_sum.assign(n_units, 0.0);
        std::vector<int> lu, cmax, alive;
        std::vector<Ent> order;
        for (size_t i = 0; i < n_units; i++) {
            if (lb.is[i * 3 + 1] != HGT_OK) continue;
            unit_keys(lb, 0, i, &order);
            sort_ranked(&order);
            uint64_t *m = keep + (size_t)lb.n_level2 * wp;
            memset(m, 0, (size_t)wp * 8);
            bool any = false;
            double psum = 0.0;
            for (size_t r = 0; r < order.size(); r++) {
                const int a = order[r].a;
                if (r >= 10 && order[r].p < 0.03) break;
                if (loc->group_off[a + 1] - loc->group_off[a] <= 1) continue;
                any = true;
                psum += order[r].p;
                for (int64_t g = loc->group_off[a]; g < loc->group_off[a + 1]; g++) {
                    const int mem = loc->group_member[g];
                    m[mem >> 6] |= 1ull << (mem & 63);
                }
            }
            if (!any) continue;
            lb.has2[i] = 1;
            lb.slot2[i] = lb.n_level2;
            lb.exon_prob_sum[i] = psum;
            ulist[lb.n_level2++] = (int32_t)i;
            lu.push_back((int)i);
            cmax.push_back(lb.ut_ncls[i * 4 + 0]);  // a projection never has more classes than its source
            int n = 0;
            for (int j = 0; j < wp; j++) n += __builtin_popcountll(m[j]);
            alive.push_back(n);
        }
        if (lb.n_level2 == 0) continue;
        const size_t n2 = (size_t)lb.n_level2;
        if (g_acct) g_acct->h2d_bytes += (int64_t)(n2 * 4 + n2 * wp * 8);
        HGT_CUDA(hgt_small_h2d(lb.d_ulist.p, ulist, n2 * 4, st));
        HGT_CUDA(hgt_small_h2d(lb.d_keep.p, keep, n2 * wp * 8, st));
        {
            b->timer.begin(ctx, st, 5);
            dim3 grid(tune_env("HGT_PROJECT_CTAS", 16), (unsigned)std::min<size_t>(n2, 16384));
            const ClassPool pool = lb.pool();
            switch (wpl_of(wp)) {
                case 1: project_kernel<1><<<grid, WARPS_PER_CTA * 32, 0, st>>>(wp, (int)n2, lb.d_ulist.as<int32_t>(), lb.d_keep.as<uint64_t>(), pool); break;
                case 2: project_kernel<2><<<grid, WARPS_PER_CTA * 32, 0, st>>>(wp, (int)n2, lb.d_ulist.as<int32_t>(), lb.d_keep.as<uint64_t>(), pool); break;
                case 4: project_kernel<4><<<grid, WARPS_PER_CTA * 32, 0, st>>>(wp, (int)n2, lb.d_ulist.as<int32_t>(), lb.d_keep.as<uint64_t>(), pool); break;
                default: project_kernel<8><<<grid, WARPS_PER_CTA * 32, 0, st>>>(wp, (int)n2, lb.d_ulist.as<int32_t>(), lb.d_keep.as<uint64_t>(), pool); break;
            }
            ctx->launches++;
            HGT_CUDA(cudaGetLastError());
            HGT_CHECK(launch_class_sort(ctx, st, lb, 3));
            b->timer.end(2);
        }
        HGT_CUDA(cudaMemsetAsync(lb.d_is2.p, 0, n_units * 12, st));
        em_problems(ctx, (int)b->units.size(), lb, 3, lu, cmax.data(), alive.data(), loc->d_allele_len, 1, lb.d_prob2, lb.d_inres2, lb.d_fk2, lb.d_is2,
                    &probs);
    }
    if (!probs.empty()) {
        b->timer.begin(ctx, st, 6);
        const int64_t l0 = ctx->launches;
        HGT_CHECK(hgt_em_batch_dev(ctx, st, (int)probs.size(), probs.data(), b->h_em_args[1].p, b->d_em_args[1].p));
        b->timer.end((int)(ctx->launches - l0));
        HGT_CHECK(fetch_results(b, st, 1));
        b->timer.resolve();
    }
    b->finished = true;
    return HGT_OK;
}

// ================================================================================================================
// C ABI: batches
// ================================================================================================================
extern "C" int hgt_batch_create(hgt_ctx *ctx, int32_t n_loci, hgt_locus *const *loci, const hgt_params *params,
                                int32_t remove_low, hgt_batch **out) {
    if (!ctx || !loci || n_loci < 1 || !params || !out) {
        hgt_set_error("hgt_batch_create: bad argument");
        return HGT_ERR_ARG;
    }
    for (int i = 0; i < n_loci; i++) {
        if (!loci[i] || !loci[i]->ctx) {
            hgt_set_error("hgt_batch_create: locus %d has no device tables", i);
            return HGT_ERR_ARG;
        }
        if (loci[i]->wp > 256) {
            hgt_set_error("typing kernels support at most 16384 alleles per locus (got %d)", loci[i]->A);
            return HGT_ERR_UNSUPPORTED;
        }
    }
    hgt_batch *b = new hgt_batch();
    b->ctx = ctx;
    b->params = *params;
    b->remove_low = remove_low;
    b->loci.assign(loci, loci + n_loci);
    *out = b;
    return HGT_OK;
}

extern "C" void hgt_batch_free(hgt_batch *b) { delete b; }

extern "C" int hgt_batch_set_pileup_hook(hgt_batch *b, hgt_pileup_hook fn, void *arg) {
    if (!b || b->prepared) {
        hgt_set_error("hgt_batch_set_pileup_hook: bad state");
        return HGT_ERR_ARG;
    }
    b->pileup_hook = fn;
    b->pileup_hook_arg = arg;
    return HGT_OK;
}

extern "C" int64_t hgt_batch_add_unit(hgt_batch *b, int32_t locus_index, const char *sam_text, size_t n_bytes) {
    if (!b || locus_index < 0 || locus_index >= (int)b->loci.size() || (!sam_text && n_bytes) || b->prepared) {
        hgt_set_error("hgt_batch_add_unit: bad argument");
        return HGT_ERR_ARG;
    }
    UnitHost u;
    u.locus = locus_index;
    u.sam = sam_text;
    u.n_bytes = n_bytes;
    b->units.push_back(std::move(u));
    return (int64_t)b->units.size() - 1;
}

extern "C" int64_t hgt_batch_add_unit_bam(hgt_batch *b, int32_t locus_index, const void *blob, size_t n_bytes) {
    if (!b || locus_index < 0 || locus_index >= (int)b->loci.size() || b->prepared) {
        hgt_set_error("hgt_batch_add_unit_bam: bad argument");
        return HGT_ERR_ARG;
    }
    hgtb::BamUnitHeader h;
    if (const char *why = hgtb::bam_unit_check(blob, n_bytes, &h)) {
        hgt_set_error("hgt_batch_add_unit_bam: not a packed BAM unit: %s", why);
        return HGT_ERR_ARG;
    }
    UnitHost u;
    u.locus = locus_index;
    u.blob = blob;
    u.blob_bytes = n_bytes;
    u.n_records = h.n_records;
    b->units.push_back(std::move(u));
    return (int64_t)b->units.size() - 1;
}

extern "C" int64_t hgt_batch_add_unit_bam_dsplit(hgt_batch *b, int32_t locus_index, const hgt_bam_dsplit *s, int32_t stream,
                                                 int32_t ref) {
    if (!b || locus_index < 0 || locus_index >= (int)b->loci.size() || b->prepared || !s) {
        hgt_set_error("hgt_batch_add_unit_bam_dsplit: bad argument");
        return HGT_ERR_ARG;
    }
    UnitHost u;
    int device = -1;
    if (bam_dsplit_unit(s, stream, ref, &u.dsu, &u.n_records, &u.n_bytes, &device) != HGT_OK) {
        hgt_set_error("hgt_batch_add_unit_bam_dsplit: stream %d / reference %d outside the split", stream, ref);
        return HGT_ERR_ARG;
    }
    if (device != b->ctx->device) {
        hgt_set_error("hgt_batch_add_unit_bam_dsplit: the split is on device %d, the batch on device %d", device, b->ctx->device);
        return HGT_ERR_ARG;
    }
    u.locus = locus_index;
    u.ds = s;
    b->units.push_back(std::move(u));
    return (int64_t)b->units.size() - 1;
}

extern "C" int hgt_batch_unit_text(const hgt_batch *b, int64_t unit, char *dst, size_t *n_bytes) {
    if (!b || !b->prepared || unit < 0 || unit >= (int64_t)b->units.size() || !n_bytes) {
        hgt_set_error("hgt_batch_unit_text: bad argument or batch not prepared");
        return HGT_ERR_ARG;
    }
    const UnitHost &U = b->units[(size_t)unit];
    if (!dst) {
        *n_bytes = U.n_bytes;
        return HGT_OK;
    }
    if (*n_bytes < U.n_bytes) {
        hgt_set_error("hgt_batch_unit_text: buffer of %zu bytes for %zu bytes of text", *n_bytes, U.n_bytes);
        return HGT_ERR_ARG;
    }
    *n_bytes = U.n_bytes;
    if (!U.n_bytes) return HGT_OK;
    HGT_CUDA(cudaSetDevice(b->ctx->device));
    g_acct = b->ctx;
    HGT_CUDA(d2h(dst, b->rd.d_text.as<char>() + b->rd.unit_off[(size_t)U.arena], U.n_bytes, b->ctx->stream));
    HGT_CUDA(cudaStreamSynchronize(b->ctx->stream));
    return HGT_OK;
}

extern "C" int64_t hgt_batch_add_units(hgt_batch *b, int64_t n, const int32_t *locus_index, const char *const *sam_text,
                                       const size_t *n_bytes) {
    if (!b || n < 0 || (n > 0 && (!locus_index || !sam_text || !n_bytes))) {
        hgt_set_error("hgt_batch_add_units: bad argument");
        return HGT_ERR_ARG;
    }
    const int64_t first = (int64_t)b->units.size();
    for (int64_t k = 0; k < n; k++) {
        const int64_t u = hgt_batch_add_unit(b, locus_index[k], sam_text[k], n_bytes[k]);
        if (u < 0) {
            b->units.resize((size_t)first);
            return u;
        }
    }
    return first;
}

extern "C" int hgt_batch_prepare(hgt_batch *b) {
    if (!b || b->prepared) {
        hgt_set_error("hgt_batch_prepare: bad state");
        return HGT_ERR_ARG;
    }
    HGT_CUDA(cudaSetDevice(b->ctx->device));
    g_acct = b->ctx;
    return batch_prepare(b);
}

extern "C" int hgt_batch_execute(hgt_batch *b, void *stream) {
    if (!b || !b->prepared) {
        hgt_set_error("hgt_batch_execute: batch is not prepared");
        return HGT_ERR_ARG;
    }
    HGT_CUDA(cudaSetDevice(b->ctx->device));
    g_acct = b->ctx;
    return batch_execute(b, stream ? static_cast<cudaStream_t>(stream) : b->ctx->stream);
}

extern "C" int hgt_batch_finish(hgt_batch *b, void *stream) {
    if (!b || !b->executed) {
        hgt_set_error("hgt_batch_finish: batch was not executed");
        return HGT_ERR_ARG;
    }
    if (b->finished) {  // a second finish would project into the same table-3 regions again and double their counts
        hgt_set_error("hgt_batch_finish: already finished; call hgt_batch_execute again first");
        return HGT_ERR_ARG;
    }
    HGT_CUDA(cudaSetDevice(b->ctx->device));
    g_acct = b->ctx;
    return batch_finish(b, stream ? static_cast<cudaStream_t>(stream) : b->ctx->stream);
}

extern "C" int hgt_batch_run(hgt_batch *b) {
    HGT_CHECK(hgt_batch_prepare(b));
    HGT_CHECK(hgt_batch_execute(b, nullptr));
    return hgt_batch_finish(b, nullptr);
}

extern "C" int hgt_batch_totals(const hgt_batch *b, int64_t *n_units, int64_t *num_reads, int64_t *num_pairs,
                                int64_t *n_haplotypes, int64_t *n_rows, int64_t *algorithmic_bytes) {
    if (!b) return HGT_ERR_ARG;
    int64_t r = 0, p = 0, h = 0, rows = 0, bytes = 0;
    for (const UnitHost &u : b->units) {
        r += u.num_reads;
        p += u.num_pairs;
    }
    for (const LocusBatch &lb : b->lb) {
        if (lb.units.empty()) continue;
        h += lb.n_haps;
        rows += lb.n_rows;
        const int n_tables = lb.loc->is_hla ? 3 : 1;
        // SURVEY.md 8d: per pair S_rec + T * wp * 8, S_rec = packed haplotype records actually read
        bytes += lb.n_haps * 12 + lb.n_rows * 4 + lb.n_jobs * 16;
        for (int u : lb.units) bytes += b->units[u].num_pairs * (int64_t)n_tables * lb.loc->wp * 8;
    }
    if (n_units) *n_units = (int64_t)b->units.size();
    if (num_reads) *num_reads = r;
    if (num_pairs) *num_pairs = p;
    if (n_haplotypes) *n_haplotypes = h;
    if (n_rows) *n_rows = rows;
    if (algorithmic_bytes) *algorithmic_bytes = bytes;
    return HGT_OK;
}

extern "C" int hgt_batch_job_stats(const hgt_batch *b, int64_t out[4]) {
    if (!b || !out || !b->prepared) {
        hgt_set_error("hgt_batch_job_stats: batch is not prepared");
        return HGT_ERR_ARG;
    }
    out[0] = out[1] = out[2] = out[3] = 0;
    for (const LocusBatch &lb : b->lb) {
        out[0] += lb.n_jobs;
        out[1] += lb.n_big;
        out[2] = std::max(out[2], lb.max_job_haps);
        out[3] += lb.n_haps;
    }
    return HGT_OK;
}

static int unit_check(const hgt_batch *b, int64_t unit, bool need_finish) {
    if (!b || unit < 0 || unit >= (int64_t)b->units.size() || (need_finish && !b->finished)) {
        hgt_set_error("batch accessor: bad unit index or batch not finished");
        return HGT_ERR_ARG;
    }
    return HGT_OK;
}

extern "C" int hgt_batch_unit_summary(const hgt_batch *b, int64_t unit, int64_t *num_reads, int64_t *num_pairs,
                                      int32_t n_classes[4], int32_t em_iters[2], int32_t em_status[2]) {
    HGT_CHECK(unit_check(b, unit, false));
    const UnitHost &U = b->units[unit];
    if (num_reads) *num_reads = U.num_reads;
    if (num_pairs) *num_pairs = U.num_pairs;
    if (b->finished) {
        const LocusBatch &lb = b->lb[U.locus];
        for (int t = 0; t < 4; t++) {
            const int64_t room = lb.ut_base[(size_t)U.local * 4 + t + 1] - lb.ut_base[(size_t)U.local * 4 + t];
            if (n_classes) n_classes[t] = (int32_t)std::min<int64_t>(lb.ut_ncls[(size_t)U.local * 4 + t], room);
        }
        if (em_iters) {
            em_iters[0] = lb.is[(size_t)U.local * 3];
            em_iters[1] = (!lb.has2.empty() && lb.has2[U.local]) ? lb.is2[(size_t)U.local * 3] : 0;
        }
        if (em_status) {
            em_status[0] = lb.is[(size_t)U.local * 3 + 1];
            em_status[1] = (!lb.has2.empty() && lb.has2[U.local]) ? lb.is2[(size_t)U.local * 3 + 1] : 0;
        }
    }
    return HGT_OK;
}

// Per-read haplotypes of a unit: what the reference's typing() holds per surviving alignment when it builds the assembly
// nodes (left_positive_hts / right_positive_hts of the read, core:1386-1406 -> :1408-1540).  Read back from the record
// stage's device arrays (the walk's output), slow records expanded to left ends x middle x right ends.
extern "C" int hgt_batch_unit_reads(hgt_batch *b, int64_t unit, int64_t *n_records, int64_t *n_haps, int64_t *n_ids,
                                    int64_t *rec_line, int32_t *rec_flag, int64_t *rec_hap_off, int32_t *hap_left,
                                    int32_t *hap_right, int64_t *hap_id_off, int32_t *ids) {
    if (!b || unit < 0 || unit >= (int64_t)b->units.size() || !b->executed) {
        hgt_set_error("hgt_batch_unit_reads: bad unit index or batch not executed");
        return HGT_ERR_ARG;
    }
    using namespace hgtd;
    HGT_CUDA(cudaSetDevice(b->ctx->device));
    cudaStream_t st = b->ctx->stream;
    ReadsDev &rd = b->rd;
    const UnitHost &U = b->units[unit];
    const size_t N = (size_t)rd.n_lines;
    int64_t l01[2] = {0, 0};
    HGT_CUDA(cudaMemcpyAsync(l01, reinterpret_cast<int64_t *>(static_cast<unsigned char *>(rd.d_units.p) + rd.o_uline0) + U.arena, 16,
                             cudaMemcpyDeviceToHost, st));
    HGT_CUDA(cudaStreamSynchronize(st));
    const size_t l0 = (size_t)l01[0], n = (size_t)(l01[1] - l01[0]);
    std::vector<uint16_t> stv(std::max<size_t>(n, 1));
    std::vector<RecFields> rec(std::max<size_t>(n, 1));
    std::vector<int32_t> hl(std::max<size_t>(n, 1)), hr(hl.size()), hn(hl.size()), slot(hl.size()), hid(hl.size() * MAXI);
    if (n > 0) {
        const int32_t *hdr = rd.d_hdr.as<int32_t>();
        HGT_CUDA(cudaMemcpyAsync(stv.data(), rd.d_st.as<uint16_t>() + l0, n * 2, cudaMemcpyDeviceToHost, st));
        HGT_CUDA(cudaMemcpyAsync(rec.data(), rd.d_rec.as<RecFields>() + l0, n * sizeof(RecFields), cudaMemcpyDeviceToHost, st));
        HGT_CUDA(cudaMemcpyAsync(hl.data(), hdr + l0, n * 4, cudaMemcpyDeviceToHost, st));
        HGT_CUDA(cudaMemcpyAsync(hr.data(), hdr + N + l0, n * 4, cudaMemcpyDeviceToHost, st));
        HGT_CUDA(cudaMemcpyAsync(hn.data(), hdr + 2 * N + l0, n * 4, cudaMemcpyDeviceToHost, st));
        HGT_CUDA(cudaMemcpyAsync(slot.data(), hdr + 3 * N + l0, n * 4, cudaMemcpyDeviceToHost, st));
        HGT_CUDA(cudaMemcpyAsync(hid.data(), rd.d_hids.as<int32_t>() + l0 * MAXI, n * MAXI * 4, cudaMemcpyDeviceToHost, st));
        HGT_CUDA(cudaStreamSynchronize(st));
    }
    std::vector<SlowRec> slow;
    std::vector<int64_t> slow_of(n, -1);
    for (size_t i = 0; i < n; i++)
        if ((stv[i] & ST_SURV) && slot[i] >= 0) {
            slow_of[i] = (int64_t)slow.size();
            slow.emplace_back();
            HGT_CUDA(cudaMemcpyAsync(&slow.back(), rd.d_slow.as<SlowRec>() + slot[i], sizeof(SlowRec), cudaMemcpyDeviceToHost, st));
            HGT_CUDA(cudaStreamSynchronize(st));  // (emplace_back may move the vector: one record at a time)
        }
    int64_t nr = 0, nh = 0, ni = 0;
    for (size_t i = 0; i < n; i++) {
        if (!(stv[i] & ST_SURV)) continue;
        if (rec_line) rec_line[nr] = (int64_t)i;
        if (rec_flag) rec_flag[nr] = rec[i].flag;
        if (rec_hap_off) rec_hap_off[nr] = nh;
        if (slow_of[i] < 0) {
            if (hap_left) hap_left[nh] = hl[i];
            if (hap_right) hap_right[nh] = hr[i];
            if (hap_id_off) hap_id_off[nh] = ni;
            for (int k = 0; k < hn[i]; k++, ni++)
                if (ids) ids[ni] = hid[i * MAXI + k];
            nh++;
        } else {
            const SlowRec &S = slow[(size_t)slow_of[i]];
            for (int a = 0; a < S.e.n_left; a++)
                for (int c = 0; c < S.e.n_right; c++) {
                    if (hap_left) hap_left[nh] = S.e.left[a].pos;
                    if (hap_right) hap_right[nh] = S.e.right[c].pos;
                    if (hap_id_off) hap_id_off[nh] = ni;
                    for (int k = 0; k < S.e.left[a].n; k++, ni++)
                        if (ids) ids[ni] = S.e.left[a].ids[k];
                    for (int k = 0; k < S.n_mid; k++, ni++)
                        if (ids) ids[ni] = S.mid[k];
                    for (int k = 0; k < S.e.right[c].n; k++, ni++)
                        if (ids) ids[ni] = S.e.right[c].ids[k];
                    nh++;
                }
        }
        nr++;
    }
    if (rec_hap_off) rec_hap_off[nr] = nh;
    if (hap_id_off) hap_id_off[nh] = ni;
    if (n_records) *n_records = nr;
    if (n_haps) *n_haps = nh;
    if (n_ids) *n_ids = ni;
    return HGT_OK;
}

extern "C" int hgt_batch_unit_table(hgt_batch *b, int64_t unit, int32_t table, uint64_t *class_bits, int64_t *class_count,
                                    int64_t *class_first, int64_t *allele_count, int64_t *allele_first) {
    HGT_CHECK(unit_check(b, unit, true));
    if (table < 0 || table > 3) {
        hgt_set_error("hgt_batch_unit_table: table must be 0..3");
        return HGT_ERR_ARG;
    }
    const UnitHost &U = b->units[unit];
    LocusBatch &lb = b->lb[U.locus];
    const hgt_locus *loc = lb.loc;
    HGT_CUDA(cudaSetDevice(b->ctx->device));
    cudaStream_t st = b->ctx->stream;
    const int ut = U.local * 4 + table;
    const int64_t base = lb.ut_base[ut];
    const int n = (int)std::min<int64_t>(lb.ut_ncls[ut], lb.ut_base[ut + 1] - base);
    const int wp = loc->wp, A = loc->A;
    std::vector<uint64_t> bits((size_t)std::max(n, 1) * wp);
    std::vector<unsigned long long> cnt(std::max(n, 1));
    std::vector<int32_t> first(std::max(n, 1));
    if (n > 0) {
        HGT_CUDA(cudaMemcpyAsync(bits.data(), lb.d_bits.as<uint64_t>() + (size_t)base * wp, (size_t)n * wp * 8,
                                 cudaMemcpyDeviceToHost, st));
        HGT_CUDA(d2h(cnt.data(), lb.d_count.as<unsigned long long>() + base, (size_t)n * 8, st));
        HGT_CUDA(d2h(first.data(), lb.d_first.as<int32_t>() + base, (size_t)n * 4, st));
    }
    std::vector<long long> ac;
    std::vector<int32_t> af;
    if ((allele_count || allele_first) && table == 0) {
        ac.resize(A);
        af.resize(A);
        HGT_CUDA(d2h(ac.data(), lb.d_acount.as<long long>() + (size_t)U.local * A, (size_t)A * 8, st));
        HGT_CUDA(d2h(af.data(), lb.d_afirst.as<int32_t>() + (size_t)U.local * A, (size_t)A * 4, st));
    }
    HGT_CUDA(cudaStreamSynchronize(st));
    // dict order = first-seen order (each pair creates at most one class per table, so `first` is a strict key)
    std::vector<int> order(n);
    std::iota(order.begin(), order.end(), 0);
    std::sort(order.begin(), order.end(), [&](int x, int y) { return first[x] < first[y]; });
    for (int k = 0; k < n; k++) {
        const int c = order[k];
        if (class_bits) memcpy(class_bits + (size_t)k * wp, &bits[(size_t)c * wp], (size_t)wp * 8);
        if (class_count) class_count[k] = (int64_t)cnt[c];
        if (class_first) class_first[k] = first[c];
    }
    if (allele_count || allele_first) {
        if (table == 0) {
            for (int a = 0; a < A; a++) {
                if (allele_count) allele_count[a] = ac[a];
                if (allele_first) allele_first[a] = ac[a] ? af[a] : -1;
            }
        } else {  // other tables: derive from the class rows just read
            for (int a = 0; a < A; a++) {
                int64_t c = 0, f = -1;
                for (int k = 0; k < n; k++)
                    if ((bits[(size_t)k * wp + (a >> 6)] >> (a & 63)) & 1ull) {
                        c += (int64_t)cnt[k];
                        if (f < 0 || first[k] < f) f = first[k];
                    }
                if (allele_count) allele_count[a] = c;
                if (allele_first) allele_first[a] = f;
            }
        }
    }
    return HGT_OK;
}

extern "C" int hgt_batch_set_skip_em(hgt_batch *b, int32_t skip) {
    if (!b) return HGT_ERR_ARG;
    b->skip_em = skip != 0;
    return HGT_OK;
}

extern "C" int hgt_batch_unit_table_dev(const hgt_batch *b, int64_t unit, int32_t table, const uint64_t **class_bits,
                                        const uint64_t **class_count, const int32_t **class_first, int32_t *n_classes) {
    HGT_CHECK(unit_check(b, unit, true));
    if (table < 0 || table > 3) {
        hgt_set_error("hgt_batch_unit_table_dev: table must be 0..3");
        return HGT_ERR_ARG;
    }
    const UnitHost &U = b->units[unit];
    const LocusBatch &lb = b->lb[U.locus];
    const int ut = U.local * 4 + table;
    const int64_t base = lb.ut_base[ut];
    if (class_bits) *class_bits = lb.d_bits.as<uint64_t>() + (size_t)base * lb.loc->wp;
    if (class_count) *class_count = lb.d_count.as<uint64_t>() + base;
    if (class_first) *class_first = lb.d_first.as<int32_t>() + base;
    if (n_classes) *n_classes = (int32_t)std::min<int64_t>(lb.ut_ncls[ut], lb.ut_base[ut + 1] - base);
    return HGT_OK;
}

// Diploid pair calls of every unit (pair_batch.cu) on table 0, 1 or 2 of a finished batch, read in place.
extern "C" int hgt_batch_pairs(hgt_batch *b, int32_t table, int64_t max_pairs, int32_t cap, int32_t *allele_lo,
                               int32_t *allele_hi, double *prob, int32_t *n_total, int32_t *iters, int32_t *status) {
    if (!b || !b->finished || table < 0 || table > 2 || max_pairs < 0 || cap < 0 || !n_total || !iters || !status ||
        (cap > 0 && (!allele_lo || !allele_hi || !prob))) {
        hgt_set_error("hgt_batch_pairs: bad argument, table outside 0..2 or batch not finished");
        return HGT_ERR_ARG;
    }
    HGT_CUDA(cudaSetDevice(b->ctx->device));
    std::vector<std::shared_ptr<NameRel>> names(b->lb.size());
    for (size_t i = 0; i < b->lb.size(); i++)
        if (!b->lb[i].units.empty()) HGT_CHECK(locus_names_dev(b->lb[i].loc, b->ctx->device, &names[i]));
    auto &pc = b->pairs;
    if (!(pc.valid && pc.table == table && pc.max_pairs == max_pairs && pc.names == names)) {
        pc.valid = false;
        std::vector<PairUnit> units(b->units.size());
        for (size_t u = 0; u < b->units.size(); u++) {
            const UnitHost &U = b->units[u];
            const LocusBatch &lb = b->lb[U.locus];
            const hgt_locus *loc = lb.loc;
            const NameRel &rel = *names[U.locus];
            const int ut = U.local * 4 + table;
            const int64_t base = lb.ut_base[ut];
            PairUnit &P = units[u];
            P.C = (int32_t)std::min<int64_t>(lb.ut_ncls[ut], lb.ut_base[ut + 1] - base);
            P.A = loc->A;
            P.wp = loc->wp;
            P.bits = lb.d_bits.as<uint64_t>() + (size_t)base * loc->wp;
            P.count = lb.d_count.as<unsigned long long>() + base;
            P.first = lb.d_first.as<int32_t>() + base;
            P.sub_off = rel.d_sub_off; P.sub_idx = rel.d_sub_idx;
            P.sup_off = rel.d_sup_off; P.sup_idx = rel.d_sup_idx;
        }
        HGT_CHECK(hgt_pair_batch_run(b->ctx, b->ctx->stream, units, max_pairs, std::max(cap, 16), &pc.r));
        pc.table = table;
        pc.max_pairs = max_pairs;
        pc.names = std::move(names);
        pc.valid = true;
    }
    const PairResult &r = pc.r;
    for (size_t u = 0; u < b->units.size(); u++) {
        n_total[u] = r.n_total[u];
        iters[u] = r.iters[u];
        status[u] = r.status[u];
        const int64_t o = r.off[u];
        for (int32_t k = 0; k < cap && k < r.n_total[u]; k++) {
            allele_lo[u * (size_t)cap + k] = r.lo[o + k];
            allele_hi[u * (size_t)cap + k] = r.hi[o + k];
            prob[u * (size_t)cap + k] = r.p[o + k];
        }
    }
    return HGT_OK;
}

extern "C" int hgt_batch_pair_sizes(const hgt_batch *b, int64_t *n_pairs) {
    if (!b || !n_pairs || !b->pairs.valid) {
        hgt_set_error("hgt_batch_pair_sizes: no hgt_batch_pairs result on this batch");
        return HGT_ERR_ARG;
    }
    std::copy(b->pairs.r.n_pairs.begin(), b->pairs.r.n_pairs.end(), n_pairs);
    return HGT_OK;
}

extern "C" int hgt_batch_unit_em(const hgt_batch *b, int64_t unit, int32_t level, double *prob, uint8_t *in_result,
                                 int32_t *first_class, int32_t *iters, int32_t *status) {
    HGT_CHECK(unit_check(b, unit, true));
    const UnitHost &U = b->units[unit];
    const LocusBatch &lb = b->lb[U.locus];
    const size_t A = (size_t)lb.loc->A, o = (size_t)U.local * A;
    // dense view of a result that came back as a key list
    auto scatter = [&](int lv) {
        if (prob) memset(prob, 0, A * 8);
        if (in_result) memset(in_result, 0, A);
        if (first_class)
            for (size_t a = 0; a < A; a++) first_class[a] = 0x7fffffff;
        std::vector<Ent> keys;
        unit_keys(lb, lv, (size_t)U.local, &keys);
        for (const Ent &e : keys) {
            if (prob) prob[e.a] = e.p;
            if (in_result) in_result[e.a] = 1;
            if (first_class) first_class[e.a] = e.fk;
        }
    };
    if (level == 0) {
        if (!lb.dense[0] && lb.is[(size_t)U.local * 3 + 1] == HGT_OK) {
            scatter(0);
        } else {
            if (prob) memcpy(prob, &lb.prob[o], A * 8);
            if (in_result) memcpy(in_result, &lb.inres[o], A);
            if (first_class) memcpy(first_class, &lb.fk[o], A * 4);
        }
        if (iters) *iters = lb.is[(size_t)U.local * 3];
        if (status) *status = lb.is[(size_t)U.local * 3 + 1];
        return HGT_OK;
    }
    if (lb.has2.empty() || !lb.has2[U.local]) {
        if (status) *status = 1;  // not run: no exon group with more than one member was selected (core:1752)
        if (iters) *iters = 0;
        return HGT_OK;
    }
    if (!lb.dense[1] && lb.is2[(size_t)U.local * 3 + 1] == HGT_OK) {
        scatter(1);
    } else {
        if (prob) memcpy(prob, &lb.prob2[o], A * 8);
        if (in_result) memcpy(in_result, &lb.inres2[o], A);
        if (first_class) memcpy(first_class, &lb.fk2[o], A * 4);
    }
    if (iters) *iters = lb.is2[(size_t)U.local * 3];
    if (status) *status = lb.is2[(size_t)U.local * 3 + 1];
    return HGT_OK;
}

// Gene_prob of one unit, ranked: the combination rule of core:1771-1782 on the hla path (first-level entries
// outside exon_alleles, then second-level entries scaled by exon_prob_sum, stable sort by probability), the plain
// EM result otherwise.  Writes at most `cap` entries; *n_total receives the full length.
extern "C" int hgt_batch_unit_abundance(const hgt_batch *b, int64_t unit, int32_t cap, int32_t *allele, double *prob,
                                        int32_t *n_total) {
    HGT_CHECK(unit_check(b, unit, true));
    const UnitHost &U = b->units[unit];
    const LocusBatch &lb = b->lb[U.locus];
    const hgt_locus *loc = lb.loc;
    const size_t A = (size_t)loc->A, o = (size_t)U.local * A;
    const int st1 = lb.is[(size_t)U.local * 3 + 1];
    if (st1 != HGT_OK) return st1;
    auto ranked = [&](int lv, std::vector<Ent> *out) {
        unit_keys(lb, lv, (size_t)U.local, out);
        sort_ranked(out);
    };
    std::vector<Ent> first, second, comb;
    ranked(0, &first);
    const bool two = loc->is_hla && !lb.has2.empty() && lb.has2[U.local];
    if (!two) {
        comb.swap(first);
    } else {
        const int st2 = lb.is2[(size_t)U.local * 3 + 1];
        if (st2 != HGT_OK) return st2;
        ranked(1, &second);
        const uint64_t *keep = lb.h_keep.as<uint64_t>() + (size_t)lb.slot2[U.local] * loc->wp;
        for (const Ent &e : first)
            if (!((keep[e.a >> 6] >> (e.a & 63)) & 1ull)) comb.push_back(e);
        for (const Ent &e : second) comb.push_back({e.a, e.p * lb.exon_prob_sum[U.local], 0});
        std::stable_sort(comb.begin(), comb.end(), [](const Ent &x, const Ent &y) { return x.p > y.p; });
    }
    if (n_total) *n_total = (int32_t)comb.size();
    for (int32_t k = 0; k < cap && k < (int32_t)comb.size(); k++) {
        if (allele) allele[k] = comb[k].a;
        if (prob) prob[k] = comb[k].p;
    }
    return HGT_OK;
}

extern "C" int hgt_batch_abundances(const hgt_batch *b, int32_t cap, int32_t *allele, double *prob, int32_t *n_total,
                                    int32_t *status) {
    if (!b || !b->finished || cap < 0 || !n_total || !status || (cap > 0 && (!allele || !prob))) {
        hgt_set_error("hgt_batch_abundances: bad argument or batch not finished");
        return HGT_ERR_ARG;
    }
    const int64_t nu = (int64_t)b->units.size();
    parallel_units(std::min<int>(batch_threads(b->params), 8), (size_t)nu, [&](size_t u) {
        status[u] = hgt_batch_unit_abundance(b, (int64_t)u, cap, allele + u * (size_t)cap, prob + u * (size_t)cap, &n_total[u]);
    });
    return HGT_OK;
}

// ================================================================================================================
// C ABI: single (sample, locus) — a batch of one unit
// ================================================================================================================
struct hgt_typing {
    hgt_batch *batch = nullptr;
};

extern "C" void hgt_typing_free(hgt_typing *t) {
    if (!t) return;
    delete t->batch;
    delete t;
}

extern "C" int hgt_typing_run(hgt_ctx *ctx, hgt_locus *loc, const char *sam, size_t n_bytes, const hgt_params *params,
                              hgt_typing **out) {
    if (!ctx || !loc || !params || !out || (!sam && n_bytes)) {
        hgt_set_error("hgt_typing_run: null argument");
        return HGT_ERR_ARG;
    }
    *out = nullptr;
    hgt_batch *b = nullptr;
    hgt_locus *loci[1] = {loc};
    HGT_CHECK(hgt_batch_create(ctx, 1, loci, params, 1, &b));
    b->keep_counts = true;
    int rc = (int)hgt_batch_add_unit(b, 0, sam, n_bytes);
    if (rc >= 0) rc = hgt_batch_prepare(b);
    if (rc == HGT_OK) rc = hgt_batch_execute(b, nullptr);
    if (rc == HGT_OK) rc = hgt_batch_finish(b, nullptr);
    if (rc != HGT_OK) {
        delete b;
        return rc;
    }
    hgt_typing *t = new hgt_typing();
    t->batch = b;
    *out = t;
    return HGT_OK;
}

extern "C" int hgt_typing_summary(const hgt_typing *t, int64_t *num_reads, int64_t *num_pairs, int32_t n_classes[3]) {
    if (!t) return HGT_ERR_ARG;
    int32_t nc[4] = {0, 0, 0, 0};
    HGT_CHECK(hgt_batch_unit_summary(t->batch, 0, num_reads, num_pairs, nc, nullptr, nullptr));
    if (n_classes)
        for (int i = 0; i < 3; i++) n_classes[i] = nc[i];
    return HGT_OK;
}

extern "C" int hgt_typing_pileup(const hgt_typing *t, uint32_t *counts, uint8_t *nt_mask) {
    if (!t) return HGT_ERR_ARG;
    const UnitHost &U = t->batch->units[0];
    if (counts) memcpy(counts, U.counts.data(), U.counts.size() * 4);
    if (nt_mask && !U.nt_mask.empty()) memcpy(nt_mask, U.nt_mask.data(), U.nt_mask.size());
    return HGT_OK;
}

extern "C" int hgt_typing_table(const hgt_typing *t, int32_t table, uint64_t *class_bits, int64_t *class_count,
                                int64_t *class_first, int64_t *allele_count, int64_t *allele_first) {
    if (!t || table < 0 || table > 2) {
        hgt_set_error("hgt_typing_table: bad argument");
        return HGT_ERR_ARG;
    }
    return hgt_batch_unit_table(t->batch, 0, table, class_bits, class_count, class_first, allele_count, allele_first);
}

extern "C" int hgt_typing_em(hgt_ctx *ctx, const hgt_typing *t, int32_t table, const uint64_t *keep_mask,
                             const double *allele_len, int32_t remove_low, double *prob, uint8_t *in_result,
                             int32_t *first_class, int32_t *iters) {
    if (!ctx || !t || table < 0 || table > 2) {
        hgt_set_error("hgt_typing_em: bad argument");
        return HGT_ERR_ARG;
    }
    const hgt_locus *loc = t->batch->loci[0];
    const int wp = loc->wp, A = loc->A;
    int32_t nc[4] = {0, 0, 0, 0};
    HGT_CHECK(hgt_batch_unit_summary(t->batch, 0, nullptr, nullptr, nc, nullptr, nullptr));
    const int n = nc[table];
    std::vector<uint64_t> bits((size_t)std::max(n, 1) * wp);
    std::vector<int64_t> cnt(std::max(n, 1));
    HGT_CHECK(hgt_batch_unit_table(t->batch, 0, table, bits.data(), cnt.data(), nullptr, nullptr, nullptr));
    int m = n;
    if (keep_mask) {
        // project classes onto the kept alleles, merge equal keys in first-seen order (core:1753-1766)
        std::unordered_map<std::string, int> where;
        std::vector<uint64_t> b2;
        std::vector<int64_t> c2;
        for (int k = 0; k < n; k++) {
            bool any = false;
            for (int j = 0; j < wp; j++) {
                bits[(size_t)k * wp + j] &= keep_mask[j];
                any |= bits[(size_t)k * wp + j] != 0;
            }
            if (!any) continue;
            std::string key(reinterpret_cast<const char *>(&bits[(size_t)k * wp]), (size_t)wp * 8);
            auto f = where.find(key);
            if (f == where.end()) {
                where.emplace(std::move(key), (int)c2.size());
                b2.insert(b2.end(), bits.begin() + (size_t)k * wp, bits.begin() + (size_t)(k + 1) * wp);
                c2.push_back(cnt[k]);
            } else {
                c2[f->second] += cnt[k];
            }
        }
        bits.swap(b2);
        cnt.swap(c2);
        m = (int)cnt.size();
    }
    return hgt_em(ctx, bits.data(), cnt.data(), m, A, wp, allele_len, remove_low, prob, in_result, first_class, iters);
}

// ================================================================================================================
// Host emulation of the record stage (tests of the device logic without a GPU)
// ================================================================================================================
// hgt_host_walk runs the SAME __host__ __device__ functions the kernels call (walk_dev.cuh) in plain loops over host
// memory, with a caller-supplied pileup.  It exists for tests/test_host_walk.py (no GPU in that environment); nothing
// on the typing path calls it.
struct hgt_walk {
    int64_t num_reads = 0, num_pairs = 0;
    struct Tab {
        std::vector<int64_t> job_off{0}, row_off{0};
        std::vector<int32_t> hap_left, hap_right, rows;
    } tb[3];
};

extern "C" int hgt_host_walk(hgt_locus *loc, const char *sam, size_t n_bytes, const hgt_params *params,
                             const uint32_t *counts, const uint8_t *nt_mask, hgt_walk **out) {
    using namespace hgtd;
    if (!loc || !params || !out || !counts || !nt_mask || (!sam && n_bytes)) {
        hgt_set_error("hgt_host_walk: null argument");
        return HGT_ERR_ARG;
    }
    *out = nullptr;
    // arena: the text plus at least one closing newline, padded to 16 bytes
    std::vector<char> text(a16(n_bytes + 1), '\n');
    if (n_bytes) memcpy(text.data(), sam, n_bytes);
    std::vector<int64_t> line_off{0};
    for (size_t i = 0; i < text.size(); i++)
        if (text[i] == '\n') line_off.push_back((int64_t)i + 1);
    const int64_t N = (int64_t)line_off.size() - 1;
    const size_t n1 = (size_t)std::max<int64_t>(N, 1);
    std::vector<uint8_t> flag(loc->L);
    for (int i = 0; i < loc->L; i++) {
        const uint32_t *c = counts + (size_t)i * 6;
        const uint64_t dels = c[5], nts = (uint64_t)c[0] + c[1] + c[2] + c[3] + c[4];
        flag[i] = dels * 6 < nts ? 1 : 0;
    }
    std::vector<int32_t> unit(n1), hdr(n1 * 4), hids(n1 * MAXI), slow_list(n1), amb_list(n1), head_list(n1);
    std::vector<RecFields> rec(n1);
    std::vector<uint16_t> stv(n1);
    std::vector<int64_t> scan((size_t)(N + 1) * 5, 0);
    int64_t unit_off[2] = {0, (int64_t)text.size()}, unit_line0[2] = {0, N}, unit_pos0[2] = {0, 0};
    int32_t unit_locus[1] = {0}, unit_local[1] = {0}, n_slow = 0, n_amb = 0, n_heads = 0, max_job = 0;
    unsigned long long err = ~0ull, unit_reads[1] = {0}, unit_pairs[1] = {0};
    LocusJobs jobs;
    memset(&jobs, 0, sizeof(jobs));
    ReadsView R;
    memset(&R, 0, sizeof(R));
    R.text = text.data(); R.n_lines = N; R.line_off = line_off.data();
    R.unit = unit.data(); R.rec = rec.data(); R.st = stv.data();
    R.h_left = hdr.data(); R.h_right = R.h_left + n1; R.h_n = R.h_right + n1; R.slow_slot = R.h_n + n1;
    R.h_ids = hids.data(); R.slow_list = slow_list.data(); R.n_slow = &n_slow;
    R.amb_list = amb_list.data(); R.n_amb = &n_amb;
    std::vector<int32_t> pair_cnt((size_t)n1 * 3);
    R.pair_cnt = pair_cnt.data();
    R.head_list = head_list.data(); R.n_heads = &n_heads;
    R.n_units = 1; R.unit_off = unit_off; R.unit_line0 = unit_line0; R.unit_locus = unit_locus; R.unit_local = unit_local;
    R.unit_pos0 = unit_pos0; R.nt_mask = nt_mask; R.del_flag = flag.data(); R.loci = &loc->wt_host;
    R.err = &err; R.unit_reads = unit_reads; R.unit_pairs = unit_pairs;
    R.s_pairs = scan.data(); R.s_haps = R.s_pairs + (N + 1); R.s_rows = R.s_haps + (N + 1); R.s_small = R.s_rows + (N + 1);
    R.s_big = R.s_small + (N + 1);
    R.max_job_haps = &max_job; R.jobs = &jobs;
    WalkParams P;
    P.num_editdist = params->num_editdist; P.error_correction = params->error_correction;
    P.allow_discordant = params->allow_discordant; P.simulation = params->simulation; P.base_locus = params->base_locus;
    auto fail = [&]() {
        int status = HGT_ERR_PARSE;
        const char *msg = walk_error_text((int)(err & 0xff), &status);
        const int64_t line = (int64_t)(err >> 8);
        hgt_set_error("%s (read %s)", msg,
                      line_name(text.data() + line_off[line], (size_t)(line_off[line + 1] - line_off[line])).c_str());
        return status;
    };
    const bool times = getenv("HGT_WALK_TIMES") != nullptr;
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto ms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
        return std::chrono::duration<double, std::milli>(b - a).count();
    };
    const auto t0 = now();
    for (int64_t i = 0; i < N; i++) parse_line(R, P, R.text, i);
    const auto t1 = now();
    for (int64_t i = 0; i < N; i++) mark_head(R, i);
    for (int64_t i = 0; i < N; i++) mark_candidate(R, i);
    const auto t2 = now();
    // HGT_EMU_NO_ECMASK: the walk reads the bases itself (the path of reads longer than 128 bases)
    const bool use_mask = getenv("HGT_EMU_NO_ECMASK") == nullptr;
    hgtd::EcMask no_mask;
    no_mask.w0 = no_mask.w1 = no_mask.w2 = no_mask.w3 = 0;
    no_mask.valid = false;
    for (int64_t i = 0; i < N; i++) walk_record<0>(R, P, R.text, i, -1, use_mask ? record_ec_mask(R, P, R.text, i) : no_mask);
    for (int k = 0; k < n_amb; k++)
        walk_record<1>(R, P, R.text, amb_list[k], -1, use_mask ? record_ec_mask(R, P, R.text, amb_list[k]) : no_mask);
    const auto t3 = now();
    if (times)
        fprintf(stderr, "emulation: %lld lines, parse %.2f ms, head+cand %.2f ms, walk %.2f ms (%d to the second pass, %d to the third)\n",
                (long long)N, ms(t0, t1), ms(t1, t2), ms(t2, t3), n_amb, n_slow);
    if (err != ~0ull) return fail();
    std::vector<SlowRec> slow((size_t)std::max(n_slow, 1));
    R.slow = slow.data();
    for (int k = 0; k < n_slow; k++)
        walk_record<2>(R, P, R.text, slow_list[k], k, use_mask ? record_ec_mask(R, P, R.text, slow_list[k]) : no_mask);
    for (int k = 0; k < n_heads; k++) pair_jobs<false>(R, head_list[k], k);
    if (err != ~0ull) return fail();
    for (int k = 0; k < 5; k++) {
        int64_t *a = scan.data() + (size_t)k * (N + 1), run = 0;
        for (int64_t i = 0; i < N; i++) {
            const int64_t v = a[i];
            a[i] = run;
            run += v;
        }
        a[N] = run;
    }
    const int T = loc->is_hla ? 3 : 1;
    const int64_t pairs = R.s_pairs[N], J = pairs * T, H = R.s_haps[N], RW = R.s_rows[N];
    std::vector<int64_t> job_off((size_t)J + 1, 0), row_off((size_t)H + 1, 0);
    std::vector<int32_t> job_ut((size_t)std::max<int64_t>(J, 1)), job_pair((size_t)std::max<int64_t>(J, 1)),
        job_list((size_t)std::max<int64_t>(J, 1)), hl((size_t)std::max<int64_t>(H, 1)), hr((size_t)std::max<int64_t>(H, 1)),
        htb((size_t)std::max<int64_t>(H, 1)), rows((size_t)std::max<int64_t>(RW, 1));
    jobs.job_off = job_off.data(); jobs.row_off = row_off.data(); jobs.job_ut = job_ut.data(); jobs.job_pair = job_pair.data();
    jobs.job_list = job_list.data(); jobs.hap_left = hl.data(); jobs.hap_right = hr.data(); jobs.hap_table = htb.data();
    jobs.rows = rows.data(); jobs.line0 = 0; jobs.n_small = R.s_small[N]; jobs.n_tables = T;
    for (int k = 0; k < n_heads; k++) pair_jobs<true>(R, head_list[k], k);
    if (err != ~0ull) return fail();
    hgt_walk *w = new hgt_walk();
    w->num_reads = (int64_t)unit_reads[0];
    w->num_pairs = (int64_t)unit_pairs[0];
    // regroup per table: job (pair p, table t) = p * T + t
    for (int64_t p = 0; p < pairs; p++)
        for (int t = 0; t < 3; t++) {
            hgt_walk::Tab &D = w->tb[t];
            if (t < T) {
                const int64_t job = p * T + t;
                for (int64_t h = job_off[job]; h < job_off[job + 1]; h++) {
                    D.hap_left.push_back(hl[h]);
                    D.hap_right.push_back(hr[h]);
                    D.rows.insert(D.rows.end(), rows.begin() + row_off[h], rows.begin() + row_off[h + 1]);
                    D.row_off.push_back((int64_t)D.rows.size());
                }
            }
            D.job_off.push_back((int64_t)D.hap_left.size());
        }
    *out = w;
    return HGT_OK;
}

extern "C" int hgt_walk_summary(const hgt_walk *w, int64_t *num_reads, int64_t *num_pairs, int64_t n_haps[3],
                                int64_t n_rows[3]) {
    if (!w) return HGT_ERR_ARG;
    if (num_reads) *num_reads = w->num_reads;
    if (num_pairs) *num_pairs = w->num_pairs;
    for (int t = 0; t < 3; t++) {
        if (n_haps) n_haps[t] = (int64_t)w->tb[t].hap_left.size();
        if (n_rows) n_rows[t] = (int64_t)w->tb[t].rows.size();
    }
    return HGT_OK;
}

extern "C" int hgt_walk_table(const hgt_walk *w, int32_t table, int64_t *job_off, int32_t *hap_left, int32_t *hap_right,
                              int64_t *row_off, int32_t *rows) {
    if (!w || table < 0 || table > 2) return HGT_ERR_ARG;
    const hgt_walk::Tab &J = w->tb[table];
    if (job_off) memcpy(job_off, J.job_off.data(), J.job_off.size() * 8);
    if (hap_left && !J.hap_left.empty()) memcpy(hap_left, J.hap_left.data(), J.hap_left.size() * 4);
    if (hap_right && !J.hap_right.empty()) memcpy(hap_right, J.hap_right.data(), J.hap_right.size() * 4);
    if (row_off) memcpy(row_off, J.row_off.data(), J.row_off.size() * 8);
    if (rows && !J.rows.empty()) memcpy(rows, J.rows.data(), J.rows.size() * 4);
    return HGT_OK;
}

extern "C" void hgt_walk_free(hgt_walk *w) { delete w; }

// ================================================================================================================
// Read-sharded locus: merge of the ranks' class tables (include/hgt.h)
// ================================================================================================================
static inline uint32_t merge_cap(int64_t n_in) {
    uint32_t cap = 64;
    while ((int64_t)cap < 2 * std::max<int64_t>(n_in, 1)) cap <<= 1;
    return cap;
}
extern "C" size_t hgt_class_merge_workspace_bytes(int64_t n_in) { return (size_t)merge_cap(n_in) * 8 + 256; }

extern "C" int hgt_class_merge_dev(hgt_ctx *ctx, void *stream, const uint64_t *rows_in, const uint64_t *count_in,
                                   const int32_t *first_in, int64_t n_in, int32_t n_alleles, int32_t wp, int32_t rank,
                                   int32_t world, uint64_t *rows_out, uint64_t *count_out, int32_t *first_out, int32_t *n_out,
                                   void *workspace) {
    if (!ctx || n_in < 0 || world < 1 || rank < 0 || rank >= world || !n_out || !workspace ||
        (n_in > 0 && (!rows_in || !count_in || !first_in || !rows_out || !count_out || !first_out))) {
        hgt_set_error("hgt_class_merge_dev: bad argument");
        return HGT_ERR_ARG;
    }
    if (wp != hgt_row_pitch(n_alleles) || n_in > POOL_MAX_ROWS) {
        hgt_set_error("hgt_class_merge_dev: need wp == hgt_row_pitch(n_alleles) and at most 2^28 rows");
        return HGT_ERR_ARG;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // workspace: ut_base[2] (int64) | pad to 256 | keys[cap]
    unsigned char *w = static_cast<unsigned char *>(workspace);
    const uint32_t cap = merge_cap(n_in);
    const int64_t base[2] = {0, n_in};
    HGT_CUDA(cudaMemcpyAsync(w, base, 16, cudaMemcpyHostToDevice, st));  // (pageable source: copied before the call returns)
    HGT_CUDA(cudaMemsetAsync(w + 256, 0, (size_t)cap * 8, st));
    HGT_CUDA(cudaMemsetAsync(n_out, 0, 4, st));
    if (n_in == 0) return HGT_OK;
    HGT_CUDA(cudaMemsetAsync(count_out, 0, (size_t)n_in * 8, st));
    HGT_CUDA(cudaMemsetAsync(first_out, 0x7f, (size_t)n_in * 4, st));
    ClassPool pool;
    pool.keys = reinterpret_cast<unsigned long long *>(w + 256);
    pool.cap_mask = cap - 1;
    pool.bits = rows_out;
    pool.count = reinterpret_cast<unsigned long long *>(count_out);
    pool.first = first_out;
    pool.ut_base = reinterpret_cast<const int64_t *>(w);
    pool.ut_ncls = n_out;
    const int ctas = (int)std::min<int64_t>((n_in + WARPS_PER_CTA - 1) / WARPS_PER_CTA, (int64_t)ctx->sm_count * 8);
    const unsigned long long *cnt = reinterpret_cast<const unsigned long long *>(count_in);
    switch (wpl_of(wp)) {
        case 1: class_merge_kernel<1><<<ctas, WARPS_PER_CTA * 32, 0, st>>>(wp, rows_in, cnt, first_in, n_in, rank, world, pool); break;
        case 2: class_merge_kernel<2><<<ctas, WARPS_PER_CTA * 32, 0, st>>>(wp, rows_in, cnt, first_in, n_in, rank, world, pool); break;
        case 4: class_merge_kernel<4><<<ctas, WARPS_PER_CTA * 32, 0, st>>>(wp, rows_in, cnt, first_in, n_in, rank, world, pool); break;
        default: class_merge_kernel<8><<<ctas, WARPS_PER_CTA * 32, 0, st>>>(wp, rows_in, cnt, first_in, n_in, rank, world, pool); break;
    }
    HGT_CUDA(cudaGetLastError());
    ctx->launches++;
    return HGT_OK;
}

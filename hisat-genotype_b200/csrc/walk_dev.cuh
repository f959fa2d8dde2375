// Stage (a), record half: alignment TEXT -> haplotypes, as code that runs on the GPU (one thread per alignment line).
//
// Restates, record by record, reference hisatgenotype_modules/hisatgenotype_typing_core.py:800-1406
//   (line split + filters :804-874, CIGAR x MD x Zs walk :876-1095, error_correct :119-243, post-filters :1117-1124,
//   novel variants :404-431 / :1126-1164, cmp_list2 :1351-1368, haplotype assembly :1386-1406, pair finalisation
//   :1238-1347 / :1545-1587, get_exon_haplotypes :718-792) and hisatgenotype_typing_common.py:1663-1955
//   (identify_ambigious_diffs) + hisatgenotype_validation_check.py:313-341 (check_amb_uniqueness).
//
// Every function is __host__ __device__: the kernels of reads.cuh call them with device pointers, and the host
// emulation behind hgt_host_walk (no GPU; tests/test_host_walk.py) calls the SAME functions in plain loops, so the
// device logic is pinned by the reference-captured goldens on a machine without a GPU as well.
//
// Data flow (all arrays indexed by line number i of the batch's text arena):
//   parse_line        text line -> RecFields (field offsets, FLAG, POS, NM, NH) + filter flags (core:804-852)
//   mark_head         run of equal read ids = one pair (core:1238; the input is name-grouped, core:458-468)
//   mark_candidate    mate de-dup: first record of its mate kind inside the run (core:855-874)
//   walk_record<0>    CIGAR x MD x Zs walk + error correction + post-filters -> ONE haplotype in the common case; records
//                     whose ends touch an Alts_left / Alts_right anchor are queued for
//   walk_record<1>    the same walk followed by identify_ambigious_diffs -> alternative left / right ends (factored form)
//   pair_jobs<0 / 1>  per run: union of the mates' haplotypes, exon clipping, count pass / fill pass of the job arrays
//                     the allele-set kernels consume (typing.cu)
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define HGT_HD __host__ __device__ __forceinline__
#define HGT_HDN __host__ __device__ __noinline__
#else
#define HGT_HD inline
#define HGT_HDN inline
#endif

namespace hgtd {

// ---- capacities (exceeding one is HGT_ERR_UNSUPPORTED, never a silent truncation) -------------------------------------
constexpr int MAXC = 96;   // cmp_list entries of one record
constexpr int MAXI = 32;   // variant ids of a haplotype's middle part (between the ambiguous ends)
constexpr int MAXS = 16;   // alternative ends per side of one record
constexpr int MAXA = 16;   // variant ids of one alternative end
constexpr int MAXHID = MAXI + 2 * MAXA;  // ids of a full haplotype
constexpr int MAX_PAIR_HTS = 255;        // haplotypes of one pair and table (8 bit planes in class_kernel)

enum : uint8_t { T_SINGLE = 0, T_DELETION = 1, T_INSERTION = 2 };
enum : uint8_t { C_MATCH = 0, C_MISMATCH = 1, C_INSERTION = 2, C_DELETION = 3 };
constexpr int32_t VAR_UNKNOWN = -1;
// novel indel (type, pos, len) packed into a negative id: -2 - (ins << 29 | pos << 10 | len); pos < 2^19, len < 2^10
HGT_HD bool novel_fits(int32_t pos, int32_t len) { return pos >= 0 && pos < (1 << 19) && len >= 0 && len < (1 << 10); }
HGT_HD int32_t novel_code(bool ins, int32_t pos, int32_t len) { return -2 - (int32_t)(((ins ? 1u : 0u) << 29) | ((uint32_t)pos << 10) | (uint32_t)len); }
HGT_HD bool is_novel(int32_t v) { return v <= -2; }

enum : uint16_t {
    ST_VALID = 1,   // the line is an alignment record (not blank, not a header)
    ST_PRE = 2,     // passes the filters in front of the mate de-dup (core:814-852)
    ST_PU = 4,      // passes the weaker filters of get_mpileup (common:1084-1098)
    ST_HEAD = 8,    // first record of a run of equal read ids
    ST_CAND = 16,   // first record of its mate kind in the run: goes through the walk
    ST_SURV = 32,   // survived the walk and the post-filters: counts in num_reads, contributes haplotypes
    ST_SLOW = 64,   // its ends touch Alts anchors: haplotypes live in a SlowRec
};

// error codes written by the device code (first failing line wins); messages and hgt_status on the host side
enum : int {
    E_NONE = 0, E_RECORD = 1, E_NO_NM_NH, E_MATE_KIND, E_NO_MD, E_CIGAR, E_ZS_ITEM, E_ZS_OFFSET, E_MD_SHORT, E_MD_PAST_READ,
    E_MD_BASE, E_ZS_NOT_S, E_ZS_ID, E_ZS_NOT_I, E_MD_CARET, E_CLIP_MIDDLE, E_CIGAR_OP, E_EMPTY, E_ALT_INDEX, E_ALT_TOKEN,
    E_AMBIGUITY, E_CAP_CMP, E_CAP_ENDS, E_CAP_IDS, E_LINE_LONG, E_NOVEL_RANGE, E_PAIR_HTS, E_COUNT_
};

// ---- atomics on both sides -----------------------------------------------------------------------------------------------
HGT_HD void hd_min_u64(unsigned long long *p, unsigned long long v) {
#ifdef __CUDA_ARCH__
    atomicMin(p, v);
#else
    if (v < *p) *p = v;
#endif
}
HGT_HD unsigned long long hd_add_u64(unsigned long long *p, unsigned long long v) {
#ifdef __CUDA_ARCH__
    return atomicAdd(p, v);
#else
    const unsigned long long o = *p;
    *p += v;
    return o;
#endif
}
HGT_HD int32_t hd_add_i32(int32_t *p, int32_t v) {
#ifdef __CUDA_ARCH__
    return atomicAdd(p, v);
#else
    const int32_t o = *p;
    *p += v;
    return o;
#endif
}
HGT_HD void hd_max_i32(int32_t *p, int32_t v) {
#ifdef __CUDA_ARCH__
    atomicMax(p, v);
#else
    if (v > *p) *p = v;
#endif
}

// ---- per-locus tables of the walk (one blob per locus; pointers into host or device memory) ---------------------------
struct VarTab {
    int V;
    const int32_t *pos, *len;   // [V] Var_list order
    const int32_t *lb;          // [L+2] number of variants with pos < x (lower_bound by position as a table)
    int L;
    const uint8_t *type;        // [V] T_*
    const char *base;           // [V] alt base of a single
    const uint8_t *flags;       // [V] bit0 id is a key of Links, bit1 id starts with "hv"
    const int32_t *id_off;      // [V+1] into id_pool
    const char *id_pool;
    const int32_t *id_hash;     // open addressing: row or -1
    uint32_t id_hash_mask;
    // "regular" ids (every id is "hv<decimal>", no leading zeros, unique - what extract_vars writes, process:1088-1102):
    // row = num_row[number - num_lo]; num_n == 0 when the locus has any other id (the hash table is used then)
    const int32_t *num_row;
    const int32_t *id_num;      // [V] the number of every id (regular ids only)
    int32_t num_lo, num_n;
    int32_t tok_regular;        // regular ids and every token of the Alts keys is a number or an id of the locus
};
struct AltTab {  // Alts_left or Alts_right (common:1424-1657), entries sorted by anchor position
    int n;
    const int32_t *anchor;      // [n]
    const int32_t *below;       // [L+2] number of anchors < x
    const uint8_t *end_flag;    // [L+2] 1 where a read END (left end for Alts_left, right end for Alts_right) can make
                                //       identify_ambigious_diffs do anything: bound_j <= x <= anchor_j for some entry j
    const int32_t *key_off;     // [n+1] key string "529-hv8-hv22-606" in key_pool
    const char *key_pool;
    const int32_t *tok_off;     // [n+1] tokens of the key
    const int32_t *tok_row;     // row of the token when it is a variant id of the locus, else -1
    const int32_t *tok_num;     // atoi(token)
    const int32_t *alt_off;     // [n+1] alternatives of the entry
    const int32_t *alt_left, *alt_right;
    const int32_t *altrow_off;  // [n_alts+1]
    const int32_t *altrow;
};
struct LocusWalk {
    const char *ref;
    int L, is_hla;
    VarTab v;
    AltTab al, ar;
    int n_exons, n_pexons;
    const int32_t *exons, *pexons;  // [2*n] left,right inclusive
};

struct WalkParams {
    int num_editdist, error_correction, allow_discordant, simulation, base_locus;
};

struct RecFields {  // 32 bytes per line
    int32_t flag, pos;  // pos: 0-based on the backbone, after subtracting base_locus + 1
    int16_t nm, nh;
    uint16_t qn_off, qn_len, cig_off, cig_len, seq_off, seq_len, md_off, md_len, zs_off, zs_len;
};

struct AltEnd {  // element of left_alt_set (pos-ids) / right_alt_set (ids-pos)
    int32_t pos, n;
    int32_t ids[MAXA];
};
template <int NS>
struct EndSets {  // result of identify_ambigious_diffs: alternative left ends x alternative right ends
    int32_t n_left, n_right;
    AltEnd left[NS + 1], right[NS + 1];  // + 1: the spare slot a candidate element is built in
};
struct SlowRec {  // a record with more than one haplotype, factored: left end x middle x right end
    int32_t n_mid, pad;
    int32_t mid[MAXI];
    EndSets<MAXS> e;
};

struct LocusJobs {  // job arrays of one locus batch (typing.cu consumes them), all device (or host-emulation) pointers
    int64_t *job_off, *row_off;                                        // [J+1], [H+1]
    int32_t *job_ut, *job_pair, *job_list, *hap_left, *hap_right, *hap_table, *rows;
    int64_t line0;     // first line of the locus in the arena
    int64_t n_small;   // small jobs of the locus (<= 7 haplotypes) come first in job_list
    int32_t n_tables, pad;
};

struct ReadsView {
    const char *text;
    int64_t n_lines;
    const int64_t *line_off;   // [n_lines+1]; line i = [line_off[i], line_off[i+1] - 1), the byte before the end is '\n'
    int32_t *unit;             // [n_lines]
    RecFields *rec;
    uint16_t *st;
    // haplotype of a surviving common-case record
    int32_t *h_left, *h_right, *h_n, *slow_slot;  // slow_slot >= 0: index into slow[]
    int32_t *h_ids;            // [n_lines][MAXI]
    SlowRec *slow;
    int32_t *amb_list, *slow_list;  // lines queued for the second pass (an Alts anchor in reach) / the third (several haplotypes)
    int32_t *n_amb, *n_slow;
    int32_t *head_list, *n_heads;   // run heads (any order): the pair stage runs one thread per run
    // units
    int n_units;
    const int64_t *unit_off;   // [n_units+1] byte range of every unit in the arena
    int64_t *unit_line0;       // [n_units+1] first line of every unit
    const int32_t *unit_locus, *unit_local;
    const int64_t *unit_pos0;  // first position of the unit in the batch-wide pileup arrays
    const uint8_t *nt_mask, *del_flag;
    const LocusWalk *loci;
    unsigned long long *err;   // (line << 8 | code), smallest wins; ~0 = none
    unsigned long long *unit_reads, *unit_pairs;
    // pair stage: per-line counts (non-zero at run heads), exclusive scans in place
    int64_t *s_pairs, *s_haps, *s_rows, *s_small, *s_big;  // [n_lines+1]
    int32_t *pair_cnt;  // [n_heads][3]: per run and table, haplotypes | rows << 8 (count pass -> fill pass)
    int32_t *max_job_haps;
    LocusJobs *jobs;           // [n_loci]
};

// index of a new entry of the slow list; on the device the lanes of a warp that arrive together share one atomic
HGT_HD int32_t slow_list_push(int32_t *counter) {
#ifdef __CUDA_ARCH__
    const unsigned act = __activemask();
    const int lane = threadIdx.x & 31, leader = __ffs((int)act) - 1;
    int32_t base = 0;
    if (lane == leader) base = atomicAdd(counter, __popc(act));
    base = __shfl_sync(act, base, leader);
    return base + __popc(act & ((1u << lane) - 1u));
#else
    return (*counter)++;
#endif
}

HGT_HD void set_error(const ReadsView &R, int64_t line, int code) {
    hd_min_u64(R.err, ((unsigned long long)line << 8) | (unsigned long long)code);
}

// ---- small helpers -------------------------------------------------------------------------------------------------------
HGT_HD bool is_ws(char c) { return c == ' ' || c == '\t' || c == '\r' || c == '\n' || c == '\v' || c == '\f'; }
HGT_HD bool is_dig(char c) { return c >= '0' && c <= '9'; }
HGT_HD bool is_nt(char c) { return c == 'A' || c == 'C' || c == 'G' || c == 'T'; }
HGT_HD int nt_code(char c) { return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : 4; }
HGT_HD int ctz32(uint32_t m) {
#ifdef __CUDA_ARCH__
    return __ffs((int)m) - 1;
#else
    return __builtin_ctz(m);
#endif
}

HGT_HD bool parse_int(const char *s, int n, int32_t *out) {
    if (n <= 0) return false;
    int i = 0;
    bool neg = false;
    if (s[0] == '-' || s[0] == '+') {
        neg = s[0] == '-';
        i = 1;
    }
    if (i >= n) return false;
    int64_t v = 0;
    for (; i < n; i++) {
        if (!is_dig(s[i])) return false;
        v = v * 10 + (s[i] - '0');
        if (v > 2000000000LL) return false;
    }
    *out = (int32_t)(neg ? -v : v);
    return true;
}

HGT_HD int lower_bound_i32(const int32_t *a, int n, int key) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (a[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

HGT_HD int32_t var_right(const VarTab &v, int r) { return v.type[r] == T_DELETION ? v.pos[r] + v.len[r] - 1 : v.pos[r]; }

// Known `single` variant at pos with this base (core:159-169, 204-214, 949-961) else VAR_UNKNOWN.
HGT_HD int var_lower_bound(const VarTab &v, int32_t pos) { return pos < 0 ? 0 : (pos > v.L + 1 ? v.V : v.lb[pos]); }
HGT_HD int32_t known_single(const VarTab &v, int32_t pos, char base) {
    for (int j = var_lower_bound(v, pos); j < v.V && v.pos[j] == pos; j++)
        if (v.type[j] == T_SINGLE && v.base[j] == base) return j;
    return VAR_UNKNOWN;
}
HGT_HD int32_t known_indel(const VarTab &v, int32_t pos, uint8_t type, int32_t len) {
    for (int j = var_lower_bound(v, pos); j < v.V && v.pos[j] == pos; j++)
        if (v.type[j] == type && v.len[j] == len) return j;
    return VAR_UNKNOWN;
}

HGT_HD uint64_t fnv1a(const char *p, int n) {
    uint64_t h = 1469598103934665603ull;
    for (int i = 0; i < n; i++) {
        h ^= (unsigned char)p[i];
        h *= 1099511628211ull;
    }
    return h;
}
HGT_HD uint32_t id_slot(const char *p, int n, uint32_t mask) {  // FNV-1a alone clusters on "hv<N>": finish with a mixer
    uint64_t h = fnv1a(p, n);
    h ^= h >> 33;
    h *= 0xff51afd7ed558ccdull;
    h ^= h >> 33;
    h *= 0xc4ceb9fe1a85ec53ull;
    h ^= h >> 33;
    return (uint32_t)h & mask;
}
// "hv<decimal>" without leading zeros -> the number, else -1
HGT_HD int64_t regular_id_number(const char *p, int n) {
    if (n < 3 || n > 11 || p[0] != 'h' || p[1] != 'v') return -1;
    if (p[2] == '0' && n > 3) return -1;
    int64_t x = 0;
    for (int k = 2; k < n; k++) {
        if (!is_dig(p[k])) return -1;
        x = x * 10 + (p[k] - '0');
    }
    return x;
}
// row of a variant id given as characters (Zs tag), -3 when it is not a variant of this locus
HGT_HDN int32_t row_of_chars(const VarTab &v, const char *p, int n) {
    if (v.V <= 0) return -3;
    if (v.num_n > 0) {
        const int64_t x = regular_id_number(p, n) - v.num_lo;
        if (x < 0 || x >= v.num_n) return -3;
        const int32_t r = v.num_row[x];
        return r < 0 ? -3 : r;
    }
    uint32_t slot = id_slot(p, n, v.id_hash_mask);
    while (true) {
        const int32_t r = v.id_hash[slot];
        if (r < 0) return -3;
        const int32_t o = v.id_off[r], m = v.id_off[r + 1] - o;
        if (m == n) {
            bool eq = true;
            for (int k = 0; k < n && eq; k++) eq = v.id_pool[o + k] == p[k];
            if (eq) return r;
        }
        slot = (slot + 1) & v.id_hash_mask;
    }
}

// ---- line -> record fields + filters (core:804-852, common:1084-1098) ----------------------------------------------------
HGT_HD void parse_line(const ReadsView &R, const WalkParams &P, const char *text, int64_t i) {
    const int64_t b = R.line_off[i], e = R.line_off[i + 1] - 1;
    int lo = 0, hi = R.n_units;  // unit = last u with unit_off[u] <= b
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (R.unit_off[mid] <= b) lo = mid;
        else hi = mid;
    }
    R.unit[i] = lo;
    R.st[i] = 0;
    R.slow_slot[i] = -1;
    const char *s = text + b;
    const int64_t n64 = e - b;
    int64_t a = 0;
    while (a < n64 && is_ws(s[a])) a++;
    if (a >= n64 || s[a] == '@') return;  // blank line (arena padding) or header
    if (n64 > 65535) {
        set_error(R, i, E_LINE_LONG);
        return;
    }
    const int n = (int)n64;
    RecFields f;
    f.flag = f.pos = 0;
    f.nm = f.nh = 0;
    f.qn_off = f.qn_len = f.cig_off = f.cig_len = f.seq_off = f.seq_len = f.md_off = f.md_len = f.zs_off = f.zs_len = 0;
    bool has_nm = false, has_nh = false, bad = false;
    int col = 0, p = (int)a;
    while (p < n) {
        while (p < n && is_ws(s[p])) p++;
        if (p >= n) break;
        int q = p;
        while (q < n && !is_ws(s[q])) q++;
        const int m = q - p;
        if (col == 0) {
            f.qn_off = (uint16_t)p;
            int len = m;
            if (P.simulation) {  // read_id.split('|')[0]  (core:808-809)
                for (int k = 0; k < m; k++)
                    if (s[p + k] == '|') {
                        len = k;
                        break;
                    }
            }
            f.qn_len = (uint16_t)len;
        } else if (col == 1) {
            if (!parse_int(s + p, m, &f.flag)) bad = true;
        } else if (col == 3) {
            if (!parse_int(s + p, m, &f.pos)) bad = true;
            f.pos -= P.base_locus + 1;
        } else if (col == 5) {
            f.cig_off = (uint16_t)p;
            f.cig_len = (uint16_t)m;
        } else if (col == 9) {
            f.seq_off = (uint16_t)p;
            f.seq_len = (uint16_t)m;
        } else if (col >= 11 && m >= 5) {
            const char c0 = s[p], c1 = s[p + 1];
            int32_t v = 0;
            if (c0 == 'Z' && c1 == 's') {
                f.zs_off = (uint16_t)(p + 5);
                f.zs_len = (uint16_t)(m - 5);
            } else if (c0 == 'M' && c1 == 'D') {
                f.md_off = (uint16_t)(p + 5);
                f.md_len = (uint16_t)(m - 5);
            } else if (c0 == 'N' && c1 == 'M') {
                has_nm = parse_int(s + p + 5, m - 5, &v);
                f.nm = (int16_t)(v > 32767 ? 32767 : (v < -32768 ? -32768 : v));
            } else if (c0 == 'N' && c1 == 'H') {
                has_nh = parse_int(s + p + 5, m - 5, &v);
                f.nh = (int16_t)(v > 32767 ? 32767 : (v < -32768 ? -32768 : v));
            }
        }
        if (bad) break;
        col++;
        p = q;
    }
    if (bad || col < 11) {
        set_error(R, i, E_RECORD);
        return;
    }
    R.rec[i] = f;
    uint16_t st = ST_VALID;
    const bool aligned = !(f.flag & 0x4), inside = f.pos >= 0, conc = P.allow_discordant || (f.flag & 0x2);
    if (aligned && inside && conc) {  // get_mpileup's filters (common:1084-1098)
        st |= ST_PU;
        // CIGAR must parse: digits then an op character, repeatedly
        bool have = false, ok = true;
        for (int k = 0; k < f.cig_len && ok; k++) {
            const char c = s[f.cig_off + k];
            if (is_dig(c)) have = true;
            else {
                ok = have;
                have = false;
            }
        }
        if (!ok || have) {
            set_error(R, i, E_CIGAR);
            return;
        }
    }
    if (inside && aligned) {  // main loop filters, in the reference's order (core:814-852)
        if (!has_nm || !has_nh) {
            set_error(R, i, E_NO_NM_NH);
            return;
        }
        if (f.nm <= P.num_editdist && f.nh <= 1 && conc) {
            if (!(f.flag & 0x40) && !(f.flag & 0x80) && !P.allow_discordant) {
                set_error(R, i, E_MATE_KIND);
                return;
            }
            st |= ST_PRE;
        }
    }
    R.st[i] = st;
}

HGT_HD int mate_kind(int32_t flag) { return (flag & 0x40) ? 0 : ((flag & 0x80) ? 1 : 2); }

// previous alignment record of the same unit, -1 if none
HGT_HD int64_t prev_valid(const ReadsView &R, int64_t i) {
    const int64_t first = R.unit_line0[R.unit[i]];
    for (int64_t j = i - 1; j >= first; j--)
        if (R.st[j] & ST_VALID) return j;
    return -1;
}

// A run of consecutive records with the same read id is one pair (core:1238: the pair closes when a kept record
// carries a new id; the text is grouped by name, core:458-468).
HGT_HD void mark_head(const ReadsView &R, int64_t i) {
    if (!(R.st[i] & ST_VALID)) return;
    const int64_t j = prev_valid(R, i);
    bool head = j < 0;
    if (!head) {
        const RecFields &x = R.rec[i], &y = R.rec[j];
        head = x.qn_len != y.qn_len;
        if (!head) {
            const char *p = R.text + R.line_off[i] + x.qn_off, *q = R.text + R.line_off[j] + y.qn_off;
            for (int k = 0; k < x.qn_len && !head; k++) head = p[k] != q[k];
        }
    }
    if (head) {
        R.st[i] |= ST_HEAD;
        R.head_list[slow_list_push(R.n_heads)] = (int32_t)i;
    }
}

// Mate de-dup (core:855-874): a record is dropped when an earlier record of the run with the same mate kind passed
// the filters in front of the de-dup.
HGT_HD void mark_candidate(const ReadsView &R, int64_t i) {
    const uint16_t st = R.st[i];
    if (!(st & ST_PRE)) return;
    const int kind = mate_kind(R.rec[i].flag);
    bool dup = false;
    if (!(st & ST_HEAD)) {
        const int64_t first = R.unit_line0[R.unit[i]];
        for (int64_t j = i - 1; j >= first && !dup; j--) {
            const uint16_t sj = R.st[j];
            if (!(sj & ST_VALID)) continue;
            if ((sj & ST_PRE) && mate_kind(R.rec[j].flag) == kind) dup = true;
            if (sj & ST_HEAD) break;
        }
    }
    if (!dup) R.st[i] = st | ST_CAND;
}

// ---- the walk ---------------------------------------------------------------------------------------------------------------
struct CmpList {  // three words per entry: the touched part of a thread's list stays small (local memory, L1-resident)
    int32_t pos[MAXC], var[MAXC];
    uint32_t lt[MAXC];  // len << 2 | type
    int n;
};
HGT_HD uint8_t c_type(const CmpList &c, int k) { return (uint8_t)(c.lt[k] & 3u); }
HGT_HD int32_t c_len(const CmpList &c, int k) { return (int32_t)(c.lt[k] >> 2); }
HGT_HD void c_set(CmpList &c, int k, uint8_t type, int32_t pos, int32_t len, int32_t var) {
    c.pos[k] = pos;
    c.var[k] = var;
    c.lt[k] = ((uint32_t)len << 2) | type;
}

struct ZsCursor {  // streaming reader of "off|K|id,off|K|id,..."
    const char *s;
    int p, end;
    bool have;
    int32_t off;
    char kind;
    int id_p, id_n;
};
HGT_HD void zs_next(ZsCursor &z) {
    if (z.p >= z.end) {
        z.have = false;
        return;
    }
    int q = z.p;
    while (q < z.end && z.s[q] != ',') q++;
    int b1 = z.p;
    while (b1 < q && z.s[b1] != '|') b1++;
    int32_t off = 0;
    parse_int(z.s + z.p, b1 - z.p, &off);  // validated by zs_validate
    z.off = off;
    z.kind = z.s[b1 + 1];
    z.id_p = b1 + 3;
    z.id_n = q - (b1 + 3);
    z.have = true;
    z.p = q + 1;
}
// format check of every item up front (the host parser split the whole tag before the walk)
HGT_HD int zs_validate(const char *s, int n) {
    int p = 0;
    while (p < n) {
        int q = p;
        while (q < n && s[q] != ',') q++;
        int b1 = p;
        while (b1 < q && s[b1] != '|') b1++;
        if (b1 >= q) return E_ZS_ITEM;
        if (b1 + 2 >= q || s[b1 + 2] != '|') return E_ZS_ITEM;
        int32_t off;
        if (!parse_int(s + p, b1 - p, &off)) return E_ZS_OFFSET;
        p = q + 1;
    }
    return E_NONE;
}

HGT_HD bool cmp_push(CmpList &c, uint8_t type, int32_t pos, int32_t len, int32_t var) {
    if (c.n >= MAXC) return false;
    c_set(c, c.n, type, pos, len, var);
    c.n++;
    return true;
}

// error_correct (core:119-243), streamed: the entries of one M segment are fed one by one as the walk produces them and
// the corrected entries go straight to `out` (adjacent matches of the corrected segment merge, core:226-240).
// Mismatch-with-the-pileup bits of a read, one per SEQ index (bit set: the aligned backbone position has a non-empty
// representative-base set that does not hold the read's base, core:146-151 / 190-195).  They depend on the CIGAR alone, so
// the lanes of a warp compute them together, coalesced, for each of the warp's records (reads.cuh: warp_ec_masks) and the
// serial walk scans bits instead of bases.  valid = false (reads longer than 128 bases): the walk reads the bases itself.
struct EcMask {
    uint32_t w0, w1, w2, w3;
    bool valid;
};
HGT_HD uint32_t ecm_word(const EcMask &m, int k) { return k == 0 ? m.w0 : k == 1 ? m.w1 : k == 2 ? m.w2 : m.w3; }
HGT_HD void ecm_or(EcMask &m, int k, uint32_t b) {
    if (k == 0) m.w0 |= b;
    else if (k == 1) m.w1 |= b;
    else if (k == 2) m.w2 |= b;
    else if (k == 3) m.w3 |= b;
}
constexpr int ECM_MAX_SEQ = 128;
HGT_HD bool ec_flag(const char *seq, int seq_len, const uint8_t *nt_mask, int L, int32_t rp, int32_t ep) {
    if (rp >= seq_len || ep < 0 || ep >= L) return false;
    const uint32_t m = nt_mask[ep];
    const int c = nt_code(seq[rp]);
    return m != 0 && !(c < 4 && ((m >> c) & 1u));
}
// one record, one thread (host emulation; the device computes the same bits with warp_ec_masks)
HGT_HD EcMask ec_mask_serial(const char *cig, int cig_n, const char *seq, int seq_len, const uint8_t *nt_mask, int L, int32_t pos) {
    EcMask m;
    m.w0 = m.w1 = m.w2 = m.w3 = 0;
    m.valid = seq_len <= ECM_MAX_SEQ;
    if (!m.valid) return m;
    int cp = 0;
    int32_t read_pos = 0, right_pos = pos;
    while (cp < cig_n) {
        int32_t length = 0;
        while (cp < cig_n && is_dig(cig[cp])) {
            if (length < (1 << 24)) length = length * 10 + (cig[cp] - '0');
            cp++;
        }
        if (cp >= cig_n) break;
        const char op = cig[cp++];
        if (op == 'M')
            for (int32_t j = 0; j < length && read_pos + j < seq_len; j++)
                if (ec_flag(seq, seq_len, nt_mask, L, read_pos + j, right_pos + j)) ecm_or(m, (read_pos + j) >> 5, 1u << ((read_pos + j) & 31));
        if (op == 'M' || op == 'N' || op == 'D') right_pos += length;
        if (op == 'M' || op == 'I' || op == 'S') read_pos += length;
    }
    return m;
}

struct EcState {
    int seg_start;     // out.n when the segment began
    int32_t read_pos;  // read cursor inside the segment
    int ncorr;
    bool verbatim;     // an entry beyond the backbone was met: the rest of the segment is copied (core:136-139)
    bool ok;           // false when `out` overflowed
};
HGT_HD void ec_emit(EcState &E, CmpList &out, uint8_t type, int32_t pos, int32_t len, int32_t var) {
    if (type == C_MATCH && out.n > E.seg_start && c_type(out, out.n - 1) == C_MATCH)
        out.lt[out.n - 1] += (uint32_t)len << 2;
    else E.ok &= cmp_push(out, type, pos, len, var);
}
// the correction of one base of a match entry (core:146-169)
HGT_HD void ec_fix_base(const LocusWalk &L, const uint8_t *nt_mask, EcState &E, CmpList &out, int32_t epos, int32_t j, int32_t &last) {
    const uint32_t m = nt_mask[epos + j];
    const char nb = (m & (m - 1)) ? 'N' : "ACGT"[ctz32(m)];
    E.ncorr++;
    const int32_t vid = nb != 'N' ? known_single(L.v, epos + j, nb) : VAR_UNKNOWN;
    if (j > last) ec_emit(E, out, C_MATCH, epos + last, j - last, -1);
    ec_emit(E, out, C_MISMATCH, epos + j, 1, vid);
    last = j + 1;
}
HGT_HD void ec_feed(const LocusWalk &L, const char *seq, int seq_len, const uint8_t *nt_mask, const EcMask &M, EcState &E,
                    CmpList &out, uint8_t ty, int32_t epos, int32_t elen, int32_t var) {
    if (!E.verbatim && epos >= L.L) E.verbatim = true;
    if (E.verbatim) {
        ec_emit(E, out, ty, epos, elen, var);
        return;
    }
    const int32_t read_pos = E.read_pos;
    if (ty == C_MATCH) {
        int32_t last = 0;
        if (M.valid) {
            const int32_t end = read_pos + elen < ECM_MAX_SEQ ? read_pos + elen : ECM_MAX_SEQ;  // bits at or past seq_len are 0
            for (int w = read_pos >> 5; (w << 5) < end; w++) {
                uint32_t bits = ecm_word(M, w);
                if ((w << 5) < read_pos) bits &= ~0u << (read_pos & 31);
                if (((w + 1) << 5) > end) bits &= ~0u >> (((w + 1) << 5) - end);
                while (bits) {
                    const int b = ctz32(bits);
                    bits &= bits - 1;
                    ec_fix_base(L, nt_mask, E, out, epos, (w << 5) + b - read_pos, last);
                }
            }
        } else {
            for (int32_t j = 0; j < elen; j++)
                if (ec_flag(seq, seq_len, nt_mask, L.L, read_pos + j, epos + j)) ec_fix_base(L, nt_mask, E, out, epos, j, last);
        }
        if (last < elen) ec_emit(E, out, C_MATCH, epos + last, elen - last, -1);
    } else {
        uint8_t t2 = ty;
        int32_t v2 = var;
        // the walk checked read_pos < seq_len for a mismatch entry; epos < L.L here
        const bool off = M.valid ? ((ecm_word(M, read_pos >> 5) >> (read_pos & 31)) & 1u) != 0
                                 : ec_flag(seq, seq_len, nt_mask, L.L, read_pos, epos);
        if (off) {
            const uint32_t m = nt_mask[epos];
            const char nb = (m & (m - 1)) ? 'N' : "ACGT"[ctz32(m)];
            if (nb == 'N') v2 = VAR_UNKNOWN;
            else if (nb == L.ref[epos]) {
                t2 = C_MATCH;
                v2 = -1;
                E.ncorr++;
            } else v2 = known_single(L.v, epos, nb);
        }
        ec_emit(E, out, t2, epos, t2 == C_MATCH ? 1 : elen, v2);
    }
    E.read_pos += elen;  // the ORIGINAL entry length (core:222)
}

struct WalkOut {
    int32_t right_pos;
    int ncorr;
    bool misaligned;
};

// CIGAR x MD x Zs walk (core:876-1095).  Returns E_NONE or the error code.
HGT_HDN int walk_cigar(const LocusWalk &L, const WalkParams &P, const char *line, const RecFields &f,
                       const uint8_t *nt_mask, const uint8_t *del_flag, const EcMask M, CmpList &cmp, WalkOut &w) {
    if (f.md_len == 0) return E_NO_MD;
    const char *MD = line + f.md_off;
    const int MDn = f.md_len;
    const char *seq = line + f.seq_off;
    const int seq_len = f.seq_len;
    const char *cig = line + f.cig_off;
    const int cig_n = f.cig_len;
    ZsCursor z;
    z.s = line + f.zs_off;
    z.p = 0;
    z.end = f.zs_len;
    z.have = false;
    if (f.zs_len > 0) {
        const int ze = zs_validate(z.s, f.zs_len);
        if (ze != E_NONE) return ze;
        zs_next(z);
    }
    int32_t zs_pos = z.have ? z.off : 0;
    int md_i = 0;
    int32_t md_len = 0, read_pos = 0, right_pos = f.pos;
    cmp.n = 0;
    w.ncorr = 0;
    w.misaligned = false;
    int cp = 0, ci = 0;
    while (cp < cig_n) {
        int32_t length = 0;
        bool have = false;
        while (cp < cig_n && is_dig(cig[cp])) {
            length = length * 10 + (cig[cp] - '0');
            have = true;
            cp++;
        }
        if (!have || cp >= cig_n) return E_CIGAR;
        const char op = cig[cp++];
        const bool last_op = cp >= cig_n;
        if (op == 'M') {
            bool first = true;
            int32_t used = 0;
            EcState E;
            E.seg_start = cmp.n;
            E.read_pos = read_pos;
            E.ncorr = 0;
            E.verbatim = false;
            E.ok = true;
            // Each turn of the loop yields up to two entries (a match run, then a mismatch or nothing); they go through the
            // error correction - or straight to the list when it is off - at ONE place (the code of ec_feed exists once).
            bool more = true;
            while (more) {
                if (!first || md_len == 0) {
                    if (md_i >= MDn) return E_MD_SHORT;
                    if (is_dig(MD[md_i])) {
                        int32_t num = 0;
                        while (md_i < MDn && is_dig(MD[md_i])) num = num * 10 + (MD[md_i++] - '0');
                        md_len += num;
                    }
                }
                int32_t m_pos = 0, m_len = 0, x_pos = 0, x_var = VAR_UNKNOWN;
                bool have_x = false;
                if (md_len >= length) {
                    md_len -= length;
                    m_pos = right_pos + used;
                    m_len = length - used;
                    more = false;
                } else {
                    first = false;
                    if (read_pos + md_len >= seq_len) return E_MD_PAST_READ;
                    const char base = seq[read_pos + md_len];
                    if (md_i >= MDn || !is_nt(MD[md_i])) return E_MD_BASE;
                    md_i++;
                    m_pos = right_pos + used;
                    m_len = md_len - used;
                    if (read_pos + md_len == zs_pos && z.have) {
                        if (z.kind != 'S') return E_ZS_NOT_S;
                        x_var = row_of_chars(L.v, z.s + z.id_p, z.id_n);
                        if (x_var < 0) return E_ZS_ID;
                        zs_next(z);
                        zs_pos += 1;
                        if (z.have) zs_pos += z.off;
                    } else {
                        x_var = known_single(L.v, right_pos + md_len, base);
                    }
                    have_x = true;
                    x_pos = right_pos + md_len;
                    used = md_len + 1;
                    md_len += 1;
                    if (md_len == length) {
                        md_len = 0;
                        more = false;
                    }
                }
                for (int e = 0; e < 2; e++) {
                    const bool is_x = e == 1;
                    if (is_x ? !have_x : m_len <= 0) continue;
                    const uint8_t ty = is_x ? C_MISMATCH : C_MATCH;
                    const int32_t pos = is_x ? x_pos : m_pos, len = is_x ? 1 : m_len, var = is_x ? x_var : -1;
                    bool fed;
                    if (P.error_correction) {
                        ec_feed(L, seq, seq_len, nt_mask, M, E, cmp, ty, pos, len, var);
                        fed = E.ok;
                    } else fed = cmp_push(cmp, ty, pos, len, var);
                    if (!fed) return E_CAP_CMP;
                }
            }
            w.ncorr += E.ncorr;
        } else if (op == 'I') {
            int32_t vid = VAR_UNKNOWN;
            if (read_pos == zs_pos && z.have) {
                if (z.kind != 'I') return E_ZS_NOT_I;
                vid = row_of_chars(L.v, z.s + z.id_p, z.id_n);
                if (vid < 0) return E_ZS_ID;
                zs_next(z);
                if (z.have) zs_pos += z.off;
            } else {
                vid = known_indel(L.v, right_pos, T_INSERTION, length);
            }
            if (!cmp_push(cmp, C_INSERTION, right_pos, length, vid)) return E_CAP_CMP;
            for (int32_t j = read_pos; j < read_pos + length && j < seq_len; j++)
                if (seq[j] == 'N') w.misaligned = true;
        } else if (op == 'D') {
            if (md_i < MDn && MD[md_i] == '0') md_i++;
            if (md_i >= MDn || MD[md_i] != '^') return E_MD_CARET;
            md_i++;
            while (md_i < MDn && is_nt(MD[md_i])) md_i++;
            int32_t vid = VAR_UNKNOWN;
            if (read_pos == zs_pos && z.have && z.kind == 'D') {
                vid = row_of_chars(L.v, z.s + z.id_p, z.id_n);
                if (vid < 0) return E_ZS_ID;
                zs_next(z);
                if (z.have) zs_pos += z.off;
            } else {
                vid = known_indel(L.v, right_pos, T_DELETION, length);
            }
            if (!cmp_push(cmp, C_DELETION, right_pos, length, vid)) return E_CAP_CMP;
            // artificial-deletion rule, hla only (core:1064-1077)
            if (right_pos >= 0 && right_pos < L.L && L.is_hla && del_flag[right_pos]) w.misaligned = true;
        } else if (op == 'S') {
            if (ci == 0) zs_pos += length;
            else if (!last_op) return E_CLIP_MIDDLE;
        } else {
            return E_CIGAR_OP;
        }
        if (op == 'M' || op == 'N' || op == 'D') right_pos += length;
        if (op == 'M' || op == 'I' || op == 'S') read_pos += length;
        ci++;
    }
    w.right_pos = right_pos;
    return E_NONE;
}

HGT_HD bool any_anchor(const AltTab &t, int L, int32_t lo, int32_t hi) {  // conservative outside the backbone
    if (lo < 0 || hi >= L) return true;
    if (hi < lo) return false;
    return t.below[hi + 1] - t.below[lo] > 0;
}
HGT_HD bool id_is_hv(const VarTab &v, int32_t var) { return var >= 0 && ((v.flags[var] >> 1) & 1); }

// Totals of a slice of the list that identify_ambigious_diffs asks for at every entry (get_haplotype_and_seq,
// common:1679-1700): known ids, novel ids, read bases.  The walk over the entries adds / removes one entry at a time.
struct SliceTotals {
    int known, novel;
    int32_t seq_len;
};
HGT_HD void slice_add(SliceTotals &t, const CmpList &c, int k, int L, int sign) {
    const uint8_t ty = c_type(c, k);
    if (ty == C_MATCH) {
        const int32_t a = c.pos[k] < 0 ? 0 : (c.pos[k] > L ? L : c.pos[k]);
        const int32_t e = c.pos[k] + c_len(c, k);
        const int32_t b = e < 0 ? 0 : (e > L ? L : e);
        t.seq_len += sign * (b > a ? b - a : 0);
    } else {
        if (ty == C_MISMATCH) t.seq_len += sign;
        if (c.var[k] >= 0) t.known += sign;
        else if (c.var[k] < -1) t.novel += sign;
    }
}
HGT_HD int anchors_below(const AltTab &t, int L, int32_t x) {  // number of anchors < x
    return (x >= 0 && x <= L + 1) ? t.below[x] : lower_bound_i32(t.anchor, t.n, x);
}

// Does the '-'-joined id string of the known ids of c[lo..hi] occur inside the entry's key (common:1734, 1856: str.find)?
// Character form: any ids.
HGT_HD bool key_contains_ids_chars(const VarTab &v, const AltTab &t, int e, const CmpList &c, int lo, int hi, int m) {
    const char *key = t.key_pool + t.key_off[e];
    const int kn = t.key_off[e + 1] - t.key_off[e];
    int total = m - 1;
    for (int k = lo; k <= hi; k++)
        if (c_type(c, k) != C_MATCH && c.var[k] >= 0) total += v.id_off[c.var[k] + 1] - v.id_off[c.var[k]];
    for (int s = 0; s + total <= kn; s++) {
        int p = s;
        bool ok = true, first = true;
        for (int k = lo; k <= hi && ok; k++) {
            if (c_type(c, k) == C_MATCH || c.var[k] < 0) continue;
            if (!first) ok = key[p++] == '-';
            first = false;
            const int32_t o = v.id_off[c.var[k]], n = v.id_off[c.var[k] + 1] - o;
            for (int q = 0; q < n && ok; q++) ok = key[p++] == v.id_pool[o + q];
        }
        if (ok) return true;
    }
    return false;
}
HGT_HD bool id_is_prefix(const VarTab &v, int32_t a, int32_t b) {  // id string of row a is a prefix of the id string of row b
    if (v.num_n > 0) {  // "hv<x>" vs "hv<y>", no leading zeros: x is y with trailing digits cut off
        const int32_t x = v.id_num[a];
        int32_t y = v.id_num[b];
        if (x == y) return true;
        if (x == 0) return false;
        while (y > x) y /= 10;
        return y == x;
    }
    const int32_t oa = v.id_off[a], na = v.id_off[a + 1] - oa, ob = v.id_off[b], nb = v.id_off[b + 1] - ob;
    if (na > nb) return false;
    for (int q = 0; q < na; q++)
        if (v.id_pool[oa + q] != v.id_pool[ob + q]) return false;
    return true;
}
// Token form, exact when the ids are regular ("hv<N>", unique) and every key token is a number or an id of the locus
// (VarTab::tok_regular): 'h' occurs only at the start of an id token, so a match starts at a token; every id but the last
// must then equal its key token, and the last must be a PREFIX of its key token ("hv1" is found inside "hv12").
// k0 = the entry of the first known id of the slice (the caller keeps it while it walks the entries).
HGT_HD bool key_contains_ids(const VarTab &v, const AltTab &t, int e, const CmpList &c, int lo, int hi, int m, int k0) {
    if (!v.tok_regular) return key_contains_ids_chars(v, t, e, c, lo, hi, m);
    const int32_t *tr = t.tok_row + t.tok_off[e];
    const int nt = t.tok_off[e + 1] - t.tok_off[e];
    if (m > nt) return false;
    const int32_t r0 = c.var[k0];
    for (int s = 0; s + m <= nt; s++) {
        const int32_t t0 = tr[s];
        if (t0 < 0) continue;
        if (m == 1) {
            if (t0 == r0 || id_is_prefix(v, r0, t0)) return true;
            continue;
        }
        if (t0 != r0) continue;
        int p = s + 1, seen = 1;
        bool ok = true;
        for (int k = k0 + 1; k <= hi && ok; k++) {
            if (c_type(c, k) == C_MATCH || c.var[k] < 0) continue;
            const int32_t row = tr[p++];
            seen++;
            if (row < 0) ok = false;
            else if (row != c.var[k]) ok = seen == m && id_is_prefix(v, c.var[k], row);
        }
        if (ok) return true;
    }
    return false;
}

// A candidate element of left_alt_set / right_alt_set is built in the spare slot set[n_set] and committed unless an equal
// element is already there (set semantics); returns false when the set is full.
HGT_HD bool end_id(AltEnd &x, int32_t id) {
    if (x.n >= MAXA) return false;
    x.ids[x.n++] = id;
    return true;
}
HGT_HD bool end_commit(AltEnd *set, int32_t &n_set, int cap) {
    const AltEnd &x = set[n_set];
    for (int k = 0; k < n_set; k++) {
        if (set[k].pos != x.pos || set[k].n != x.n) continue;
        bool eq = true;
        for (int q = 0; q < x.n && eq; q++) eq = set[k].ids[q] == x.ids[q];
        if (eq) return true;
    }
    if (n_set >= cap) return false;
    n_set++;
    return true;
}

// identify_ambigious_diffs (common:1663-1955) on cmp_list2 `c`; alternative ends go to S.left / S.right, the kept
// entry range to *cmp_left / *cmp_right.  Returns E_NONE or an error code (E_CAP_ENDS: S is too small).
template <int NS>
HGT_HDN int identify_ambiguous(const LocusWalk &L, const CmpList &c, EndSets<NS> &S, int32_t *cmp_left_out, int32_t *cmp_right_out) {
    const VarTab &V = L.v;
    const int n = c.n;
    int32_t cmp_left = 0, cmp_right = n - 1;
    S.n_left = S.n_right = 0;
    const int32_t left = c.pos[0], right = c.pos[n - 1] + c_len(c, n - 1) - 1;
    bool cap_ok = true;
    // ---- left end ------------------------------------------------------------------------------------------
    bool found = false;
    if (L.al.n > 0) {
        const AltTab &T = L.al;
        SliceTotals tot;  // of c[0..i]
        tot.known = tot.novel = 0;
        tot.seq_len = 0;
        int first_known = n;  // entry of the first known id of the list (every left slice starts at entry 0)
        for (int k = n - 1; k >= 0; k--) {
            slice_add(tot, c, k, L.L, +1);
            if (c_type(c, k) != C_MATCH && c.var[k] >= 0) first_known = k;
        }
        for (int i = n - 1; i >= 0; slice_add(tot, c, i, L.L, -1), i--) {
            const uint8_t ty = c_type(c, i);
            if (ty != C_MATCH) {
                if (ty == C_INSERTION || !id_is_hv(V, c.var[i])) continue;
            }
            const int32_t cur_left = c.pos[i];
            const int32_t cur_right = (ty == C_MATCH || ty == C_DELETION) ? c.pos[i] + c_len(c, i) - 1 : c.pos[i];
            if (!any_anchor(T, L.L, cur_left, cur_right)) continue;
            int start = anchors_below(T, L.L, cur_right + 1) + 1;
            if (start > T.n) start = T.n;
            const bool novel = tot.novel > 0;
            const int32_t cur_len = tot.seq_len;
            const int n_cur = tot.known;
            const int n_ids = n_cur + (novel ? 1 : 0);  // novel ids count as ids that never match
            bool hit = false;
            for (int j = start - 1; j >= 0; j--) {
                if (T.anchor[j] < cur_left) break;
                if (T.anchor[j] > cur_right) continue;
                // The extent test (common:1745-1760) first - a few loads, and it rejects most entries - then the substring
                // test; the error returns of the extent test only count once the substring test has passed, as before.
                const int32_t *tok_row = T.tok_row + T.tok_off[j], *tok_num = T.tok_num + T.tok_off[j];
                const int ntok = T.tok_off[j + 1] - T.tok_off[j] - 1;  // key.split('-')[:-1]
                int extent_err = E_NONE;
                bool extent_ok = true;
                if (n_cur + 1 == ntok) {
                    extent_ok = !(left < tok_num[0]);
                } else {
                    int k = ntok - n_cur - 1;
                    if (k < 0) k += ntok;  // Python negative index
                    if (k < 0 || k >= ntok) extent_err = E_ALT_INDEX;
                    else if (tok_row[k] < 0) extent_err = E_ALT_TOKEN;
                    else extent_ok = !(left <= var_right(V, tok_row[k]));
                }
                if (extent_err == E_NONE && !extent_ok) continue;
                if (n_ids > 0) {
                    if (novel || !key_contains_ids(V, T, j, c, 0, i, n_cur, first_known)) continue;
                }
                if (extent_err != E_NONE) return extent_err;
                hit = true;
                for (int a = T.alt_off[j]; a < T.alt_off[j + 1]; a++) {
                    const int32_t *rows = T.altrow + T.altrow_off[a];
                    const int nrow = T.altrow_off[a + 1] - T.altrow_off[a];
                    int32_t seq_pos = cur_right - T.alt_right[a], cur_pos = T.alt_right[a];
                    int first_kept = nrow;  // rows[first_kept..nrow) form the part covered by the read
                    for (int t = nrow - 1; t >= 0; t--) {
                        const int32_t r = rows[t];
                        const int32_t vp = var_right(V, r);
                        int32_t nxt = seq_pos + (cur_pos - vp);
                        if (nxt >= cur_len) break;
                        int32_t npos;
                        if (V.type[r] == T_SINGLE) {
                            nxt += 1;
                            npos = vp - 1;
                        } else npos = vp - V.len[r];
                        first_kept = t;
                        if (nxt >= cur_len) break;
                        seq_pos = nxt;
                        cur_pos = npos;
                    }
                    if (first_kept < nrow) {
                        const int32_t seq_left = cur_len - seq_pos - 1;
                        AltEnd &x = S.left[S.n_left];
                        x.pos = cur_pos - seq_left;
                        x.n = 0;
                        bool ok = true;
                        for (int t = first_kept; t < nrow; t++) ok &= end_id(x, rows[t]);
                        if (found)
                            for (int q = i + 1; q < cmp_left; q++)
                                if (c_type(c, q) != C_MATCH && id_is_hv(V, c.var[q])) ok &= end_id(x, c.var[q]);
                        cap_ok &= ok && end_commit(S.left, S.n_left, NS);
                    }
                }
            }
            if (hit) {
                if (!found) {
                    cmp_left = i + 1;
                    // cur_ht_str; a hit implies the slice holds no novel id (the substring test would fail)
                    AltEnd &x = S.left[S.n_left];
                    x.pos = left;
                    x.n = 0;
                    bool ok = true;
                    for (int q = 0; q <= i; q++)
                        if (c_type(c, q) != C_MATCH && c.var[q] >= 0) ok &= end_id(x, c.var[q]);
                    cap_ok &= ok && end_commit(S.left, S.n_left, NS);
                }
                found = true;
            }
        }
    }
    if (!found) {
        S.left[S.n_left].pos = left;
        S.left[S.n_left].n = 0;
        cap_ok &= end_commit(S.left, S.n_left, NS);
    }
    // ---- right end -----------------------------------------------------------------------------------------
    found = false;
    if (L.ar.n > 0) {
        const AltTab &T = L.ar;
        SliceTotals tot;  // of c[i..n-1]
        tot.known = tot.novel = 0;
        tot.seq_len = 0;
        for (int k = 0; k < n; k++) slice_add(tot, c, k, L.L, +1);
        int next_known = 0;  // entry of the first known id at or after entry i
        for (int i = 0; i < n; slice_add(tot, c, i, L.L, -1), i++) {
            const uint8_t ty = c_type(c, i);
            if (ty != C_MATCH) {
                if (ty == C_INSERTION || !id_is_hv(V, c.var[i])) continue;
            }
            const int32_t cur_left = c.pos[i];
            const int32_t cur_right = (ty == C_MATCH || ty == C_DELETION) ? c.pos[i] + c_len(c, i) - 1 : c.pos[i];
            if (!any_anchor(T, L.L, cur_left, cur_right)) continue;
            const int start = anchors_below(T, L.L, cur_left);
            if (start >= T.n || T.anchor[start] > cur_right) continue;
            const bool novel = tot.novel > 0;
            const int32_t cur_len = tot.seq_len;
            const int n_cur = tot.known;
            const int n_ids = n_cur + (novel ? 1 : 0);
            if (next_known < i) next_known = i;
            while (next_known < n && (c_type(c, next_known) == C_MATCH || c.var[next_known] < 0)) next_known++;
            bool hit = false;
            for (int j = start; j < T.n; j++) {
                if (T.anchor[j] > cur_right) break;
                if (T.anchor[j] < cur_left) continue;
                const int32_t *tok_row = T.tok_row + T.tok_off[j], *tok_num = T.tok_num + T.tok_off[j];
                const int ntok = T.tok_off[j + 1] - T.tok_off[j] - 1;  // key.split('-')[1:]
                int extent_err = E_NONE;
                bool extent_ok = true;
                if (n_cur + 1 == ntok) {
                    extent_ok = !(right > tok_num[ntok]);
                } else {
                    const int k = n_cur;
                    if (k >= ntok) extent_err = E_ALT_INDEX;
                    else if (tok_row[1 + k] < 0) extent_err = E_ALT_TOKEN;
                    else extent_ok = !(right >= V.pos[tok_row[1 + k]]);
                }
                if (extent_err == E_NONE && !extent_ok) continue;
                if (n_ids > 0) {
                    if (novel || !key_contains_ids(V, T, j, c, i, n - 1, n_cur, next_known)) continue;
                }
                if (extent_err != E_NONE) return extent_err;
                hit = true;
                for (int a = T.alt_off[j]; a < T.alt_off[j + 1]; a++) {
                    const int32_t *rows = T.altrow + T.altrow_off[a];
                    const int nrow = T.altrow_off[a + 1] - T.altrow_off[a];
                    int32_t seq_pos = T.alt_left[a] - cur_left, cur_pos = T.alt_left[a];
                    int kept = 0;
                    for (int t = 0; t < nrow; t++) {
                        const int32_t r = rows[t];
                        int32_t nxt = seq_pos + (V.pos[r] - cur_pos);
                        if (nxt >= cur_len) break;
                        int32_t npos;
                        if (V.type[r] == T_SINGLE) {
                            nxt += 1;
                            npos = V.pos[r] + 1;
                        } else npos = V.pos[r] + V.len[r];
                        kept = t + 1;
                        if (nxt >= cur_len) break;
                        seq_pos = nxt;
                        cur_pos = npos;
                    }
                    if (kept > 0) {
                        const int32_t seq_left = cur_len - seq_pos - 1;
                        AltEnd &x = S.right[S.n_right];
                        x.pos = cur_pos + seq_left;
                        x.n = 0;
                        bool ok = true;
                        if (found)
                            for (int q = cmp_right + 1; q < i; q++)
                                if (c_type(c, q) != C_MATCH && id_is_hv(V, c.var[q])) ok &= end_id(x, c.var[q]);
                        for (int t = 0; t < kept; t++) ok &= end_id(x, rows[t]);
                        cap_ok &= ok && end_commit(S.right, S.n_right, NS);
                    }
                }
            }
            if (hit) {
                if (!found) {
                    cmp_right = i - 1;
                    AltEnd &x = S.right[S.n_right];
                    x.pos = right;
                    x.n = 0;
                    bool ok = true;
                    for (int q = i; q < n; q++)
                        if (c_type(c, q) != C_MATCH && c.var[q] >= 0) ok &= end_id(x, c.var[q]);
                    cap_ok &= ok && end_commit(S.right, S.n_right, NS);
                }
                found = true;
            }
        }
    }
    if (!found) {
        S.right[S.n_right].pos = right;
        S.right[S.n_right].n = 0;
        cap_ok &= end_commit(S.right, S.n_right, NS);
    }
    if (cmp_right < cmp_left) {
        cmp_left = 0;
        S.left[0].pos = left;
        S.left[0].n = 0;
        S.n_left = 1;
    }
    if (!cap_ok) return E_CAP_ENDS;
    // check_amb_uniqueness (validation_check.py:313-341): no non-empty id list twice across both sides
    for (int x = 0; x < S.n_left + S.n_right; x++) {
        const AltEnd &ex = x < S.n_left ? S.left[x] : S.right[x - S.n_left];
        if (ex.n == 0) continue;
        for (int y = 0; y < x; y++) {
            const AltEnd &ey = y < S.n_left ? S.left[y] : S.right[y - S.n_left];
            if (ey.n != ex.n) continue;
            bool eq = true;
            for (int k = 0; k < ex.n && eq; k++) eq = ex.ids[k] == ey.ids[k];
            if (eq) return E_AMBIGUITY;
        }
    }
    *cmp_left_out = cmp_left;
    *cmp_right_out = cmp_right;
    return E_NONE;
}

// EcMask of record i by one thread (host emulation of warp_ec_masks)
HGT_HD EcMask record_ec_mask(const ReadsView &R, const WalkParams &P, const char *text, int64_t i) {
    EcMask m;
    m.w0 = m.w1 = m.w2 = m.w3 = 0;
    m.valid = false;
    if (!(R.st[i] & ST_CAND) || !P.error_correction) return m;
    const RecFields f = R.rec[i];
    const int u = R.unit[i];
    const char *line = text + R.line_off[i];
    return ec_mask_serial(line + f.cig_off, f.cig_len, line + f.seq_off, f.seq_len, R.nt_mask + R.unit_pos0[u],
                          R.loci[R.unit_locus[u]].L, f.pos);
}

// One candidate record through the walk, in up to three passes (each a kernel whose warps do one kind of work):
//   MODE 0  every candidate record: walk -> ONE haplotype when no Alts anchor lies inside an eligible entry (most records);
//           the others are queued (amb_list)
//   MODE 1  a queued record: the walk again, then identify_ambigious_diffs with room for two ends per side - nearly every
//           read that covers an anchor still comes out with ONE haplotype; the others (and only they) are queued (slow_list)
//   MODE 2  a record of the slow list (slot = its SlowRec): the full-size identify_ambigious_diffs, haplotypes factored as
//           left ends x middle x right ends
// `text` = base the line offsets are relative to (the arena, or its shared-memory image).
template <int MODE>
HGT_HD void walk_record(const ReadsView &R, const WalkParams &P, const char *text, int64_t i, int32_t slot, const EcMask &M) {
    const uint16_t st = R.st[i];
    if (!(st & ST_CAND)) return;
    const RecFields f = R.rec[i];
    const int u = R.unit[i];
    const LocusWalk &L = R.loci[R.unit_locus[u]];
    const char *line = text + R.line_off[i];
    const uint8_t *nt_mask = R.nt_mask + R.unit_pos0[u], *del_flag = R.del_flag + R.unit_pos0[u];
    CmpList cmp;
    WalkOut w;
    const int rc = walk_cigar(L, P, line, f, nt_mask, del_flag, M, cmp, w);
    if (rc != E_NONE) {
        set_error(R, i, rc);
        return;
    }
    // post-filters (core:1117-1124)
    if (w.right_pos > L.L) return;
    if (w.ncorr > (P.num_editdist > 1 ? P.num_editdist : 1)) return;
    if (w.misaligned) return;
    // novel variants (core:1126-1164): only indels keep an identity, (type, pos, len); unknown mismatches turn into
    // matches below.  cmp_list2 (core:1351-1368) in place.
    int n2 = 0;
    for (int k = 0; k < cmp.n; k++) {
        const uint8_t ty = c_type(cmp, k);
        const int32_t pos = cmp.pos[k], len = c_len(cmp, k);
        int32_t var = cmp.var[k];
        if ((ty == C_INSERTION || ty == C_DELETION) && var == VAR_UNKNOWN) {
            if (!novel_fits(pos, len)) {
                set_error(R, i, E_NOVEL_RANGE);
                return;
            }
            var = novel_code(ty == C_INSERTION, pos, len);
        }
        if (ty == C_MATCH || (ty == C_MISMATCH && var < 0)) {
            const int32_t ln = ty == C_MATCH ? len : 1;
            if (n2 > 0 && c_type(cmp, n2 - 1) == C_MATCH) cmp.lt[n2 - 1] += (uint32_t)ln << 2;
            else c_set(cmp, n2++, C_MATCH, pos, ln, -1);
        } else {
            c_set(cmp, n2++, ty, pos, len, var);
        }
    }
    cmp.n = n2;
    if (n2 == 0) {
        set_error(R, i, E_EMPTY);
        return;
    }
    if (MODE == 0) {
        int32_t *ids_out = R.h_ids + i * MAXI;
        int m = 0;
        bool ok = true;
        for (int k = 0; k < n2; k++)
            if (c_type(cmp, k) != C_MATCH) {
                if (m < MAXI) ids_out[m++] = cmp.var[k];
                else ok = false;
            }
        // Does identify_ambigious_diffs have anything to do?  An entry j of Alts_left only acts on a read whose left end
        // lies between the entry's bound and its anchor (the extent tests of common:1745-1760: left >= first token, or
        // left > right end of a key variant; the anchor lies inside the read), and symmetrically for Alts_right and the
        // right end (common:1867-1882).  end_flag marks those positions (typing.cu: build_walk_tables).
        const int32_t h_left = cmp.pos[0], h_right = cmp.pos[n2 - 1] + c_len(cmp, n2 - 1) - 1;
        bool amb = h_left < 0 || h_right >= L.L || h_right < h_left;
        if (!amb) amb = (L.al.n > 0 && L.al.end_flag[h_left]) || (L.ar.n > 0 && L.ar.end_flag[h_right]);
        if (amb) {
            R.amb_list[slow_list_push(R.n_amb)] = (int32_t)i;
            return;
        }
        if (!ok) {
            set_error(R, i, E_CAP_IDS);
            return;
        }
        R.h_left[i] = h_left;
        R.h_right[i] = h_right;
        R.h_n[i] = m;
        R.st[i] = st | ST_SURV;
        hd_add_u64(&R.unit_reads[u], 1ull);
    } else if (MODE == 1) {
        int32_t *ids_out = R.h_ids + i * MAXI;
        int m = 0;
        int32_t cl = 0, cr = n2 - 1;
        bool ok = true;
        EndSets<2> S;
        const int e = identify_ambiguous<2>(L, cmp, S, &cl, &cr);
        if (e == E_CAP_ENDS || (e == E_NONE && S.n_left * S.n_right > 1)) {
            R.slow_list[slow_list_push(R.n_slow)] = (int32_t)i;
            return;
        }
        if (e != E_NONE) {
            set_error(R, i, e);
            return;
        }
        for (int k = 0; k < S.left[0].n; k++) ids_out[m++] = S.left[0].ids[k];  // MAXA <= MAXI
        for (int k = cl; k <= cr; k++)
            if (c_type(cmp, k) != C_MATCH) {
                if (m < MAXI) ids_out[m++] = cmp.var[k];
                else ok = false;
            }
        for (int k = 0; k < S.right[0].n; k++) {
            if (m < MAXI) ids_out[m++] = S.right[0].ids[k];
            else ok = false;
        }
        if (!ok) {
            set_error(R, i, E_CAP_IDS);
            return;
        }
        R.h_left[i] = S.left[0].pos;
        R.h_right[i] = S.right[0].pos;
        R.h_n[i] = m;
        R.st[i] = st | ST_SURV;
        hd_add_u64(&R.unit_reads[u], 1ull);
    } else {
        SlowRec &S = R.slow[slot];
        int32_t cl = 0, cr = n2 - 1;
        const int e = identify_ambiguous<MAXS>(L, cmp, S.e, &cl, &cr);
        if (e != E_NONE) {
            set_error(R, i, e);
            return;
        }
        int m = 0;
        for (int k = cl; k <= cr; k++)
            if (c_type(cmp, k) != C_MATCH) {
                if (m >= MAXI) {
                    set_error(R, i, E_CAP_IDS);
                    return;
                }
                S.mid[m++] = cmp.var[k];
            }
        S.n_mid = m;
        R.slow_slot[i] = slot;
        R.st[i] = st | ST_SURV | ST_SLOW;
        hd_add_u64(&R.unit_reads[u], 1ull);
    }
}

// ---- pair stage ------------------------------------------------------------------------------------------------------------
// One haplotype of a record, materialised: bounds + variant ids in read order.  The common-case record has exactly one
// (h_left / h_right / h_ids of its line); a SlowRec has n_left x n_right (left end a, middle, right end b).
struct Hap {
    int32_t left, right;
    int n;
    int32_t ids[MAXHID];
};
HGT_HD int haps_of(const ReadsView &R, int64_t line) {
    const int32_t slot = R.slow_slot[line];
    return slot < 0 ? 1 : R.slow[slot].e.n_left * R.slow[slot].e.n_right;
}
// haplotype g of the record on `line`; false when it has more than MAXHID ids
HGT_HDN bool hap_load(const ReadsView &R, int64_t line, int g, Hap &h) {
    const int32_t slot = R.slow_slot[line];
    if (slot < 0) {
        h.left = R.h_left[line];
        h.right = R.h_right[line];
        h.n = R.h_n[line];  // <= MAXI
        const int32_t *src = R.h_ids + line * MAXI;
#pragma unroll 1
        for (int k = 0; k < h.n; k++) h.ids[k] = src[k];
        return true;
    }
    const SlowRec &S = R.slow[slot];
    const AltEnd &A = S.e.left[g / S.e.n_right], &B = S.e.right[g % S.e.n_right];
    h.left = A.pos;
    h.right = B.pos;
    h.n = A.n + S.n_mid + B.n;
    if (h.n > MAXHID) return false;
    int m = 0;
#pragma unroll 1
    for (int k = 0; k < A.n; k++) h.ids[m++] = A.ids[k];
#pragma unroll 1
    for (int k = 0; k < S.n_mid; k++) h.ids[m++] = S.mid[k];
#pragma unroll 1
    for (int k = 0; k < B.n; k++) h.ids[m++] = B.ids[k];
    return true;
}
HGT_HD bool hap_equal(const Hap &x, const Hap &y) {
    if (x.left != y.left || x.right != y.right || x.n != y.n) return false;
#pragma unroll 1
    for (int k = 0; k < x.n; k++)
        if (x.ids[k] != y.ids[k]) return false;
    return true;
}

struct VarLite {
    uint8_t type;
    int32_t pos, len;
};
HGT_HD VarLite var_lite(const VarTab &v, int32_t id) {
    VarLite x;
    if (id >= 0) {
        x.type = v.type[id];
        x.pos = v.pos[id];
        x.len = v.len[id];
    } else {
        const uint32_t c = (uint32_t)(-2 - id);
        x.type = (c >> 29) & 1u ? T_INSERTION : T_DELETION;
        x.pos = (int32_t)((c >> 10) & 0x7ffffu);
        x.len = (int32_t)(c & 0x3ffu);
    }
    return x;
}

// get_exon_haplotypes (core:718-792) for ONE exon: false when the haplotype does not overlap it, else the clipped
// bounds and the kept id range [lo, hi).
HGT_HDN bool exon_clip(const VarTab &V, const Hap &h, int32_t e_left, int32_t e_right, int32_t *left_out, int32_t *right_out,
                       int *lo_out, int *hi_out) {
    int32_t left = h.left, right = h.right;
    if (e_left > right || e_right < left) return false;
    const int n = h.n;
    int lo = 0, hi = n;
    if (left < e_left) {
        bool split = false;
        for (int k = 0; k < n; k++) {
            const VarLite v = var_lite(V, h.ids[k]);
            if ((v.type != T_DELETION && v.pos >= e_left) || (v.type == T_DELETION && v.pos - 1 >= e_left)) {
                left = e_left;
                lo = k;
                split = true;
                break;
            }
            if (v.type == T_DELETION && v.pos + v.len >= e_left) {
                left = v.pos + v.len;
                lo = k + 1;
                split = true;
                break;
            }
        }
        if (!split) {
            left = e_left;
            lo = hi = 0;
        }
    }
    if (right > e_right) {
        bool split = false;
        for (int k = hi; k-- > lo;) {
            const VarLite v = var_lite(V, h.ids[k]);
            const int32_t r = v.type == T_DELETION ? v.pos + v.len - 1 : v.pos;
            if ((v.type != T_DELETION && r <= e_right) || (v.type == T_DELETION && r + 1 <= e_right)) {
                right = e_right;
                hi = k + 1;
                split = true;
                break;
            }
            if (v.type == T_DELETION && r - v.len <= e_right) {
                right = r - v.len;
                hi = k;
                split = true;
                break;
            }
        }
        if (!split) {
            right = e_right;
            lo = hi = 0;
        }
    }
    *left_out = left;
    *right_out = right;
    *lo_out = lo;
    *hi_out = hi;
    return true;
}

// rows of Links the allele-set kernel ANDs: ids [lo, hi) that are known variants present in Links, sorted, unique
// (ids come in read order, i.e. nearly sorted: the insertion rarely moves anything)
HGT_HDN int hap_rows(const VarTab &V, const Hap &h, int lo, int hi, int32_t *rows) {
    int m = 0;
    for (int k = lo; k < hi; k++) {
        const int32_t id = h.ids[k];
        if (id < 0 || !(V.flags[id] & 1)) continue;
        int p = m;
        while (p > 0 && rows[p - 1] > id) p--;
        if (p > 0 && rows[p - 1] == id) continue;
        for (int q = m; q > p; q--) rows[q] = rows[q - 1];
        rows[p] = id;
        m++;
    }
    return m;
}

// Pair finalisation (core:1238-1347, 1545-1587) for the run that starts at head line i.
//   FILL = false: count pass - pairs, haplotypes, rows, small / big jobs of the run into the s_* arrays (scanned later)
//   FILL = true : write the job arrays of the locus at the scanned offsets
// Both passes walk the same sequence: distinct haplotypes of the run (union of the mates' sets, core:1250-1251), each
// materialised once; per haplotype the Gene-table entry, then its clips to the exons and to the primary exons.  Each
// table of the pair keeps its own contiguous range of the job arrays (job_off), so the fill pass first repeats the
// counting (cheap: one or two haplotypes in the common run) to place its three cursors, then writes.
template <bool FILL>
HGT_HD void pair_jobs(const ReadsView &R, int64_t i, int64_t head_k) {
    if (!(R.st[i] & ST_HEAD)) return;  // (the s_* arrays are zeroed before the count pass)
    const int u = R.unit[i];
    const int locus = R.unit_locus[u];
    const LocusWalk &L = R.loci[locus];
    const VarTab &V = L.v;
    const int T = L.is_hla ? 3 : 1;
    // surviving records of the run: the first-mate record feeds left_positive_hts, the others right_positive_hts
    int64_t recs[3];
    int nrec = 0;
    {
        int64_t left_rec = -1, others[2];
        int no = 0;
        const int64_t end = R.unit_line0[u + 1];
        for (int64_t j = i; j < end; j++) {
            const uint16_t sj = R.st[j];
            if (j > i && (sj & ST_HEAD)) break;
            if (!(sj & ST_SURV)) continue;
            if (mate_kind(R.rec[j].flag) == 0) left_rec = j;
            else if (no < 2) others[no++] = j;
        }
        if (left_rec >= 0) recs[nrec++] = left_rec;
        for (int k = 0; k < no; k++) recs[nrec++] = others[k];
    }
    if (nrec == 0) return;
    int total = 0;
    for (int r = 0; r < nrec; r++) total += haps_of(R, recs[r]);
    // per-table cursors of the fill pass
    int64_t hap_cur[3] = {0, 0, 0}, row_cur[3] = {0, 0, 0};
    int64_t kt[3] = {0, 0, 0}, rt[3] = {0, 0, 0};
    int64_t pair_in_locus = 0;
    Hap h, other;
    int32_t rows[MAXHID];
    // Count pass: per-table totals of the run, kept in pair_cnt (haplotypes | rows << 8 per table).  Fill pass: cursors from
    // those totals, then ONE walk over the haplotypes that writes (it used to repeat the counting walk first).
    if (FILL) {
        for (int tb = 0; tb < 3; tb++) {
            const int32_t c = R.pair_cnt[head_k * 3 + tb];
            kt[tb] = c & 255;
            rt[tb] = c >> 8;
        }
        // job headers and the three cursors (tables of a pair are laid out one after the other)
        const LocusJobs &J = R.jobs[locus];
        const int64_t l0 = J.line0;
        pair_in_locus = R.s_pairs[i] - R.s_pairs[l0];
        const int64_t pair_in_unit = R.s_pairs[i] - R.s_pairs[R.unit_line0[u]];
        int64_t hap = R.s_haps[i] - R.s_haps[l0], row = R.s_rows[i] - R.s_rows[l0];
        int64_t small = R.s_small[i] - R.s_small[l0], big = J.n_small + (R.s_big[i] - R.s_big[l0]);
        for (int tb = 0; tb < T; tb++) {
            const int64_t job = pair_in_locus * T + tb;
            J.job_ut[job] = R.unit_local[u] * 4 + tb;
            J.job_pair[job] = (int32_t)pair_in_unit;
            if (kt[tb] <= 7) J.job_list[small++] = (int32_t)job;
            else J.job_list[big++] = (int32_t)job;
            hap_cur[tb] = hap;
            row_cur[tb] = row;
            hap += kt[tb];
            row += rt[tb];
            J.job_off[job + 1] = hap;
        }
    }
    const bool write = FILL;
    int64_t kt_run[3] = {0, 0, 0};
    int flat = 0;  // index of the haplotype over all records of the run
    for (int r = 0; r < nrec; r++) {
        const int cnt = haps_of(R, recs[r]);
        for (int g = 0; g < cnt; g++, flat++) {
            if (!hap_load(R, recs[r], g, h)) {
                set_error(R, i, E_CAP_IDS);
                return;
            }
            // an earlier equal haplotype of the run makes this one a duplicate (set union)
            bool dup = false;
            if (total > 1) {
                int f2 = 0;
                for (int r2 = 0; r2 <= r && !dup; r2++) {
                    const int cnt2 = haps_of(R, recs[r2]);
                    for (int g2 = 0; g2 < cnt2 && f2 < flat && !dup; g2++, f2++)
                        dup = hap_load(R, recs[r2], g2, other) && hap_equal(other, h);
                }
            }
            if (dup) continue;
            for (int tb = 0; tb < T; tb++) {
                const int ne = tb == 0 ? 1 : (tb == 2 ? L.n_pexons : L.n_exons);
                const int32_t *ex = tb == 2 ? L.pexons : L.exons;
                for (int x = 0; x < ne; x++) {
                    int32_t l2 = h.left, r2 = h.right;
                    int lo = 0, hi = h.n;
                    if (tb > 0 && !exon_clip(V, h, ex[2 * x], ex[2 * x + 1], &l2, &r2, &lo, &hi)) continue;
                    const int m = hap_rows(V, h, lo, hi, rows);
                    if (write) {
                        const LocusJobs &J = R.jobs[locus];
                        const int64_t hp = hap_cur[tb]++;
                        J.hap_left[hp] = l2;
                        J.hap_right[hp] = r2;
                        J.hap_table[hp] = tb;
                        for (int k = 0; k < m; k++) J.rows[row_cur[tb] + k] = rows[k];
                        row_cur[tb] += m;
                        J.row_off[hp + 1] = row_cur[tb];
                    } else {
                        kt_run[tb]++;
                        rt[tb] += m;
                    }
                }
            }
        }
    }
    if (!FILL) {
        for (int tb = 0; tb < 3; tb++) kt[tb] = kt_run[tb];
        int n_small = 0;
        int64_t kmax = 0;
        for (int tb = 0; tb < T; tb++) {
            if (kt[tb] > MAX_PAIR_HTS) {
                set_error(R, i, E_PAIR_HTS);
                return;
            }
            n_small += kt[tb] <= 7;
            kmax = kt[tb] > kmax ? kt[tb] : kmax;
        }
        for (int tb = 0; tb < 3; tb++) R.pair_cnt[head_k * 3 + tb] = (int32_t)(kt[tb] | (rt[tb] << 8));
        R.s_pairs[i] = 1;
        R.s_haps[i] = kt[0] + kt[1] + kt[2];
        R.s_rows[i] = rt[0] + rt[1] + rt[2];
        R.s_small[i] = n_small;
        R.s_big[i] = T - n_small;
        hd_add_u64(&R.unit_pairs[u], 1ull);
        hd_max_i32(R.max_job_haps, (int32_t)kmax);
    }
}

}  // namespace hgtd

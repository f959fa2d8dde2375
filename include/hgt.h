/* libhgt — C ABI of the B200-native HISAT-genotype typing hot path.
 *
 * The reference (DaehwanKimLab/hisat-genotype v1.3.2) is pure Python and has no FFI for this path; the
 * seam is the module-level Python API (SURVEY.md §8b).  Each entry point below names the reference code it
 * replaces; INTEGRATION.md shows the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions: plain pointers and sizes only; caller-owned buffers; every function returns 0 on success or a
 * negative hgt_status; hgt_last_error() gives a message for the calling thread.  One hgt_ctx per (process,
 * device); a context is not thread-safe, distinct contexts are independent.  Functions whose name ends in
 * `_dev` take DEVICE pointers and a CUDA stream and never synchronise; all others take HOST pointers, do their
 * own host<->device copies and return when the result is in the caller's buffers.
 *
 * Bit layout: allele sets are arrays of uint64 words, bit (a & 63) of word (a >> 6) = allele a, where alleles
 * of a locus are numbered in sorted-name order with the backbone excluded (the order of names inside a
 * Gene_cmpt key, reference hisatgenotype_typing_core.py:1229-1230).  Row pitch `wp` is in 64-bit words and
 * must be even (16-byte rows for bulk copies); use hgt_row_pitch(n_alleles).
 */
#ifndef HGT_H
#define HGT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hgt_ctx hgt_ctx;
typedef struct hgt_locus hgt_locus;
typedef struct hgt_typing hgt_typing;

typedef enum {
    HGT_OK = 0,
    HGT_ERR_CUDA = -1,          /* CUDA runtime error (message has the call site) */
    HGT_ERR_KEY = -2,           /* reference would raise KeyError in the SQUAREM step (common:1365-1369) */
    HGT_ERR_ZERODIV = -3,       /* reference would raise ZeroDivisionError in normalize (common:1285-1297) */
    HGT_ERR_ARG = -4,           /* bad argument */
    HGT_ERR_UNSUPPORTED = -5,   /* shape outside what the kernels are built for (message says which) */
    HGT_ERR_PARSE = -6,         /* malformed alignment record (the reference would assert) */
    HGT_ERR_AMBIGUITY = -7,     /* check_amb_uniqueness would exit(1) (validation_check.py:313-341) */
    HGT_ERR_NOMEM = -8,
    HGT_ERR_PEER = -9           /* a rank of a read-sharded locus did not reach an exchange in time (hgt_em_peer_dev) */
} hgt_status;

const char *hgt_last_error(void);
int hgt_abi_version(void);
/* words per allele-set row (even, >= 2) for n_alleles */
int hgt_row_pitch(int n_alleles);

/* ---- context ------------------------------------------------------------------------------------------- */
int hgt_init(int device, hgt_ctx **out);
void hgt_free(hgt_ctx *ctx);
/* number of kernels this context has launched so far (bench.py reports it as gpu_launches) */
int64_t hgt_launch_count(const hgt_ctx *ctx);
int hgt_sm_count(const hgt_ctx *ctx);
/* Measurement hooks for bench.py: with profiling on, batch execute/finish bracket each GPU stage with CUDA
 * events on the launching stream.  stage_ms / stage_launches [8]: [0] line index + record parse + pileup, [1]
 * haplotype->allele-set (compat), [2] per-pair class + de-duplication, [3] Gene_counts, [4] first-level EM, [5]
 * projection, [6] second-level EM, [7] run heads + mate de-dup + walk + ambiguity pass + pair jobs.
 * h2d/d2h_bytes count every host<->device copy the library issued since the last reset (a BAM unit counts its blob
 * bytes, not the text rendered from it). */
void hgt_profile_enable(hgt_ctx *ctx, int on);
void hgt_profile_reset(hgt_ctx *ctx);
void hgt_profile_read(const hgt_ctx *ctx, double *stage_ms, int64_t *stage_launches, int64_t *h2d_bytes,
                      int64_t *d2h_bytes);
/* wall-clock milliseconds the host stages of prepare/execute/finish took since the last reset, host_ms[8]: [0] text to
 * the device (issue of the copies, staging of pageable input), [1] unit tables + line count (includes the wait for the
 * copies), [5] table / pool allocation, [6] finish-side host work; the others are unused */
void hgt_profile_host(const hgt_ctx *ctx, double *host_ms);

/* Phase tracing of the EM kernels (tooling, not on the typing path): returns in cycles16 the SM clock cycles CTA 0 of
 * every em_kernel launch since the last call spent in [0] staging p, [1] the s_k pass, [2] the per-allele pass, [3] the
 * cross-CTA reduction, [4] normalisation, [5] set-up, [6] SQUAREM/diff/prune, [7] the <=64-allele loop, [8] the whole
 * kernel, then [9] sweeps and [10] launches, and over all CTAs [11] the sum and [12] the maximum of their lifetimes in
 * ns and [13] their number; clears the counters and switches tracing on/off.  cycles16 may be NULL. */
int hgt_em_trace(hgt_ctx *ctx, int32_t enable, uint64_t *cycles16);

/* Page-locked host memory for alignment text: hgt_batch_add_unit() accepts any host pointer, but text that lives in
 * memory from hgt_host_alloc() (or any other page-locked allocation, e.g. cudaHostAlloc / torch pin_memory) is read by
 * the GPU's copy engine directly; pageable text is first assembled in a page-locked staging arena by host threads. */
int hgt_host_alloc(size_t n_bytes, void **out);
void hgt_host_free(void *p);

/* ---- stage (b): EM abundance ----------------------------------------------------------------------------
 * Replaces single_abundance(Gene_cmpt, remove_low_abundance_allele, Gene_length)
 *   reference hisatgenotype_modules/hisatgenotype_typing_common.py:1282-1410 (+ prob_diff :1272-1279).
 * class_bits [n_classes][wp]: member alleles of each Gene_cmpt key, classes in dict (first-seen) order;
 * class_count[n_classes]: the dict values; allele_len[n_alleles] or NULL (Gene_length == {}).
 * Outputs: prob[n_alleles] (0 for alleles not in the result), in_result[n_alleles] (1 if the allele is a key
 * of the reference's final Gene_prob), first_class[n_alleles] (index of the first class that inserted the
 * allele into the final dict — the tie-break of the reference's stable sort), iters (loop count, :1351). */
int hgt_em(hgt_ctx *ctx, const uint64_t *class_bits, const int64_t *class_count, int32_t n_classes,
           int32_t n_alleles, int32_t wp, const double *allele_len, int32_t remove_low, double *prob,
           uint8_t *in_result, int32_t *first_class, int32_t *iters);
/* The same with class counts as doubles: the reference does float(count) (common:1304, 1318), so fractional counts are
 * legal input of single_abundance. */
int hgt_em_f64(hgt_ctx *ctx, const uint64_t *class_bits, const double *class_count, int32_t n_classes,
           int32_t n_alleles, int32_t wp, const double *allele_len, int32_t remove_low, double *prob,
           uint8_t *in_result, int32_t *first_class, int32_t *iters);

/* Batched form: n_problems independent EM problems in one launch (one CTA per problem).  Problem i uses
 * classes [class_off[i], class_off[i+1]) of the concatenated class arrays and alleles
 * [allele_off[i], allele_off[i+1]) of the concatenated per-allele arrays; all rows share pitch wp.
 * status[i] receives the per-problem hgt_status. */
int hgt_em_batch(hgt_ctx *ctx, int32_t n_problems, const uint64_t *class_bits, const int64_t *class_count,
                 const int64_t *class_off, const int64_t *allele_off, int32_t wp, const double *allele_len,
                 const uint8_t *remove_low, double *prob, uint8_t *in_result, int32_t *first_class,
                 int32_t *iters, int32_t *status);

/* Device-pointer form of hgt_em for inputs already resident in HBM (class_count as double).  `workspace` must
 * hold hgt_em_workspace_bytes() bytes.  n_ctas = 0 lets the library choose (1 CTA for small problems, one per
 * SM for large ones).  fixed_iters > 0 runs exactly that many loop iterations ignoring convergence (bench). */
size_t hgt_em_workspace_bytes(const hgt_ctx *ctx, int32_t n_classes, int32_t n_alleles);
int hgt_em_dev(hgt_ctx *ctx, void *stream, const uint64_t *class_bits, const double *class_count,
               int32_t n_classes, int32_t n_alleles, int32_t wp, const double *allele_len, int32_t remove_low,
               int32_t fixed_iters, int32_t n_ctas, double *prob, uint8_t *in_result, int32_t *first_class,
               int32_t *iters_status /* [3]: iters, status, next_prob sweeps */, void *workspace);

/* The execution form hgt_em_dev chooses for a problem of this size, from the host's planning alone (nothing is launched):
 * the allele-compacted shared-memory layout (one CTA), one CTA streaming the class rows in slabs of slab_rows rows, or
 * a cooperative launch over `grid` CTAs (each owns ceil(n_classes / grid) rows, streamed when that exceeds slab_rows).
 * na = allele slots per thread of the kernel variant.  slab_bytes = shared-memory bytes of the compacted matrix (0 for
 * the streaming forms); the kernel stores that matrix sparse (16 bytes per non-zero 32-bit word plus an index) when it
 * fits there, dense otherwise.  merge = a compacted problem merges alleles with identical columns (no lengths,
 * a_live_max <= 6144, wp <= 128 and room for the tables).  collapse = one CTA can switch to the <= 64-key loop.
 * batch_coop = typing's batched launch of n_problems problems would run this one cooperatively on all SMs.
 * wp may be wider than hgt_row_pitch(n_alleles) (batched problems share the widest pitch); a_live_max < 1 means
 * n_alleles.  Fails like hgt_em_dev on sizes the kernel does not support. */
enum { HGT_EM_FORM_COMPACT = 0, HGT_EM_FORM_STREAM = 1, HGT_EM_FORM_COOP = 2 };
typedef struct {
    int32_t form, grid, na, slab_rows;
    int64_t slab_bytes;
    int32_t merge, collapse, batch_coop;
} hgt_em_form_info;
int hgt_em_form(const hgt_ctx *ctx, int32_t n_classes, int32_t n_alleles, int32_t wp, int32_t has_lengths, int32_t n_ctas,
                int32_t a_live_max, int32_t n_problems, hgt_em_form_info *out);

/* Read-sharded locus (SURVEY.md 8e): ONE partial sweep of next_prob() over the class rows that live on this device.
 * mode 0: initial mass (common:1299-1309; p_in unused), 1: next_prob E/M sums (common:1311-1331), 2: smallest class
 * key per allele (dict insertion order of the output, common:1324-1331).  p_in[n_alleles] holds the GLOBAL current
 * probabilities with 0 for alleles that are not keys.  acc_out[a] = sum over local classes k with s_k > 0 that hold a
 * of n_k / s_k (n_k / |class| in mode 0); aux_out[a] = 1 if any such class exists (modes 0, 1) or the smallest
 * class_key + key_offset (mode 2; class_key NULL = class index).  The caller all-reduces acc_out (sum) and aux_out
 * (max / min) over the ranks and finishes the step (hisat-genotype_b200/em_dist.py).  Exactly one of the two count
 * arrays is non-NULL.  Device pointers, no synchronisation. */
size_t hgt_em_partial_workspace_bytes(const hgt_ctx *ctx, int32_t n_alleles);
int hgt_em_partial_dev(hgt_ctx *ctx, void *stream, const uint64_t *class_bits, const double *class_count_f64,
                       const uint64_t *class_count_u64, const int32_t *class_key, int32_t key_offset, int32_t n_classes,
                       int32_t n_alleles, int32_t wp, const double *p_in, int32_t mode, double *acc_out, int32_t *aux_out,
                       void *workspace);

/* Read-sharded locus, device-resident loop: the O(A) vector half of the reference loop (common:1351-1409) as kernels, so
 * that one iteration costs 3 x (sweep, all-reduce, finish) + squarem + advance and one 64-byte host read.
 * `state` (device, hgt_em_shard_state_bytes(n_alleles), zeroed by the caller before the loop) holds, in this order,
 *   double vec[6][A]  0 Gene_prob, 1 next, 2 next2, 3 extrapolated, 4 next of extrapolated, 5 input of the last next_prob
 *   double red[2A]    the buffer the caller all-reduces (sum): per-allele sums | hit counts of the sweep
 *   double scal[8]    0 sum r^2, 1 sum v^2, 2 KeyError, 3 ZeroDivisionError, 4 prob_diff, 5 third sweep used, 6 keys left
 *   int32 fk[A]       (A rounded up to even) smallest class key of the mode-2 sweep, all-reduced with min
 *   uint8 live[5][A]  key flags of vec 0, 1, 2, 4 and 5
 * hgt_em_shard_sweep_dev = hgt_em_partial_dev with p_in = vec[src] (src < 0 or mode 0: none), results into red (modes 0, 1)
 * or fk (mode 2).  hgt_em_shard_vec_dev op 0 FINISH: vec[dst] = normalize(vec[src] * sums) over keys = live(src) & hit
 * (src < 0: initial mass; src 3 is masked by the keys of vec 2), 1 SQUAREM (common:1361-1383; vec[3], scal 0, 1, 2, 5),
 * 2 ADVANCE (prob_diff into scal[4], Gene_prob = next, select_alleles when iteration >= 10 and remove_low), 3 FINAL
 * (select_alleles + normalize: prob into vec[1], keys in live[0]).  Device pointers, no synchronisation. */
size_t hgt_em_shard_state_bytes(int32_t n_alleles);
int hgt_em_shard_sweep_dev(hgt_ctx *ctx, void *stream, const uint64_t *class_bits, const double *class_count_f64,
                           const uint64_t *class_count_u64, const int32_t *class_key, int32_t key_offset, int32_t n_classes,
                           int32_t n_alleles, int32_t wp, int32_t mode, int32_t src, void *state, void *workspace);
int hgt_em_shard_vec_dev(hgt_ctx *ctx, void *stream, int32_t op, int32_t n_alleles, void *state, const double *allele_len,
                         int32_t src, int32_t dst, int32_t iteration, int32_t remove_low);

/* Read-sharded locus, the whole loop as ONE cooperative launch per rank (one process per GPU).  The reference has no
 * counterpart: it is single_abundance (common:1282-1410) run on class rows that live on several GPUs.  Every rank owns an
 * exchange block (hgt_em_peer_alloc; its 64-byte CUDA IPC handle is passed to the other ranks by the caller, e.g. with
 * torch.distributed.all_gather, and mapped there with hgt_em_peer_open).  hgt_em_peer_dev then runs hgt_em_dev's loop on
 * this rank's rows; after every partial sweep the per-allele sums (8 * n_alleles bytes per rank) are summed over the ranks
 * in rank order through the peer-mapped blocks (NVLink loads, flags with release / acquire at system scope), so every
 * rank holds bit-identical vectors, takes the same branches and writes the same prob / in_result / first_class.
 * blocks[r] = rank r's block as mapped in THIS process (blocks[rank] = the own block).  All ranks must call it with the
 * same n_alleles, remove_low and allele_len; n_classes may be 0.  class_key + key_offset = global index of the class's
 * first read pair (dict order of the reference).  iters_status[1] = HGT_ERR_PEER when a rank does not reach an exchange
 * within 4 s (the kernel gives up instead of hanging the GPU).  `workspace` as for hgt_em_dev. */
size_t hgt_em_peer_block_bytes(int32_t n_alleles);
int hgt_em_peer_alloc(hgt_ctx *ctx, int32_t n_alleles, void **block, unsigned char handle[64]);
int hgt_em_peer_open(hgt_ctx *ctx, const unsigned char handle[64], void **block);
int hgt_em_peer_close(hgt_ctx *ctx, void *block);
int hgt_em_peer_free(hgt_ctx *ctx, void *block);
int hgt_em_peer_dev(hgt_ctx *ctx, void *stream, const uint64_t *class_bits, const double *class_count_f64,
                    const uint64_t *class_count_u64, const int32_t *class_key, int32_t key_offset, int32_t n_classes,
                    int32_t n_alleles, int32_t wp, const double *allele_len, int32_t remove_low, int32_t rank, int32_t world,
                    void *const *blocks, double *prob, uint8_t *in_result, int32_t *first_class,
                    int32_t *iters_status /* [3]: iters, status, sweeps */, void *workspace);

/* Read-sharded locus: class tables of all ranks -> the rows THIS rank owns, duplicates merged (Gene_cmpt[key] += count
 * of core:1171-1236 across shards; first = smallest first-pair index).  A class belongs to rank (hash of its row) mod
 * world, so after the call the ranks hold disjoint row sets whose union is the Gene_cmpt of all reads - the EM then costs
 * 1 / world of the rows per rank instead of nearly all of them on every rank.  rows_in[n_in][wp], count_in[n_in],
 * first_in[n_in] (global pair indices): the gathered tables (e.g. torch.distributed.all_gather of every rank's
 * hgt_batch_unit_table_dev).  Output arrays must hold n_in entries; *n_out (device int32) receives the row count.
 * `workspace`: hgt_class_merge_workspace_bytes(n_in).  Device pointers, no synchronisation. */
size_t hgt_class_merge_workspace_bytes(int64_t n_in);
int hgt_class_merge_dev(hgt_ctx *ctx, void *stream, const uint64_t *rows_in, const uint64_t *count_in, const int32_t *first_in,
                        int64_t n_in, int32_t n_alleles, int32_t wp, int32_t rank, int32_t world, uint64_t *rows_out,
                        uint64_t *count_out, int32_t *first_out, int32_t *n_out, void *workspace);

/* ---- stage (b'): diploid allele-pair model ---------------------------------------------------------------
 * Replaces joint_abundance(HLA_cmpt, HLA_length) of the reference's legacy typer
 *   etc/hisatgenotype_hla_cyp.py:236-302 (pair mass :243-254, choose_top_alleles :259-270, next_prob :273-287).
 * The live typing() never calls it (SURVEY.md 0.3); it is offered next to single_abundance as the reference's
 * own pair scoring.  The caller (hisat-genotype_b200/typing_common.py: joint_abundance) enumerates the pairs that
 * survive the first choose_top_alleles and hands over, per pair, p0 (normalised) and the bitset of the alleles whose
 * NAME occurs inside the pair's key string - the legacy code tests `allele in allele_pair` on strings.
 * class_bits [n_classes][wp], class_count [n_classes], pair_bits [n_pairs][wp]; prob [n_pairs] = final pair
 * probabilities, 0 for pruned pairs; *iters = loop iterations.  Host pointers. */
int hgt_pair_em(hgt_ctx *ctx, const uint64_t *class_bits, const int64_t *class_count, int32_t n_classes, int32_t wp,
                const uint64_t *pair_bits, int32_t n_pairs, const double *p0, double *prob, int32_t *iters);

/* ---- stage (a): per-read allele compatibility -----------------------------------------------------------
 * Replaces the per-read loop of typing() for index_type == "graph"
 *   reference hisatgenotype_modules/hisatgenotype_typing_core.py:598-1596 (add_count :626-677, add_stat
 *   :1171-1236, get_exon_haplotypes :718-792, error_correct :119-243) together with
 *   hisatgenotype_typing_common.py get_mpileup :1059-1184 and identify_ambigious_diffs :1663-1955.
 *
 * A locus is described once (hgt_locus_desc mirrors the per-locus state typing() derives at core:385-596);
 * hgt_typing_run consumes the alignment lines of one (sample, locus) exactly as the reference reads them from
 * `samtools view <aln> <backbone> | sort -k1,1 -s` (core:436-468) and leaves Gene_cmpt / Gene_counts for the
 * three tables on the device.  Table ids: 0 = Gene (all alleles), 1 = exon (allele_rep_set),
 * 2 = primary exon (primary_exon_allele_rep_set); tables 1 and 2 exist only when is_hla != 0 (core:1274-1291). */
typedef struct {
    int32_t n_alleles;           /* alleles of the locus, backbone excluded, sorted-name order */
    int32_t n_vars;              /* variants in Var_list order (sorted by position, file order inside one) */
    int32_t ref_len;
    const char *ref_seq;         /* backbone sequence */
    const int32_t *var_pos;      /* [n_vars] 0-based backbone position */
    const int32_t *var_len;      /* [n_vars] deletion length / inserted length / 1 for single */
    const uint8_t *var_type;     /* [n_vars] 0 single, 1 deletion, 2 insertion */
    const char *var_base;        /* [n_vars] alternative base of a single, else 0 */
    const uint8_t *var_flags;    /* [n_vars] bit0: id is a key of Links, bit1: id starts with "hv" */
    const char *var_ids;         /* n_vars NUL-terminated id strings, concatenated */
    const int64_t *link_off;     /* [n_vars+1] CSR offsets into link_allele */
    const int32_t *link_allele;  /* allele indices linked to each variant (Links[var_id]) */
    int32_t n_exons;
    const int32_t *exons;        /* [2*n_exons] left,right inclusive (ref_exons) */
    int32_t n_primary_exons;
    const int32_t *primary_exons;
    const uint64_t *exon_rep_mask;     /* [wp] allele_rep_set, NULL when is_hla == 0 */
    const uint64_t *primary_rep_mask;  /* [wp] primary_exon_allele_rep_set */
    const int32_t *gene_names_rank;    /* [n_alleles] position of the allele in Gene_names[gene] (dict order of the
                                          per-read count tables, core:1338-1347) */
    int32_t is_hla;              /* base_fname == "hla" */
    const char *alts_text;       /* get_alternatives() tables: lines "L\tkey\talt,alt,...\n" / "R\t..." */
    const int64_t *group_off;    /* [n_alleles+1] CSR: members of allele_rep_groups[a] (empty unless a is a
                                    representative), used by the two-level EM driver (core:1739-1749); may be NULL */
    const int32_t *group_member;
    const double *allele_len;    /* [n_alleles] Gene_lengths[gene][allele] (core:2480-2485); may be NULL */
} hgt_locus_desc;

typedef struct {
    int32_t num_editdist;      /* --num-editdist (args.py:294-299), default 2 */
    int32_t error_correction;  /* default on */
    int32_t allow_discordant;  /* --discordant */
    int32_t simulation;        /* read ids are cut at the first '|' (core:808-809) */
    int32_t base_locus;        /* 0 unless typing inside a genotype genome (core:437-441) */
    int32_t n_threads;         /* host threads that stage PAGEABLE input text into page-locked memory; <= 0 = library
                                  default; unused when the text is already page-locked */
    int32_t chunk_bytes;       /* unused (kept for ABI stability: the record walk no longer runs in host tasks) */
} hgt_params;

/* ctx may be NULL: the locus then only carries the host tables (used by hgt_host_walk). */
int hgt_locus_create(hgt_ctx *ctx, const hgt_locus_desc *desc, hgt_locus **out);
void hgt_locus_free(hgt_locus *locus);

int hgt_typing_run(hgt_ctx *ctx, hgt_locus *locus, const char *sam_text, size_t n_bytes, const hgt_params *params,
                   hgt_typing **out);
void hgt_typing_free(hgt_typing *t);
/* num_reads / num_pairs (core:1168, 1240, 1546) and number of classes per table */
int hgt_typing_summary(const hgt_typing *t, int64_t *num_reads, int64_t *num_pairs, int32_t n_classes[3]);
/* Gene_cmpt of one table in dict (first-seen) order: class_bits [n_classes][wp], class_count, class_first
 * (pair index that created the key); Gene_counts as allele_count[n_alleles] plus allele_first[n_alleles]
 * (pair index that inserted the allele; ties follow gene_names_rank).  Any output pointer may be NULL. */
int hgt_typing_table(const hgt_typing *t, int32_t table, uint64_t *class_bits, int64_t *class_count,
                     int64_t *class_first, int64_t *allele_count, int64_t *allele_first);
/* pileup of the locus: counts [ref_len][6] for A,C,G,T,other,D and the nt_set mask (bit i = "ACGT"[i]) */
int hgt_typing_pileup(const hgt_typing *t, uint32_t *counts, uint8_t *nt_mask);
/* EM directly on a device-resident table.  keep_mask (nullable, [wp]) projects every class onto a subset of
 * alleles first, merging classes that become equal and dropping empty ones (core:1753-1766). */
int hgt_typing_em(hgt_ctx *ctx, const hgt_typing *t, int32_t table, const uint64_t *keep_mask,
                  const double *allele_len, int32_t remove_low, double *prob, uint8_t *in_result,
                  int32_t *first_class, int32_t *iters);

/* ---- batches of (sample, locus) units ----------------------------------------------------------------------
 * The production shape of the path: the reference types one (sample, locus) at a time inside Pool workers
 * (hisatgenotype:613-665, core:370); here any number of units over any number of loci go through the GPU
 * together.  prepare = the alignment text goes to the device as it is (one arena, one line count; BAM units go as
 * packed records and are rendered into their arena slices on the device, hgt_batch_add_unit_bam);
 * execute = GPU only: line index, record parse + filters, pileup, mate de-dup, CIGAR x MD x Zs walk with error
 * correction, ambiguity expansion, pair jobs, haplotype->allele-set, per-pair class, class de-duplication, Gene_counts
 * and the first-level EM (exon table on the hla path, Gene table otherwise) for every unit; the host only reads back
 * sizes (three small synchronisations) to allocate the next buffers;
 * finish = results back and, on the hla path, projection + second-level EM (core:1739-1782).
 * execute and finish may be repeated on a prepared batch (bench: text resident in HBM).  Table 3 = the projected Gene
 * table the second-level EM ran on.  sam_text buffers must stay valid until prepare returns.  The text of one unit
 * must be grouped by read name like the reference's input (`samtools view | sort -k1,1 -s`, core:458-468): a run of
 * consecutive lines with one read id is one pair. */
typedef struct hgt_batch hgt_batch;
int hgt_batch_create(hgt_ctx *ctx, int32_t n_loci, hgt_locus *const *loci, const hgt_params *params,
                     int32_t remove_low_abundance_alleles, hgt_batch **out);
void hgt_batch_free(hgt_batch *b);
int64_t hgt_batch_add_unit(hgt_batch *b, int32_t locus_index, const char *sam_text, size_t n_bytes);
/* n units in one call; returns the index of the first one (the others follow) or a negative status */
int64_t hgt_batch_add_units(hgt_batch *b, int64_t n, const int32_t *locus_index, const char *const *sam_text,
                            const size_t *n_bytes);
/* A unit given as a packed BAM unit (hgt_bam_split_write_records) instead of text: prepare copies the blob to the device
 * and renders its records there into the unit's slice of the text arena, byte for byte what hgt_bam_split_write_text
 * gives; everything after that is the text path.  The blob's header, name table and offset table are checked here
 * (HGT_ERR_ARG when an offset leaves the blob); blob must be 8-byte aligned and stay valid until prepare returns.
 * Page-locked blobs are copied directly, pageable ones staged like text.  BAM and text units mix in one batch; a batch
 * without BAM units does exactly what it did before. */
int64_t hgt_batch_add_unit_bam(hgt_batch *b, int32_t locus_index, const void *blob, size_t n_bytes);
/* After prepare: the unit's slice of the device text arena (the rendered text of a BAM unit, the caller's text of a text
 * unit).  dst NULL: *n_bytes = its length; else *n_bytes (capacity in, length out) must hold it. */
int hgt_batch_unit_text(const hgt_batch *b, int64_t unit, char *dst, size_t *n_bytes);
/* Read-sharded locus (several processes hold disjoint reads of the same (sample, locus), SURVEY.md 8e): error
 * correction depends on the pileup of ALL reads (common:1124-1134), so prepare calls the hook once, after the raw
 * base counts of this process are on the device and before nt_set is derived; the hook sums dev_counts
 * (n_u32 uint32 values: every unit's [ref_len][6] histogram, units in add order) over the ranks in place, e.g. with
 * ncclAllReduce, and returns 0.  `stream` is idle when the hook runs. */
typedef int (*hgt_pileup_hook)(void *arg, void *dev_counts, size_t n_u32, void *stream);
int hgt_batch_set_pileup_hook(hgt_batch *b, hgt_pileup_hook fn, void *arg);
int hgt_batch_prepare(hgt_batch *b);
int hgt_batch_execute(hgt_batch *b, void *stream);
int hgt_batch_finish(hgt_batch *b, void *stream);
int hgt_batch_run(hgt_batch *b); /* prepare + execute + finish */
/* totals over the batch (valid after execute); algorithmic_bytes = SURVEY.md 8d figure for stage (a): packed records read plus one
 * allele-set row per pair and table */
int hgt_batch_totals(const hgt_batch *b, int64_t *n_units, int64_t *num_reads, int64_t *num_pairs,
                     int64_t *n_haplotypes, int64_t *n_rows, int64_t *algorithmic_bytes);
/* (pair, table) jobs of a prepared batch: out[0] jobs, out[1] jobs with more than 7 haplotypes (the 8-bit-plane class
 * kernel, core:1171-1236 with > 7 add_count calls per pair), out[2] largest haplotype count of a job, out[3] haplotypes */
int hgt_batch_job_stats(const hgt_batch *b, int64_t out[4]);
int hgt_batch_unit_summary(const hgt_batch *b, int64_t unit, int64_t *num_reads, int64_t *num_pairs,
                           int32_t n_classes[4], int32_t em_iters[2], int32_t em_status[2]);
int hgt_batch_unit_table(hgt_batch *b, int64_t unit, int32_t table, uint64_t *class_bits, int64_t *class_count,
                         int64_t *class_first, int64_t *allele_count, int64_t *allele_first);
/* level 0: first-level EM; level 1: second-level EM (status 1 = not run for this unit, core:1752) */
/* device pointers of one table of a finished (or executed) batch: class rows [n][wp], counts [n] (uint64) and
 * first-seen pair indices [n]; valid until the batch is freed or executed again */
int hgt_batch_unit_table_dev(const hgt_batch *b, int64_t unit, int32_t table, const uint64_t **class_bits,
                             const uint64_t **class_count, const int32_t **class_first, int32_t *n_classes);
/* skip != 0: execute/finish stop after the class tables (the caller runs the EM itself, e.g. the sharded EM) */
int hgt_batch_set_skip_em(hgt_batch *b, int32_t skip);
int hgt_batch_unit_em(const hgt_batch *b, int64_t unit, int32_t level, double *prob, uint8_t *in_result,
                      int32_t *first_class, int32_t *iters, int32_t *status);

/* Per-read haplotypes of a unit, for callers that continue with the reference's assembly (SURVEY.md 8f-4): for every
 * surviving alignment record, in text order, the haplotypes typing() holds for it when it builds the assembly nodes
 * (left_positive_hts / right_positive_hts, core:1386-1406 -> :1408-1540).  Call once with NULL arrays for the sizes, then
 * with arrays of n_records (+1 for rec_hap_off), n_haps (+1 for hap_id_off) and n_ids entries.  rec_line = line of
 * the unit's text; ids = variant rows (Var_list order) in haplotype order, or a novel indel as
 * -2 - (is_insertion << 29 | pos << 10 | len).  Valid after execute. */
int hgt_batch_unit_reads(hgt_batch *b, int64_t unit, int64_t *n_records, int64_t *n_haps, int64_t *n_ids, int64_t *rec_line,
                         int32_t *rec_flag, int64_t *rec_hap_off, int32_t *hap_left, int32_t *hap_right,
                         int64_t *hap_id_off, int32_t *ids);

/* Gene_prob of one unit as typing() ranks it (core:1771-1782 on the hla path, core:1789 otherwise): allele indices and
 * probabilities in report order; at most cap entries are written, *n_total is the full length.  Returns the EM
 * status of the unit (HGT_ERR_KEY / HGT_ERR_ZERODIV mirror the reference's exceptions). */
int hgt_batch_unit_abundance(const hgt_batch *b, int64_t unit, int32_t cap, int32_t *allele, double *prob,
                             int32_t *n_total);
/* The same for every unit of the batch in one call (a typing service reads the calls of thousands of units per batch):
 * allele / prob are [n_units][cap], n_total / status [n_units]; status[u] is what hgt_batch_unit_abundance returns for
 * unit u (0, HGT_ERR_KEY, HGT_ERR_ZERODIV).  The function itself fails only on bad arguments. */
int hgt_batch_abundances(const hgt_batch *b, int32_t cap, int32_t *allele, double *prob, int32_t *n_total,
                         int32_t *status);

/* ---- native SAM intake (host) -------------------------------------------------------------------------------
 * Replaces, for all loci of a sample at once, the external pipe the reference runs per locus
 *   samtools view <bam> <backbone> | sort -k1,1 -s     (hisatgenotype_typing_core.py:436-468)
 * on the coordinate-sorted BAM of hisatgenotype_typing_common.py:1038-1054: the aligner's SAM text (any record
 * order, header lines allowed) is bucketed by RNAME into the given backbones and every bucket is ordered by
 * (read name bytewise, position, input order) - the order of the reference's two stable sorts under LC_ALL=C.
 * hgt_sam_split_write() emits a bucket as the name-grouped alignment text hgt_batch_add_unit() takes; dst may be
 * page-locked memory (hgt_host_alloc).  sam_text must stay valid until the handle is freed. */
typedef struct hgt_sam_split hgt_sam_split;
int hgt_sam_split_create(const char *sam_text, size_t n_bytes, int32_t n_refs, const char *const *ref_names,
                         int32_t n_threads, hgt_sam_split **out);
/* The same with options: HGT_SPLIT_DROP_QUAL writes '*' for the QUAL column of every record (legal SAM; the typing path
 * - the reference's and this one - never reads base qualities, and the column is 27 % of a 2x100 bp record that would
 * otherwise travel to the GPU). */
enum { HGT_SPLIT_DROP_QUAL = 1 };
int hgt_sam_split_create_opts(const char *sam_text, size_t n_bytes, int32_t n_refs, const char *const *ref_names,
                              int32_t n_threads, int32_t flags, hgt_sam_split **out);
int hgt_sam_split_sizes(const hgt_sam_split *s, size_t *bytes_per_ref, int64_t *lines_per_ref);
int hgt_sam_split_write(const hgt_sam_split *s, int32_t ref, char *dst);
void hgt_sam_split_free(hgt_sam_split *s);

/* ---- native BAM intake (host split, device render) ------------------------------------------------------------
 * The same replacement for a BAM file.  bam = the DECOMPRESSED BAM stream (magic "BAM\1", header, records; BGZF is
 * inflated by the caller, e.g. sam_intake.read_bgzf).  Every record is validated completely: a block_size that disagrees
 * with l_read_name / n_cigar_op / l_seq / the aux bytes, a read name without NUL, an aux tag of unknown type or past the
 * record end, a refID outside the header give HGT_ERR_PARSE naming the read; float tags (f, d, B:f) and the long-CIGAR
 * placeholder CG give HGT_ERR_UNSUPPORTED naming the read and the tag.  Records are bucketed by refID into the given
 * backbones (the SAM split's RNAME rule) and ordered by the same rule as hgt_sam_split_*.  flags: HGT_SPLIT_DROP_QUAL
 * leaves the QUAL bytes out (the text then carries '*').  `bam` must stay valid until the handle is freed.
 * A bucket leaves as a packed unit (layout: csrc/bam_dev.cuh) for hgt_batch_add_unit_bam (hgt_bam_split_write_records;
 * dst 8-byte aligned, e.g. page-locked memory) or as the SAM text `samtools view` prints for its records
 * (hgt_bam_split_write_text, rendered on the host by the functions the device render runs).  sizes: blob bytes, text
 * bytes (rendered on demand: pass NULL when not needed) and records per reference; any pointer may be NULL. */
typedef struct hgt_bam_split hgt_bam_split;
int hgt_bam_split_create(const void *bam, size_t n_bytes, int32_t n_refs, const char *const *ref_names, int32_t n_threads,
                         int32_t flags, hgt_bam_split **out);
int hgt_bam_split_sizes(const hgt_bam_split *s, size_t *blob_bytes, size_t *text_bytes, int64_t *records);
int hgt_bam_split_write_records(const hgt_bam_split *s, int32_t ref, void *dst);
int hgt_bam_split_write_text(const hgt_bam_split *s, int32_t ref, char *dst);
void hgt_bam_split_free(hgt_bam_split *s);

/* ---- BGZF inflate (BAM's compression) on the GPU ----------------------------------------------------------------
 * Replaces read_bgzf's zlib thread pool (sam_intake.py) for the native BAM intake.  open: host walk of the block headers
 * of n_streams BGZF streams (the rules of sam_intake._bgzf_blocks: gzip magic, FEXTRA, BC subfield, BSIZE within the
 * stream) plus ISIZE <= 65536 -> per stream the inflated size (sum of ISIZE), block count, and whether it ends in the EOF
 * marker block.  A malformed header gives HGT_ERR_PARSE naming the stream and byte offset, with read_bgzf's wording.
 * ISIZE > 65536 is the one input read_bgzf accepts and this path refuses: the BGZF spec caps a block at 64 KiB, htslib
 * never writes more, and the cap bounds the output a block can claim.
 * inflate: compressed bytes to the device, ONE kernel launch per call (bgzf_inflate_kernel: one warp per block, all
 * blocks of all streams; none when there is no block), CRC32 + ISIZE checked on the device, stream i's bytes into dst[i]
 * (page-locked dst is written by the copy engine directly), one synchronisation.  A block is accepted exactly when zlib's
 * raw inflate accepts it with nothing left over and the trailer agrees (read_bgzf's decision).  The first failing block
 * gives HGT_ERR_PARSE "stream %d: BGZF block at byte %d: <rule>", with zlib's or read_bgzf's wording where the rule is
 * the same; dst then holds unspecified bytes and the context stays usable.  h2d_bytes grows by the streams' bytes plus
 * 16 * (blocks + 1) bytes of block offsets, d2h_bytes by the inflated bytes plus an 8-byte status word.
 * Input must stay valid until the handle is freed. */
typedef struct hgt_bgzf hgt_bgzf;
int hgt_bgzf_open(int32_t n_streams, const void *const *data, const size_t *n_bytes, hgt_bgzf **out);
int hgt_bgzf_sizes(const hgt_bgzf *z, size_t *out_bytes, int64_t *n_blocks, int32_t *has_eof);   /* [n_streams] each */
int hgt_bgzf_inflate(hgt_ctx *ctx, const hgt_bgzf *z, void *const *dst);
/* Host EMULATION (test infrastructure, not on the typing path): the same bgzf_dev.cuh functions on host threads
 * (n_threads <= 0: all cores), the same decisions and messages. */
int hgt_bgzf_inflate_host(const hgt_bgzf *z, int32_t n_threads, void *const *dst);
void hgt_bgzf_free(hgt_bgzf *z);

/* Host EMULATION of the record stage with a caller-supplied pileup (no GPU needed; test infrastructure, not on the
 * typing path): the same __host__ __device__ functions the kernels call (csrc/walk_dev.cuh: parse, filters, mate
 * de-dup, walk, error correction, ambiguity expansion, exon clipping, pair jobs) run in plain loops.  Output is the
 * job list the allele-set kernels consume, regrouped per table: jobs tb_job_off[n_pairs+1] -> haplotypes (left,
 * right, row_off[..+1] -> rows).  Buffers are owned by the returned handle. */
typedef struct hgt_walk hgt_walk;
int hgt_host_walk(hgt_locus *locus, const char *sam_text, size_t n_bytes, const hgt_params *params,
                  const uint32_t *counts, const uint8_t *nt_mask, hgt_walk **out);
int hgt_walk_summary(const hgt_walk *w, int64_t *num_reads, int64_t *num_pairs, int64_t n_haps[3],
                     int64_t n_rows[3]);
int hgt_walk_table(const hgt_walk *w, int32_t table, int64_t *job_off, int32_t *hap_left, int32_t *hap_right,
                   int64_t *row_off, int32_t *rows);
void hgt_walk_free(hgt_walk *w);

/* ---- (f)-2: typing database text files, native reader -------------------------------------------------------
 * Reads what genotyping_locus reads (core:2417-2485 through common:279-309 read_locus, :313-334 read_backbone_alleles,
 * :339-368 read_variants, :388-403 read_links) - <prefix>_backbone.fa, .locus, .snp, .link, .allele, .partial - and, when
 * present, the index-side files .index.snp and .haplotype (formats: process.py:1055-1063, 1088-1106, 1215-1220, 1242-1244).
 * A missing mandatory file gives HGT_ERR_ARG with the reference's message ("index files missing", common:572-575), a
 * malformed line HGT_ERR_PARSE (the reference would fail an assert or a split).  Genes come in .locus order; the variants
 * of a gene in Var_list order (by position, file order inside one position).
 * hgt_db_sizes: out = backbone length, exons, variants, .allele entries, .partial entries, haplotypes, locus left, right.
 * hgt_db_ints copies one numeric table (at most `cap` values): EXONS = (left, right, primary) triples, VAR_TYPE = 0 single /
 * 1 deletion / 2 insertion, HAP_RANGE = (left, right) pairs.  hgt_db_text returns one string table as '\n'-terminated
 * entries (BACKBONE: the bare sequence; GENE: gene, backbone name, chromosome, strand; VAR_LINKS: the allele names of each
 * variant, blank separated, an empty line for a variant without a .link line; HAP_VARS: comma separated variant ids); the
 * pointer stays valid until the next hgt_db_text call on the handle. */
typedef struct hgt_db hgt_db;
enum {
    HGT_DB_EXONS = 0, HGT_DB_VAR_TYPE = 1, HGT_DB_VAR_POS = 2, HGT_DB_VAR_IN_INDEX = 3, HGT_DB_HAP_RANGE = 4,
    HGT_DB_GENE = 16, HGT_DB_BACKBONE = 17, HGT_DB_VAR_ID = 18, HGT_DB_VAR_DATA = 19, HGT_DB_VAR_LINKS = 20,
    HGT_DB_ALLELES = 21, HGT_DB_PARTIAL = 22, HGT_DB_HAP_ID = 23, HGT_DB_HAP_VARS = 24
};
int hgt_db_open(const char *prefix, hgt_db **out);
void hgt_db_close(hgt_db *db);
int32_t hgt_db_n_genes(const hgt_db *db);
int hgt_db_sizes(const hgt_db *db, int32_t gene, int64_t out[8]);
int hgt_db_ints(const hgt_db *db, int32_t gene, int32_t what, int64_t *out, int64_t cap);
int hgt_db_text(hgt_db *db, int32_t gene, int32_t what, const char **text, size_t *n_bytes);
/* The writer of the same formats: the handle's tables as <prefix>.locus, .snp, .link, _backbone.fa, .allele, .partial (and
 * .index.snp / .haplotype when the handle holds such entries); hgt_db_open(prefix) reads the same tables back. */
int hgt_db_write(const hgt_db *db, const char *prefix);

#ifdef __cplusplus
}
#endif
#endif /* HGT_H */

// Stage (b): EM abundance with SQUAREM acceleration, whole loop inside one kernel launch.
//
// Replaces single_abundance() of the reference
//   (hisatgenotype_modules/hisatgenotype_typing_common.py:1282-1410; matrix form in SURVEY.md appendix A.9).
//
// Data layout in HBM: class x allele membership as a row-major bit matrix bits[C][wp] (uint64 words, wp even
// so a row slab is a multiple of 16 bytes and moves with one cp.async.bulk / TMA bulk copy), class counts
// cnt[C] (double), optional allele lengths len[A].  Probability vectors are A doubles and live in a small
// global workspace that stays L2-resident; the vector a pass reads is staged in shared memory.
//
// One next_prob() evaluation = one sweep over the bit matrix.  A CTA owns a contiguous range of class rows and
// walks it in slabs that are bulk-copied into shared memory; while a slab is resident BOTH halves of the E/M
// step run on it:
//   phase 1 (warp per class row)   s_k = sum_{a in S_k} p[a],  w_k = n_k / s_k
//   phase 2 (thread per allele)    acc[a] += w_k for every row of the slab that has bit a set
// so the matrix is read from HBM/L2 once per next_prob() (algorithmic bytes 3*C*(wp*8+8)+6*A*8 per loop
// iteration, SURVEY.md 8d).  If a CTA's rows fit its slab buffer they are loaded once and stay in shared
// memory for every iteration (small loci: zero HBM traffic inside the loop).
//
// Two launch shapes share the code: batched (grid = problems, one CTA each) and cooperative (grid = one CTA
// per SM on ONE problem; partial accumulators are reduced through global memory in a fixed order with two
// grid syncs per sweep, so results are bit-reproducible run to run).  All sums use a fixed association.
#include <cooperative_groups.h>
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int EM_THREADS = 1024;
constexpr int EM_WARPS = EM_THREADS / 32;
constexpr int MODE_INIT = 0, MODE_NEXT = 1, MODE_FIRSTK = 2;
constexpr int32_t FK_NONE = 0x7fffffff;

// ---- phase tracing (hgt_em_trace): CTA 0 of every em_kernel launch adds the SM clock cycles its thread 0 spends in
// each phase; off by default (one uniform branch per phase boundary).
// slots: 0 stage p, 1 phase 1 (s_k), 2 phase 2 (acc), 3 cross-CTA reduction, 4 normalise, 5 set-up, 6 SQUAREM/diff/prune,
//        7 <=64-allele loop, 8 kernel total, 9 sweeps, 10 launches; over ALL CTAs: 11 sum of CTA lifetimes (ns), 12 longest
//        CTA lifetime (ns), 13 CTAs
__device__ unsigned long long g_em_trace[16];
__device__ int g_em_trace_on;
struct Trace {
    bool on;
    long long t;
    unsigned long long ns0;
    __device__ __forceinline__ void start() {
        on = g_em_trace_on && blockIdx.x == 0 && threadIdx.x == 0;
        t = on ? clock64() : 0;
        ns0 = 0;
        if (g_em_trace_on && threadIdx.x == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns0));
    }
    __device__ __forceinline__ void finish() {  // every CTA
        if (g_em_trace_on && threadIdx.x == 0) {
            unsigned long long ns1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns1));
            atomicAdd(&g_em_trace[11], ns1 - ns0);
            atomicMax(&g_em_trace[12], ns1 - ns0);
            atomicAdd(&g_em_trace[13], 1ull);
        }
    }
    __device__ __forceinline__ void mark(int k) {
        if (on) {
            const long long n = clock64();
            atomicAdd(&g_em_trace[k], (unsigned long long)(n - t));
            t = n;
        }
    }
    __device__ __forceinline__ void count(int k) {
        if (on) atomicAdd(&g_em_trace[k], 1ull);
    }
};

// ---- read-sharded locus: the per-allele sums of a sweep are exchanged through NVLink peer memory -------------------------
// Every rank (one process per GPU) owns one exchange block, cudaMalloc'ed by hgt_em_peer_alloc and mapped into the other
// processes through CUDA IPC: uint32 flags[EM_PEER_MAX][EM_PEER_G] | int32 abort | uint32 seq | pad to 256 B |
// double data[2][Apad]  (seq = exchanges done so far: a launch continues the numbering of the previous one, so stale
// flags can never satisfy a wait).
// One exchange (sequence number q, parity q & 1), per CTA g - all ranks run the same grid, so CTA g owns the same slice of
// the alleles everywhere: the CTA stores its slice of the locally reduced sums into ITS OWN rank's data[parity]; after a
// system-scope fence it writes q into flags[own rank][g] of every peer's block (one remote store per peer), waits until
// its own block holds flags[r][g] >= q for every peer r, and adds up the slice over the ranks in rank order straight from
// the peers' blocks (remote loads, all in flight together) - so all ranks obtain bit-identical sums and take the same
// branches of the loop, and the only grid-wide step of the exchange is the sync the single-GPU kernel has anyway.
// data[parity] is rewritten two exchanges later, by which time CTA g of every peer has signalled the exchange in
// between, i.e. finished reading.  A peer that does not arrive within EM_PEER_TIMEOUT_NS raises the abort word: the wait
// ends, every CTA sees the word after the next grid sync and the kernel returns HGT_ERR_PEER instead of hanging the GPU.
constexpr int EM_PEER_MAX = 16, EM_PEER_G = 256;  // ranks, CTAs per rank
constexpr unsigned long long EM_PEER_TIMEOUT_NS = 4000000000ull;
constexpr size_t EM_PEER_FLAG_BYTES = (size_t)EM_PEER_MAX * EM_PEER_G * 4, EM_PEER_HDR = EM_PEER_FLAG_BYTES + 256;
struct EmPeer {
    int rank, world;
    unsigned char *block[EM_PEER_MAX];  // block[r] = rank r's exchange block as mapped in this process
};
__device__ __forceinline__ void st_release_sys(uint32_t *p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ double ld_sys_f64(const double *p) {
    double v;
    asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ int32_t ld_sys_s32(const int32_t *p) {
    int32_t v;
    asm volatile("ld.relaxed.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

struct EmArgs {
    const uint64_t *bits;
    const double *cnt;
    const double *len;
    int C, A, wp, remove_low, fixed_iters;
    int slab_rows;  // rows per slab buffer
    int compact;     // host plan: keep an allele-compacted copy of ALL class rows in shared memory (batched launches)
    int A_live_max;  // upper bound of the alleles that are members of any class (sizes the compact buffers)
    unsigned slab_bytes;  // compact layout: bytes of the slab region (>= slab_rows x pitch x 8; the sparse form may use more)
    uint64_t *dense_ws;  // compact layout: global scratch for the gathered dense rows, slab_rows x pitch(A_live_max) words
    uint64_t *mv_ws;     // compact layout: global scratch, 6 x wp words (bit-compress masks of every source word)
    int32_t *rep_ws;     // compact layout: global scratch [64 wp]: representative allele of every member allele, -1 = none
    double *mult_ws;     // compact layout: global scratch [64 wp]: alleles represented by compact column j
    const unsigned long long *cnt_u64;  // class counts as integers (device-resident tables); overrides cnt
    const int32_t *C_ptr;               // number of classes read on the device at launch; overrides C
    const int32_t *class_first;         // tie-break key of each class (first pair index); default = class index
    int32_t key_offset;                 // added to every class key (read-sharded locus: pairs of the lower ranks)
    const EmPeer *peer;                 // cooperative launch on a read-sharded locus: exchange blocks of all ranks (else null)
    double *prob;
    uint8_t *in_result;
    int32_t *first_class;
    int32_t *iters_status;  // [3]: iters, status, sweeps
    // workspace
    double *vec;     // 4 x [Apad]
    uint8_t *live;   // 4 x [Apad]
    double *part_acc;   // [G][Apad]   (cooperative only)
    int32_t *part_aux;  // [G][Apad]   hit flag or first-class index
    double *red_acc;    // [Apad]
    int32_t *red_aux;   // [Apad]
};

struct Smem {
    uint64_t *mbar;
    double *red;
    double *p;
    double *w;
    uint8_t *valid;
    uint64_t *slab;
    // allele-compacted layout only (null otherwise)
    const int32_t *lv;   // [A'] original allele index of compact column j (ascending)
    double *cnt;         // [C] class counts as doubles
    uint64_t *cm64;      // [C] row masks of the <= 64-allele mode
    unsigned char *c64;  // 4 KB block for the small vectors of the <= 64-allele mode
    // sparse form of the compacted matrix (null when the dense slab is used): the non-zero 32-bit words of every
    // class row (row-major, for s_k) and of every 32-allele column (column-major, for acc[a]); rows/columns in
    // ascending order, so all sums keep a fixed association
    const int32_t *row_off;   // [C+1]
    const int32_t *col_off;   // [2*wp+1]
    const uint64_t *r_ent;    // [nnzw] row-major:    low 32 bits = the word, high 32 bits = byte offset of slot p_slot(32 * column)
    const uint64_t *c_ent;    // [nnzw] column-major: low 32 bits = the word, high 32 bits = byte offset of w[row]
    const double *mult;       // [A'] alleles merged into compact column j (identical membership columns); null = all 1
    const uint64_t *dense_g;  // global copy of the compacted dense rows (pitch = wp words), kept for one-off gathers
};

// The staged probability vector is skewed by one slot per 32 alleles (slot of allele a = a + a/32): lanes that walk the
// same bit of 32 different words then fall into different banks (stride 33 doubles instead of 32).
__device__ __forceinline__ int p_slot(int a) { return a + (a >> 5); }
__host__ __device__ constexpr size_t p_slots(size_t Apad) { return Apad + Apad / 32; }

__device__ __forceinline__ int orig_allele(const Smem &sm, int al) { return sm.lv ? sm.lv[al] : al; }

__device__ __forceinline__ double block_sum(double v, double *red) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) red[warp] = v;
    __syncthreads();
    if (warp == 0) {
        double x = red[lane];  // EM_WARPS == 32
        x = warp_sum(x);
        if (lane == 0) red[32] = x;
    }
    __syncthreads();
    double r = red[32];
    __syncthreads();
    return r;
}
__device__ __forceinline__ double block_max(double v, double *red) {
    v = warp_max(v);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) red[warp] = v;
    __syncthreads();
    if (warp == 0) {
        double x = red[lane];
        x = warp_max(x);
        if (lane == 0) red[32] = x;
    }
    __syncthreads();
    double r = red[32];
    __syncthreads();
    return r;
}
__device__ __forceinline__ int block_or(int v) { return __syncthreads_or(v); }

// First half of a sweep: stage the input vector, then both halves of the E/M step over this CTA's rows.  Leaves the
// per-allele sums in acc[] (thread tid, slot i <-> allele tid + i*EM_THREADS), the "met by a class with s_k > 0"
// flags in `hit` and, in FIRSTK mode, the smallest class key in fk[].
template <int NA>
__device__ __forceinline__ void em_accumulate(const EmArgs &a, const Smem &sm, int mode, const double *pin,
                                              const uint8_t *livein, int row_lo, int row_hi, bool resident, bool &loaded,
                                              uint32_t &parity, double (&acc)[NA], int32_t (&fk)[NA], uint32_t &hit,
                                              Trace &tr) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int A = a.A, wp = a.wp;
    const int Apad = wp * 64;
    // stage the input vector (0 for alleles that are not keys of the input dict)
    // (merged columns: the vectors hold the MASS of a column's alleles; the initial mass needs |class| = sum of the
    // multiplicities, so INIT stages them and takes the weighted-sum path)
    const bool weighted_init = mode == MODE_INIT && sm.mult != nullptr;
    if (mode != MODE_INIT) {
        for (int i = tid; i < Apad; i += EM_THREADS) sm.p[p_slot(i)] = (i < A && (!livein || livein[i])) ? pin[i] : 0.0;
    } else if (weighted_init) {
        for (int i = tid; i < Apad; i += EM_THREADS) sm.p[p_slot(i)] = i < A ? sm.mult[i] : 0.0;
    }
    hit = 0;
#pragma unroll
    for (int i = 0; i < NA; i++) {
        acc[i] = 0.0;
        fk[i] = FK_NONE;
    }
    __syncthreads();
    tr.mark(0);
    const uint32_t *slab32 = reinterpret_cast<const uint32_t *>(sm.slab);
    if (sm.row_off) {
        // ---- sparse resident form: cost follows the number of non-zero 32-bit words, not C x A -------------------
        // One packed 64-bit entry per non-zero word; a whole warp takes an entry (word broadcast, lane = bit), so an
        // entry costs LDS.64 + address add + LDS.64 + bit test + predicated DADD.  Four independent partial sums per
        // row hide the DADD latency there; a column keeps ONE running sum (see below); the association is fixed, so
        // results are reproducible.
        const int C = row_hi;
        const unsigned char *p_lane = reinterpret_cast<const unsigned char *>(sm.p + lane);
        int any_skipped = 0;
        for (int r = warp; r < C; r += EM_WARPS) {
            const int e0 = sm.row_off[r], e1 = sm.row_off[r + 1];
            double s = 0.0;
            if (mode == MODE_INIT && !weighted_init) {
                int pc = 0;
                for (int e = e0 + lane; e < e1; e += 32) pc += __popc((uint32_t)sm.r_ent[e]);
                for (int o = 16; o > 0; o >>= 1) pc += __shfl_xor_sync(0xffffffffu, pc, o);
                s = (double)pc;
            } else {
                double s1 = 0.0, s2 = 0.0, s3 = 0.0;
                int e = e0;
                if ((e & 1) && e < e1) {  // entries are fetched in 16-byte pairs from here on (one broadcast wavefront each)
                    const uint64_t x0 = sm.r_ent[e];
                    const double p0 = *reinterpret_cast<const double *>(p_lane + (uint32_t)(x0 >> 32));
                    if (((uint32_t)x0 >> lane) & 1u) s += p0;
                    e++;
                }
                for (; e + 3 < e1; e += 4) {
                    const ulonglong2 q01 = *reinterpret_cast<const ulonglong2 *>(sm.r_ent + e);
                    const ulonglong2 q23 = *reinterpret_cast<const ulonglong2 *>(sm.r_ent + e + 2);
                    const uint64_t x0 = q01.x, x1 = q01.y, x2 = q23.x, x3 = q23.y;
                    const double p0 = *reinterpret_cast<const double *>(p_lane + (uint32_t)(x0 >> 32));
                    const double p1 = *reinterpret_cast<const double *>(p_lane + (uint32_t)(x1 >> 32));
                    const double p2 = *reinterpret_cast<const double *>(p_lane + (uint32_t)(x2 >> 32));
                    const double p3 = *reinterpret_cast<const double *>(p_lane + (uint32_t)(x3 >> 32));
                    if (((uint32_t)x0 >> lane) & 1u) s += p0;
                    if (((uint32_t)x1 >> lane) & 1u) s1 += p1;
                    if (((uint32_t)x2 >> lane) & 1u) s2 += p2;
                    if (((uint32_t)x3 >> lane) & 1u) s3 += p3;
                }
                for (; e < e1; e++) {
                    const uint64_t x0 = sm.r_ent[e];
                    const double p0 = *reinterpret_cast<const double *>(p_lane + (uint32_t)(x0 >> 32));
                    if (((uint32_t)x0 >> lane) & 1u) s += p0;
                }
                s = warp_sum((s + s1) + (s2 + s3));
            }
            if (lane == 0) {
                sm.w[r] = s > 0.0 ? sm.cnt[r] / s : -1.0;  // negative = class skipped (s_k <= 0)
                if (!(s > 0.0)) any_skipped = 1;
            }
        }
        const int skipped = __syncthreads_or(any_skipped);
        tr.mark(1);
        const unsigned char *w_base = reinterpret_cast<const unsigned char *>(sm.w);
#pragma unroll
        for (int i = 0; i < NA; i++) {
            const int c = warp + 32 * i;  // thread (warp, lane), slot i  <->  allele c*32 + lane = tid + i*EM_THREADS
            if (c >= 2 * wp) continue;
            const int e0 = sm.col_off[c], e1 = sm.col_off[c + 1];
            if (mode == MODE_FIRSTK) {
                for (int e = e0; e < e1; e++) {
                    const uint64_t x = sm.c_ent[e];
                    const int r = (int)((uint32_t)(x >> 32) >> 3);
                    if (sm.w[r] < 0.0) continue;
                    if (((uint32_t)x >> lane) & 1u) fk[i] = min(fk[i], (a.class_first ? a.class_first[r] : r) + a.key_offset);
                }
            } else if (!skipped) {
                // ONE running sum per allele, rows in ascending order: alleles with identical membership columns must end
                // with bit-identical sums (the reference's ties are exact and decide the ranking), and with partial sums
                // chosen by entry parity the association would depend on the OTHER alleles of the 32-allele word.  The
                // loads of four entries are issued together; only the predicated adds form the chain.
                double x0 = 0.0;
                uint32_t seen = 0u;
                int e = e0;
                if ((e & 1) && e < e1) {
                    const uint64_t y0 = sm.c_ent[e];
                    const double w0 = *reinterpret_cast<const double *>(w_base + (uint32_t)(y0 >> 32));
                    if (((uint32_t)y0 >> lane) & 1u) x0 += w0;
                    seen |= (uint32_t)y0;
                    e++;
                }
                for (; e + 3 < e1; e += 4) {
                    const ulonglong2 q01 = *reinterpret_cast<const ulonglong2 *>(sm.c_ent + e);
                    const ulonglong2 q23 = *reinterpret_cast<const ulonglong2 *>(sm.c_ent + e + 2);
                    const double w0 = *reinterpret_cast<const double *>(w_base + (uint32_t)(q01.x >> 32));
                    const double w1 = *reinterpret_cast<const double *>(w_base + (uint32_t)(q01.y >> 32));
                    const double w2 = *reinterpret_cast<const double *>(w_base + (uint32_t)(q23.x >> 32));
                    const double w3 = *reinterpret_cast<const double *>(w_base + (uint32_t)(q23.y >> 32));
                    if (((uint32_t)q01.x >> lane) & 1u) x0 += w0;
                    if (((uint32_t)q01.y >> lane) & 1u) x0 += w1;
                    if (((uint32_t)q23.x >> lane) & 1u) x0 += w2;
                    if (((uint32_t)q23.y >> lane) & 1u) x0 += w3;
                    seen |= (uint32_t)q01.x | (uint32_t)q01.y | (uint32_t)q23.x | (uint32_t)q23.y;
                }
                for (; e < e1; e++) {
                    const uint64_t y0 = sm.c_ent[e];
                    const double w0 = *reinterpret_cast<const double *>(w_base + (uint32_t)(y0 >> 32));
                    if (((uint32_t)y0 >> lane) & 1u) x0 += w0;
                    seen |= (uint32_t)y0;
                }
                acc[i] = x0;
                if ((seen >> lane) & 1u) hit |= 1u << i;
            } else {
                double x = 0.0;
                bool h = false;
                for (int e = e0; e < e1; e++) {
                    const uint64_t y = sm.c_ent[e];
                    const double w = *reinterpret_cast<const double *>(w_base + (uint32_t)(y >> 32));
                    if (w < 0.0) continue;
                    if (((uint32_t)y >> lane) & 1u) {
                        x += w;
                        h = true;
                    }
                }
                acc[i] = x;
                if (h) hit |= 1u << i;
            }
        }
        __syncthreads();
        tr.mark(2);
        row_lo = row_hi;  // nothing left for the slab loop
    }
    for (int r0 = row_lo; r0 < row_hi; r0 += a.slab_rows) {
        const int nr = min(a.slab_rows, row_hi - r0);
        if (!(resident && loaded)) {
            if (tid == 0) {
                const uint32_t bytes = (uint32_t)nr * (uint32_t)wp * 8u;
                mbar_expect_tx(sm.mbar, bytes);
                bulk_g2s(sm.slab, a.bits + (size_t)r0 * wp, bytes, sm.mbar);
            }
            mbar_wait(sm.mbar, parity);
            parity ^= 1u;
            loaded = true;
        }
        // ---- phase 1: warp per row ---------------------------------------------------------------------
        int any_skipped = 0;
        for (int r = warp; r < nr; r += EM_WARPS) {
            const uint64_t *row = sm.slab + (size_t)r * wp;
            double s = 0.0;
            if (mode == MODE_INIT && !weighted_init) {
                int pc = 0;
                for (int j = lane; j < wp; j += 32) pc += __popcll(row[j]);
                for (int o = 16; o > 0; o >>= 1) pc += __shfl_xor_sync(0xffffffffu, pc, o);
                s = (double)pc;
            } else {
                // 32 words at a time: every lane fetches one word, the non-zero ones are then taken one by one by the whole
                // warp (word broadcast by shuffle, lane = bit, conflict-free read of 32 consecutive p slots), so the cost
                // follows the number of non-zero words and not the per-lane maximum of set bits
                const uint32_t *row32 = reinterpret_cast<const uint32_t *>(row);
                double s1 = 0.0;
                for (int j0 = 0; j0 < 2 * wp; j0 += 32) {
                    const int j = j0 + lane;
                    const uint32_t mine = j < 2 * wp ? row32[j] : 0u;
                    unsigned nz = __ballot_sync(0xffffffffu, mine != 0u);
                    const double *pb = sm.p + j0 * 33 + lane;
                    while (nz) {
                        const int k0 = __ffs((int)nz) - 1;
                        nz &= nz - 1;
                        const uint32_t w0 = __shfl_sync(0xffffffffu, mine, k0);
                        const double v0 = pb[k0 * 33];
                        if ((w0 >> lane) & 1u) s += v0;
                        if (nz) {
                            const int k1 = __ffs((int)nz) - 1;
                            nz &= nz - 1;
                            const uint32_t w1 = __shfl_sync(0xffffffffu, mine, k1);
                            const double v1 = pb[k1 * 33];
                            if ((w1 >> lane) & 1u) s1 += v1;
                        }
                    }
                }
                s += s1;
                s = warp_sum(s);
            }
            if (lane == 0) {
                const bool ok = s > 0.0;
                sm.valid[r] = ok ? 1 : 0;
                const double n = sm.cnt ? sm.cnt[r0 + r] : (a.cnt_u64 ? (double)a.cnt_u64[r0 + r] : a.cnt[r0 + r]);
                sm.w[r] = ok ? n / s : -1.0;  // negative = class skipped (s_k <= 0)
                if (!ok) any_skipped = 1;
            }
        }
        const int skipped = __syncthreads_or(any_skipped);
        tr.mark(1);
        // ---- phase 2: thread per allele column -----------------------------------------------------------
        // thread (warp, lane), slot i  <->  allele (warp + 32 i) * 32 + lane: all lanes of a warp read the same 32-bit
        // word of a row (shared-memory broadcast) and test their own bit.  Rows are walked with one running pointer and
        // the slot offsets are compile-time constants, so a (row, slot) step is LDS + bit test + predicated DADD.
        if (mode == MODE_FIRSTK) {
            for (int r = 0; r < nr; r++) {
                if (!sm.valid[r]) continue;
                const int32_t key = (a.class_first ? a.class_first[r0 + r] : r0 + r) + a.key_offset;
#pragma unroll
                for (int i = 0; i < NA; i++) {
                    const int al = tid + i * EM_THREADS;
                    if (al < A) {
                        const uint32_t w32 = slab32[(size_t)r * wp * 2 + (al >> 5)];
                        if ((w32 >> (al & 31)) & 1u) fk[i] = min(fk[i], key);
                    }
                }
            }
        } else {
            const uint32_t *pr = slab32 + warp;
            const int stride = 2 * wp;
            uint32_t seen[NA];
#pragma unroll
            for (int i = 0; i < NA; i++) seen[i] = 0u;
            const int nslot = min(NA, (stride - warp + 31) >> 5);  // slots whose word column lies inside the row
            if (nslot == NA) {
                for (int r = 0; r < nr; r++, pr += stride) {
                    const double w = sm.w[r];
                    if (skipped && w < 0.0) continue;
#pragma unroll
                    for (int i = 0; i < NA; i++) {
                        const uint32_t w32 = pr[32 * i];
                        if ((w32 >> lane) & 1u) acc[i] += w;
                        seen[i] |= w32;
                    }
                }
            } else {
                for (int r = 0; r < nr; r++, pr += stride) {
                    const double w = sm.w[r];
                    if (skipped && w < 0.0) continue;
#pragma unroll
                    for (int i = 0; i < NA; i++) {
                        if (i < nslot) {
                            const uint32_t w32 = pr[32 * i];
                            if ((w32 >> lane) & 1u) acc[i] += w;
                            seen[i] |= w32;
                        }
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < NA; i++)
                if ((seen[i] >> lane) & 1u) hit |= 1u << i;
        }
        __syncthreads();
        tr.mark(2);
    }
}

// The exchange step of a sweep on a read-sharded locus (see EmPeer).  Not inlined: it runs once per sweep, and inlined its
// sixteen in-flight remote loads would raise the register pressure of every em_kernel<.., true> instance.
__device__ __noinline__ void peer_exchange(const EmArgs &a, const EmPeer *px, int mode, uint32_t q, int a_lo, int a_hi, int Apad,
                                           int g) {
    const int tid = threadIdx.x;
    // slice g of this rank <-> slice g of every peer (same grid on every rank): no grid-wide step in between
    // the slice was written by lane 0 of every warp: those lanes fence at system scope, the CTA barrier orders them before the
    // release store of the flag (release is cumulative over what happens-before it)
    if ((tid & 31) == 0) __threadfence_system();
    __syncthreads();
    uint32_t *my_flags = reinterpret_cast<uint32_t *>(px->block[px->rank]);
    int32_t *my_abort = reinterpret_cast<int32_t *>(px->block[px->rank] + EM_PEER_FLAG_BYTES);
    if (tid < px->world && tid != px->rank) {
        st_release_sys(reinterpret_cast<uint32_t *>(px->block[tid]) + px->rank * EM_PEER_G + g, q);
        unsigned long long t0, t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        while (ld_acquire_sys(my_flags + tid * EM_PEER_G + g) < q) {
            if (*reinterpret_cast<volatile int32_t *>(my_abort)) break;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            if (t1 - t0 > EM_PEER_TIMEOUT_NS) {
                atomicExch(my_abort, 1);
                break;
            }
        }
    }
    __syncthreads();
    const size_t off = EM_PEER_HDR + (size_t)(q & 1u) * Apad * 8;
    for (int al = a_lo + tid; al < a_hi; al += EM_THREADS) {
        // all remote loads in flight together, then the sum in rank order (the same association on every rank)
        if (mode == MODE_FIRSTK) {
            int32_t x = FK_NONE;
            for (int r0 = 0; r0 < px->world; r0 += 8) {
                int32_t v[8];
#pragma unroll
                for (int r = 0; r < 8; r++)
                    v[r] = r0 + r < px->world ? ld_sys_s32(reinterpret_cast<const int32_t *>(px->block[r0 + r] + off) + al) : FK_NONE;
#pragma unroll
                for (int r = 0; r < 8; r++) x = min(x, v[r]);
            }
            a.red_aux[al] = x;
        } else {
            double s = -0.0;
            for (int r0 = 0; r0 < px->world; r0 += 8) {
                double v[8];
#pragma unroll
                for (int r = 0; r < 8; r++)
                    v[r] = r0 + r < px->world ? ld_sys_f64(reinterpret_cast<const double *>(px->block[r0 + r] + off) + al) : -0.0;
#pragma unroll
                for (int r = 0; r < 8; r++) s += v[r];  // (-0.0 is the neutral element, also for the sign-of-zero flag)
            }
            a.red_acc[al] = s;
        }
    }
}

// One sweep over this CTA's class rows.  mode INIT: initial mass (common:1299-1309); NEXT: next_prob
// (common:1311-1336); FIRSTK: only the dict insertion order of next_prob's output.
template <int NA, bool COOP>
__device__ void em_sweep(const EmArgs &a, const Smem &sm, int mode, const double *pin, const uint8_t *livein,
                         double *pout, uint8_t *liveout, int32_t *fkout, int row_lo, int row_hi, bool resident,
                         bool &loaded, uint32_t &parity, int *status, Trace &tr, uint32_t &xseq) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int A = a.A, wp = a.wp;
    const int Apad = wp * 64;
    double acc[NA];
    int32_t fk[NA];
    uint32_t hit = 0;
    em_accumulate<NA>(a, sm, mode, pin, livein, row_lo, row_hi, resident, loaded, parity, acc, fk, hit, tr);
    tr.count(9);
    // ---- cross-CTA reduction (cooperative launch only) ------------------------------------------------------
    if (COOP) {
        // Partials are laid out [CTA][allele]: coalesced stores, and the reducing warps read whole sectors (below).  In the
        // INIT / NEXT modes the "met by a valid class" flag rides in the sign of zero: a CTA that did not meet the allele
        // contributes -0.0, one that did contributes its sum (>= +0.0), and -0.0 survives an IEEE sum only if every
        // term is -0.0.  FIRSTK exchanges the int32 keys instead of sums.
        cg::grid_group grid = cg::this_grid();
        const int G = gridDim.x, g = blockIdx.x;
#pragma unroll
        for (int i = 0; i < NA; i++) {
            const int al = tid + i * EM_THREADS;
            if (al < A) {
                if (mode == MODE_FIRSTK) a.part_aux[(size_t)g * Apad + al] = fk[i];
                else a.part_acc[(size_t)g * Apad + al] = ((hit >> i) & 1u) ? acc[i] : -0.0;
            }
        }
        grid.sync();
        tr.mark(14);  // (cooperative launches: partials written + first grid sync; the batched form uses the slot for the merge)
        // slices of whole 4-allele groups: a reducing warp takes four alleles at a time, lane = CTA, so that every 32-byte
        // sector of the partials is written once (coalesced, [CTA][allele]) and read once
        const int Ag = (((A + G - 1) / G) + 3) & ~3;
        const int a_lo = min(A, g * Ag), a_hi = min(A, a_lo + Ag);
        // (read-sharded locus: the slice goes to this rank's exchange block first, see EmPeer)
        const EmPeer *px = a.peer;
        const uint32_t q = xseq + 1;
        double *x_acc = px ? reinterpret_cast<double *>(px->block[px->rank] + EM_PEER_HDR) + (size_t)(q & 1u) * Apad : a.red_acc;
        int32_t *x_aux = px ? reinterpret_cast<int32_t *>(x_acc) : a.red_aux;
        for (int al = a_lo + 4 * warp; al < a_hi; al += 4 * EM_WARPS) {
            if (mode == MODE_FIRSTK) {
                int32_t x0 = FK_NONE, x1 = FK_NONE, x2 = FK_NONE, x3 = FK_NONE;
                for (int gg = lane; gg < G; gg += 32) {
                    const int4 v = __ldcg(reinterpret_cast<const int4 *>(a.part_aux + (size_t)gg * Apad + al));
                    x0 = min(x0, v.x); x1 = min(x1, v.y); x2 = min(x2, v.z); x3 = min(x3, v.w);
                }
                for (int o = 16; o > 0; o >>= 1) {
                    x0 = min(x0, __shfl_xor_sync(0xffffffffu, x0, o));
                    x1 = min(x1, __shfl_xor_sync(0xffffffffu, x1, o));
                    x2 = min(x2, __shfl_xor_sync(0xffffffffu, x2, o));
                    x3 = min(x3, __shfl_xor_sync(0xffffffffu, x3, o));
                }
                if (lane == 0) {
                    x_aux[al] = x0;
                    if (al + 1 < a_hi) x_aux[al + 1] = x1;
                    if (al + 2 < a_hi) x_aux[al + 2] = x2;
                    if (al + 3 < a_hi) x_aux[al + 3] = x3;
                }
            } else {
                double s0 = -0.0, s1 = -0.0, s2 = -0.0, s3 = -0.0;
                for (int gg = lane; gg < G; gg += 32) {
                    const double2 *src = reinterpret_cast<const double2 *>(a.part_acc + (size_t)gg * Apad + al);
                    const double2 u = __ldcg(src), v = __ldcg(src + 1);
                    s0 += u.x; s1 += u.y; s2 += v.x; s3 += v.y;
                }
                s0 = warp_sum(s0); s1 = warp_sum(s1); s2 = warp_sum(s2); s3 = warp_sum(s3);
                if (lane == 0) {
                    x_acc[al] = s0;
                    if (al + 1 < a_hi) x_acc[al + 1] = s1;
                    if (al + 2 < a_hi) x_acc[al + 2] = s2;
                    if (al + 3 < a_hi) x_acc[al + 3] = s3;
                }
            }
        }
        if (px) {
            xseq = q;
            peer_exchange(a, px, mode, q, a_lo, a_hi, Apad, g);
        }
        tr.mark(15);  // (cooperative launches: slice reduction + exchange)
        grid.sync();
        if (px && *reinterpret_cast<volatile int32_t *>(px->block[px->rank] + EM_PEER_FLAG_BYTES)) {
            if (tid == 0) *status = HGT_ERR_PEER;  // (every CTA reads the same word after the grid sync)
            __syncthreads();
        }
        hit = 0;
#pragma unroll
        for (int i = 0; i < NA; i++) {
            const int al = tid + i * EM_THREADS;
            if (al < A) {
                if (mode == MODE_FIRSTK) {
                    fk[i] = __ldcg(&a.red_aux[al]);
                } else {
                    acc[i] = __ldcg(&a.red_acc[al]);
                    if (!signbit(acc[i])) hit |= 1u << i;
                }
            }
        }
    }
    if (COOP) tr.mark(3);
    if (mode == MODE_FIRSTK) {
#pragma unroll
        for (int i = 0; i < NA; i++) {
            const int al = tid + i * EM_THREADS;
            if (al < A) fkout[orig_allele(sm, al)] = livein[al] ? fk[i] : FK_NONE;
        }
        __syncthreads();
        return;
    }
    // ---- q = p * acc, keys = live & hit, normalize (common:1285-1297) ----------------------------------------
    double part = 0.0;
    int nkeys = 0;
#pragma unroll
    for (int i = 0; i < NA; i++) {
        const int al = tid + i * EM_THREADS;
        bool key = false;
        double q = 0.0;
        if (al < A) {
            key = ((hit >> i) & 1u) && (mode == MODE_INIT || livein[al]);
            if (key) {
                q = (mode == MODE_INIT && !sm.mult) ? acc[i] : sm.p[p_slot(al)] * acc[i];  // INIT on merged columns: x multiplicity
                if (a.len) q = q / a.len[orig_allele(sm, al)];
                part += q;
                nkeys = 1;
            }
        }
        acc[i] = q;
        hit = key ? (hit | (1u << i)) : (hit & ~(1u << i));
    }
    const double total = block_sum(part, sm.red);
    const int any = block_or(nkeys);
    if (any && !(total > 0.0) && !(total < 0.0)) {
        if (tid == 0) *status = HGT_ERR_ZERODIV;
    }
#pragma unroll
    for (int i = 0; i < NA; i++) {
        const int al = tid + i * EM_THREADS;
        if (al < A) {
            const bool key = (hit >> i) & 1u;
            pout[al] = key ? acc[i] / total : 0.0;
            liveout[al] = key ? 1 : 0;
        }
    }
    __syncthreads();
    tr.mark(4);
}

// select_alleles (common:1338-1346): keep p >= max/10
__device__ void em_prune(const EmArgs &a, const Smem &sm, double *p, uint8_t *live) {
    // merged columns: p holds the mass of sm.mult[al] equal alleles, the rule is per allele
    double mx = -1.0;
    for (int al = threadIdx.x; al < a.A; al += EM_THREADS)
        if (live[al]) mx = fmax(mx, sm.mult ? p[al] / sm.mult[al] : p[al]);
    mx = block_max(mx, sm.red);
    if (mx < 0.0) return;
    const double thr = mx / 10.0;
    for (int al = threadIdx.x; al < a.A; al += EM_THREADS) {
        if (live[al] && !((sm.mult ? p[al] / sm.mult[al] : p[al]) >= thr)) {
            live[al] = 0;
            p[al] = 0.0;
        }
    }
    __syncthreads();
}


// ---- compact mode ------------------------------------------------------------------------------------------------
// Once at most 64 alleles are still keys of Gene_prob (typically right after the first select_alleles() at
// iteration 10, common:1390-1391) every class row collapses to ONE 64-bit word over those alleles.  The rest of
// the loop then runs entirely out of shared memory: cm[C] (row masks), cnt[C], w[C] and 64-entry vectors.
// Sums run in a fixed order (ascending allele / fixed lane stride + butterfly), so results are reproducible.
struct Compact {
    uint64_t *cm;   // [C] membership of the compact alleles in each class
    double *cnt;    // [C]
    double *w;      // [C] n_k / s_k, negative = class skipped (s_k <= 0)
    int *lv;        // [64] allele id of compact slot j (ascending)
    double *v;      // [4][64] p0, p1, p2, extrapolated
    int *l;         // [3][64] key flags of p0, p1, p2
    double *len;    // [64]
    double *q;      // [64] scratch
    int n;          // compact alleles
};

__device__ void compact_sweep(const EmArgs &a, const Compact &c, const double *pin, const int *lin, double *pout,
                              int *lout, int *status) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int C = a.C;
    for (int r = tid; r < C; r += EM_THREADS) {
        uint64_t m = c.cm[r];
        double s = 0.0;
        while (m) {
            const int j = __ffsll((long long)m) - 1;
            m &= m - 1;
            if (lin[j]) s += pin[j];
        }
        c.w[r] = s > 0.0 ? c.cnt[r] / s : -1.0;
    }
    __syncthreads();
    for (int j = warp; j < c.n; j += EM_WARPS) {
        double acc = 0.0;
        int hit = 0;
        for (int r = lane; r < C; r += 32) {
            const double w = c.w[r];
            if (((c.cm[r] >> j) & 1ull) && w >= 0.0) {
                acc += w;
                hit = 1;
            }
        }
        acc = warp_sum(acc);
        hit = __any_sync(0xffffffffu, hit);
        if (lane == 0) {
            const int key = lin[j] && hit;
            double q = key ? pin[j] * acc : 0.0;
            if (a.len && key) q = q / c.len[j];
            c.q[j] = q;
            lout[j] = key;
        }
    }
    __syncthreads();
    if (warp == 0) {
        double part = 0.0;
        int any = 0;
        for (int j = lane; j < c.n; j += 32)
            if (lout[j]) {
                part += c.q[j];
                any = 1;
            }
        const double total = warp_sum(part);
        any = __any_sync(0xffffffffu, any);
        if (any && !(total > 0.0) && !(total < 0.0) && lane == 0) *status = HGT_ERR_ZERODIV;
        for (int j = lane; j < c.n; j += 32) pout[j] = lout[j] ? c.q[j] / total : 0.0;
    }
    __syncthreads();
}

// Runs the remaining loop iterations in compact form.  On return slot 0 holds Gene_prob, `last` tells which
// slot fed the last next_prob() (0 or 3) with key flags in l[last == 3 ? 2 : 0].
__device__ void compact_loop(const EmArgs &a, Compact &c, double &diff, int &iter, int &sweeps, int &last,
                             bool &have_last, int *status) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double *v0 = c.v, *v1 = c.v + 64, *v2 = c.v + 128, *v3 = c.v + 192;
    int *l0 = c.l, *l1 = c.l + 64, *l2 = c.l + 128;
    __shared__ double s_diff;
    __shared__ int s_flag;
    while (a.fixed_iters > 0 ? iter < a.fixed_iters : (diff > 0.0001 && iter < 1000)) {
        if (*status != HGT_OK) break;
        compact_sweep(a, c, v0, l0, v1, l1, status);
        compact_sweep(a, c, v1, l1, v2, l2, status);
        sweeps += 2;
        if (warp == 0) {
            double ssr = 0.0, ssv = 0.0;
            int keyerr = 0;
            for (int j = lane; j < c.n; j += 32)
                if (l0[j]) {
                    if (!l1[j] || !l2[j]) keyerr = 1;
                    const double r = v1[j] - v0[j];
                    const double v = v2[j] - v1[j] - r;
                    ssr += r * r;
                    ssv += v * v;
                }
            ssr = warp_sum(ssr);
            ssv = warp_sum(ssv);
            keyerr = __any_sync(0xffffffffu, keyerr);
            int flag = 0;
            if (keyerr) flag = 2;
            else if (ssv > 0.0) {
                flag = 1;
                const double g = -sqrt(ssr / ssv);
                for (int j = lane; j < c.n; j += 32) {
                    double x = 0.0;
                    if (l0[j]) {
                        const double r = v1[j] - v0[j];
                        const double v = v2[j] - v1[j] - r;
                        x = v0[j] - 2 * g * r + g * g * v;
                        x = x > 0.0 ? x : 0.0;
                    }
                    v3[j] = x;
                }
            }
            if (lane == 0) s_flag = flag;
        }
        __syncthreads();
        const int flag = s_flag;
        if (flag == 2) {
            if (tid == 0) *status = HGT_ERR_KEY;
            __syncthreads();
            break;
        }
        if (flag == 1) {
            compact_sweep(a, c, v3, l2, v1, l1, status);
            sweeps += 1;
            last = 3;
        } else {
            last = 0;
        }
        have_last = true;
        if (warp == 0) {
            double d = 0.0;
            for (int j = lane; j < c.n; j += 32)
                if (l0[j]) d += l1[j] ? fabs(v0[j] - v1[j]) : v0[j];
            d = warp_sum(d);
            if (lane == 0) s_diff = d;
        }
        __syncthreads();
        diff = s_diff;
        // Gene_prob = Gene_prob_next: slot 0 <- slot 1 (a copy keeps `last == 0` pointing at the old vector in slot 1)
        if (tid < 64) {
            const double t = v0[tid];
            const int tl = l0[tid];
            v0[tid] = v1[tid];
            l0[tid] = l1[tid];
            v1[tid] = t;
            l1[tid] = tl;
        }
        __syncthreads();
        if (last == 0) last = 1;  // the input of the last next_prob() now sits in slot 1
        if (iter >= 10 && a.remove_low) {
            if (warp == 0) {
                double mx = -1.0;
                for (int j = lane; j < c.n; j += 32)
                    if (l0[j]) mx = fmax(mx, v0[j]);
                mx = warp_max(mx);
                if (mx >= 0.0) {
                    const double thr = mx / 10.0;
                    for (int j = lane; j < c.n; j += 32)
                        if (l0[j] && !(v0[j] >= thr)) {
                            l0[j] = 0;
                            v0[j] = 0.0;
                        }
                }
            }
            __syncthreads();
        }
        iter++;
    }
}

constexpr int DEDUP_CAP = 8192;         // hash slots; at most 6144 live alleles (load factor 0.75)
constexpr int DEDUP_MAX_LIVE = 6144;
constexpr int DEDUP_COLS = 4;           // 64-allele word columns per warp: wp <= 128
// Sizes under which an allele-compacted problem without lengths merges identical columns (kernel and hgt_em_form).
__host__ __device__ inline bool em_merge_fits(int wp, int A_live_max, size_t slab_bytes) {
    return wp <= DEDUP_COLS * EM_WARPS && A_live_max <= DEDUP_MAX_LIVE && slab_bytes >= (size_t)wp * 64 * 12 + DEDUP_CAP * 4 &&
           slab_bytes >= (size_t)wp * 8 * 32;
}
// Whether a one-CTA problem can switch to the <= 64-key loop: the allele-compacted layout has buffers for it, the
// streaming layout re-uses its staged vector and slab (C class masks, counts and weights) (kernel and hgt_em_form).
__host__ __device__ inline bool em_collapse_fits(bool compacted, int C, int wp, int slab_rows) {
    return compacted || (size_t)C * 24 + 64 * 64 <= p_slots((size_t)wp * 64) * 8 + (size_t)slab_rows * 8 + (size_t)slab_rows * wp * 8;
}
__device__ __forceinline__ unsigned long long dedup_mix(unsigned long long x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
    return x;
}

// Builds the allele-compacted problem in shared memory: the alleles that are members of at least one class
// (every other allele keeps probability 0 for the whole run, common:1299-1309) are renumbered 0..A'-1 in
// ascending order and every class row is gathered into A' bits.  Returns A'.
__device__ int em_compact_build(const EmArgs &a, Smem &sm, int32_t *lv, int C, int *s_int, bool dedup, Trace &tr) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wp = a.wp;  // <= 256
    uint64_t *lw = reinterpret_cast<uint64_t *>(sm.c64);           // [256] OR of all rows
    int32_t *base = reinterpret_cast<int32_t *>(sm.c64 + 2048);    // [256] live alleles before word j
    for (int j = tid; j < 256; j += EM_THREADS) lw[j] = 0ull;
    __syncthreads();
    {
        uint64_t acc[8];
#pragma unroll
        for (int i = 0; i < 8; i++) acc[i] = 0ull;
        for (int r = warp; r < C; r += EM_WARPS) {
            const uint64_t *row = a.bits + (size_t)r * wp;
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const int j = lane + 32 * i;
                if (j < wp) acc[i] |= row[j];
            }
        }
#pragma unroll
        for (int i = 0; i < 8; i++)
            if (acc[i]) atomicOr(reinterpret_cast<unsigned long long *>(&lw[lane + 32 * i]), (unsigned long long)acc[i]);
    }
    __syncthreads();
    tr.mark(5);
    if (dedup) {
        // ---- merge alleles with identical membership columns --------------------------------------------------------------
        // Such alleles start with the same mass and receive the same factor in every next_prob(), so they stay equal for
        // the whole run: only the smallest one of each set (the representative) stays in the live mask and carries the
        // set's total mass (em_kernel keeps track of the multiplicities where a per-allele quantity is needed).
        // Columns are compared through a 96-bit GF(2)-linear signature: bit t of allele a = parity of the rows that hold a
        // and whose random word has bit t set (two distinct columns collide with probability 2^-96).  It is computed 64
        // alleles at a time: a warp owns a 64-allele word column, lane t keeps the three 64-bit planes t, t+32 and t+64
        // (plane ^= row word where the row's random word has that bit), the class rows come through shared memory in
        // tiles, and a ballot transpose turns the planes into per-allele signatures.
        int32_t *cnt32 = reinterpret_cast<int32_t *>(a.dense_ws);  // [64 wp] members merged into allele a (dense scratch)
        const int Atot = wp * 64;
        for (int al = tid; al < Atot; al += EM_THREADS) { cnt32[al] = 0; a.rep_ws[al] = -1; }
        unsigned long long *xs = reinterpret_cast<unsigned long long *>(sm.w);  // per-row random words (free until the sweeps)
        uint32_t *ys = reinterpret_cast<uint32_t *>(sm.cnt);
        for (int r = tid; r < C; r += EM_THREADS) {
            const unsigned long long x = dedup_mix((unsigned long long)r + 1ull);
            xs[r] = x;
            ys[r] = (uint32_t)dedup_mix(x ^ 0x9e3779b97f4a7c15ull);
        }
        uint64_t *tile = sm.slab;
        const int T = min(C, (int)(a.slab_bytes / ((size_t)wp * 8)));
        uint64_t pa[DEDUP_COLS], pb[DEDUP_COLS], pc[DEDUP_COLS];
#pragma unroll
        for (int c = 0; c < DEDUP_COLS; c++) pa[c] = pb[c] = pc[c] = 0ull;
        for (int t0 = 0; t0 < C; t0 += T) {
            const int nr = min(T, C - t0);
            __syncthreads();
            {  // wp is even and the rows are 16-byte aligned: 16-byte copies, four in flight per thread
                const ulonglong2 *src = reinterpret_cast<const ulonglong2 *>(a.bits + (size_t)t0 * wp);
                ulonglong2 *dst = reinterpret_cast<ulonglong2 *>(tile);
                const int n2 = nr * wp / 2;
#pragma unroll 4
                for (int i = tid; i < n2; i += EM_THREADS) dst[i] = __ldg(&src[i]);
            }
            __syncthreads();
            // a warp owns the 4 adjacent word columns 4 warp .. 4 warp + 3: two 16-byte loads fetch them, and a row that is
            // zero in all four (most rows of most column groups) costs nothing else
            const int j0 = warp * DEDUP_COLS;
            if (j0 < wp) {
                const bool v1 = j0 + 1 < wp, v2 = j0 + 2 < wp, v3 = j0 + 3 < wp;
                for (int r = 0; r < nr; r++) {
                    const ulonglong2 *trow = reinterpret_cast<const ulonglong2 *>(tile + (size_t)r * wp + j0);
                    const ulonglong2 q01 = trow[0], q23 = trow[1];
                    const uint64_t w0 = q01.x, w1 = v1 ? q01.y : 0ull, w2 = v2 ? q23.x : 0ull, w3 = v3 ? q23.y : 0ull;
                    if ((w0 | w1 | w2 | w3) == 0ull) continue;
                    const unsigned long long x = xs[t0 + r];
                    const uint32_t y = ys[t0 + r];
                    const uint64_t m0 = ((x >> lane) & 1ull) ? ~0ull : 0ull, m1 = ((x >> (lane + 32)) & 1ull) ? ~0ull : 0ull,
                                   m2 = ((y >> lane) & 1u) ? ~0ull : 0ull;
                    pa[0] ^= w0 & m0; pb[0] ^= w0 & m1; pc[0] ^= w0 & m2;
                    pa[1] ^= w1 & m0; pb[1] ^= w1 & m1; pc[1] ^= w1 & m2;
                    pa[2] ^= w2 & m0; pb[2] ^= w2 & m1; pc[2] ^= w2 & m2;
                    pa[3] ^= w3 & m0; pb[3] ^= w3 & m1; pc[3] ^= w3 & m2;
                }
            }
        }
        __syncthreads();
        tr.mark(14);
        unsigned long long *sig1 = reinterpret_cast<unsigned long long *>(sm.slab);  // [64 wp], the tile is done with
        uint32_t *sig2 = reinterpret_cast<uint32_t *>(sig1 + Atot);
#pragma unroll
        for (int c = 0; c < DEDUP_COLS; c++) {
            const int j = warp * DEDUP_COLS + c;
            if (j >= wp) continue;
            const uint64_t live = lw[j];
            for (int b = 0; b < 64; b++) {
                if (!((live >> b) & 1ull)) continue;  // warp-uniform
                const unsigned m0 = __ballot_sync(0xffffffffu, (pa[c] >> b) & 1ull);
                const unsigned m1 = __ballot_sync(0xffffffffu, (pb[c] >> b) & 1ull);
                const unsigned m2 = __ballot_sync(0xffffffffu, (pc[c] >> b) & 1ull);
                if (lane == 0) {
                    sig1[j * 64 + b] = (unsigned long long)m0 | ((unsigned long long)m1 << 32);
                    sig2[j * 64 + b] = m2;
                }
            }
        }
        __syncthreads();
        // hash table in shared memory next to the signatures, one 32-bit word per slot: high half = the allele that
        // claimed the slot (its signature is the slot's key), low half = the smallest allele met with that signature
        // (atomicMin on the whole word: the high half is fixed once claimed)
        uint32_t *occ = sig2 + Atot;
        for (int i = tid; i < DEDUP_CAP; i += EM_THREADS) occ[i] = 0xffffffffu;
        __syncthreads();
        for (int al = tid; al < Atot; al += EM_THREADS) {
            if (!((lw[al >> 6] >> (al & 63)) & 1ull)) continue;
            const unsigned long long h1 = sig1[al];
            const uint32_t h2 = sig2[al];
            unsigned slot = (unsigned)dedup_mix(h1 + h2) & (DEDUP_CAP - 1);
            while (true) {
                const uint32_t prev = atomicCAS(&occ[slot], 0xffffffffu, ((uint32_t)al << 16) | (uint32_t)al);
                if (prev == 0xffffffffu) break;
                const int owner = (int)(prev >> 16);
                if (sig1[owner] == h1 && sig2[owner] == h2) {
                    atomicMin(&occ[slot], ((uint32_t)owner << 16) | (uint32_t)al);
                    break;
                }
                slot = (slot + 1) & (DEDUP_CAP - 1);
            }
            a.rep_ws[al] = (int)slot;  // resolved to the representative allele below
        }
        __syncthreads();
        for (int al = tid; al < Atot; al += EM_THREADS) {
            const int slot = a.rep_ws[al];
            if (slot < 0) continue;
            const int rp = (int)(occ[slot] & 0xffffu);
            a.rep_ws[al] = rp;
            if (rp != al) atomicAdd(&cnt32[rp], 1);
        }
        __syncthreads();
        // only the representatives stay live
        for (int al = tid; al < Atot; al += EM_THREADS) {
            const int rp = a.rep_ws[al];
            if (rp >= 0 && rp != al) atomicAnd(reinterpret_cast<unsigned long long *>(&lw[al >> 6]), ~(1ull << (al & 63)));
        }
        __syncthreads();
        tr.mark(15);
    }
    if (warp == 0) {
        int run = 0;
        for (int j0 = 0; j0 < wp; j0 += 32) {
            const int j = j0 + lane;
            const int c = j < wp ? __popcll(lw[j]) : 0;
            int incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += y;
            }
            if (j < wp) base[j] = run + incl - c;
            run += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (lane == 0) *s_int = run;
    }
    __syncthreads();
    const int An = *s_int;
    if (An > a.A_live_max) return An;  // caller reports the broken bound
    for (int j = tid; j < wp; j += EM_THREADS) {
        uint64_t m = lw[j];
        int n = base[j];
        while (m) {
            const int b = __ffsll((long long)m) - 1;
            m &= m - 1;
            lv[n++] = j * 64 + b;
        }
    }
    __syncthreads();
    if (dedup) {  // alleles carried by compact column j (the merge counters live in the scratch that is zero-filled next)
        const int32_t *cnt32 = reinterpret_cast<const int32_t *>(a.dense_ws);
        for (int j = tid; j < An; j += EM_THREADS) a.mult_ws[j] = 1.0 + (double)cnt32[lv[j]];
        __syncthreads();
        sm.mult = a.mult_ws;
    }
    const int wpc = max(2, ((An + 63) / 64 + 1) & ~1);
    // ---- gather every class row to A' bits (dense, in global scratch) ------------------------------------------------
    // bit-compress of a 64-bit word under the fixed mask live[j] (Hacker's Delight 7-4): the six move masks depend
    // only on the mask, so they are computed once per source word and reused for all rows
    for (int j = tid; j < wp; j += EM_THREADS) {
        uint64_t m = lw[j], mk = ~m << 1;
#pragma unroll
        for (int i = 0; i < 6; i++) {
            uint64_t mp = mk ^ (mk << 1);
            mp ^= mp << 2; mp ^= mp << 4; mp ^= mp << 8; mp ^= mp << 16; mp ^= mp << 32;
            const uint64_t mv = mp & m;
            a.mv_ws[(size_t)j * 6 + i] = mv;
            m = (m ^ mv) | (mv >> (1 << i));
            mk &= ~mp;
        }
    }
    uint64_t *dense = a.dense_ws;
    for (int i = tid; i < C * wpc; i += EM_THREADS) dense[i] = 0ull;
    __syncthreads();
    for (int j = lane; j < wp; j += 32) {  // source word (slot-outer: its masks stay in registers)
        const uint64_t m = lw[j];
        if (m == 0ull) continue;
        uint64_t mv[6];
#pragma unroll
        for (int i = 0; i < 6; i++) mv[i] = a.mv_ws[(size_t)j * 6 + i];
        const int o = base[j], n = __popcll(m);
        const int wi = o >> 6, sh = o & 63;
        for (int r = warp; r < C; r += EM_WARPS) {
            uint64_t x = a.bits[(size_t)r * wp + j] & m;
            if (x == 0ull) continue;
#pragma unroll
            for (int i = 0; i < 6; i++) {
                const uint64_t t = x & mv[i];
                x = (x ^ t) | (t >> (1 << i));
            }
            atomicOr(reinterpret_cast<unsigned long long *>(&dense[(size_t)r * wpc + wi]), (unsigned long long)(x << sh));
            if (sh + n > 64)
                atomicOr(reinterpret_cast<unsigned long long *>(&dense[(size_t)r * wpc + wi + 1]),
                         (unsigned long long)(x >> (64 - sh)));
        }
    }
    for (int r = tid; r < C; r += EM_THREADS) sm.cnt[r] = a.cnt_u64 ? (double)a.cnt_u64[r] : a.cnt[r];
    __threadfence();
    __syncthreads();
    sm.dense_g = dense;
    // ---- sparse form: count the non-zero 32-bit words per row and per column ---------------------------------------------
    const int wq = 2 * wpc, nb = (C + 31) / 32;
    const uint32_t *dense32 = reinterpret_cast<const uint32_t *>(dense);
    unsigned char *R = reinterpret_cast<unsigned char *>(sm.slab);
    const size_t R_bytes = a.slab_bytes;
    int32_t *row_off = reinterpret_cast<int32_t *>(R);
    int32_t *col_off = row_off + (C + 1);
    uint32_t *nzbits = reinterpret_cast<uint32_t *>(col_off + (wq + 1));  // [wq][nb] rows with a non-zero word in column c
    uint32_t *nzpre = nzbits + (size_t)wq * nb;                           // [wq][nb] such rows before block w
    const size_t fixed = ((size_t)(C + 1) + (wq + 1) + 2 * (size_t)wq * nb) * 4;
    if (fixed + 64 > R_bytes) {  // not even the index fits: dense slab
        for (int i = tid; i < C * wpc; i += EM_THREADS) sm.slab[i] = __ldcg(&dense[i]);
        __syncthreads();
        return An;
    }
    for (int i = tid; i < wq * nb; i += EM_THREADS) nzbits[i] = 0u;
    __syncthreads();
    for (int r = warp; r < C; r += EM_WARPS) {
        int n = 0;
        for (int c0 = 0; c0 < wq; c0 += 32) {
            const int c = c0 + lane;
            const bool nz = c < wq && __ldcg(&dense32[(size_t)r * wq + c]) != 0u;
            if (nz) atomicOr(&nzbits[(size_t)c * nb + (r >> 5)], 1u << (r & 31));
            n += __popc(__ballot_sync(0xffffffffu, nz));
        }
        if (lane == 0) row_off[r + 1] = n;
    }
    __syncthreads();
    if (warp == 0) {  // exclusive scans (fixed order)
        int run = 0;
        for (int r0 = 0; r0 < C; r0 += 32) {
            const int r = r0 + lane;
            const int c = r < C ? row_off[r + 1] : 0;
            int incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += y;
            }
            if (r < C) row_off[r + 1] = run + incl;
            run += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (lane == 0) row_off[0] = 0;
    }
    for (int c = tid; c < wq; c += EM_THREADS) {
        int n = 0;
        for (int w = 0; w < nb; w++) {
            nzpre[(size_t)c * nb + w] = (uint32_t)n;
            n += __popc(nzbits[(size_t)c * nb + w]);
        }
        col_off[c + 1] = n;
    }
    __syncthreads();
    if (warp == 0) {
        int run = 0;
        for (int c0 = 0; c0 < wq; c0 += 32) {
            const int c = c0 + lane;
            const int v = c < wq ? col_off[c + 1] : 0;
            int incl = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += y;
            }
            if (c < wq) col_off[c + 1] = run + incl;
            run += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (lane == 0) col_off[0] = 0;
    }
    __syncthreads();
    const int nnzw = row_off[C];
    const size_t need = ((fixed + 15) & ~(size_t)15) + (size_t)nnzw * 16 + 32;
    if (need > R_bytes || C > 65535) {  // too dense for the sparse form: dense slab (overwrites the index)
        __syncthreads();
        for (int i = tid; i < C * wpc; i += EM_THREADS) sm.slab[i] = __ldcg(&dense[i]);
        __syncthreads();
        return An;
    }
    uint64_t *r_ent = reinterpret_cast<uint64_t *>(R + ((fixed + 15) & ~(size_t)15));
    uint64_t *c_ent = r_ent + ((nnzw + 1) & ~1);  // both lists 16-byte aligned: entries are read in pairs
    for (int r = warp; r < C; r += EM_WARPS) {
        int pos = row_off[r];
        for (int c0 = 0; c0 < wq; c0 += 32) {
            const int c = c0 + lane;
            const uint32_t word = c < wq ? __ldcg(&dense32[(size_t)r * wq + c]) : 0u;
            const unsigned nzm = __ballot_sync(0xffffffffu, word != 0u);
            if (word != 0u) {
                const int e = pos + __popc(nzm & ((1u << lane) - 1u));
                r_ent[e] = (uint64_t)word | ((uint64_t)((uint32_t)c * 264u) << 32);  // 33 slots per 32 alleles (p_slot)
                const int ce = col_off[c] + (int)nzpre[(size_t)c * nb + (r >> 5)] +
                               __popc(nzbits[(size_t)c * nb + (r >> 5)] & ((1u << (r & 31)) - 1u));
                c_ent[ce] = (uint64_t)word | ((uint64_t)((uint32_t)r * 8u) << 32);
            }
            pos += __popc(nzm);
        }
    }
    __syncthreads();
    sm.row_off = row_off; sm.col_off = col_off;
    sm.r_ent = r_ent; sm.c_ent = c_ent;
    return An;
}

template <int NA, bool COOP>
__global__ void __launch_bounds__(EM_THREADS, 1) em_kernel(const EmArgs *__restrict__ args_arr) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    EmArgs a = COOP ? args_arr[0] : args_arr[blockIdx.x];
    if (a.C_ptr) a.C = min(*a.C_ptr, a.C);
    const int tid = threadIdx.x;
    const int A_orig = a.A;
    __shared__ int s_status;
    __shared__ int s_int;
    if (tid == 0) s_status = HGT_OK;
    Trace tr, tr_all;
    tr.start();
    tr_all = tr;
    tr.count(10);
    Smem sm;
    sm.mbar = reinterpret_cast<uint64_t *>(smem_raw);
    sm.red = reinterpret_cast<double *>(smem_raw + 16);
    sm.lv = nullptr; sm.cnt = nullptr; sm.cm64 = nullptr; sm.c64 = nullptr;
    sm.row_off = nullptr; sm.col_off = nullptr; sm.r_ent = nullptr; sm.c_ent = nullptr; sm.dense_g = nullptr;
    sm.mult = nullptr;
    bool compacted = false;
    if (!COOP && a.compact) {
        // ---- allele-compacted, fully shared-memory-resident problem ---------------------------------------------
        const int wpc_max = max(2, ((a.A_live_max + 63) / 64 + 1) & ~1);
        const size_t Apadc = (size_t)wpc_max * 64, Cpad = (size_t)a.slab_rows;
        unsigned char *q = smem_raw + 16 + 40 * 8;
        sm.c64 = q; q += 4096;
        int32_t *lv = reinterpret_cast<int32_t *>(q); q += Apadc * 4;
        sm.p = reinterpret_cast<double *>(q); q += p_slots(Apadc) * 8;
        sm.w = reinterpret_cast<double *>(q); q += Cpad * 8;
        sm.cnt = reinterpret_cast<double *>(q); q += Cpad * 8;
        sm.cm64 = reinterpret_cast<uint64_t *>(q); q += Cpad * 8;
        sm.slab = reinterpret_cast<uint64_t *>(q); q += a.slab_bytes;
        sm.valid = q;
        for (int al = tid; al < A_orig; al += EM_THREADS) {
            a.prob[al] = 0.0;
            a.in_result[al] = 0;
            a.first_class[al] = FK_NONE;
        }
        // identical columns are merged when there are no allele lengths (lengths differ inside a set) and the sizes fit
        // the merge tables
        const bool dedup = !a.len && a.rep_ws && em_merge_fits(a.wp, a.A_live_max, a.slab_bytes);
        const int An = em_compact_build(a, sm, lv, a.C, &s_int, dedup, tr);
        if (An > a.A_live_max) {
            if (tid == 0) {
                a.iters_status[0] = 0;
                a.iters_status[1] = HGT_ERR_ARG;
                a.iters_status[2] = 0;
            }
            return;
        }
        sm.lv = lv;
        a.A = An;
        a.wp = max(2, ((An + 63) / 64 + 1) & ~1);
        compacted = true;
    } else {
        const int Apad0 = a.wp * 64;
        sm.p = sm.red + 40;
        sm.w = sm.p + p_slots(Apad0);
        sm.slab = reinterpret_cast<uint64_t *>(sm.w + a.slab_rows);  // offset stays a multiple of 16 (slab_rows even)
        sm.valid = reinterpret_cast<uint8_t *>(sm.slab + (size_t)a.slab_rows * a.wp);
    }
    const int Apad = a.wp * 64;
    if (tid == 0) {
        mbar_init(sm.mbar, 1);
        fence_barrier_init();
    }
    __syncthreads();
    int row_lo = 0, row_hi = a.C;
    if (COOP) {
        const int G = gridDim.x;
        const int per = (a.C + G - 1) / G;
        row_lo = min(a.C, (int)blockIdx.x * per);
        row_hi = min(a.C, row_lo + per);
    }
    const bool resident = compacted || (row_hi - row_lo) <= a.slab_rows;
    bool loaded = compacted;
    uint32_t parity = 0;
    uint32_t xseq = 0;  // exchanges done (read-sharded locus); continues from the block's last sequence number
    if (COOP && a.peer) xseq = *reinterpret_cast<const volatile uint32_t *>(a.peer->block[a.peer->rank] + EM_PEER_FLAG_BYTES + 4);
    double *v0 = a.vec, *v1 = a.vec + Apad, *v2 = a.vec + 2 * (size_t)Apad, *v3 = a.vec + 3 * (size_t)Apad;
    uint8_t *l0 = a.live, *l1 = a.live + Apad, *l2 = a.live + 2 * (size_t)Apad;
    // In cooperative mode every CTA computes the same vectors and writes identical values to the shared
    // workspace; reads of those values are ordered by the sweep's grid syncs / __syncthreads.
    tr.mark(5);
    em_sweep<NA, COOP>(a, sm, MODE_INIT, nullptr, nullptr, v0, l0, nullptr, row_lo, row_hi, resident, loaded,
                       parity, &s_status, tr, xseq);
    double diff = 1.0;
    int iter = 0, sweeps = 0;
    const double *last_in = v0;
    const uint8_t *last_live = l0;
    bool have_last = false;
    // bytes from sm.p to the end of the slab buffer can be re-used by the compact mode
    // (the allele-compacted layout has dedicated buffers for it instead, so its slab stays intact)
    const bool compact_ok = !COOP && em_collapse_fits(compacted, a.C, a.wp, a.slab_rows);
    while (a.fixed_iters > 0 ? iter < a.fixed_iters : (diff > 0.0001 && iter < 1000)) {
        if (s_status != HGT_OK) break;
        if (compact_ok && (iter == 0 || (iter > 10 && a.remove_low))) {
            int cnt_live = 0;
            for (int al = tid; al < a.A; al += EM_THREADS)
                if (l0[al]) cnt_live += (sm.mult && sm.mult[al] != 1.0) ? 1000 : 1;  // merged columns stay on the sweeps
            cnt_live = (int)block_sum((double)cnt_live, sm.red);
            if (cnt_live > 0 && cnt_live <= 64) {
                // ---- build the compact problem ---------------------------------------------------------------
                Compact c;
                unsigned char *base = compacted ? sm.c64 : reinterpret_cast<unsigned char *>(sm.p);
                c.v = reinterpret_cast<double *>(base);
                c.len = c.v + 256;
                c.q = c.len + 64;
                c.lv = reinterpret_cast<int *>(c.q + 64);
                c.l = c.lv + 64;
                if (compacted) {
                    c.cnt = sm.cnt;
                    c.w = sm.w;
                    c.cm = sm.cm64;
                } else {
                    c.cnt = reinterpret_cast<double *>(c.l + 192);
                    c.w = c.cnt + a.C;
                    c.cm = reinterpret_cast<uint64_t *>(c.w + a.C);
                }
                c.n = cnt_live;
                __syncthreads();
                if (tid < 32) {  // ordered list of key alleles
                    int n = 0;
                    for (int a0 = 0; a0 < a.A; a0 += 32) {
                        const int al = a0 + tid;
                        const bool k = al < a.A && l0[al];
                        const unsigned m = __ballot_sync(0xffffffffu, k);
                        if (k) c.lv[n + __popc(m & ((1u << tid) - 1u))] = al;
                        n += __popc(m);
                    }
                }
                __syncthreads();
                if (tid < 64) {
                    const bool k = tid < c.n;
                    const int al = k ? c.lv[tid] : 0;
                    c.v[tid] = k ? v0[al] : 0.0;
                    c.v[64 + tid] = c.v[128 + tid] = c.v[192 + tid] = 0.0;
                    c.l[tid] = k ? 1 : 0;
                    c.l[64 + tid] = c.l[128 + tid] = 0;
                    c.len[tid] = (k && a.len) ? a.len[orig_allele(sm, al)] : 1.0;
                }
                // row masks straight from global memory: warp per class row, lane per compact allele
                {
                    const int lane = tid & 31, warp = tid >> 5;
                    const int a_lo = lane < c.n ? c.lv[lane] : -1, a_hi = lane + 32 < c.n ? c.lv[lane + 32] : -1;
                    for (int r = warp; r < a.C; r += EM_WARPS) {
                        const uint64_t *row = (compacted ? sm.dense_g : a.bits) + (size_t)r * a.wp;
                        const bool b_lo = a_lo >= 0 && ((__ldcg(&row[a_lo >> 6]) >> (a_lo & 63)) & 1ull);
                        const bool b_hi = a_hi >= 0 && ((__ldcg(&row[a_hi >> 6]) >> (a_hi & 63)) & 1ull);
                        const unsigned m_lo = __ballot_sync(0xffffffffu, b_lo), m_hi = __ballot_sync(0xffffffffu, b_hi);
                        if (lane == 0) {
                            c.cm[r] = (uint64_t)m_lo | ((uint64_t)m_hi << 32);
                            if (!compacted) c.cnt[r] = a.cnt_u64 ? (double)a.cnt_u64[r] : a.cnt[r];
                        }
                    }
                }
                __syncthreads();
                int last = 0;
                const int iter_before = iter;
                tr.mark(6);
                compact_loop(a, c, diff, iter, sweeps, last, have_last, &s_status);
                tr.mark(7);
                const bool ran = iter > iter_before;  // otherwise the dense last_in / last_live stay valid
                // ---- back to the dense representation for the epilogue ----------------------------------------
                for (int al = tid; al < a.A; al += EM_THREADS) {
                    v0[al] = 0.0; l0[al] = 0;
                    if (ran) { v3[al] = 0.0; l2[al] = 0; }
                }
                __syncthreads();
                if (tid < c.n) {
                    const int al = c.lv[tid];
                    v0[al] = c.v[tid];
                    l0[al] = (uint8_t)c.l[tid];
                    if (ran) {
                        const int slot = last;  // 1 or 3
                        v3[al] = c.v[slot * 64 + tid];
                        l2[al] = (uint8_t)(slot == 3 ? c.l[128 + tid] : c.l[64 + tid]);
                    }
                }
                __syncthreads();
                if (ran) {
                    last_in = v3;
                    last_live = l2;
                }
                if (!compacted) loaded = false;  // the slab buffer was overwritten
                break;
            }
        }
        tr.mark(6);
        em_sweep<NA, COOP>(a, sm, MODE_NEXT, v0, l0, v1, l1, nullptr, row_lo, row_hi, resident, loaded, parity,
                           &s_status, tr, xseq);
        em_sweep<NA, COOP>(a, sm, MODE_NEXT, v1, l1, v2, l2, nullptr, row_lo, row_hi, resident, loaded, parity,
                           &s_status, tr, xseq);
        sweeps += 2;
        // SQUAREM extrapolation (common:1361-1383)
        double ssr = 0.0, ssv = 0.0;
        int keyerr = 0;
        for (int al = tid; al < a.A; al += EM_THREADS) {
            if (l0[al]) {
                if (!l1[al] || !l2[al]) keyerr = 1;
                const double r = v1[al] - v0[al];
                const double v = v2[al] - v1[al] - r;
                if (sm.mult) {  // m equal alleles with r / m each: sum of squares = r^2 / m
                    const double m = sm.mult[al];
                    ssr += r * r / m;
                    ssv += v * v / m;
                } else {
                    ssr += r * r;
                    ssv += v * v;
                }
            }
        }
        ssr = block_sum(ssr, sm.red);
        ssv = block_sum(ssv, sm.red);
        if (block_or(keyerr)) {
            if (tid == 0) s_status = HGT_ERR_KEY;
            __syncthreads();
            break;
        }
        if (ssv > 0.0) {
            // extrapolated vector goes to a 4th buffer: slower CTAs may still be reading v2 (cooperative mode)
            const double g = -sqrt(ssr / ssv);
            for (int al = tid; al < a.A; al += EM_THREADS) {
                double x = 0.0;
                if (l0[al]) {
                    const double r = v1[al] - v0[al];
                    const double v = v2[al] - v1[al] - r;
                    x = v0[al] - 2 * g * r + g * g * v;
                    x = x > 0.0 ? x : 0.0;
                }
                v3[al] = x;
            }
            __syncthreads();
            tr.mark(6);
            em_sweep<NA, COOP>(a, sm, MODE_NEXT, v3, l2, v1, l1, nullptr, row_lo, row_hi, resident, loaded,
                               parity, &s_status, tr, xseq);
            sweeps += 1;
            last_in = v3;
            last_live = l2;
        } else {
            last_in = v0;
            last_live = l0;
        }
        have_last = true;
        // prob_diff (common:1272-1279)
        double d = 0.0;
        for (int al = tid; al < a.A; al += EM_THREADS)
            if (l0[al]) d += l1[al] ? fabs(v0[al] - v1[al]) : v0[al];
        diff = block_sum(d, sm.red);
        // (cooperative mode) v0 becomes the next sweep's target; that sweep only writes after its own grid
        // syncs, which every CTA reaches after the reads above, so no extra sync is needed here
        // Gene_prob = Gene_prob_next
        {
            double *tv = v0; v0 = v1; v1 = tv;
            uint8_t *tl = l0; l0 = l1; l1 = tl;
        }
        if (iter >= 10 && a.remove_low) {
            em_prune(a, sm, v0, l0);
        }
        iter++;
    }
    if (s_status == HGT_OK) {
        if (a.remove_low) em_prune(a, sm, v0, l0);
        // final normalize (common:1404-1407)
        double part = 0.0;
        int nk = 0;
        for (int al = tid; al < a.A; al += EM_THREADS)
            if (l0[al]) {
                part += a.len ? v0[al] / a.len[orig_allele(sm, al)] : v0[al];
                nk = 1;
            }
        const double total = block_sum(part, sm.red);
        if (block_or(nk) && !(total > 0.0) && !(total < 0.0)) {
            if (tid == 0) s_status = HGT_ERR_ZERODIV;
            __syncthreads();
        }
        const bool writer = !COOP || blockIdx.x == 0;
        if (writer) {
            for (int al = tid; al < a.A; al += EM_THREADS) {
                const bool key = l0[al];
                const int ao = orig_allele(sm, al);
                a.prob[ao] = key ? (a.len ? v0[al] / a.len[ao] / total : (sm.mult ? v0[al] / sm.mult[al] / total : v0[al] / total)) : 0.0;
                a.in_result[ao] = key ? 1 : 0;
            }
        }
        // dict insertion order of the final Gene_prob = order in which the last next_prob() call met the
        // alleles (common:1324-1331); needed for the stable sort's tie-break (common:1409)
        if (have_last) {
            em_sweep<NA, COOP>(a, sm, MODE_FIRSTK, last_in, last_live, nullptr, nullptr, a.first_class, row_lo,
                               row_hi, resident, loaded, parity, &s_status, tr, xseq);
        } else if (writer) {
            for (int al = tid; al < A_orig; al += EM_THREADS) a.first_class[al] = FK_NONE;
        }
        if (sm.mult) {  // merged columns: every member gets its representative's result
            __syncthreads();
            for (int al = tid; al < A_orig; al += EM_THREADS) {
                const int rp = a.rep_ws[al];
                if (rp >= 0 && rp != al) {
                    a.prob[al] = a.prob[rp];
                    a.in_result[al] = a.in_result[rp];
                    a.first_class[al] = a.first_class[rp];
                }
            }
        }
    }
    tr.mark(6);
    tr_all.mark(8);
    tr_all.finish();
    if (tid == 0 && (!COOP || blockIdx.x == 0)) {
        a.iters_status[0] = iter;
        a.iters_status[1] = s_status;
        a.iters_status[2] = sweeps;
        if (COOP && a.peer) *reinterpret_cast<uint32_t *>(a.peer->block[a.peer->rank] + EM_PEER_FLAG_BYTES + 4) = xseq;
    }
}

// ---- partial sweeps for a read-sharded locus (SURVEY.md 8e) ---------------------------------------------------------
// The class rows of one locus are spread over several GPUs; one next_prob() is then: every rank runs em_part_kernel +
// em_part_reduce_kernel over ITS rows with the global probability vector, the per-allele sums are all-reduced (NCCL),
// and every rank finishes the step identically (hisat-genotype_b200/em_dist.py).
template <int NA>
__global__ void __launch_bounds__(EM_THREADS, 1) em_part_kernel(EmArgs a, int mode, const double *__restrict__ pin) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x;
    Smem sm;
    sm.mbar = reinterpret_cast<uint64_t *>(smem_raw);
    sm.red = reinterpret_cast<double *>(smem_raw + 16);
    sm.lv = nullptr; sm.cnt = nullptr; sm.cm64 = nullptr; sm.c64 = nullptr;
    sm.row_off = nullptr; sm.col_off = nullptr; sm.r_ent = nullptr; sm.c_ent = nullptr; sm.dense_g = nullptr;
    sm.mult = nullptr;
    const int Apad = a.wp * 64;
    sm.p = sm.red + 40;
    sm.w = sm.p + p_slots(Apad);
    sm.slab = reinterpret_cast<uint64_t *>(sm.w + a.slab_rows);
    sm.valid = reinterpret_cast<uint8_t *>(sm.slab + (size_t)a.slab_rows * a.wp);
    if (tid == 0) {
        mbar_init(sm.mbar, 1);
        fence_barrier_init();
    }
    __syncthreads();
    const int G = gridDim.x, g = blockIdx.x;
    const int per = (a.C + G - 1) / G;
    const int row_lo = min(a.C, g * per), row_hi = min(a.C, row_lo + per);
    bool loaded = false;
    uint32_t parity = 0;
    double acc[NA];
    int32_t fk[NA];
    uint32_t hit = 0;
    Trace tr;
    tr.on = false; tr.t = 0; tr.ns0 = 0;
    em_accumulate<NA>(a, sm, mode, pin, nullptr, row_lo, row_hi, false, loaded, parity, acc, fk, hit, tr);
#pragma unroll
    for (int i = 0; i < NA; i++) {
        const int al = tid + i * EM_THREADS;
        if (al < a.A) {
            a.part_acc[(size_t)g * Apad + al] = acc[i];
            a.part_aux[(size_t)g * Apad + al] = (mode == MODE_FIRSTK) ? fk[i] : (int32_t)((hit >> i) & 1u);
        }
    }
}

__global__ void em_part_reduce_kernel(int G, int A, int Apad, int mode, const double *__restrict__ part_acc,
                                      const int32_t *__restrict__ part_aux, double *__restrict__ acc_out,
                                      int32_t *__restrict__ aux_out, double *__restrict__ hit_out) {
    const int al = blockIdx.x * blockDim.x + threadIdx.x;
    if (al >= A) return;
    double s = 0.0;
    int32_t x = (mode == MODE_FIRSTK) ? FK_NONE : 0;
    for (int g = 0; g < G; g++) {  // fixed order: reproducible
        s += part_acc[(size_t)g * Apad + al];
        const int32_t y = part_aux[(size_t)g * Apad + al];
        x = (mode == MODE_FIRSTK) ? min(x, y) : (x | y);
    }
    if (acc_out) acc_out[al] = s;
    if (aux_out) aux_out[al] = x;
    if (hit_out) hit_out[al] = (double)x;  // modes 0, 1: the flag as a summable number (one all-reduce for both)
}

struct EmPlan {
    int na;
    int slab_rows;
    size_t smem;
};

int em_plan(const hgt_ctx *ctx, int rows_per_cta, int A, int wp, EmPlan *plan) {
    const int Apad = wp * 64;
    if (A > 16 * EM_THREADS) {
        hgt_set_error("EM kernel supports at most %d alleles per problem (got %d)", 16 * EM_THREADS, A);
        return HGT_ERR_UNSUPPORTED;
    }
    int na = 1;
    while (na * EM_THREADS < Apad) na *= 2;
    const size_t fixed = 16 + 40 * 8 + p_slots(Apad) * 8;
    const size_t budget = ctx->smem_optin > 1024 ? ctx->smem_optin - 1024 : 0;
    if (fixed + 2 * ((size_t)wp * 8 + 9) > budget) {
        hgt_set_error("EM kernel: %d alleles do not fit shared memory", A);
        return HGT_ERR_UNSUPPORTED;
    }
    size_t rows = (budget - fixed) / ((size_t)wp * 8 + 9);
    rows &= ~(size_t)1;
    int want = rows_per_cta < 2 ? 2 : ((rows_per_cta + 1) & ~1);
    if ((size_t)want < rows) rows = want;
    plan->na = na;
    plan->slab_rows = (int)rows;
    plan->smem = fixed + rows * ((size_t)wp * 8 + 8) + rows + 16;
    return HGT_OK;
}

template <bool COOP>
int em_launch(hgt_ctx *ctx, cudaStream_t st, const EmArgs *d_args, int grid, int na, size_t smem) {
    void (*kern)(const EmArgs *) = nullptr;
    switch (na) {
        case 1: kern = em_kernel<1, COOP>; break;
        case 2: kern = em_kernel<2, COOP>; break;
        case 4: kern = em_kernel<4, COOP>; break;
        case 8: kern = em_kernel<8, COOP>; break;
        default: kern = em_kernel<16, COOP>; break;
    }
    HGT_CUDA(hgt_smem_at_least((const void *)kern, smem));
    if (COOP) {
        void *params[] = {(void *)&d_args};
        HGT_CUDA(cudaLaunchCooperativeKernel((void *)kern, dim3(grid), dim3(EM_THREADS), params, smem, st));
    } else {
        kern<<<grid, EM_THREADS, smem, st>>>(d_args);
        HGT_CUDA(cudaGetLastError());
    }
    ctx->launches++;
    return HGT_OK;
}

// Plan of one batched problem (one CTA): the allele-compacted shared-memory-resident layout when it fits, else the
// streaming layout of em_plan().
constexpr size_t EM_DENSE_SCRATCH = 232448;
struct EmShape {
    int C, A, wp, A_live_max;
};
int em_plan_batched(const hgt_ctx *ctx, const EmShape &sh, EmArgs *a, int *na, size_t *smem) {
    const size_t budget = ctx->smem_optin > 1024 ? ctx->smem_optin - 1024 : 0;
    int alive = sh.A_live_max < sh.A ? sh.A_live_max : sh.A;
    if (alive < 1) alive = 1;
    const int wpc = hgt_row_pitch(alive);
    const size_t Apadc = (size_t)wpc * 64;
    const size_t Cpad = sh.C < 2 ? 2 : (size_t)((sh.C + 1) & ~1);
    const size_t dense = Cpad * (size_t)wpc * 8;
    const size_t other = 16 + 40 * 8 + 4096 + Apadc * 4 + p_slots(Apadc) * 8 + Cpad * 25 + 16;
    size_t need = other + dense;
    if (sh.wp <= 256 && need <= budget && dense <= EM_DENSE_SCRATCH && Apadc <= (size_t)16 * EM_THREADS) {
        // room for the sparse form (16 B per non-zero 32-bit word + index) up to full density, if the SM has it
        const size_t nb = (Cpad + 31) / 32;
        size_t want = 4 * dense + (Cpad + 1 + 2 * (size_t)wpc + 1 + 4 * (size_t)wpc * nb) * 4 + 64;
        want = (want + 15) & ~(size_t)15;
        size_t slab = dense;
        if (other + want <= budget) slab = want;
        else if (budget - other > dense) slab = (budget - other) & ~(size_t)15;
        need = other + slab;
        a->slab_bytes = (unsigned)slab;
        a->compact = 1;
        a->A_live_max = alive;
        a->slab_rows = (int)Cpad;
        int n = 1;
        while ((size_t)n * EM_THREADS < Apadc) n *= 2;
        *na = n;
        *smem = need;
        return HGT_OK;
    }
    EmPlan plan;
    HGT_CHECK(em_plan(ctx, sh.C < 1 ? 1 : sh.C, sh.A, sh.wp, &plan));
    a->compact = 0;
    a->slab_bytes = 0;
    a->A_live_max = sh.A;
    a->slab_rows = plan.slab_rows;
    *na = plan.na;
    *smem = plan.smem;
    return HGT_OK;
}

// Launches n planned problems (one CTA each): grouped by register variant, heaviest problems first inside a group.
// h_args (host, pinned or otherwise alive until the stream has passed the copy) and d_args hold n EmArgs.
int em_launch_batched(hgt_ctx *ctx, cudaStream_t st, int n, const EmArgs *planned, const int *na, const size_t *smem,
                      EmArgs *h_args, EmArgs *d_args, bool h_pinned) {
    std::vector<int> order(n);
    for (int i = 0; i < n; i++) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) {
        if (planned[x].compact != planned[y].compact) return planned[x].compact < planned[y].compact;
        return (double)planned[x].C * planned[x].A_live_max > (double)planned[y].C * planned[y].A_live_max;
    });
    for (int i = 0; i < n; i++) h_args[i] = planned[order[i]];
    if (h_pinned) HGT_CUDA(hgt_small_h2d(d_args, h_args, (size_t)n * sizeof(EmArgs), st));
    else HGT_CUDA(cudaMemcpyAsync(d_args, h_args, (size_t)n * sizeof(EmArgs), cudaMemcpyHostToDevice, st));
    // one launch: the widest register variant serves every problem (narrower ones just skip slots), so all SMs
    // stay busy instead of running the variants back to back
    int na_max = 1;
    size_t sm = 0;
    for (int i = 0; i < n; i++) {
        if (na[i] > na_max) na_max = na[i];
        if (smem[i] > sm) sm = smem[i];
    }
    HGT_CHECK(em_launch<false>(ctx, st, d_args, n, na_max, sm));
    return HGT_OK;
}

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
// global scratch of one allele-compacted problem: the gathered dense rows (never larger than the shared-memory
// budget they were planned into) + the bit-compress masks
inline size_t em_compact_scratch_bytes(int wp) { return align_up(EM_DENSE_SCRATCH + (size_t)wp * 48 + (size_t)wp * 64 * 12, 256); }
inline void em_set_scratch(EmArgs *a, void *scratch) {  // a->wp must be set
    unsigned char *b = static_cast<unsigned char *>(scratch);
    a->dense_ws = reinterpret_cast<uint64_t *>(b);
    a->mv_ws = reinterpret_cast<uint64_t *>(b + EM_DENSE_SCRATCH);
    a->mult_ws = reinterpret_cast<double *>(b + EM_DENSE_SCRATCH + (size_t)a->wp * 48);
    a->rep_ws = reinterpret_cast<int32_t *>(b + EM_DENSE_SCRATCH + (size_t)a->wp * 48 + (size_t)a->wp * 64 * 8);
}

// workspace carve-up (device pointers) for one problem
struct EmWs {
    EmArgs *d_args;
    double *vec;
    uint8_t *live;
    double *part_acc;
    int32_t *part_aux;
    double *red_acc;
    int32_t *red_aux;
    void *scratch;
};
size_t em_ws_bytes(int sm_count, int A) {
    const size_t Apad = (size_t)hgt_row_pitch(A) * 64;
    size_t b = 512;                                   // args (+ the EmPeer of a read-sharded launch)
    b += align_up(4 * Apad * 8, 256);                 // vec
    b += align_up(4 * Apad, 256);                     // live
    b += align_up((size_t)sm_count * Apad * 8, 256);  // part_acc
    b += align_up((size_t)sm_count * Apad * 4, 256);  // part_aux
    b += align_up(Apad * 8, 256) + align_up(Apad * 4, 256);
    b += em_compact_scratch_bytes(hgt_row_pitch(A));
    return b;
}
EmWs em_ws_carve(void *ws, int sm_count, int A) {
    const size_t Apad = (size_t)hgt_row_pitch(A) * 64;
    unsigned char *p = static_cast<unsigned char *>(ws);
    EmWs w;
    w.d_args = reinterpret_cast<EmArgs *>(p); p += 512;
    w.vec = reinterpret_cast<double *>(p); p += align_up(4 * Apad * 8, 256);
    w.live = p; p += align_up(4 * Apad, 256);
    w.part_acc = reinterpret_cast<double *>(p); p += align_up((size_t)sm_count * Apad * 8, 256);
    w.part_aux = reinterpret_cast<int32_t *>(p); p += align_up((size_t)sm_count * Apad * 4, 256);
    w.red_acc = reinterpret_cast<double *>(p); p += align_up(Apad * 8, 256);
    w.red_aux = reinterpret_cast<int32_t *>(p); p += align_up(Apad * 4, 256);
    w.scratch = p;
    return w;
}

// Grid and plan of hgt_em_dev (hgt_em_form reports the same decisions).  One CTA takes the batched plan: the
// allele-compacted layout when it fits, else one streaming CTA; more CTAs run the cooperative streaming plan.
int em_dev_plan(const hgt_ctx *ctx, int n_classes, int n_alleles, int wp, int n_ctas, int A_live_max, EmArgs *a,
                EmPlan *plan, int *grid) {
    int G = n_ctas;
    if (G <= 0) {
        // one CTA until the matrix stops fitting comfortably in a single SM's shared memory
        const size_t bytes = (size_t)n_classes * wp * 8;
        G = bytes <= 160 * 1024 ? 1 : ctx->sm_count;
    }
    if (G > ctx->sm_count) G = ctx->sm_count;
    if (G > n_classes) G = n_classes;
    if (G < 1) G = 1;
    if (G == 1) {
        const EmShape sh{n_classes, n_alleles, wp, A_live_max};
        int na = 1;
        size_t smem = 0;
        HGT_CHECK(em_plan_batched(ctx, sh, a, &na, &smem));
        plan->na = na; plan->smem = smem; plan->slab_rows = a->slab_rows;
    } else {
        HGT_CHECK(em_plan(ctx, (n_classes + G - 1) / G, n_alleles, wp, plan));
        a->compact = 0; a->A_live_max = n_alleles; a->slab_bytes = 0;
        a->slab_rows = plan->slab_rows;
    }
    *grid = G;
    return HGT_OK;
}

}  // namespace

extern "C" size_t hgt_em_workspace_bytes(const hgt_ctx *ctx, int32_t n_classes, int32_t n_alleles) {
    (void)n_classes;
    return em_ws_bytes(ctx ? ctx->sm_count : 148, n_alleles);
}

extern "C" int hgt_em_dev(hgt_ctx *ctx, void *stream, const uint64_t *class_bits, const double *class_count,
                          int32_t n_classes, int32_t n_alleles, int32_t wp, const double *allele_len,
                          int32_t remove_low, int32_t fixed_iters, int32_t n_ctas, double *prob,
                          uint8_t *in_result, int32_t *first_class, int32_t *iters_status, void *workspace) {
    if (!ctx || !class_bits || !class_count || !prob || !in_result || !first_class || !iters_status || !workspace) {
        hgt_set_error("hgt_em_dev: null argument");
        return HGT_ERR_ARG;
    }
    if (wp != hgt_row_pitch(n_alleles) || n_classes < 1 || n_alleles < 1) {
        hgt_set_error("hgt_em_dev: need n_classes >= 1, n_alleles >= 1 and wp == hgt_row_pitch(n_alleles)");
        return HGT_ERR_ARG;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    EmPlan plan;
    EmWs w = em_ws_carve(workspace, ctx->sm_count, n_alleles);
    EmArgs a;
    a.bits = class_bits; a.cnt = class_count; a.len = allele_len;
    a.C = n_classes; a.A = n_alleles; a.wp = wp; a.remove_low = remove_low; a.fixed_iters = fixed_iters;
    a.cnt_u64 = nullptr; a.C_ptr = nullptr; a.class_first = nullptr; a.key_offset = 0; a.peer = nullptr;
    a.prob = prob; a.in_result = in_result; a.first_class = first_class; a.iters_status = iters_status;
    a.vec = w.vec; a.live = w.live; a.part_acc = w.part_acc; a.part_aux = w.part_aux;
    a.red_acc = w.red_acc; a.red_aux = w.red_aux;
    em_set_scratch(&a, w.scratch);
    int G = 1;
    HGT_CHECK(em_dev_plan(ctx, n_classes, n_alleles, wp, n_ctas, n_alleles, &a, &plan, &G));
    HGT_CUDA(cudaMemcpyAsync(w.d_args, &a, sizeof(a), cudaMemcpyHostToDevice, st));
    if (G == 1) return em_launch<false>(ctx, st, w.d_args, 1, plan.na, plan.smem);
    return em_launch<true>(ctx, st, w.d_args, G, plan.na, plan.smem);
}

// ---- read-sharded locus across GPUs: the whole loop as ONE cooperative launch per rank (EmPeer) ----------------------------
extern "C" size_t hgt_em_peer_block_bytes(int32_t n_alleles) {
    const size_t Apad = (size_t)hgt_row_pitch(n_alleles < 1 ? 1 : n_alleles) * 64;
    return EM_PEER_HDR + 2 * Apad * 8;
}
extern "C" int hgt_em_peer_alloc(hgt_ctx *ctx, int32_t n_alleles, void **block, unsigned char handle[64]) {
    if (!ctx || !block || !handle || n_alleles < 1) {
        hgt_set_error("hgt_em_peer_alloc: bad argument");
        return HGT_ERR_ARG;
    }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    HGT_CUDA(cudaSetDevice(ctx->device));
    void *p = nullptr;
    const size_t n = hgt_em_peer_block_bytes(n_alleles);
    HGT_CUDA(cudaMalloc(&p, n));  // (own allocation, not the pool: an IPC handle names a whole cudaMalloc block)
    HGT_CUDA(cudaMemset(p, 0, n));
    HGT_CUDA(cudaDeviceSynchronize());
    cudaIpcMemHandle_t h;
    HGT_CUDA(cudaIpcGetMemHandle(&h, p));
    memcpy(handle, &h, 64);
    *block = p;
    return HGT_OK;
}
extern "C" int hgt_em_peer_open(hgt_ctx *ctx, const unsigned char handle[64], void **block) {
    if (!ctx || !block || !handle) {
        hgt_set_error("hgt_em_peer_open: bad argument");
        return HGT_ERR_ARG;
    }
    HGT_CUDA(cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    HGT_CUDA(cudaIpcOpenMemHandle(block, h, cudaIpcMemLazyEnablePeerAccess));
    return HGT_OK;
}
extern "C" int hgt_em_peer_close(hgt_ctx *ctx, void *block) {
    if (!ctx || !block) return HGT_ERR_ARG;
    HGT_CUDA(cudaSetDevice(ctx->device));
    HGT_CUDA(cudaIpcCloseMemHandle(block));
    return HGT_OK;
}
extern "C" int hgt_em_peer_free(hgt_ctx *ctx, void *block) {
    if (!ctx || !block) return HGT_ERR_ARG;
    HGT_CUDA(cudaSetDevice(ctx->device));
    HGT_CUDA(cudaFree(block));
    return HGT_OK;
}

extern "C" int hgt_em_peer_dev(hgt_ctx *ctx, void *stream, const uint64_t *class_bits, const double *class_count_f64,
                               const uint64_t *class_count_u64, const int32_t *class_key, int32_t key_offset,
                               int32_t n_classes, int32_t n_alleles, int32_t wp, const double *allele_len, int32_t remove_low,
                               int32_t rank, int32_t world, void *const *blocks, double *prob, uint8_t *in_result,
                               int32_t *first_class, int32_t *iters_status, void *workspace) {
    if (!ctx || !blocks || !prob || !in_result || !first_class || !iters_status || !workspace || world < 1 ||
        world > EM_PEER_MAX || rank < 0 || rank >= world || n_classes < 0 ||
        (n_classes > 0 && (!class_bits || (!class_count_f64 && !class_count_u64)))) {
        hgt_set_error("hgt_em_peer_dev: bad argument (at most %d ranks)", EM_PEER_MAX);
        return HGT_ERR_ARG;
    }
    if (wp != hgt_row_pitch(n_alleles) || n_alleles < 1) {
        hgt_set_error("hgt_em_peer_dev: need n_alleles >= 1 and wp == hgt_row_pitch(n_alleles)");
        return HGT_ERR_ARG;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int G = ctx->sm_count;  // all SMs even for a handful of rows; the SAME grid on every rank (slices pair up by CTA)
    if (G > EM_PEER_G) {
        hgt_set_error("hgt_em_peer_dev: more than %d SMs", EM_PEER_G);
        return HGT_ERR_UNSUPPORTED;
    }
    EmPlan plan;
    HGT_CHECK(em_plan(ctx, std::max(1, (n_classes + G - 1) / G), n_alleles, wp, &plan));
    EmWs w = em_ws_carve(workspace, ctx->sm_count, n_alleles);
    EmArgs a;
    memset(&a, 0, sizeof(a));
    a.bits = class_bits; a.cnt = class_count_f64; a.len = allele_len;
    a.cnt_u64 = reinterpret_cast<const unsigned long long *>(class_count_u64);
    a.class_first = class_key; a.key_offset = key_offset;
    a.C = n_classes; a.A = n_alleles; a.wp = wp; a.remove_low = remove_low; a.fixed_iters = 0;
    a.prob = prob; a.in_result = in_result; a.first_class = first_class; a.iters_status = iters_status;
    a.vec = w.vec; a.live = w.live; a.part_acc = w.part_acc; a.part_aux = w.part_aux;
    a.red_acc = w.red_acc; a.red_aux = w.red_aux;
    em_set_scratch(&a, w.scratch);
    a.compact = 0; a.A_live_max = n_alleles; a.slab_bytes = 0; a.slab_rows = plan.slab_rows;
    // EmArgs at d_args, EmPeer right behind it (the 256-byte args slot of the workspace holds both)
    static_assert(sizeof(EmArgs) + sizeof(EmPeer) <= 512, "args slot");
    EmPeer px;
    memset(&px, 0, sizeof(px));
    px.rank = rank; px.world = world;
    for (int r = 0; r < world; r++) {
        if (!blocks[r]) {
            hgt_set_error("hgt_em_peer_dev: exchange block of rank %d is null", r);
            return HGT_ERR_ARG;
        }
        px.block[r] = static_cast<unsigned char *>(blocks[r]);
    }
    EmPeer *d_px = reinterpret_cast<EmPeer *>(reinterpret_cast<unsigned char *>(w.d_args) + 256);
    a.peer = d_px;
    HGT_CUDA(cudaMemcpyAsync(d_px, &px, sizeof(px), cudaMemcpyHostToDevice, st));
    HGT_CUDA(cudaMemcpyAsync(w.d_args, &a, sizeof(a), cudaMemcpyHostToDevice, st));
    return em_launch<true>(ctx, st, w.d_args, G, plan.na, plan.smem);
}

extern "C" int hgt_em(hgt_ctx *ctx, const uint64_t *class_bits, const int64_t *class_count, int32_t n_classes,
                      int32_t n_alleles, int32_t wp, const double *allele_len, int32_t remove_low, double *prob,
                      uint8_t *in_result, int32_t *first_class, int32_t *iters) {
    if (n_classes > 0 && !class_count) {
        hgt_set_error("hgt_em: null class_count");
        return HGT_ERR_ARG;
    }
    std::vector<double> cnt((size_t)std::max(n_classes, 0));
    for (int i = 0; i < n_classes; i++) cnt[i] = (double)class_count[i];
    return hgt_em_f64(ctx, class_bits, cnt.data(), n_classes, n_alleles, wp, allele_len, remove_low, prob, in_result, first_class,
                      iters);
}

extern "C" int hgt_em_f64(hgt_ctx *ctx, const uint64_t *class_bits, const double *class_count, int32_t n_classes,
                          int32_t n_alleles, int32_t wp, const double *allele_len, int32_t remove_low, double *prob,
                          uint8_t *in_result, int32_t *first_class, int32_t *iters) {
    if (!ctx) {
        hgt_set_error("hgt_em: null context");
        return HGT_ERR_ARG;
    }
    HGT_CUDA(cudaSetDevice(ctx->device));
    if (n_classes == 0) {  // empty Gene_cmpt: the reference loop runs once on empty dicts and returns []
        for (int i = 0; i < n_alleles; i++) { prob[i] = 0.0; in_result[i] = 0; first_class[i] = FK_NONE; }
        if (iters) *iters = 1;
        return HGT_OK;
    }
    cudaStream_t st = ctx->stream;
    const size_t nb = (size_t)n_classes * wp * 8;
    const size_t wsb = em_ws_bytes(ctx->sm_count, n_alleles);
    unsigned char *d = nullptr;
    const size_t o_bits = 0, o_cnt = align_up(nb, 256), o_len = o_cnt + align_up((size_t)n_classes * 8, 256),
                 o_prob = o_len + align_up((size_t)n_alleles * 8, 256),
                 o_in = o_prob + align_up((size_t)n_alleles * 8, 256), o_fk = o_in + align_up(n_alleles, 256),
                 o_is = o_fk + align_up((size_t)n_alleles * 4, 256), o_ws = o_is + 256, total = o_ws + wsb;
    HGT_CUDA(cudaMalloc(&d, total));
    const double *cnt_h = class_count;
    int rc = HGT_OK;
    int32_t is[3] = {0, 0, 0};
    do {
#define TRY(call)                                                                                 \
    {                                                                                             \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess) {                                                                  \
            hgt_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            rc = HGT_ERR_CUDA;                                                                    \
            break;                                                                                \
        }                                                                                         \
    }
        TRY(cudaMemcpyAsync(d + o_bits, class_bits, nb, cudaMemcpyHostToDevice, st));
        TRY(cudaMemcpyAsync(d + o_cnt, cnt_h, (size_t)n_classes * 8, cudaMemcpyHostToDevice, st));
        if (allele_len) TRY(cudaMemcpyAsync(d + o_len, allele_len, (size_t)n_alleles * 8, cudaMemcpyHostToDevice, st));
        rc = hgt_em_dev(ctx, st, reinterpret_cast<uint64_t *>(d + o_bits), reinterpret_cast<double *>(d + o_cnt),
                        n_classes, n_alleles, wp, allele_len ? reinterpret_cast<double *>(d + o_len) : nullptr,
                        remove_low, 0, 0, reinterpret_cast<double *>(d + o_prob), d + o_in,
                        reinterpret_cast<int32_t *>(d + o_fk), reinterpret_cast<int32_t *>(d + o_is), d + o_ws);
        if (rc != HGT_OK) break;
        TRY(cudaMemcpyAsync(prob, d + o_prob, (size_t)n_alleles * 8, cudaMemcpyDeviceToHost, st));
        TRY(cudaMemcpyAsync(in_result, d + o_in, (size_t)n_alleles, cudaMemcpyDeviceToHost, st));
        TRY(cudaMemcpyAsync(first_class, d + o_fk, (size_t)n_alleles * 4, cudaMemcpyDeviceToHost, st));
        TRY(cudaMemcpyAsync(is, d + o_is, sizeof(is), cudaMemcpyDeviceToHost, st));
        TRY(cudaStreamSynchronize(st));
#undef TRY
    } while (0);
    cudaFree(d);
    if (rc != HGT_OK) return rc;
    if (iters) *iters = is[0];
    if (is[1] == HGT_ERR_KEY) hgt_set_error("KeyError: allele vanished from next_prob output during SQUAREM step");
    if (is[1] == HGT_ERR_ZERODIV) hgt_set_error("ZeroDivisionError: float division by zero in normalize");
    return is[1];
}

extern "C" int hgt_em_batch(hgt_ctx *ctx, int32_t n_problems, const uint64_t *class_bits, const int64_t *class_count,
                            const int64_t *class_off, const int64_t *allele_off, int32_t wp, const double *allele_len,
                            const uint8_t *remove_low, double *prob, uint8_t *in_result, int32_t *first_class,
                            int32_t *iters, int32_t *status) {
    if (!ctx || n_problems < 0 || !class_off || !allele_off) {
        hgt_set_error("hgt_em_batch: bad argument");
        return HGT_ERR_ARG;
    }
    if (n_problems == 0) return HGT_OK;
    HGT_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int64_t Ctot = class_off[n_problems], Atot = allele_off[n_problems];
    const size_t Apad = (size_t)wp * 64;
    std::vector<EmArgs> args(n_problems);
    std::vector<double> cnt((size_t)Ctot);
    for (int64_t i = 0; i < Ctot; i++) cnt[i] = (double)class_count[i];
    // device arena
    const size_t o_bits = 0, o_cnt = align_up((size_t)Ctot * wp * 8, 256), o_len = o_cnt + align_up((size_t)Ctot * 8, 256),
                 o_prob = o_len + align_up((size_t)Atot * 8, 256), o_in = o_prob + align_up((size_t)Atot * 8, 256),
                 o_fk = o_in + align_up((size_t)Atot, 256), o_is = o_fk + align_up((size_t)Atot * 4, 256),
                 o_args = o_is + align_up((size_t)n_problems * 12, 256),
                 o_vec = o_args + align_up((size_t)n_problems * sizeof(EmArgs), 256),
                 o_live = o_vec + (size_t)n_problems * 4 * Apad * 8,
                 o_scr = align_up(o_live + (size_t)n_problems * 4 * Apad, 256),
                 total = o_scr + (size_t)n_problems * em_compact_scratch_bytes(wp);
    unsigned char *d = nullptr;
    HGT_CUDA(cudaMalloc(&d, total));
    int rc = HGT_OK;
    std::vector<int> nas(n_problems, 1);
    std::vector<size_t> smems(n_problems, 0);
    std::vector<EmArgs> h_args(n_problems);
    std::vector<int32_t> is((size_t)n_problems * 3, 0);
    for (int i = 0; i < n_problems && rc == HGT_OK; i++) {
        const int C = (int)(class_off[i + 1] - class_off[i]), A = (int)(allele_off[i + 1] - allele_off[i]);
        if (A < 1 || hgt_row_pitch(A) > wp) {
            hgt_set_error("hgt_em_batch: problem %d has %d alleles, pitch %d too small", i, A, wp);
            rc = HGT_ERR_ARG;
            break;
        }
        EmArgs &a = args[i];
        const EmShape sh{C, A, wp, A};
        rc = em_plan_batched(ctx, sh, &a, &nas[i], &smems[i]);
        if (rc != HGT_OK) break;
        a.bits = reinterpret_cast<uint64_t *>(d + o_bits) + (size_t)class_off[i] * wp;
        a.cnt = reinterpret_cast<double *>(d + o_cnt) + class_off[i];
        a.len = allele_len ? reinterpret_cast<double *>(d + o_len) + allele_off[i] : nullptr;
        a.C = C; a.A = A; a.wp = wp; a.remove_low = remove_low ? remove_low[i] : 0; a.fixed_iters = 0;
        a.cnt_u64 = nullptr; a.C_ptr = nullptr; a.class_first = nullptr; a.key_offset = 0; a.peer = nullptr;
        a.prob = reinterpret_cast<double *>(d + o_prob) + allele_off[i];
        a.in_result = d + o_in + allele_off[i];
        a.first_class = reinterpret_cast<int32_t *>(d + o_fk) + allele_off[i];
        a.iters_status = reinterpret_cast<int32_t *>(d + o_is) + (size_t)i * 3;
        a.vec = reinterpret_cast<double *>(d + o_vec) + (size_t)i * 4 * Apad;
        a.live = d + o_live + (size_t)i * 4 * Apad;
        em_set_scratch(&a, d + o_scr + (size_t)i * em_compact_scratch_bytes(wp));
        a.part_acc = nullptr; a.part_aux = nullptr; a.red_acc = nullptr; a.red_aux = nullptr;
    }
    do {
        if (rc != HGT_OK) break;
#define TRY(call)                                                                                 \
    {                                                                                             \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess) {                                                                  \
            hgt_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            rc = HGT_ERR_CUDA;                                                                    \
            break;                                                                                \
        }                                                                                         \
    }
        TRY(cudaMemcpyAsync(d + o_bits, class_bits, (size_t)Ctot * wp * 8, cudaMemcpyHostToDevice, st));
        TRY(cudaMemcpyAsync(d + o_cnt, cnt.data(), (size_t)Ctot * 8, cudaMemcpyHostToDevice, st));
        if (allele_len) TRY(cudaMemcpyAsync(d + o_len, allele_len, (size_t)Atot * 8, cudaMemcpyHostToDevice, st));
        TRY(cudaMemsetAsync(d + o_is, 0, (size_t)n_problems * 12, st));
        rc = em_launch_batched(ctx, st, n_problems, args.data(), nas.data(), smems.data(), h_args.data(),
                               reinterpret_cast<EmArgs *>(d + o_args), false);
        if (rc != HGT_OK) break;
        TRY(cudaMemcpyAsync(prob, d + o_prob, (size_t)Atot * 8, cudaMemcpyDeviceToHost, st));
        TRY(cudaMemcpyAsync(in_result, d + o_in, (size_t)Atot, cudaMemcpyDeviceToHost, st));
        TRY(cudaMemcpyAsync(first_class, d + o_fk, (size_t)Atot * 4, cudaMemcpyDeviceToHost, st));
        TRY(cudaMemcpyAsync(is.data(), d + o_is, (size_t)n_problems * 12, cudaMemcpyDeviceToHost, st));
        TRY(cudaStreamSynchronize(st));
#undef TRY
    } while (0);
    cudaFree(d);
    if (rc != HGT_OK) return rc;
    for (int i = 0; i < n_problems; i++) {
        if (iters) iters[i] = is[(size_t)i * 3];
        if (status) status[i] = is[(size_t)i * 3 + 1];
    }
    return HGT_OK;
}

extern "C" size_t hgt_em_partial_workspace_bytes(const hgt_ctx *ctx, int32_t n_alleles) {
    const size_t Apad = (size_t)hgt_row_pitch(n_alleles) * 64;
    const int G = ctx ? ctx->sm_count : 148;
    return align_up((size_t)G * Apad * 8, 256) + align_up((size_t)G * Apad * 4, 256);
}

static int em_partial_impl(hgt_ctx *ctx, void *stream, const uint64_t *class_bits, const double *class_count_f64,
                           const uint64_t *class_count_u64, const int32_t *class_key, int32_t key_offset,
                           int32_t n_classes, int32_t n_alleles, int32_t wp, const double *p_in, int32_t mode,
                           double *acc_out, int32_t *aux_out, double *hit_out, void *workspace);

extern "C" int hgt_em_partial_dev(hgt_ctx *ctx, void *stream, const uint64_t *class_bits, const double *class_count_f64,
                                  const uint64_t *class_count_u64, const int32_t *class_key, int32_t key_offset,
                                  int32_t n_classes, int32_t n_alleles, int32_t wp, const double *p_in, int32_t mode,
                                  double *acc_out, int32_t *aux_out, void *workspace) {
    return em_partial_impl(ctx, stream, class_bits, class_count_f64, class_count_u64, class_key, key_offset, n_classes,
                           n_alleles, wp, p_in, mode, acc_out, aux_out, nullptr, workspace);
}

static int em_partial_impl(hgt_ctx *ctx, void *stream, const uint64_t *class_bits, const double *class_count_f64,
                           const uint64_t *class_count_u64, const int32_t *class_key, int32_t key_offset,
                           int32_t n_classes, int32_t n_alleles, int32_t wp, const double *p_in, int32_t mode,
                           double *acc_out, int32_t *aux_out, double *hit_out, void *workspace) {
    if (!ctx || (!acc_out && !aux_out) || !workspace || (!class_count_f64 && !class_count_u64 && n_classes > 0) ||
        (mode != MODE_INIT && !p_in) || mode < 0 || mode > 2 || (n_classes > 0 && !class_bits)) {
        hgt_set_error("hgt_em_partial_dev: bad argument");
        return HGT_ERR_ARG;
    }
    if (wp != hgt_row_pitch(n_alleles) || n_alleles < 1 || n_classes < 0) {
        hgt_set_error("hgt_em_partial_dev: need n_alleles >= 1 and wp == hgt_row_pitch(n_alleles)");
        return HGT_ERR_ARG;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t Apad = (size_t)wp * 64;
    int G = ctx->sm_count;
    if (G > n_classes) G = n_classes < 1 ? 1 : n_classes;
    EmPlan plan;
    HGT_CHECK(em_plan(ctx, (n_classes + G - 1) / G, n_alleles, wp, &plan));
    EmArgs a;
    memset(&a, 0, sizeof(a));
    a.bits = class_bits; a.cnt = class_count_f64; a.cnt_u64 = reinterpret_cast<const unsigned long long *>(class_count_u64);
    a.class_first = class_key; a.key_offset = key_offset;
    a.C = n_classes; a.A = n_alleles; a.wp = wp; a.slab_rows = plan.slab_rows;
    unsigned char *w = static_cast<unsigned char *>(workspace);
    a.part_acc = reinterpret_cast<double *>(w);
    a.part_aux = reinterpret_cast<int32_t *>(w + align_up((size_t)ctx->sm_count * Apad * 8, 256));
    void (*kern)(EmArgs, int, const double *) = nullptr;
    switch (plan.na) {
        case 1: kern = em_part_kernel<1>; break;
        case 2: kern = em_part_kernel<2>; break;
        case 4: kern = em_part_kernel<4>; break;
        case 8: kern = em_part_kernel<8>; break;
        default: kern = em_part_kernel<16>; break;
    }
    HGT_CUDA(hgt_smem_at_least((const void *)kern, plan.smem));
    kern<<<G, EM_THREADS, plan.smem, st>>>(a, mode, p_in);
    HGT_CUDA(cudaGetLastError());
    em_part_reduce_kernel<<<(n_alleles + 255) / 256, 256, 0, st>>>(G, n_alleles, (int)Apad, mode, a.part_acc, a.part_aux,
                                                                   acc_out, aux_out, hit_out);
    HGT_CUDA(cudaGetLastError());
    ctx->launches += 2;
    return HGT_OK;
}


// ---- read-sharded locus: the O(A) vector half of the loop on the device ---------------------------------------------
// State block (device, caller-allocated, hgt_em_shard_state_bytes): doubles vec[6][A] (0 p0, 1 p1, 2 p2, 3 p3, 4 p1', 5
// last input), red[2A] (all-reduce buffer: sums | hit counts), scal[8] (0 sum r^2, 1 sum v^2, 2 key error, 3 division by
// zero, 4 diff, 5 third sweep used, 6 keys left, 7 -), then int32 fk[A], then bytes live[5][A] (0 l0, 1 l1, 2 l2, 3 l1', 4
// last).  Every vector op is ONE single-CTA kernel (A <= 16 k), so an iteration of the reference loop (common:1351-1400)
// is 3 x (sweep, all-reduce, finish) + squarem + advance and ONE host read of scal.
struct ShardState {
    double *vec, *red, *scal;
    int32_t *fk;
    uint8_t *live;
};
__host__ __device__ inline ShardState shard_state(void *base, int A) {
    ShardState s;
    unsigned char *b = static_cast<unsigned char *>(base);
    s.vec = reinterpret_cast<double *>(b);
    s.red = s.vec + 6 * (size_t)A;
    s.scal = s.red + 2 * (size_t)A;
    s.fk = reinterpret_cast<int32_t *>(s.scal + 8);
    s.live = reinterpret_cast<uint8_t *>(s.fk + (((size_t)A + 1) & ~(size_t)1));
    return s;
}
enum { SHARD_FINISH = 0, SHARD_SQUAREM = 1, SHARD_ADVANCE = 2, SHARD_FINAL = 3 };

__device__ void shard_prune(int A, double *p, uint8_t *live, double *red) {  // select_alleles (common:1338-1346)
    double mx = -1.0;
    for (int al = threadIdx.x; al < A; al += EM_THREADS)
        if (live[al]) mx = fmax(mx, p[al]);
    mx = block_max(mx, red);
    if (mx < 0.0) return;
    const double thr = mx / 10.0;
    for (int al = threadIdx.x; al < A; al += EM_THREADS)
        if (live[al] && !(p[al] >= thr)) {
            live[al] = 0;
            p[al] = 0.0;
        }
    __syncthreads();
}

__global__ void __launch_bounds__(EM_THREADS, 1)
    em_shard_vec_kernel(int op, int A, void *state, const double *__restrict__ len, int src, int dst, int it, int remove_low) {
    __shared__ double red[40];
    const ShardState s = shard_state(state, A);
    const int tid = threadIdx.x;
    if (op == SHARD_FINISH) {
        // normalize (common:1285-1297) of q = p * sums over keys = live & hit; src < 0: initial mass (q = sums, keys = hit)
        const double *pin = src >= 0 ? s.vec + (size_t)(src == 3 ? 3 : src) * A : nullptr;
        const uint8_t *lin = src < 0 ? nullptr : s.live + (size_t)(src == 3 ? 2 : src) * A;  // p3 is masked by l2
        double *pout = s.vec + (size_t)dst * A;
        uint8_t *lout = s.live + (size_t)(dst == 4 ? 3 : dst) * A;
        double part = 0.0;
        int any = 0;
        for (int al = tid; al < A; al += EM_THREADS) {
            const bool key = s.red[A + al] > 0.0 && (!lin || lin[al]);
            double q = 0.0;
            if (key) {
                q = pin ? pin[al] * s.red[al] : s.red[al];
                if (len) q = q / len[al];
                any = 1;
            }
            pout[al] = q;
            lout[al] = key ? 1 : 0;
            part += q;
        }
        const double total = block_sum(part, red);
        any = block_or(any);
        if (any && !(total > 0.0) && !(total < 0.0) && tid == 0) s.scal[3] = 1.0;
        for (int al = tid; al < A; al += EM_THREADS) pout[al] = lout[al] ? pout[al] / total : 0.0;
    } else if (op == SHARD_SQUAREM) {
        // common:1361-1383
        const double *p0 = s.vec, *p1 = s.vec + A, *p2 = s.vec + 2 * (size_t)A;
        double *p3 = s.vec + 3 * (size_t)A;
        const uint8_t *l0 = s.live, *l1 = s.live + A, *l2 = s.live + 2 * (size_t)A;
        double ssr = 0.0, ssv = 0.0;
        int keyerr = 0;
        for (int al = tid; al < A; al += EM_THREADS)
            if (l0[al]) {
                if (!l1[al] || !l2[al]) keyerr = 1;
                const double r = p1[al] - p0[al], v = p2[al] - p1[al] - r;
                ssr += r * r;
                ssv += v * v;
            }
        ssr = block_sum(ssr, red);
        ssv = block_sum(ssv, red);
        keyerr = block_or(keyerr);
        const double g = ssv > 0.0 ? -sqrt(ssr / ssv) : 0.0;
        for (int al = tid; al < A; al += EM_THREADS) {
            double x = 0.0;
            if (l0[al] && l2[al] && ssv > 0.0) {
                const double r = p1[al] - p0[al], v = p2[al] - p1[al] - r;
                x = p0[al] - 2 * g * r + g * g * v;
                x = x > 0.0 ? x : 0.0;
            }
            p3[al] = x;
        }
        if (tid == 0) {
            s.scal[0] = ssr; s.scal[1] = ssv;
            if (keyerr) s.scal[2] = 1.0;
            s.scal[5] = ssv > 0.0 ? 1.0 : 0.0;
        }
    } else if (op == SHARD_ADVANCE) {
        // prob_diff (common:1272-1279), Gene_prob = Gene_prob_next, select_alleles from iteration 10 on
        const bool use3 = s.scal[5] != 0.0;
        double *p0 = s.vec, *lastp = s.vec + 5 * (size_t)A;
        const double *pn = s.vec + (size_t)(use3 ? 4 : 1) * A, *p3 = s.vec + 3 * (size_t)A;
        uint8_t *l0 = s.live, *lastl = s.live + 4 * (size_t)A;
        const uint8_t *ln = s.live + (size_t)(use3 ? 3 : 1) * A, *l2 = s.live + 2 * (size_t)A;
        double d = 0.0;
        for (int al = tid; al < A; al += EM_THREADS) {
            const double a0 = p0[al], an = pn[al];
            const uint8_t k0 = l0[al], kn = ln[al];
            if (k0) d += kn ? fabs(a0 - an) : a0;
            lastp[al] = use3 ? (l2[al] ? p3[al] : 0.0) : (k0 ? a0 : 0.0);
            lastl[al] = use3 ? l2[al] : k0;
            p0[al] = an;
            l0[al] = kn;
        }
        d = block_sum(d, red);
        if (it >= 10 && remove_low) shard_prune(A, p0, l0, red);
        if (tid == 0) s.scal[4] = d;
    } else {  // SHARD_FINAL: last select_alleles + normalize (common:1402-1407); prob -> vec[1], keys stay in live[0]
        double *p0 = s.vec, *prob = s.vec + A;
        uint8_t *l0 = s.live;
        if (remove_low) shard_prune(A, p0, l0, red);
        double part = 0.0;
        int any = 0;
        for (int al = tid; al < A; al += EM_THREADS)
            if (l0[al]) {
                part += len ? p0[al] / len[al] : p0[al];
                any = 1;
            }
        const double total = block_sum(part, red);
        any = block_or(any);
        if (any && !(total > 0.0) && !(total < 0.0) && tid == 0) s.scal[3] = 1.0;
        for (int al = tid; al < A; al += EM_THREADS)
            prob[al] = l0[al] ? (len ? p0[al] / len[al] / total : p0[al] / total) : 0.0;
        if (tid == 0) s.scal[6] = any ? 1.0 : 0.0;
    }
}

extern "C" size_t hgt_em_shard_state_bytes(int32_t n_alleles) {
    const size_t A = (size_t)(n_alleles < 1 ? 1 : n_alleles);
    return align_up((8 * A + 8) * 8 + ((A + 1) & ~(size_t)1) * 4 + 5 * A, 256);
}

extern "C" int hgt_em_shard_sweep_dev(hgt_ctx *ctx, void *stream, const uint64_t *class_bits, const double *class_count_f64,
                                      const uint64_t *class_count_u64, const int32_t *class_key, int32_t key_offset,
                                      int32_t n_classes, int32_t n_alleles, int32_t wp, int32_t mode, int32_t src,
                                      void *state, void *workspace) {
    if (!state || src > 5) {
        hgt_set_error("hgt_em_shard_sweep_dev: bad argument");
        return HGT_ERR_ARG;
    }
    const ShardState s = shard_state(state, n_alleles);
    const double *pin = (mode == MODE_INIT || src < 0) ? nullptr : s.vec + (size_t)src * n_alleles;
    if (mode == MODE_FIRSTK)
        return em_partial_impl(ctx, stream, class_bits, class_count_f64, class_count_u64, class_key, key_offset, n_classes,
                               n_alleles, wp, pin, mode, nullptr, s.fk, nullptr, workspace);
    return em_partial_impl(ctx, stream, class_bits, class_count_f64, class_count_u64, class_key, key_offset, n_classes,
                           n_alleles, wp, pin, mode, s.red, nullptr, s.red + n_alleles, workspace);
}

extern "C" int hgt_em_shard_vec_dev(hgt_ctx *ctx, void *stream, int32_t op, int32_t n_alleles, void *state,
                                    const double *allele_len, int32_t src, int32_t dst, int32_t iteration,
                                    int32_t remove_low) {
    if (!ctx || !state || op < SHARD_FINISH || op > SHARD_FINAL || n_alleles < 1 || n_alleles > 16 * EM_THREADS ||
        (op == SHARD_FINISH && (src > 3 || dst < 0 || dst > 4 || dst == 3))) {
        hgt_set_error("hgt_em_shard_vec_dev: bad argument");
        return HGT_ERR_ARG;
    }
    em_shard_vec_kernel<<<1, EM_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(op, n_alleles, state, allele_len, src, dst,
                                                                                 iteration, remove_low);
    HGT_CUDA(cudaGetLastError());
    ctx->launches++;
    return HGT_OK;
}

// ---- internal: batched EM on device-resident class tables (used by typing.cu) ----------------------------------
#include "em_internal.h"

size_t hgt_em_problem_ws_bytes(int wp) {
    const size_t Apad = (size_t)wp * 64;
    return align_up(4 * Apad * 8 + 4 * Apad, 256) + em_compact_scratch_bytes(wp);
}
extern "C" int hgt_em_trace(hgt_ctx *ctx, int32_t enable, uint64_t *cycles16) {
    if (!ctx) return HGT_ERR_ARG;
    HGT_CUDA(cudaSetDevice(ctx->device));
    HGT_CUDA(cudaDeviceSynchronize());
    unsigned long long z[16];
    if (cycles16) {
        HGT_CUDA(cudaMemcpyFromSymbol(z, g_em_trace, sizeof(z)));
        for (int i = 0; i < 16; i++) cycles16[i] = z[i];
    }
    memset(z, 0, sizeof(z));
    HGT_CUDA(cudaMemcpyToSymbol(g_em_trace, z, sizeof(z)));
    const int on = enable ? 1 : 0;
    HGT_CUDA(cudaMemcpyToSymbol(g_em_trace_on, &on, sizeof(on)));
    return HGT_OK;
}

size_t hgt_em_args_bytes(int n_problems) { return align_up((size_t)n_problems * sizeof(EmArgs), 256); }

bool hgt_em_wants_coop(const hgt_ctx *ctx, int C, int A, int wp, int A_live_max, int n_problems) {
    EmArgs a;
    int na = 1;
    size_t smem = 0;
    const EmShape sh{C < 1 ? 1 : C, A, wp, A_live_max};
    if (em_plan_batched(ctx, sh, &a, &na, &smem) != HGT_OK) return false;
    if (a.compact || C < 2) return false;
    const size_t bytes = (size_t)C * wp * 8;
    // cooperative launches run one after the other: worth it for a big matrix, or when there are too few problems to fill
    // the SMs with one streaming CTA each
    return bytes > ((size_t)4 << 20) || (n_problems <= 6 && bytes > ((size_t)256 << 10));
}
size_t hgt_em_coop_ws_bytes(const hgt_ctx *ctx, int A) { return em_ws_bytes(ctx->sm_count, A); }

extern "C" int hgt_em_form(const hgt_ctx *ctx, int32_t n_classes, int32_t n_alleles, int32_t wp, int32_t has_lengths,
                           int32_t n_ctas, int32_t a_live_max, int32_t n_problems, hgt_em_form_info *out) {
    if (!ctx || !out || n_classes < 1 || n_alleles < 1 || wp < hgt_row_pitch(n_alleles) || (wp & 1)) {
        hgt_set_error("hgt_em_form: need a context, an output, n_classes >= 1, n_alleles >= 1 and an even wp >= "
                      "hgt_row_pitch(n_alleles)");
        return HGT_ERR_ARG;
    }
    if (a_live_max < 1 || a_live_max > n_alleles) a_live_max = n_alleles;
    EmArgs a;
    EmPlan plan;
    int G = 1;
    HGT_CHECK(em_dev_plan(ctx, n_classes, n_alleles, wp, n_ctas, a_live_max, &a, &plan, &G));
    out->form = G > 1 ? HGT_EM_FORM_COOP : (a.compact ? HGT_EM_FORM_COMPACT : HGT_EM_FORM_STREAM);
    out->grid = G;
    out->na = plan.na;
    out->slab_rows = plan.slab_rows;
    out->slab_bytes = a.slab_bytes;
    out->merge = a.compact && !has_lengths && em_merge_fits(wp, a.A_live_max, a.slab_bytes);
    out->collapse = G == 1 && em_collapse_fits(a.compact, n_classes, wp, plan.slab_rows);
    out->batch_coop = hgt_em_wants_coop(ctx, n_classes, n_alleles, wp, a_live_max, n_problems);
    return HGT_OK;
}

int hgt_em_batch_dev(hgt_ctx *ctx, cudaStream_t st, int n_problems, const EmDevProblem *pr, void *h_args, void *d_args) {
    if (n_problems <= 0) return HGT_OK;
    std::vector<EmArgs> args, coop;
    std::vector<int> nas, coop_na, coop_g;
    std::vector<size_t> smems, coop_smem;
    for (int i = 0; i < n_problems; i++) {
        EmArgs a;
        const size_t Apad = (size_t)pr[i].wp * 64;
        a.bits = pr[i].bits; a.cnt = nullptr; a.len = pr[i].len;
        a.C = pr[i].C_max; a.A = pr[i].A; a.wp = pr[i].wp; a.remove_low = pr[i].remove_low; a.fixed_iters = 0;
        a.cnt_u64 = pr[i].cnt; a.C_ptr = pr[i].C_ptr; a.class_first = pr[i].class_first; a.key_offset = 0; a.peer = nullptr;
        a.prob = pr[i].prob; a.in_result = pr[i].in_result; a.first_class = pr[i].first_class;
        a.iters_status = pr[i].iters_status;
        a.part_acc = nullptr; a.part_aux = nullptr; a.red_acc = nullptr; a.red_aux = nullptr;
        if (pr[i].coop_ws && pr[i].C_max > 1) {
            // one problem on every SM (cooperative launch): the class matrix streams from HBM once per next_prob
            int G = ctx->sm_count;
            if (G > pr[i].C_max) G = pr[i].C_max;
            EmPlan plan;
            HGT_CHECK(em_plan(ctx, (pr[i].C_max + G - 1) / G, pr[i].A, pr[i].wp, &plan));
            EmWs w = em_ws_carve(pr[i].coop_ws, ctx->sm_count, pr[i].A);
            a.vec = w.vec; a.live = w.live; a.part_acc = w.part_acc; a.part_aux = w.part_aux;
            a.red_acc = w.red_acc; a.red_aux = w.red_aux;
            em_set_scratch(&a, w.scratch);
            a.compact = 0; a.A_live_max = pr[i].A; a.slab_bytes = 0;
            a.slab_rows = plan.slab_rows;
            coop.push_back(a);
            coop_na.push_back(plan.na);
            coop_smem.push_back(plan.smem);
            coop_g.push_back(G);
            continue;
        }
        const EmShape sh{pr[i].C_max < 1 ? 1 : pr[i].C_max, pr[i].A, pr[i].wp, pr[i].A_live_max};
        int na = 1;
        size_t smem = 0;
        HGT_CHECK(em_plan_batched(ctx, sh, &a, &na, &smem));
        a.vec = static_cast<double *>(pr[i].ws);
        a.live = reinterpret_cast<uint8_t *>(a.vec + 4 * Apad);
        em_set_scratch(&a, static_cast<unsigned char *>(pr[i].ws) + align_up(4 * Apad * 8 + 4 * Apad, 256));
        args.push_back(a);
        nas.push_back(na);
        smems.push_back(smem);
    }
    EmArgs *h = static_cast<EmArgs *>(h_args), *d = static_cast<EmArgs *>(d_args);
    const int nb = (int)args.size();
    if (nb > 0) HGT_CHECK(em_launch_batched(ctx, st, nb, args.data(), nas.data(), smems.data(), h, d, true));
    for (size_t k = 0; k < coop.size(); k++) {
        h[nb + k] = coop[k];
        HGT_CUDA(hgt_small_h2d(d + nb + k, h + nb + k, sizeof(EmArgs), st));
        HGT_CHECK(em_launch<true>(ctx, st, d + nb + k, coop_g[k], coop_na[k], coop_smem[k]));
    }
    return HGT_OK;
}

// Diploid allele-pair model for every unit of a finished batch, on the class tables the batch keeps in HBM
//   (the legacy typer's joint_abundance, etc/hisatgenotype_hla_cyp.py:236-302; host path: typing_common.joint_abundance
//   + hgt_pair_em in pair.cu, which stays the reference of this one).
//
// Two launches, one CTA per (unit, table) problem, with one read-back of the pair counts in between:
//   pair_count_kernel   ranks the region's rows by `first` into its own scratch (the batch's rows are not moved), sums the
//                       per-allele mass m[a] = sum_k n_k / popc(S_k) in that (dict) order - the association of the host
//                       loop, so the masses and with them the pruned pair set are the host's exactly - sorts the alleles
//                       that can be in a surviving pair by (-m, index) and counts every one's partners by binary search.
//   pair_loop_kernel    (heaviest problems first) enumerates the pairs at scanned offsets, in the host's order, and runs
//                       the loop of pair_em_kernel in factorised form.  With U_q = sub(lo) u sub(hi) the legacy weight is
//                       w[k][q] = |S_k n U_q|, so one iteration needs only per-allele vectors:
//                         V[a] = sum of P over the pairs holding a          (row of a + column of a in the pair layout)
//                         T[x] = sum_{q: x in U_q} P_q = sum_{a in sup(x)} V[a] - P of the pairs with both members in sup(x)
//                         prob_k = sum_{x in S_k} T[x];  coef_k = prob_k > 0 ? n_k / prob_k : 0;  R[x] = sum_{k ni x} coef_k
//                         next_q = P_q * sum_{x in U_q} R[x]
//                       O(nnz(S restricted to the names of the candidates) + sum |U_q|) per iteration; no weight matrix.
//                       The rest is pair_em_kernel statement for statement: prob_diff (an alive pair is always touched
//                       here, since its own allele is a class member), normalise, choose_top_alleles, renormalise,
//                       diff > 1e-4 && iter < 1000.
// Every sum runs in a fixed order (thread-strided partials, fixed reduction trees, CSR lists in dict order; no floating-point
// atomics), so repeated calls give bit-identical results.  Scratch comes from the context's pool.
#include <algorithm>
#include <numeric>
#include <vector>

#include "pair_batch.h"

namespace {

constexpr int PB = 512, PBW = PB / 32;

struct PairJob {
    PairUnit u;
    int32_t unit = 0;
    int64_t oc = 0, oa = 0;  // offsets of the class-sized and allele-sized scratch slots
};
struct PairState {
    int64_t Q = 0, nnz = 0;   // pairs after the first pruning, class members that are names of the candidates
    int64_t chk = 0;          // largest running pair count at which the host enumeration tests its limit (0: never)
    int32_t n_cand = 0, pad = 0;
};
// Scratch arrays of all problems; a problem's slice starts at its offset of the array's kind.
struct PairArena {
    int32_t *ord, *pc, *ck;          // class slots: row of dict rank k, popcount, members inside X
    int64_t *coff;                   //   CSR offsets of the class -> X-member lists [C + 1]
    double *cn, *coef;               //   count as double, n_k / prob_k
    double *m, *sm, *V, *T, *R;      // allele slots: mass, sorted masses, per-allele sums of the loop
    int32_t *cidx, *pos, *e, *rr, *xl;  // sorted candidates, position of an allele there, partner ends, column lengths, X
    int64_t *off, *xoff, *tmp;       //   pair offsets per candidate, CSR offsets of the X-member -> class lists, scan space
    uint64_t *xb;                    //   X as a bit set [wp]
    int32_t *pi, *pj, *sv;           // pair slots: candidate positions of the two members, survivors
    int32_t *rlo, *rhi;              //   the result in (-p, lo, hi) order (all of it; the [unit][cap] arrays hold its head)
    double *P, *nx, *rp;
    uint8_t *alive;
    int32_t *cmem, *xcls;            // member slots: CSR lists
};
struct PairSlots {
    int64_t oq = 0, on = 0;
};

__device__ __forceinline__ double pb_sum(double v, double *red) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) red[warp] = v;
    __syncthreads();
    if (warp == 0) {
        double x = lane < PBW ? red[lane] : 0.0;
        x = warp_sum(x);
        if (lane == 0) red[32] = x;
    }
    __syncthreads();
    const double r = red[32];
    __syncthreads();
    return r;
}
__device__ __forceinline__ double pb_max(double v, double *red) {
    v = warp_max(v);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) red[warp] = v;
    __syncthreads();
    if (warp == 0) {
        double x = lane < PBW ? red[lane] : 0.0;
        x = warp_max(x);
        if (lane == 0) red[32] = x;
    }
    __syncthreads();
    const double r = red[32];
    __syncthreads();
    return r;
}

// Exclusive scan of val(0..n-1) into out[0..n] (out[n] = total); returns the total.  red: shared [PBW].
template <class F>
__device__ __forceinline__ int64_t pb_scan(int64_t n, F val, int64_t *out, long long *red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long carry = 0;
    for (int64_t b = 0; b < n; b += PB) {
        const int64_t i = b + threadIdx.x;
        const long long v = i < n ? (long long)val(i) : 0;
        long long x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) red[warp] = x;
        __syncthreads();
        if (warp == 0) {
            long long w = lane < PBW ? red[lane] : 0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const long long y = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += y;
            }
            if (lane < PBW) red[lane] = w;
        }
        __syncthreads();
        if (i < n) out[i] = carry + (warp ? red[warp - 1] : 0) + x - v;
        const long long tot = red[PBW - 1];
        __syncthreads();
        carry += tot;
    }
    if (threadIdx.x == 0) out[n] = carry;
    __syncthreads();
    return carry;
}

// Bitonic sort of the distinct indices a[0..n) by less(); a has room for the next power of two >= n (padded with -1,
// which sorts last).  Global memory, one CTA.
template <class Less>
__device__ __forceinline__ void pb_sort(int32_t *a, int n, Less less) {
    int n2 = 1;
    while (n2 < n) n2 <<= 1;
    for (int i = n + threadIdx.x; i < n2; i += PB) a[i] = -1;
    __syncthreads();
    for (int k = 2; k <= n2; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n2; i += PB) {
                const int l = i ^ j;
                if (l <= i) continue;
                const int32_t x = a[i], y = a[l];
                const bool y_first = x < 0 ? y >= 0 : (y >= 0 && less(y, x));
                if (y_first == ((i & k) == 0)) {
                    a[i] = y;
                    a[l] = x;
                }
            }
            __syncthreads();
        }
}

// first j in [0, n) with pred(j) (pred monotone false..true), n if none
template <class F>
__device__ __forceinline__ int first_true(int n, F pred) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (pred(mid)) hi = mid;
        else lo = mid + 1;
    }
    return lo;
}

__global__ void __launch_bounds__(PB, 1) pair_count_kernel(const PairJob *__restrict__ jobs, PairArena S, PairState *state) {
    __shared__ double red[33];
    __shared__ long long sred[PBW];
    const PairJob J = jobs[blockIdx.x];
    const int C = J.u.C, A = J.u.A, wp = J.u.wp, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint64_t *bits = J.u.bits;
    int32_t *ord = S.ord + J.oc, *pc = S.pc + J.oc, *ck = S.ck + J.oc;
    int64_t *coff = S.coff + J.oc;
    double *cn = S.cn + J.oc, *m = S.m + J.oa, *sm = S.sm + J.oa;
    int32_t *cidx = S.cidx + J.oa, *pos = S.pos + J.oa, *e = S.e + J.oa, *rr = S.rr + J.oa;
    int64_t *off = S.off + J.oa;
    uint64_t *xb = S.xb + J.oa;
    // rows in dict order = ascending `first`
    for (int r = tid; r < C; r += PB) ord[r] = r;
    __syncthreads();
    const int32_t *first = J.u.first;
    pb_sort(ord, C, [first](int32_t x, int32_t y) { return first[x] < first[y]; });
    for (int k = tid; k < C; k += PB) {
        const uint64_t *row = bits + (size_t)ord[k] * wp;
        int p = 0;
        for (int j = 0; j < wp; j++) p += __popcll(row[j]);
        pc[k] = p;
        cn[k] = (double)J.u.count[ord[k]];
    }
    __syncthreads();
    // m[a]: a warp per 64-allele word, a lane per two alleles, classes in dict order: share = (double)n_k / popc added one
    // after the other, as typing_common.joint_abundance does
    for (int j = warp; j < wp; j += PBW) {
        double m0 = 0.0, m1 = 0.0;
        for (int k0 = 0; k0 < C; k0 += 32) {
            const int k = k0 + lane;
            uint64_t w = 0;
            double s = 0.0;
            if (k < C) {
                w = bits[(size_t)ord[k] * wp + j];
                s = cn[k] / (double)pc[k];
            }
            const int nk = min(32, C - k0);
            for (int t = 0; t < nk; t++) {
                const uint64_t wt = __shfl_sync(0xffffffffu, w, t);
                const double st = __shfl_sync(0xffffffffu, s, t);
                if ((wt >> lane) & 1ull) m0 += st;
                if ((wt >> (lane + 32)) & 1ull) m1 += st;
            }
        }
        const int a0 = j * 64 + lane, a1 = a0 + 32;
        if (a0 < A) m[a0] = m0;
        if (a1 < A) m[a1] = m1;
    }
    __syncthreads();
    // ms[0], ms[1] of the host's sorted masses (alleles of the table only: m > 0, every count is >= 1)
    double mx = 0.0, nl = 0.0;
    for (int a = tid; a < A; a += PB) {
        const double v = m[a];
        pos[a] = -1;
        if (v > 0.0) {
            mx = fmax(mx, v);
            nl += 1.0;
        }
    }
    const double ms0 = pb_max(mx, red), n_live = pb_sum(nl, red);
    double n0 = 0.0, mx2 = 0.0;
    for (int a = tid; a < A; a += PB) {
        const double v = m[a];
        if (v > 0.0 && v == ms0) n0 += 1.0;
        if (v > 0.0 && v < ms0) mx2 = fmax(mx2, v);
    }
    const double n_top = pb_sum(n0, red), below = pb_max(mx2, red);
    const double ms1 = n_top >= 2.0 ? ms0 : below;
    double best = n_live >= 2.0 ? ms0 + ms1 : ms0;
    best = fmax(best, ms0);
    // candidates: the host's loop over the sorted alleles stops at the first (ms[i] + ms[0]) * 2 <= best (and then also
    // ms[i] * 2 <= best); every partner of a surviving pair passes the same test
    auto cand = [m, ms0, best](int64_t a) { return m[a] > 0.0 && !((m[a] + ms0) * 2.0 <= best); };
    const int n_cand = (int)pb_scan(A, cand, off, sred);
    for (int a = tid; a < A; a += PB)
        if (cand(a)) cidx[off[a]] = a;
    __syncthreads();
    pb_sort(cidx, n_cand, [m](int32_t x, int32_t y) { return m[x] > m[y] || (m[x] == m[y] && x < y); });
    double mnc = 0.0, hnc = 0.0;  // largest mass below the candidates (the host's next sorted allele), and whether one exists
    for (int a = tid; a < A; a += PB)
        if (m[a] > 0.0 && !cand(a)) {
            mnc = fmax(mnc, m[a]);
            hnc = 1.0;
        }
    const double m_next = pb_max(mnc, red), has_next = pb_max(hnc, red);
    for (int i = tid; i < n_cand; i += PB) {
        sm[i] = m[cidx[i]];
        pos[cidx[i]] = i;
    }
    __syncthreads();
    // partners of position i: j in (i, e_i), e_i = min(first j with ms[j] <= best/2 - ms[i] (the host's searchsorted),
    // first j with (ms[i] + ms[j]) * 2 <= best (its filter)); both bounds are monotone in j and non-increasing in i
    for (int i = tid; i < n_cand; i += PB) {
        const double mi = sm[i], t = best / 2.0 - mi;
        const int hia = first_true(n_cand, [sm, t](int j) { return sm[j] <= t; });
        const int hib = first_true(n_cand, [sm, mi, best](int j) { return (mi + sm[j]) * 2.0 <= best; });
        e[i] = min(hia, hib);
        // the host tests its pair limit after position i exactly when its searchsorted bound over ALL sorted alleles
        // exceeds i + 1 (that bound may run past the candidates by one allele)
        const int hia_all = hia < n_cand ? hia : (has_next > 0.0 && m_next > t ? n_cand + 1 : n_cand);
        rr[i] = hia_all > i + 1;
    }
    __syncthreads();
    const int64_t Q = pb_scan(
        n_cand, [e, sm, best](int64_t i) { return (int64_t)max(e[i] - (int)i - 1, 0) + (!(sm[i] * 2.0 <= best) ? 1 : 0); }, off, sred);
    // ... where its running count is all pairs of the positions before i plus i's partners
    double ck_part = 0.0;
    for (int i = tid; i < n_cand; i += PB)
        if (rr[i]) ck_part = fmax(ck_part, (double)(off[i] + max(e[i] - i - 1, 0)));
    const double chk = pb_max(ck_part, red);
    // X = names inside the candidates' names: the alleles whose T / R the loop needs
    for (int j = tid; j < wp; j += PB) xb[j] = 0;
    __syncthreads();
    for (int i = tid; i < n_cand; i += PB) {
        const int a = cidx[i];
        for (int64_t s = J.u.sub_off[a]; s < J.u.sub_off[a + 1]; s++) {
            const int x = J.u.sub_idx[s];
            atomicOr(reinterpret_cast<unsigned long long *>(&xb[x >> 6]), 1ull << (x & 63));
        }
    }
    __syncthreads();
    for (int k = tid; k < C; k += PB) {
        const uint64_t *row = bits + (size_t)ord[k] * wp;
        int p = 0;
        for (int j = 0; j < wp; j++) p += __popcll(row[j] & xb[j]);
        ck[k] = p;
    }
    __syncthreads();
    const int64_t nnz = pb_scan(C, [ck](int64_t k) { return ck[k]; }, coff, sred);
    if (tid == 0) {
        state[blockIdx.x].Q = Q;
        state[blockIdx.x].nnz = nnz;
        state[blockIdx.x].n_cand = n_cand;
        state[blockIdx.x].chk = (int64_t)chk;
    }
}

__global__ void __launch_bounds__(PB, 1)
    pair_loop_kernel(const PairJob *__restrict__ jobs, const int32_t *__restrict__ order, const PairSlots *__restrict__ slots,
                     const PairState *__restrict__ state, PairArena S, int cap, int32_t *out_lo, int32_t *out_hi,
                     double *out_p, int32_t *meta) {
    __shared__ double red[33];
    __shared__ long long sred[PBW];
    const int jb = order[blockIdx.x];
    const PairJob J = jobs[jb];
    const PairSlots Z = slots[jb];
    const PairState ps = state[jb];
    const int C = J.u.C, A = J.u.A, wp = J.u.wp, n_cand = ps.n_cand, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t Q = ps.Q;
    const uint64_t *bits = J.u.bits;
    const int64_t *sub_off = J.u.sub_off, *sup_off = J.u.sup_off;
    const int32_t *sub_idx = J.u.sub_idx, *sup_idx = J.u.sup_idx;
    const int32_t *ord = S.ord + J.oc;
    const int64_t *coff = S.coff + J.oc;
    const double *cn = S.cn + J.oc, *sm = S.sm + J.oa;
    double *coef = S.coef + J.oc, *V = S.V + J.oa, *T = S.T + J.oa, *R = S.R + J.oa;
    const int32_t *cidx = S.cidx + J.oa, *pos = S.pos + J.oa, *e = S.e + J.oa;
    int32_t *rr = S.rr + J.oa, *xl = S.xl + J.oa;
    const int64_t *off = S.off + J.oa;
    int64_t *xoff = S.xoff + J.oa, *tmp = S.tmp + J.oa;
    const uint64_t *xb = S.xb + J.oa;
    int32_t *pi = S.pi + Z.oq, *pj = S.pj + Z.oq, *sv = S.sv + Z.oq, *cmem = S.cmem + Z.on, *xcls = S.xcls + Z.on;
    double *P = S.P + Z.oq, *nx = S.nx + Z.oq;
    uint8_t *alive = S.alive + Z.oq;

    // ---- set-up: class -> X-member lists (dict order of classes, members ascending) -------------------------------
    for (int k = tid; k < C; k += PB) {
        const uint64_t *row = bits + (size_t)ord[k] * wp;
        int64_t p = coff[k];
        for (int j = 0; j < wp; j++) {
            uint64_t w = row[j] & xb[j];
            while (w) {
                cmem[p++] = j * 64 + __ffsll((long long)w) - 1;
                w &= w - 1;
            }
        }
    }
    // X-member -> classes in dict order: counts, scan, fill (a warp per word, a lane per two alleles, as the mass pass)
    for (int pass = 0; pass < 2; pass++) {
        for (int j = warp; j < wp; j += PBW) {
            const uint64_t xw = xb[j];
            const int a0 = j * 64 + lane, a1 = a0 + 32;
            int64_t c0 = pass ? (a0 < A ? xoff[a0] : 0) : 0, c1 = pass ? (a1 < A ? xoff[a1] : 0) : 0;
            const bool in0 = (xw >> lane) & 1ull, in1 = (xw >> (lane + 32)) & 1ull;
            if (xw)
                for (int k0 = 0; k0 < C; k0 += 32) {
                    const int k = k0 + lane;
                    const uint64_t w = k < C ? bits[(size_t)ord[k] * wp + j] & xw : 0;
                    const int nk = min(32, C - k0);
                    for (int t = 0; t < nk; t++) {
                        const uint64_t wt = __shfl_sync(0xffffffffu, w, t);
                        if (in0 && ((wt >> lane) & 1ull)) {
                            if (pass) xcls[c0] = k0 + t;
                            c0++;
                        }
                        if (in1 && ((wt >> (lane + 32)) & 1ull)) {
                            if (pass) xcls[c1] = k0 + t;
                            c1++;
                        }
                    }
                }
            if (!pass) {
                if (a0 < A) tmp[a0] = c0;
                if (a1 < A) tmp[a1] = c1;
            }
        }
        __syncthreads();
        if (!pass) pb_scan(A, [tmp](int64_t a) { return tmp[a]; }, xoff, sred);
    }
    // X as a list in index order
    pb_scan(wp, [xb](int64_t j) { return __popcll(xb[j]); }, tmp, sred);
    const int nX = (int)tmp[wp];
    for (int j = tid; j < wp; j += PB) {
        uint64_t w = xb[j];
        int64_t p = tmp[j];
        while (w) {
            xl[p++] = j * 64 + __ffsll((long long)w) - 1;
            w &= w - 1;
        }
    }
    for (int a = tid; a < A; a += PB) T[a] = 0.0;
    // pairs in the host's order: per candidate position i its partners i+1 .. e_i-1, then (i, i); p0 = mass / sum
    for (int i = tid; i < n_cand; i += PB) {
        const int64_t q0 = off[i];
        const int cnt = max(e[i] - i - 1, 0);
        for (int t = 0; t < cnt; t++) {
            pi[q0 + t] = i;
            pj[q0 + t] = i + 1 + t;
            P[q0 + t] = sm[i] + sm[i + 1 + t];
            alive[q0 + t] = 1;
        }
        if (off[i + 1] > q0 + cnt) {
            pi[q0 + cnt] = i;
            pj[q0 + cnt] = i;
            P[q0 + cnt] = sm[i];
            alive[q0 + cnt] = 1;
        }
        // column of position i: the pairs (i', i) with i' < i, i.e. the i' with e_{i'} > i (a prefix: e is non-increasing)
        rr[i] = min(i, first_true(n_cand, [e, i](int x) { return e[x] <= i; }));
    }
    __syncthreads();
    double part = 0.0;
    for (int64_t q = tid; q < Q; q += PB) part += P[q];
    const double mass = pb_sum(part, red);
    for (int64_t q = tid; q < Q; q += PB) P[q] = P[q] / mass;
    __syncthreads();

    // ---- the loop -------------------------------------------------------------------------------------------------
    double diff = 1.0;
    int iter = 0;
    while (diff > 0.0001 && iter < 1000) {
        for (int p = warp; p < n_cand; p += PBW) {
            double s = 0.0;
            for (int64_t q = off[p] + lane; q < off[p + 1]; q += 32) s += P[q];
            for (int i = lane; i < rr[p]; i += 32) s += P[off[i] + (p - i - 1)];
            s = warp_sum(s);
            if (lane == 0) V[p] = s;
        }
        __syncthreads();
        for (int t = tid; t < nX; t += PB) {
            const int x = xl[t];
            double s = 0.0;
            const int64_t b0 = sup_off[x], b1 = sup_off[x + 1];
            for (int64_t u = b0; u < b1; u++) {
                const int pa = pos[sup_idx[u]];
                if (pa >= 0) s += V[pa];
            }
            // a pair whose two members both contain x was counted twice
            for (int64_t u = b0; u < b1; u++) {
                const int pa = pos[sup_idx[u]];
                if (pa < 0) continue;
                for (int64_t w = u + 1; w < b1; w++) {
                    const int pb = pos[sup_idx[w]];
                    if (pb < 0) continue;
                    const int i = min(pa, pb), j = max(pa, pb);
                    if (j < e[i]) s -= P[off[i] + (j - i - 1)];
                }
            }
            T[x] = s;
        }
        __syncthreads();
        for (int k = tid; k < C; k += PB) {
            double s = 0.0;
            for (int64_t c = coff[k]; c < coff[k + 1]; c++) s += T[cmem[c]];
            coef[k] = s > 0.0 ? cn[k] / s : 0.0;
        }
        __syncthreads();
        for (int t = tid; t < nX; t += PB) {
            const int x = xl[t];
            double s = 0.0;
            for (int64_t c = xoff[x]; c < xoff[x + 1]; c++) s += coef[xcls[c]];
            R[x] = s;
        }
        __syncthreads();
        double npart = 0.0;
        for (int64_t q = tid; q < Q; q += PB) {
            if (!alive[q]) continue;
            const int a = cidx[pi[q]], b = cidx[pj[q]];
            double acc = 0.0;
            int64_t u = sub_off[a], ue = sub_off[a + 1], w = sub_off[b], we = sub_off[b + 1];
            if (a == b) w = we;
            while (u < ue || w < we) {  // U_q = sub(a) u sub(b), both lists ascending
                const int xa = u < ue ? sub_idx[u] : 0x7fffffff, xw = w < we ? sub_idx[w] : 0x7fffffff;
                const int x = min(xa, xw);
                acc += R[x];
                if (xa == x) u++;
                if (xw == x) w++;
            }
            const double v = P[q] * acc;
            nx[q] = v;
            npart += v;
        }
        const double total = pb_sum(npart, red);
        double dpart = 0.0, bst = 0.0;
        for (int64_t q = tid; q < Q; q += PB) {
            if (!alive[q]) continue;
            const double v = nx[q] / total;
            nx[q] = v;
            dpart += fabs(P[q] - v);
            bst = fmax(bst, v);
        }
        diff = pb_sum(dpart, red);
        const double best = pb_max(bst, red);
        double kpart = 0.0;
        for (int64_t q = tid; q < Q; q += PB) {
            const bool keep = alive[q] && !(nx[q] * 2.0 <= best);
            alive[q] = keep ? 1 : 0;
            if (keep) kpart += nx[q];
        }
        const double ktotal = pb_sum(kpart, red);
        for (int64_t q = tid; q < Q; q += PB) P[q] = alive[q] ? nx[q] / ktotal : 0.0;
        __syncthreads();
        iter++;
    }

    // ---- pairs with p > 0 in (-p, lo, hi) order ----------------------------------------------------------------------
    int64_t *spos = reinterpret_cast<int64_t *>(nx);  // (the loop is over: nx has room for Q + 1 offsets)
    const int n_s = (int)pb_scan(Q, [P](int64_t q) { return P[q] > 0.0 ? 1 : 0; }, spos, sred);
    for (int64_t q = tid; q < Q; q += PB)
        if (P[q] > 0.0) sv[spos[q]] = (int32_t)q;
    __syncthreads();
    auto lo_of = [cidx, pi, pj](int32_t q) { return min(cidx[pi[q]], cidx[pj[q]]); };
    auto hi_of = [cidx, pi, pj](int32_t q) { return max(cidx[pi[q]], cidx[pj[q]]); };
    pb_sort(sv, n_s, [P, lo_of, hi_of](int32_t x, int32_t y) {
        if (P[x] != P[y]) return P[x] > P[y];
        const int lx = lo_of(x), ly = lo_of(y);
        if (lx != ly) return lx < ly;
        return hi_of(x) < hi_of(y);
    });
    const int unit = J.unit;
    int32_t *rlo = S.rlo + Z.oq, *rhi = S.rhi + Z.oq;
    double *rp = S.rp + Z.oq;
    for (int r = tid; r < n_s; r += PB) {
        const int32_t q = sv[r];
        rlo[r] = lo_of(q);
        rhi[r] = hi_of(q);
        rp[r] = P[q];
        if (r < cap) {
            out_lo[(size_t)unit * cap + r] = rlo[r];
            out_hi[(size_t)unit * cap + r] = rhi[r];
            out_p[(size_t)unit * cap + r] = rp[r];
        }
    }
    if (tid == 0) {
        meta[unit * 3 + 0] = n_s;
        meta[unit * 3 + 1] = iter;
        meta[unit * 3 + 2] = HGT_OK;
    }
}

// Device / page-locked blocks of the context's pool, returned when the call ends.  The stream is synchronised first, so a
// return on an error path cannot hand out a block that a queued kernel or copy still uses.
struct PoolHold {
    hgt_ctx *ctx;
    cudaStream_t st;
    std::vector<std::pair<void *, std::pair<bool, size_t>>> held;
    PoolHold(hgt_ctx *c, cudaStream_t s) : ctx(c), st(s) {}
    int get(bool pinned, size_t n, void **out) {
        size_t cap = 0;
        HGT_CHECK(ctx->pool.get(pinned, n ? n : 16, out, &cap));
        held.push_back({*out, {pinned, cap}});
        return HGT_OK;
    }
    ~PoolHold() {
        if (!held.empty()) cudaStreamSynchronize(st);
        for (auto &h : held) ctx->pool.put(h.second.first, h.first, h.second.second);
    }
};

inline int64_t pow2_at_least(int64_t n) {
    int64_t p = 1;
    while (p < n) p <<= 1;
    return p;
}
inline size_t a256(size_t x) { return (x + 255) & ~(size_t)255; }

}  // namespace

int hgt_pair_batch_run(hgt_ctx *ctx, cudaStream_t st, const std::vector<PairUnit> &units, int64_t max_pairs, int32_t cap,
                       PairResult *res) {
    const int64_t nu = (int64_t)units.size();
    res->off.assign(nu + 1, 0);
    res->lo.clear(); res->hi.clear(); res->p.clear();
    res->n_total.assign(nu, 0); res->iters.assign(nu, 0); res->status.assign(nu, HGT_OK); res->n_pairs.assign(nu, 0);
    int32_t *n_total = res->n_total.data(), *iters = res->iters.data(), *status = res->status.data();
    cap = std::min(std::max(cap, 1), 4096);  // rows read back at once; longer results follow unit by unit
    std::vector<PairJob> jobs;
    int64_t nc = 0, na = 0;
    for (int64_t u = 0; u < nu; u++) {
        const PairUnit &U = units[u];
        if (U.C <= 0) continue;  // empty table: no pair, status OK
        PairJob J;
        J.u = U;
        J.unit = (int32_t)u;
        J.oc = nc;
        J.oa = na;
        nc += pow2_at_least(U.C) + 1;
        na += pow2_at_least(U.A) + 1;
        jobs.push_back(J);
    }
    if (jobs.empty()) return HGT_OK;
    const int64_t nj = (int64_t)jobs.size();
    PoolHold hold(ctx, st);
    // class- and allele-sized scratch, job descriptors, states: one device block
    const size_t o_jobs = 0, o_state = a256(o_jobs + nj * sizeof(PairJob)), o_slots = a256(o_state + nj * sizeof(PairState)),
                 o_order = a256(o_slots + nj * sizeof(PairSlots)), o_c = a256(o_order + nj * 4),
                 c_bytes = (size_t)nc * (3 * 4 + 8 + 2 * 8), o_a = a256(o_c + c_bytes),
                 a_bytes = (size_t)na * (5 * 8 + 5 * 4 + 3 * 8 + 8), bytes = a256(o_a + a_bytes);
    void *dv = nullptr, *hv = nullptr;
    HGT_CHECK(hold.get(false, bytes, &dv));
    const size_t h_bytes = a256(nj * sizeof(PairJob)) + a256(nj * sizeof(PairState)) + a256(nj * sizeof(PairSlots)) + a256(nj * 4);
    HGT_CHECK(hold.get(true, h_bytes, &hv));
    unsigned char *d = static_cast<unsigned char *>(dv), *h = static_cast<unsigned char *>(hv);
    PairJob *h_jobs = reinterpret_cast<PairJob *>(h);
    PairState *h_state = reinterpret_cast<PairState *>(h + a256(nj * sizeof(PairJob)));
    PairSlots *h_slots = reinterpret_cast<PairSlots *>(reinterpret_cast<unsigned char *>(h_state) + a256(nj * sizeof(PairState)));
    int32_t *h_order = reinterpret_cast<int32_t *>(reinterpret_cast<unsigned char *>(h_slots) + a256(nj * sizeof(PairSlots)));
    std::copy(jobs.begin(), jobs.end(), h_jobs);
    PairArena S{};
    {
        unsigned char *p = d + o_c;
        auto take = [&p](size_t elem, int64_t n) {
            unsigned char *r = p;
            p += elem * (size_t)n;
            return r;
        };
        S.coff = (int64_t *)take(8, nc); S.cn = (double *)take(8, nc); S.coef = (double *)take(8, nc);
        S.ord = (int32_t *)take(4, nc); S.pc = (int32_t *)take(4, nc); S.ck = (int32_t *)take(4, nc);
        p = d + o_a;
        S.m = (double *)take(8, na); S.sm = (double *)take(8, na); S.V = (double *)take(8, na); S.T = (double *)take(8, na);
        S.R = (double *)take(8, na);
        S.off = (int64_t *)take(8, na); S.xoff = (int64_t *)take(8, na); S.tmp = (int64_t *)take(8, na);
        S.xb = (uint64_t *)take(8, na);
        S.cidx = (int32_t *)take(4, na); S.pos = (int32_t *)take(4, na); S.e = (int32_t *)take(4, na); S.rr = (int32_t *)take(4, na);
        S.xl = (int32_t *)take(4, na);
    }
    HGT_CUDA(cudaMemcpyAsync(d + o_jobs, h_jobs, nj * sizeof(PairJob), cudaMemcpyHostToDevice, st));
    ctx->h2d_bytes += nj * (int64_t)sizeof(PairJob);
    PairState *d_state = reinterpret_cast<PairState *>(d + o_state);
    pair_count_kernel<<<(unsigned)nj, PB, 0, st>>>(reinterpret_cast<const PairJob *>(d + o_jobs), S, d_state);
    ctx->launches++;
    HGT_CUDA(cudaGetLastError());
    // the sizing read-back: pairs and CSR members of every problem
    HGT_CUDA(cudaMemcpyAsync(h_state, d_state, nj * sizeof(PairState), cudaMemcpyDeviceToHost, st));
    ctx->d2h_bytes += nj * (int64_t)sizeof(PairState);
    HGT_CUDA(cudaStreamSynchronize(st));
    std::vector<int32_t> run;
    int64_t nq = 0, nn = 0;
    for (int64_t j = 0; j < nj; j++) {
        const int u = h_jobs[j].unit;
        res->n_pairs[u] = h_state[j].Q;
        if (h_state[j].chk > max_pairs) {  // typing_common.joint_abundance's rule, test point for test point
            status[u] = HGT_ERR_UNSUPPORTED;
            continue;
        }
        h_slots[j].oq = nq;
        h_slots[j].on = nn;
        nq += pow2_at_least(h_state[j].Q) + 1;
        nn += std::max<int64_t>(h_state[j].nnz, 1);
        run.push_back((int32_t)j);
    }
    // heaviest problems first (pairs, then class members), ties by unit: the tail of the launch is short problems
    std::stable_sort(run.begin(), run.end(), [&](int32_t x, int32_t y) {
        if (h_state[x].Q != h_state[y].Q) return h_state[x].Q > h_state[y].Q;
        return h_state[x].nnz > h_state[y].nnz;
    });
    std::copy(run.begin(), run.end(), h_order);
    const size_t cp = (size_t)std::max(cap, 1);
    const size_t o_q = 0, q_bytes = (size_t)nq * (5 * 4 + 3 * 8 + 1), o_n = a256(o_q + q_bytes),
                 o_lo = a256(o_n + (size_t)nn * 8), o_hi = a256(o_lo + (size_t)nu * cp * 4),
                 o_p = a256(o_hi + (size_t)nu * cp * 4), o_meta = a256(o_p + (size_t)nu * cp * 8),
                 bytes2 = a256(o_meta + (size_t)nu * 12);
    void *dv2 = nullptr;
    HGT_CHECK(hold.get(false, bytes2, &dv2));
    unsigned char *d2 = static_cast<unsigned char *>(dv2);
    {
        unsigned char *p = d2 + o_q;
        S.P = (double *)p; p += 8 * (size_t)nq;
        S.nx = (double *)p; p += 8 * (size_t)nq;
        S.rp = (double *)p; p += 8 * (size_t)nq;
        S.rlo = (int32_t *)p; p += 4 * (size_t)nq;
        S.rhi = (int32_t *)p; p += 4 * (size_t)nq;
        S.pi = (int32_t *)p; p += 4 * (size_t)nq;
        S.pj = (int32_t *)p; p += 4 * (size_t)nq;
        S.sv = (int32_t *)p; p += 4 * (size_t)nq;
        S.alive = p;
        S.cmem = (int32_t *)(d2 + o_n);
        S.xcls = S.cmem + nn;
    }
    int32_t *d_lo = (int32_t *)(d2 + o_lo), *d_hi = (int32_t *)(d2 + o_hi), *d_meta = (int32_t *)(d2 + o_meta);
    double *d_p = (double *)(d2 + o_p);
    HGT_CUDA(cudaMemsetAsync(d2 + o_lo, 0, o_meta + (size_t)nu * 12 - o_lo, st));
    if (!run.empty()) {
        HGT_CUDA(cudaMemcpyAsync(d + o_slots, h_slots, nj * sizeof(PairSlots), cudaMemcpyHostToDevice, st));
        HGT_CUDA(cudaMemcpyAsync(d + o_order, h_order, run.size() * 4, cudaMemcpyHostToDevice, st));
        ctx->h2d_bytes += nj * (int64_t)sizeof(PairSlots) + (int64_t)run.size() * 4;
        pair_loop_kernel<<<(unsigned)run.size(), PB, 0, st>>>(reinterpret_cast<const PairJob *>(d + o_jobs),
                                                              reinterpret_cast<const int32_t *>(d + o_order),
                                                              reinterpret_cast<const PairSlots *>(d + o_slots), d_state, S, cap,
                                                              d_lo, d_hi, d_p, d_meta);
        ctx->launches++;
        HGT_CUDA(cudaGetLastError());
    }
    std::vector<int32_t> meta((size_t)nu * 3), clo((size_t)nu * cap), chi((size_t)nu * cap);
    std::vector<double> cpr((size_t)nu * cap);
    HGT_CUDA(cudaMemcpyAsync(clo.data(), d_lo, (size_t)nu * cap * 4, cudaMemcpyDeviceToHost, st));
    HGT_CUDA(cudaMemcpyAsync(chi.data(), d_hi, (size_t)nu * cap * 4, cudaMemcpyDeviceToHost, st));
    HGT_CUDA(cudaMemcpyAsync(cpr.data(), d_p, (size_t)nu * cap * 8, cudaMemcpyDeviceToHost, st));
    HGT_CUDA(cudaMemcpyAsync(meta.data(), d_meta, (size_t)nu * 12, cudaMemcpyDeviceToHost, st));
    ctx->d2h_bytes += (int64_t)nu * cap * 16 + nu * 12;
    HGT_CUDA(cudaStreamSynchronize(st));
    for (int64_t u = 0; u < nu; u++) {
        if (status[u] == HGT_OK) {  // (over max_pairs: empty result)
            n_total[u] = meta[u * 3];
            iters[u] = meta[u * 3 + 1];
            status[u] = meta[u * 3 + 2];
        }
        res->off[u + 1] = res->off[u] + n_total[u];
    }
    const size_t nt = (size_t)res->off[nu];
    res->lo.resize(nt); res->hi.resize(nt); res->p.resize(nt);
    bool more = false;
    for (int64_t u = 0; u < nu; u++) {
        const size_t o = (size_t)res->off[u], k = (size_t)std::min(n_total[u], cap);
        std::copy(clo.begin() + u * cap, clo.begin() + u * cap + k, res->lo.begin() + o);
        std::copy(chi.begin() + u * cap, chi.begin() + u * cap + k, res->hi.begin() + o);
        std::copy(cpr.begin() + u * cap, cpr.begin() + u * cap + k, res->p.begin() + o);
        more |= n_total[u] > cap;
    }
    if (more) {  // the rare unit with more than `cap` pairs in its result: its whole list, from the loop's output
        for (int64_t j = 0; j < nj; j++) {
            const int u = h_jobs[j].unit;
            if (status[u] != HGT_OK || n_total[u] <= cap) continue;
            const size_t o = (size_t)res->off[u], n = (size_t)n_total[u], q = (size_t)h_slots[j].oq;
            HGT_CUDA(cudaMemcpyAsync(res->lo.data() + o, S.rlo + q, n * 4, cudaMemcpyDeviceToHost, st));
            HGT_CUDA(cudaMemcpyAsync(res->hi.data() + o, S.rhi + q, n * 4, cudaMemcpyDeviceToHost, st));
            HGT_CUDA(cudaMemcpyAsync(res->p.data() + o, S.rp + q, n * 8, cudaMemcpyDeviceToHost, st));
            ctx->d2h_bytes += (int64_t)n * 16;
        }
        HGT_CUDA(cudaStreamSynchronize(st));
    }
    return HGT_OK;
}

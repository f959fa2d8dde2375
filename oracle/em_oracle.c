/* CPU oracle for stage (b), the EM abundance estimate — TEST INFRASTRUCTURE ONLY.
 *
 * Plain-C restatement of single_abundance()
 *   (reference hisatgenotype_modules/hisatgenotype_typing_common.py:1282-1410, prob_diff :1272-1279)
 * that keeps the reference's *operation order*: Python dicts are modelled as (value array, presence
 * array, insertion-order list), sums run in dict insertion order, and every expression is evaluated
 * with the same association as the Python source, so results agree with the reference to the last
 * bit on the golden vectors (tests/test_oracle_golden.py).  Parity: PINNED by tests/golden/*.json.gz.
 *
 * Classes come as CSR: members of class k are mem[off[k] .. off[k+1]) in the order of the names in the
 * Gene_cmpt key; cnt[k] is the class count; len[] (nullable) the allele lengths (Gene_length).
 *
 * Build: gcc -O2 -shared -fPIC -o oracle/libem_oracle.so oracle/em_oracle.c -lm   (see oracle/Makefile)
 * Only tests/, __graft_entry__.smoke() and bench.py (cpu_baseline / --impl reference) may load it.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct {
    double *val;   /* value per allele */
    uint8_t *in;   /* key present? */
    int32_t *ord;  /* keys in insertion order */
    int32_t n;
} pdict;

static void pd_init(pdict *d, int A) {
    d->val = (double *)calloc((size_t)A, sizeof(double));
    d->in = (uint8_t *)calloc((size_t)A, 1);
    d->ord = (int32_t *)malloc((size_t)(A > 0 ? A : 1) * sizeof(int32_t));
    d->n = 0;
}
static void pd_free(pdict *d) { free(d->val); free(d->in); free(d->ord); }
static void pd_clear(pdict *d) {
    for (int32_t i = 0; i < d->n; i++) { d->in[d->ord[i]] = 0; d->val[d->ord[i]] = 0.0; }
    d->n = 0;
}
static inline void pd_touch(pdict *d, int32_t a) {
    if (!d->in[a]) { d->in[a] = 1; d->val[a] = 0.0; d->ord[d->n++] = a; }
}

/* normalize / normalize_len (common:1285-1297) */
static int normalize(pdict *d, const double *len) {
    double total = 0.0;
    if (len) {
        for (int32_t i = 0; i < d->n; i++) total += d->val[d->ord[i]] / len[d->ord[i]];
        /* ZeroDivisionError in the reference; an empty dict divides by nothing (e.g. an empty Gene_cmpt with lengths) */
        if (total == 0.0 && d->n > 0) return -3;
        for (int32_t i = 0; i < d->n; i++) { int32_t a = d->ord[i]; d->val[a] = d->val[a] / len[a] / total; }
    } else {
        /* `sum(prob.values())`: CPython >= 3.12 sums floats with Neumaier compensation (Python/bltinmodule.c,
         * builtin_sum); the goldens were captured under 3.12, so the same recurrence is used here. */
        double c = 0.0;
        for (int32_t i = 0; i < d->n; i++) {
            double x = d->val[d->ord[i]], t = total + x;
            if (fabs(total) >= fabs(x)) c += (total - t) + x;
            else c += (x - t) + total;
            total = t;
        }
        if (c != 0.0 && isfinite(c)) total += c;
        if (total == 0.0 && d->n > 0) return -3;
        for (int32_t i = 0; i < d->n; i++) d->val[d->ord[i]] /= total;
    }
    return 0;
}

/* next_prob (common:1311-1336) */
static int next_prob(int C, const int64_t *off, const int32_t *mem, const double *cnt, const pdict *p, pdict *q,
                     const double *len) {
    pd_clear(q);
    for (int k = 0; k < C; k++) {
        double s = 0.0;
        for (int64_t j = off[k]; j < off[k + 1]; j++)
            if (p->in[mem[j]]) s += p->val[mem[j]];
        if (s <= 0.0) continue;
        for (int64_t j = off[k]; j < off[k + 1]; j++) {
            int32_t a = mem[j];
            if (!p->in[a]) continue;
            pd_touch(q, a);
            q->val[a] += cnt[k] * p->val[a] / s;
        }
    }
    return normalize(q, len);
}

/* select_alleles (common:1338-1346) */
static void select_alleles(pdict *d) {
    if (d->n == 0) return;
    double mx = d->val[d->ord[0]];
    for (int32_t i = 1; i < d->n; i++) if (d->val[d->ord[i]] > mx) mx = d->val[d->ord[i]];
    int32_t m = 0;
    for (int32_t i = 0; i < d->n; i++) {
        int32_t a = d->ord[i];
        if (d->val[a] >= mx / 10.0) d->ord[m++] = a;
        else { d->in[a] = 0; d->val[a] = 0.0; }
    }
    d->n = m;
}

static void pd_swap(pdict *a, pdict *b) { pdict t = *a; *a = *b; *b = t; }

/* Returns number of output alleles (>= 0) or a negative error:
 *   -2  KeyError in the SQUAREM step (an allele vanished from next_prob's output)
 *   -3  ZeroDivisionError in normalize
 * out_allele/out_prob: result list sorted by probability, descending, stable (common:1408-1409).
 * max_iter/eps reproduce `while diff > 0.0001 and iter < 1000`. */
int em_oracle_single_abundance(int C, int A, const int64_t *off, const int32_t *mem, const double *cnt,
                               const double *len, int remove_low, int32_t *out_allele, double *out_prob,
                               int32_t *out_iters) {
    pdict p, p1, p2;
    pd_init(&p, A); pd_init(&p1, A); pd_init(&p2, A);
    double *r = (double *)malloc((size_t)(A > 0 ? A : 1) * sizeof(double));
    double *v = (double *)malloc((size_t)(A > 0 ? A : 1) * sizeof(double));
    int rc = 0;
    /* initial mass (common:1299-1309) */
    for (int k = 0; k < C; k++) {
        int64_t n = off[k + 1] - off[k];
        for (int64_t j = off[k]; j < off[k + 1]; j++) {
            pd_touch(&p, mem[j]);
            p.val[mem[j]] += cnt[k] / (double)n;
        }
    }
    rc = normalize(&p, len);
    double diff = 1.0;
    int iter = 0;
    while (rc == 0 && diff > 0.0001 && iter < 1000) {
        if ((rc = next_prob(C, off, mem, cnt, &p, &p1, len)) != 0) break;
        if ((rc = next_prob(C, off, mem, cnt, &p1, &p2, len)) != 0) break;
        double ssr = 0.0, ssv = 0.0;
        for (int32_t i = 0; i < p.n; i++) {
            int32_t a = p.ord[i];
            if (!p1.in[a] || !p2.in[a]) { rc = -2; break; }
            r[a] = p1.val[a] - p.val[a];
            ssr += r[a] * r[a];
            v[a] = p2.val[a] - p1.val[a] - r[a];
            ssv += v[a] * v[a];
        }
        if (rc) break;
        if (ssv > 0.0) {
            double g = -sqrt(ssr / ssv);
            for (int32_t i = 0; i < p.n; i++) {
                int32_t a = p.ord[i];
                double x = p.val[a] - 2 * g * r[a] + g * g * v[a];
                p2.val[a] = x > 0.0 ? x : 0.0; /* max(0.0, x) */
            }
            if ((rc = next_prob(C, off, mem, cnt, &p2, &p1, len)) != 0) break;
        }
        diff = 0.0;
        for (int32_t i = 0; i < p.n; i++) {
            int32_t a = p.ord[i];
            if (p1.in[a]) diff += fabs(p.val[a] - p1.val[a]);
            else diff += p.val[a];
        }
        pd_swap(&p, &p1);
        if (iter >= 10 && remove_low) select_alleles(&p);
        iter++;
    }
    int n_out = 0;
    if (rc == 0) {
        if (remove_low) select_alleles(&p);
        rc = normalize(&p, len);
    }
    if (rc == 0) {
        /* stable insertion sort by prob descending */
        n_out = p.n;
        for (int32_t i = 0; i < p.n; i++) { out_allele[i] = p.ord[i]; out_prob[i] = p.val[p.ord[i]]; }
        /* merge sort would be nicer; n is small after pruning, but keep O(n log n) for big A */
        int32_t *idx = (int32_t *)malloc((size_t)(n_out > 0 ? n_out : 1) * sizeof(int32_t));
        int32_t *tmp = (int32_t *)malloc((size_t)(n_out > 0 ? n_out : 1) * sizeof(int32_t));
        for (int32_t i = 0; i < n_out; i++) idx[i] = i;
        for (int32_t w = 1; w < n_out; w *= 2) {
            for (int32_t lo = 0; lo < n_out; lo += 2 * w) {
                int32_t mid = lo + w < n_out ? lo + w : n_out, hi = lo + 2 * w < n_out ? lo + 2 * w : n_out;
                int32_t i = lo, j = mid, k = lo;
                while (i < mid && j < hi) tmp[k++] = (out_prob[idx[j]] > out_prob[idx[i]]) ? idx[j++] : idx[i++];
                while (i < mid) tmp[k++] = idx[i++];
                while (j < hi) tmp[k++] = idx[j++];
            }
            memcpy(idx, tmp, (size_t)n_out * sizeof(int32_t));
        }
        for (int32_t i = 0; i < n_out; i++) { tmp[i] = out_allele[idx[i]]; }
        double *pv = (double *)malloc((size_t)(n_out > 0 ? n_out : 1) * sizeof(double));
        for (int32_t i = 0; i < n_out; i++) pv[i] = out_prob[idx[i]];
        for (int32_t i = 0; i < n_out; i++) { out_allele[i] = tmp[i]; out_prob[i] = pv[i]; }
        free(pv); free(idx); free(tmp);
    }
    if (out_iters) *out_iters = iter;
    pd_free(&p); pd_free(&p1); pd_free(&p2); free(r); free(v);
    return rc ? rc : n_out;
}

/* One EM iteration's worth of work for timing (3 next_prob passes over the class table), used by the
 * cpu_baseline leg of bench.py on inputs whose convergence would otherwise end after a few iterations. */
int em_oracle_iterations(int C, int A, const int64_t *off, const int32_t *mem, const double *cnt, const double *len,
                         int n_iters, double *checksum) {
    pdict p, q;
    pd_init(&p, A); pd_init(&q, A);
    for (int k = 0; k < C; k++) {
        int64_t n = off[k + 1] - off[k];
        for (int64_t j = off[k]; j < off[k + 1]; j++) { pd_touch(&p, mem[j]); p.val[mem[j]] += cnt[k] / (double)n; }
    }
    int rc = normalize(&p, len);
    for (int it = 0; it < 3 * n_iters && rc == 0; it++) {
        rc = next_prob(C, off, mem, cnt, &p, &q, len);
        pd_swap(&p, &q);
    }
    double s = 0.0;
    for (int32_t i = 0; i < p.n; i++) s += p.val[p.ord[i]] * (double)(i + 1);
    if (checksum) *checksum = s;
    pd_free(&p); pd_free(&q);
    return rc;
}

"""Every execution form of the EM kernel (csrc/em.cu) against the C oracle (oracle/em_oracle.c), at the sizes where the
form changes.  hgt_em_form reports the form the host chooses (allele-compacted one-CTA layout, one streaming CTA, or a
cooperative grid), its register width NA and slab size; every case asserts the form it was built for, so a changed
threshold fails here instead of quietly moving the case to another form.  The two choices the kernel makes from the
data are restated from the query and the matrix: sparse or dense compacted matrix (non-zero 32-bit words against
slab_bytes, em_compact_build) and whether the <= 64-key loop ran (the EM phase trace, hgt_em_trace).

Each run must give the oracle's status (OK / KeyError / ZeroDivisionError), iteration count and ranked alleles (ties
included) with abundances within rel 1e-6 / abs 1e-12, and keep the invariants: finite prob, prob == 0 off the result,
key probabilities summing to 1, first_class < C for every key.  Lines starting with EMFORM report the form of each run
(pytest -s).  The oracle cross-check on the status cases runs without a GPU."""
import ctypes
import math

import numpy as np
import pytest

import em_oracle
import hgt_oracle as O

gpu = pytest.mark.gpu

REL, ABS = 1e-6, 1e-12  # contract tolerance of the EM abundances (BASELINE.json)
OK, KEY, ZERODIV = 0, -2, -3
STATUS_EXC = {KEY: KeyError, ZERODIV: ZeroDivisionError}
COMPACT, STREAM, COOP = 0, 1, 2
FORM_NAME = {COMPACT: "compact", STREAM: "stream", COOP: "coop"}


def allele_names(A):
    return ["A*%03d:%03d" % (i // 40 + 1, i % 40 + 1) for i in range(A)]  # name order == index order


class Problem:
    """Class matrix member[C][A] (rows distinct, no empty row, columns ascending = the key's name order), counts,
    optional lengths.  Columns that no class holds are alleles outside Gene_cmpt (wide A with few live alleles)."""

    def __init__(self, member, cnt, lengths=None, remove_low=False, label=""):
        self.member = np.asarray(member, bool)
        self.cnt = np.asarray(cnt, np.float64)
        self.C, self.A = self.member.shape
        self.ln = None if lengths is None else np.asarray(lengths, np.float64)
        self.remove_low = bool(remove_low)
        self.label = label

    @property
    def wp(self):
        return max(2, ((self.A + 63) // 64 + 1) & ~1)

    def bits(self, wp=None):
        wp = wp or self.wp
        pad = np.zeros((self.C, wp * 64), bool)
        pad[:, :self.A] = self.member
        return np.packbits(pad, axis=1, bitorder="little").view(np.uint64)

    def cmpt(self):
        names = allele_names(self.A)
        return {"-".join(names[a] for a in np.nonzero(row)[0]): c for row, c in zip(self.member, self.cnt)}

    def lengths_dict(self):
        names = allele_names(self.A)
        return {} if self.ln is None else {names[a]: float(self.ln[a]) for a in range(self.A)}


def make_problem(seed, A, C, groups=None, density=None, dense_frac=0.05, live=None, remove_low=False, lengths=False,
                 label=""):
    """random_problem of test_gpu_em.py on a matrix: classes are subsets of one allele group around a true allele (plus
    a few dense ones).  density = fraction of the group in a class (default uniform 0.05-0.9), live = number of columns
    that may be members (spread over the whole width).  Identical rows are merged like dict keys (counts added)."""
    rng = np.random.default_rng(seed)
    cols = np.arange(A) if live is None else np.sort(rng.choice(A, live, replace=False))
    n = cols.size
    groups = groups or max(1, n // 100)
    gsize = max(1, n // groups)
    truth = rng.choice(n, size=min(2, n), replace=False)
    seen, rows, cnt = {}, [], []
    for _ in range(60 * C):
        if len(rows) == C:
            break
        m = np.zeros(n, bool)
        if rng.random() < dense_frac:
            m = rng.random(n) < 0.5
        else:
            t = truth[rng.integers(0, truth.size)] if rng.random() < 0.7 else int(rng.integers(0, n))
            g0 = (t // gsize) * gsize
            hi = min(n, g0 + gsize)
            m[g0:hi] = rng.random(hi - g0) < (density if density is not None else rng.uniform(0.05, 0.9))
            m[t] = True
        if not m.any():
            continue
        c = int(rng.integers(1, 40))
        key = np.packbits(m).tobytes()
        if key in seen:
            cnt[seen[key]] += c
            continue
        seen[key] = len(rows)
        rows.append(m)
        cnt.append(c)
    member = np.zeros((len(rows), A), bool)
    member[:, cols] = np.asarray(rows)
    ln = 3000.0 + rng.integers(0, 600, A) if lengths else None
    return Problem(member, cnt, ln, remove_low, label)


def with_twins(pb, twins):
    """Column b := column a (identical membership) for every (a, b): the twins must tie bit for bit."""
    m = pb.member.copy()
    for a, b in twins:
        m[:, b] = m[:, a]
    ln = None if pb.ln is None else pb.ln.copy()
    if ln is not None:
        for a, b in twins:
            ln[b] = ln[a]
    return Problem(m, pb.cnt, ln, pb.remove_low, pb.label + "+twins")


# ---- status problems: the reference raises, or keeps zero-probability keys ---------------------------------------------
def status_zero_counts(pb):
    """Every count 0: ZeroDivisionError in the initial normalize."""
    return Problem(pb.member, np.zeros(pb.C), pb.ln, pb.remove_low, pb.label + "+zero_counts")


def _free_column(pb, skip=0):
    free = np.nonzero(~pb.member.any(axis=0))[0]
    assert free.size > skip, "no allele outside the classes to add"
    return int(free[skip])


def status_key_error(pb):
    """A class {X} with count 0 where X is in no other class: X keeps mass 0, no next_prob() output holds it, and the
    first SQUAREM step raises KeyError."""
    x = _free_column(pb)
    row = np.zeros((1, pb.A), bool)
    row[0, x] = True
    return Problem(np.vstack([pb.member, row]), np.append(pb.cnt, 0.0), pb.ln, pb.remove_low, pb.label + "+key_error")


def status_zero_keys(pb):
    """Zero-count classes that hold positive alleles and two new alleles: no error, the new alleles stay keys with
    probability 0 (ranked after the others by dict order) unless remove_low prunes them."""
    x, y = _free_column(pb, 0), _free_column(pb, 1)
    top = int(np.argmax(pb.cnt @ pb.member))  # the allele with the most reads keeps a positive mass
    rows = np.zeros((2, pb.A), bool)
    rows[0, [top, x]] = True
    rows[1, [top, x, y]] = True
    return Problem(np.vstack([pb.member, rows]), np.append(pb.cnt, [0.0, 0.0]), pb.ln, pb.remove_low,
                   pb.label + "+zero_keys")


STATUS_MAKERS = [status_zero_counts, status_key_error, status_zero_keys]


# ---- oracles ------------------------------------------------------------------------------------------------------------
def c_oracle(pb):
    """(status, iters, ranked allele indices, probabilities) of oracle/em_oracle.c."""
    off = np.zeros(pb.C + 1, np.int64)
    off[1:] = np.cumsum(pb.member.sum(axis=1))
    mem = np.nonzero(pb.member)[1].astype(np.int32)  # row-major: ascending inside each class
    out_a = np.zeros(max(pb.A, 1), np.int32)
    out_p = np.zeros(max(pb.A, 1), np.float64)
    it = ctypes.c_int32(0)
    p = em_oracle._p
    n = em_oracle.lib().em_oracle_single_abundance(
        ctypes.c_int(pb.C), ctypes.c_int(pb.A), p(off, ctypes.c_int64), p(mem, ctypes.c_int32), p(pb.cnt, ctypes.c_double),
        p(pb.ln, ctypes.c_double), ctypes.c_int(int(pb.remove_low)), p(out_a, ctypes.c_int32), p(out_p, ctypes.c_double),
        ctypes.byref(it))
    if n < 0:
        return n, it.value, None, None
    return OK, it.value, out_a[:n].copy(), out_p[:n].copy()


def py_oracle(pb):
    """(status, iters, ranked allele indices, probabilities) of the literal dict form (hgt_oracle.single_abundance)."""
    index = {nm: i for i, nm in enumerate(allele_names(pb.A))}
    try:
        res, it = O.single_abundance(pb.cmpt(), pb.remove_low, pb.lengths_dict())
    except KeyError:
        return KEY, None, None, None
    except ZeroDivisionError:
        return ZERODIV, None, None, None
    return OK, it, np.asarray([index[a] for a, _ in res], np.int32), np.asarray([p for _, p in res])


def assert_same_result(got, want, what):
    st, it, order, prob = got
    wst, wit, worder, wprob = want
    assert st == wst, "%s: status %d, oracle %d" % (what, st, wst)
    if wit is not None and it is not None:
        assert it == wit, "%s: %d iterations, oracle %d" % (what, it, wit)
    if st != OK:
        return
    assert order.tolist() == worder.tolist(), "%s: ranking differs" % what
    np.testing.assert_allclose(prob, wprob, rtol=REL, atol=ABS, err_msg=what)


def assert_zero_keys(base, res):
    """The two alleles status_zero_keys adds to `base` are keys of probability 0, in dict order (x before y)."""
    x, y = _free_column(base, 0), _free_column(base, 1)
    order = res[2].tolist()
    assert x in order and y in order and order.index(x) < order.index(y)
    assert res[3][order.index(x)] == 0.0 and res[3][order.index(y)] == 0.0


# ---- CPU: the C oracle against the literal dict form ----------------------------------------------------------------------
def _small(seed, remove_low, lengths):
    return make_problem(seed, 60, 25, groups=3, live=50, remove_low=remove_low, lengths=lengths, label="small")


@pytest.mark.parametrize("maker", [None] + STATUS_MAKERS, ids=lambda m: "plain" if m is None else m.__name__)
@pytest.mark.parametrize("remove_low", [False, True])
@pytest.mark.parametrize("lengths", [False, True])
def test_c_oracle_matches_dict_form_on_status_cases(maker, remove_low, lengths):
    pb = _small(3, remove_low, lengths)
    if maker is not None:
        pb = maker(pb)
    want = py_oracle(pb)
    assert_same_result(c_oracle(pb), want, pb.label)
    if maker is status_zero_keys and not remove_low:
        assert_zero_keys(_small(3, remove_low, lengths), want)


def test_c_oracle_empty_table_with_lengths():
    """An empty Gene_cmpt with Gene_length: the dict form divides by nothing and returns [] after one iteration; the C
    restatement used to raise ZeroDivisionError from normalize_len's total == 0."""
    assert O.single_abundance({}, True, {"A*01:01": 3000.0}) == ([], 1)
    assert em_oracle.single_abundance({}, True, {"A*01:01": 3000.0}) == ([], 1)
    assert em_oracle.single_abundance({}, False, {}) == ([], 1)


# ---- GPU runs ------------------------------------------------------------------------------------------------------------
def _torch_dev():
    import torch
    from hisatgenotype_b200 import _lib
    return torch, torch.device("cuda", _lib.default_device())


def sm_count():
    from hisatgenotype_b200 import _lib
    return int(_lib.lib().hgt_sm_count(_lib.ctx()))


def query(pb, n_ctas, n_problems=1):
    from hisatgenotype_b200 import _lib
    return _lib.em_form(pb.C, pb.A, pb.wp, pb.ln is not None, n_ctas, pb.A, n_problems)


def trace(enable):
    """hgt_em_trace: switches the EM phase counters; returns the 16 counters gathered since the last call."""
    from hisatgenotype_b200 import _lib
    out = (ctypes.c_uint64 * 16)()
    _lib.check(_lib.lib().hgt_em_trace(_lib.ctx(), int(enable), out))
    return list(out)


def run_dev(pb, n_ctas, with_trace=False):
    """hgt_em_dev on device tensors: (status, iters, ranked indices, probabilities), raw arrays, trace counters."""
    from hisatgenotype_b200 import _lib
    from hisatgenotype_b200.typing_common import rank_result
    torch, dev = _torch_dev()
    L, c = _lib.lib(), _lib.ctx()
    bits = torch.from_numpy(pb.bits().view(np.int64).reshape(-1).copy()).to(dev)
    cnt = torch.from_numpy(pb.cnt).to(dev)
    ln = None if pb.ln is None else torch.from_numpy(pb.ln).to(dev)
    prob = torch.full((pb.A,), -1.0, dtype=torch.float64, device=dev)
    inres = torch.full((pb.A,), 7, dtype=torch.uint8, device=dev)
    fk = torch.full((pb.A,), -5, dtype=torch.int32, device=dev)
    ist = torch.full((3,), -77, dtype=torch.int32, device=dev)
    ws = torch.zeros(L.hgt_em_workspace_bytes(c, pb.C, pb.A), dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    if with_trace:
        trace(1)
    _lib.check(L.hgt_em_dev(c, st, bits.data_ptr(), cnt.data_ptr(), pb.C, pb.A, pb.wp, None if ln is None else ln.data_ptr(),
                            int(pb.remove_low), 0, int(n_ctas), prob.data_ptr(), inres.data_ptr(), fk.data_ptr(),
                            ist.data_ptr(), ws.data_ptr()))
    torch.cuda.synchronize(dev)
    tr = trace(0) if with_trace else None
    it, status, _ = ist.tolist()
    p, ir, f = prob.cpu().numpy(), inres.cpu().numpy(), fk.cpu().numpy()
    if status != OK:
        return (status, it, None, None), (p, ir, f), tr
    assert set(np.unique(ir).tolist()) <= {0, 1}
    check_invariants(pb, p, ir, f)
    ranked = rank_result(list(range(pb.A)), p, ir, f)
    return (OK, it, np.asarray([a for a, _ in ranked], np.int32), np.asarray([x for _, x in ranked])), (p, ir, f), tr


def check_invariants(pb, prob, inres, fk):
    assert np.isfinite(prob).all()
    assert (prob[inres == 0] == 0.0).all()
    keys = np.nonzero(inres)[0]
    if keys.size:
        assert abs(math.fsum(prob[keys].tolist()) - 1.0) <= 1e-12
        assert (fk[keys] >= 0).all() and (fk[keys] < pb.C).all()


def compacted_sparse(pb, form):
    """em_compact_build's choice for an allele-compacted problem: True = sparse rows (16 bytes per non-zero 32-bit word
    plus the row / column index fit slab_bytes), False = dense slab."""
    live = pb.member[:, pb.member.any(axis=0)]
    if form.merge:  # identical columns collapse to one representative
        # np.unique orders the representatives differently from the kernel, which can move the count of non-zero 32-bit
        # words a little: only densities far from the threshold (the 0.5 and 0.001 cases below) decide reliably
        live = np.unique(live, axis=1)
    an = live.shape[1]
    wpc = max(2, ((an + 63) // 64 + 1) & ~1)
    wq, nb = 2 * wpc, (pb.C + 31) // 32
    pad = np.zeros((pb.C, wpc * 64), bool)
    pad[:, :an] = live
    words = np.packbits(pad, axis=1, bitorder="little").view(np.uint32)
    nnzw = int((words != 0).sum())
    fixed = ((pb.C + 1) + (wq + 1) + 2 * wq * nb) * 4
    need = ((fixed + 15) & ~15) + nnzw * 16 + 32
    return fixed + 64 <= form.slab_bytes and need <= form.slab_bytes and pb.C <= 65535


def describe(pb, n_ctas, f):
    per = -(-pb.C // f.grid)
    text = "EMFORM %-28s C=%-5d A=%-5d len=%d rl=%d n_ctas=%-3d -> %s grid=%d na=%d slab_rows=%d" % (
        pb.label, pb.C, pb.A, pb.ln is not None, pb.remove_low, n_ctas, FORM_NAME[f.form], f.grid, f.na, f.slab_rows)
    if f.form == COMPACT:
        text += " %s merge=%d" % ("sparse" if compacted_sparse(pb, f) else "dense", f.merge)
    else:
        text += " rows/cta=%d %s" % (per, "resident" if per <= f.slab_rows else "streamed x%d" % -(-per // f.slab_rows))
        if f.form == COOP:
            text += " empty_ctas=%d" % (f.grid - -(-pb.C // per))
    return text


def max_slab_rows(A):
    """Rows of one streaming slab at A alleles when the rows do not fit (the query on a tall matrix)."""
    return query(Problem(np.ones((1000, A), bool), np.ones(1000)), 1).slab_rows


def n_ctas_list():
    return [0, 1, 2, 3, sm_count()]


def expect_na(A):
    return next(n for n in (1, 2, 4, 8, 16) if n * 1024 >= max(2, ((A + 63) // 64 + 1) & ~1) * 64)


def run_forms(pb, designed, n_list=None, tie=(), collapse=None):
    """Runs pb through hgt_em_dev for every n_ctas of n_list (default 0, 1, 2, 3, SM count) against the C oracle.
    designed = {n_ctas: form} the case was built for (asserted); collapse = {n_ctas: expected <= 64-key loop}."""
    want = c_oracle(pb)
    if pb.C <= 60 and pb.A <= 300:
        assert_same_result(py_oracle(pb), want, pb.label + " dict form")
    sm = sm_count()
    seen = set()
    for n in n_list or n_ctas_list():
        f = query(pb, n)
        print(describe(pb, n, f))
        seen.add(FORM_NAME[f.form])
        if n in designed:
            assert FORM_NAME[f.form] == designed[n], describe(pb, n, f)
        assert f.na == expect_na(pb.A) or f.form == COMPACT
        if n > 1:
            assert f.form == COOP and f.grid == min(n, sm, pb.C) or pb.C == 1 or min(n, sm, pb.C) == 1
        got, (p, ir, fk), tr = run_dev(pb, n, with_trace=collapse is not None and n in collapse)
        assert_same_result(got, want, "%s n_ctas=%d" % (pb.label, n))
        if collapse is not None and n in collapse:
            assert (tr[7] > 0) == collapse[n], "%s n_ctas=%d: <= 64-key loop ran: %s" % (pb.label, n, tr[7] > 0)
        for a, b in tie:
            assert ir[a] == ir[b] and fk[a] == fk[b]
            assert p[a] == p[b], (pb.label, n, a, b, repr(p[a]), repr(p[b]))
    return seen


# ---- 1 + 2: form matrix at the NA boundaries ------------------------------------------------------------------------------
NA_CASES = [  # A, C, groups, designed form at auto G
    (1, 1, 1, "compact"), (2, 3, 1, "compact"), (63, 30, 2, "compact"), (64, 40, 2, "compact"), (65, 40, 2, "compact"),
    (1024, 200, 12, "compact"), (1025, 200, 12, "compact"), (2048, 150, 20, "compact"), (2049, 150, 20, "compact"),
    (4096, 120, 40, "compact"), (4097, 120, 40, "compact"), (8192, 150, 64, "stream"), (8193, 200, 64, "coop"),
]


# Wide problems run here with remove_low (the typing path's setting), narrow ones both ways; without remove_low, wide
# problems are compared on the abundances above a fraction of the top (test_wide_without_remove_low).
NA_RUNS = [c + (rl,) for c in NA_CASES for rl in (False, True) if rl or c[0] <= 65]


@gpu
@pytest.mark.parametrize("lengths", [False, True], ids=["nolen", "len"])
@pytest.mark.parametrize("A,C,groups,form,remove_low", NA_RUNS, ids=["A%d-%s" % (c[0], "rl" if c[4] else "all") for c in NA_RUNS])
def test_na_boundaries_every_grid(A, C, groups, form, remove_low, lengths):
    pb = make_problem(A * 7 + C, A, C, groups=groups, remove_low=remove_low, lengths=lengths, label="na_A%d" % A)
    seen = run_forms(pb, {0: form})
    if pb.C > 1:
        assert "coop" in seen


HEAD = 1e-3  # fraction of the top abundance above which a wide problem without remove_low is compared in full


def assert_same_head(got, want, what):
    """Comparison for a wide problem without remove_low: the same status and iteration count, and the oracle's alleles
    at >= HEAD x its top abundance ranked identically at the top of the kernel's list, within the contract tolerance.
    Returns (alleles compared, tail alleles outside the contract tolerance, whole ranking identical)."""
    st, it, order, prob = got
    wst, wit, worder, wprob = want
    assert st == wst == OK and it == wit, "%s: status %d / %d, iterations %d / %d" % (what, st, wst, it, wit)
    k = int((wprob >= HEAD * wprob[0]).sum())
    assert order[:k].tolist() == worder[:k].tolist(), "%s: ranking of the top %d alleles differs" % (what, k)
    np.testing.assert_allclose(prob[:k], wprob[:k], rtol=REL, atol=ABS, err_msg=what)
    mine = dict(zip(order.tolist(), prob.tolist()))
    off = sum(1 for a, q in zip(worder[k:].tolist(), wprob[k:].tolist())
              if abs(mine.get(a, 0.0) - q) > ABS + REL * abs(q))
    return k, off, order.tolist() == worder.tolist()


@gpu
@pytest.mark.parametrize("A,C,groups,form,lengths", [(4096, 120, 40, "compact", False), (8193, 200, 64, "coop", True)],
                         ids=["A4096-nolen", "A8193-len"])
def test_wide_without_remove_low(A, C, groups, form, lengths):
    """Wide problems without remove_low keep thousands of alleles that decay towards 0.  SQUAREM's max(0, x) decides on
    last-bit differences which of them reach exactly 0 (zero then stays zero), and the kernel sums in another order than
    the oracle, so values far below the top abundance and their ranks may differ beyond 1e-6 (these two shapes did, on
    some grids).  The abundances that matter must not: the alleles above HEAD x the top are compared in full, on every
    grid.  The EMFORM line counts the tail alleles outside the contract tolerance."""
    pb = make_problem(A * 7 + C, A, C, groups=groups, remove_low=False, lengths=lengths, label="wide_all_A%d" % A)
    want = c_oracle(pb)
    assert want[0] == OK and want[2].size > 1000
    for n in n_ctas_list():
        f = query(pb, n)
        if n == 0:
            assert FORM_NAME[f.form] == form
        got, _, _ = run_dev(pb, n)
        k, off, same = assert_same_head(got, want, "%s n_ctas=%d" % (pb.label, n))
        print("%s head=%d of %d tail_outside_tolerance=%d whole_ranking_identical=%d" % (
            describe(pb, n, f), k, want[2].size, off, same))


@gpu
@pytest.mark.parametrize("remove_low,lengths", [(True, False), (True, True)])
def test_na16_widest(remove_low, lengths):
    """A = 16,384 (16 slots per thread): one streaming CTA over several slabs, and cooperative."""
    pb = make_problem(16384, 16384, 100, groups=128, remove_low=remove_low, lengths=lengths, label="na_A16384")
    run_forms(pb, {0: "coop", 1: "stream"}, n_list=[0, 1, 3])
    f = query(pb, 1)
    assert f.na == 16 and pb.C > f.slab_rows


@gpu
def test_too_many_alleles_refused_before_launch():
    from hisatgenotype_b200 import _lib
    torch, dev = _torch_dev()
    L, c = _lib.lib(), _lib.ctx()
    A, C = 16385, 3
    wp = _lib.row_pitch(A)
    with pytest.raises(_lib.HgtError) as e:
        _lib.em_form(C, A, wp, False, 0, A, 1)
    assert e.value.code == _lib.HGT_ERR_UNSUPPORTED
    bits = torch.zeros(C * wp, dtype=torch.int64, device=dev)
    cnt = torch.ones(C, dtype=torch.float64, device=dev)
    out = torch.zeros(A, dtype=torch.float64, device=dev)
    b8 = torch.zeros(A, dtype=torch.uint8, device=dev)
    i32 = torch.zeros(A, dtype=torch.int32, device=dev)
    ws = torch.zeros(L.hgt_em_workspace_bytes(c, C, A), dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    for n in (0, 1, 2):
        l0 = L.hgt_launch_count(c)
        rc = L.hgt_em_dev(c, st, bits.data_ptr(), cnt.data_ptr(), C, A, wp, None, 0, 0, n, out.data_ptr(), b8.data_ptr(),
                          i32.data_ptr(), i32.data_ptr(), ws.data_ptr())
        assert rc == _lib.HGT_ERR_UNSUPPORTED and L.hgt_launch_count(c) == l0


# ---- slab boundaries of the streaming forms -------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("k,d", [(1, -1), (1, 0), (1, 1), (2, -1), (2, 0), (2, 1)])
def test_streaming_slab_boundaries(k, d):
    """One streaming CTA at C = k * slab_rows + d (rows resident, a last slab of one row, full slabs), and cooperative
    grids of 2 / 3 CTAs on the same rows (2 CTAs stream their halves once C > 2 * slab_rows)."""
    A = 8192
    rows = max_slab_rows(A)
    C = k * rows + d
    pb = make_problem(A + C, A, C, groups=64, remove_low=True, label="slab_k%d%+d" % (k, d))
    assert pb.C == C
    f = query(pb, 1)
    assert f.form == STREAM and f.slab_rows == rows
    run_forms(pb, {1: "stream", 2: "coop", 3: "coop"}, n_list=[1, 2, 3])
    streamed_pair = -(-C // 2) > query(pb, 2).slab_rows
    assert streamed_pair == (C > 2 * rows)


@gpu
def test_auto_grid_picks_streaming_cta_over_two_slabs():
    """A = 8,192, C = 160 (a 160 KB matrix): auto G = 1, not compacted, 158 + 2 rows on a B200 (227 KB opt-in)."""
    pb = make_problem(160, 8192, 160, groups=64, remove_low=True, label="auto_8192x160")
    assert pb.C == 160
    f = query(pb, 0)
    print(describe(pb, 0, f))
    assert f.form == STREAM and f.grid == 1 and pb.C > f.slab_rows
    run_forms(pb, {0: "stream"}, n_list=[0])


@gpu
def test_cooperative_grids_with_empty_ctas():
    """C = G + 1 ... 2G - 1: trailing CTAs own no rows, yet take part in every grid sync and the exit decisions."""
    sm = sm_count()
    for C, n, empty in ((3, 2, 0), (4, 3, 1), (5, 3, 0), (sm + 1, sm, sm - (sm + 2) // 2), (sm + sm // 2, sm, None),
                        (2 * sm - 1, sm, 0)):
        pb = make_problem(C * 3 + n, 700, C, groups=7, remove_low=C % 2 == 0, label="coop_C%d_G%d" % (C, n))
        assert pb.C == C
        f = query(pb, n)
        per = -(-C // f.grid)
        assert f.form == COOP and f.grid == n
        if empty is not None:
            assert f.grid - -(-C // per) == empty
        run_forms(pb, {n: "coop"}, n_list=[n])


@gpu
def test_cooperative_streamed_per_cta():
    """All SMs, more rows per CTA than a slab holds (A = 16,384: 46 rows on a B200)."""
    sm = sm_count()
    A = 16384
    C = sm * (max_slab_rows(A) + 4)
    pb = make_problem(C, A, C, groups=256, density=0.05, dense_frac=0.0, remove_low=True, label="coop_streamed")
    f = query(pb, 0)
    assert f.form == COOP and f.grid == sm and -(-pb.C // sm) > f.slab_rows
    run_forms(pb, {0: "coop"}, n_list=[0])


# ---- compacted: dense slab fallback and the merge limits --------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("density,sparse", [(0.5, False), (0.001, True)])
@pytest.mark.parametrize("lengths", [False, True], ids=["nolen", "len"])
def test_compacted_dense_and_sparse(density, sparse, lengths):
    pb = make_problem(int(density * 1000) + 5, 1000, 1200, groups=1, density=density, dense_frac=0.0, lengths=lengths,
                      remove_low=True, label="compact_d%g" % density)
    if not sparse:
        assert pb.C == 1200
    f = query(pb, 0)
    assert f.form == COMPACT
    assert compacted_sparse(pb, f) == sparse
    run_forms(pb, {0: "compact", 1: "compact"}, n_list=[0, 1, 2])


@gpu
@pytest.mark.parametrize("A,merge", [(6000, True), (6145, False), (7000, False), (8193, False)])
def test_compacted_merge_limits(A, merge):
    """Identical columns merge up to 6,144 live alleles and 128 words per row; twins tie exactly either way."""
    C = 100 if A < 8000 else 60
    pb = with_twins(make_problem(A + 1, A, C, groups=60, remove_low=True, label="merge_A%d" % A), [(5, 150), (70, 71), (33, A - 1)])
    f = query(pb, 0)
    assert f.form == COMPACT and bool(f.merge) == merge
    run_forms(pb, {0: "compact"}, n_list=[0, 1, 3], tie=[(5, 150), (70, 71), (33, A - 1)])


# ---- the <= 64-key loop entered from the streaming form ----------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("live", [63, 64, 65])
def test_streaming_collapse_at_iteration_zero(live):
    """63 / 64 / 65 live alleles spread over A = 8,192: one streaming CTA collapses to the 64-key loop at iteration 0
    iff at most 64 alleles are keys; cooperative grids never do."""
    pb = make_problem(live, 8192, 200, live=live, groups=4, label="collapse_live%d" % live)
    f = query(pb, 1)
    assert f.form == STREAM and f.collapse
    n_live = int(pb.member.any(axis=0).sum())  # every allele of a class is a key after the initial normalize
    run_forms(pb, {1: "stream", 3: "coop"}, n_list=[1, 3], collapse={1: n_live <= 64, 3: False})


@gpu
def test_streaming_collapse_after_first_prune():
    """remove_low with 400 live alleles: the prune at iteration 10 leaves <= 64 keys and the streaming CTA switches to
    the 64-key loop, then back to the dense vectors for the first-class reload."""
    pb = make_problem(11, 8192, 220, live=400, groups=8, remove_low=True, label="collapse_after_prune")
    _, it, order, _ = c_oracle(pb)
    assert it > 11 and order.size <= 64
    f = query(pb, 1)
    assert f.form == STREAM and f.collapse
    run_forms(pb, {1: "stream"}, n_list=[1, 2], collapse={1: True, 2: False})


# ---- 3: exact ties on every form ------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("A,C,n_list", [(3000, 400, "2,3,sm"), (8192, 200, "1,2,3,sm")])
@pytest.mark.parametrize("lengths", [False, True], ids=["nolen", "len"])
def test_twins_tie_exactly_on_every_form(A, C, n_list, lengths):
    rng = np.random.default_rng(A * 7 + C + lengths)
    member = rng.random((C, A)) < 0.08
    member[:, 0] = True
    twins = [(5, 150), (70, 71), (33, A - 1), (64, 129)]
    for a, b in twins:
        member[:, b] = member[:, a]
    ln = np.full(A, 1000.0) if lengths else None
    pb = Problem(member, rng.integers(1, 40, C), ln, remove_low=True, label="twins_A%d" % A)
    ns = [sm_count() if x == "sm" else int(x) for x in n_list.split(",")]
    designed = {n: ("coop" if n > 1 else "stream") for n in ns}
    run_forms(pb, designed, n_list=ns, tie=twins)


# ---- 4: statuses on every form ----------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("maker", STATUS_MAKERS, ids=lambda m: m.__name__)
@pytest.mark.parametrize("base", ["compact", "stream"])
@pytest.mark.parametrize("lengths", [False, True], ids=["nolen", "len"])
def test_statuses_every_form(maker, base, lengths):
    """Every exit decision of the loop is taken on vectors that every CTA of a cooperative grid computes identically (the
    block sums of the sweep's reduced sums), so all CTAs leave at the same iteration on an error too."""
    from hisatgenotype_b200.typing_common import single_abundance
    if base == "compact":
        base_pb = make_problem(21, 60, 25, groups=2, live=12, lengths=lengths, label="status")
        designed = {0: "compact", 1: "compact", 2: "coop", 3: "coop"}
    else:
        base_pb = make_problem(22, 8192, 200, live=300, groups=6, lengths=lengths, label="status_wide")
        designed = {1: "stream", 2: "coop", 3: "coop"}
    pb = maker(base_pb)
    run_forms(pb, designed)
    want = c_oracle(pb)
    if pb.A <= 300:
        cm, ln = pb.cmpt(), pb.lengths_dict()
        if want[0] == OK:
            res = single_abundance(cm, pb.remove_low, ln)
            assert [a for a, _ in res] == [allele_names(pb.A)[i] for i in want[2]]
        else:
            with pytest.raises(STATUS_EXC[want[0]]):
                single_abundance(cm, pb.remove_low, ln)
    if maker is status_zero_keys:
        assert want[0] == OK
        assert_zero_keys(base_pb, want)
    else:
        assert want[0] == (ZERODIV if maker is status_zero_counts else KEY)


# ---- 5: one batched launch with every NA, both batched forms and the status problems ---------------------------------------
def run_batch(pbs, wp):
    from hisatgenotype_b200 import _lib
    from hisatgenotype_b200.typing_common import rank_result
    bits = np.concatenate([pb.bits(wp) for pb in pbs])
    cnt = np.concatenate([pb.cnt for pb in pbs]).astype(np.int64)
    coff = np.cumsum([0] + [pb.C for pb in pbs]).astype(np.int64)
    aoff = np.cumsum([0] + [pb.A for pb in pbs]).astype(np.int64)
    use_len = any(pb.ln is not None for pb in pbs)
    assert all((pb.ln is not None) == use_len for pb in pbs)
    ln = np.concatenate([pb.ln for pb in pbs]) if use_len else None
    rl = np.asarray([pb.remove_low for pb in pbs], np.uint8)
    At = int(aoff[-1])
    prob, inres, fk = np.zeros(At), np.zeros(At, np.uint8), np.zeros(At, np.int32)
    iters, status = np.zeros(len(pbs), np.int32), np.zeros(len(pbs), np.int32)
    L = _lib.lib()
    l0 = L.hgt_launch_count(_lib.ctx())
    _lib.check(L.hgt_em_batch(_lib.ctx(), len(pbs), _lib.ptr(bits), _lib.ptr(cnt), _lib.ptr(coff), _lib.ptr(aoff), wp,
                              _lib.ptr(ln), _lib.ptr(rl), _lib.ptr(prob), _lib.ptr(inres), _lib.ptr(fk), _lib.ptr(iters),
                              _lib.ptr(status)))
    assert L.hgt_launch_count(_lib.ctx()) - l0 == 1  # one launch, the widest register variant serves every problem
    out = []
    for i, pb in enumerate(pbs):
        s = slice(int(aoff[i]), int(aoff[i + 1]))
        if status[i] != OK:
            out.append(((int(status[i]), int(iters[i]), None, None), None))
            continue
        check_invariants(pb, prob[s], inres[s], fk[s])
        r = rank_result(list(range(pb.A)), prob[s], inres[s], fk[s])
        out.append(((OK, int(iters[i]), np.asarray([a for a, _ in r], np.int32), np.asarray([x for _, x in r])),
                    (prob[s], inres[s], fk[s])))
    return out


@gpu
@pytest.mark.parametrize("lengths", [False, True], ids=["nolen", "len"])
def test_mixed_batched_launch(lengths):
    """One hgt_em_batch launch: problems of every NA, compacted and streaming, and the three status problems between
    them.  Each equals the oracle and its solo hgt_em_dev(n_ctas=1) run: same status, iterations, keys, first classes and
    ranking.  The values are not required to be bit-equal: the batch gives every problem the widest row pitch, which
    turns the column merge off above 128 words (sums of r^2 / m instead of m sums of (r / m)^2) and changes the word
    partition of the streaming row sums; both only move the last bits (bounded by rel 1e-9 below)."""
    from hisatgenotype_b200 import _lib
    pbs = []
    for i, (A, C, g) in enumerate([(60, 25, 3), (1000, 150, 10), (2000, 120, 20), (4000, 100, 40), (8000, 300, 60),
                                   (8000, 60, 60), (16000, 90, 128), (2000, 600, 20)]):
        pbs.append(make_problem(500 + i, A, C, groups=g, remove_low=True, lengths=lengths, label="batch_A%d" % A))
    base = make_problem(77, 300, 40, groups=2, live=12, lengths=lengths, label="batch_status")
    pbs[2:2] = [status_zero_counts(base)]
    pbs[5:5] = [status_key_error(base)]
    pbs.append(status_zero_keys(base))
    wp = max(pb.wp for pb in pbs)
    forms = set()
    for pb in pbs:
        f = _lib.em_form(pb.C, pb.A, wp, pb.ln is not None, 1, pb.A, len(pbs))
        forms.add(FORM_NAME[f.form])
        print(describe(pb, 1, f) + " (batched, wp=%d)" % wp)
    assert forms == {"compact", "stream"}
    got = run_batch(pbs, wp)
    for pb, (res, arrays) in zip(pbs, got):
        want = c_oracle(pb)
        assert_same_result(res, want, pb.label + " batched")
        solo, (p, ir, fk), _ = run_dev(pb, 1)
        assert_same_result(res, solo, pb.label + " batched vs solo")
        if res[0] == OK:
            bp, bir, bfk = arrays
            np.testing.assert_array_equal(bir, ir)
            np.testing.assert_array_equal(bfk, fk)
            np.testing.assert_allclose(bp, p, rtol=1e-9, atol=1e-300)
    # an erroring problem leaves its neighbours alone: the same launch without the status problems
    clean = [pb for pb in pbs if "batch_status" not in pb.label]
    again = run_batch(clean, wp)
    mine = [r for pb, r in zip(pbs, got) if "batch_status" not in pb.label]
    for (r1, a1), (r2, a2) in zip(mine, again):
        assert r1[1] == r2[1]
        np.testing.assert_array_equal(a1[0], a2[0])
        np.testing.assert_array_equal(a1[2], a2[2])


# ---- 6: production plumbing (integer counts, device class counts, class_first keys) --------------------------------------
PLUMB_SEED, PLUMB_A, PLUMB_PAIRS = 116, 7000, 700  # Gene table of 445 classes x 7,000 alleles: 392 KB


@gpu
@pytest.mark.parametrize("n_units", [3, 7])
def test_typing_batch_em_forms(n_units):
    """A synthetic non-hla locus whose Gene table is a 256 KB - 4 MB EM matrix: a batch of <= 6 units runs each unit
    cooperatively on all SMs, one of >= 7 units one streaming CTA per unit in a single launch.  unit_em / unit_calls
    must equal oracle/hgt_oracle.py::locus_abundance.  The Gene table's allele mask holds every allele, so here the
    problems carry A_live_max == A; A_live_max < A (the exon table of an hla locus) is not asserted by this test."""
    from hisatgenotype_b200 import _lib
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.locus import LocusTables
    from helpers import synthetic_case
    args, sam, truth = synthetic_case(PLUMB_SEED, PLUMB_A, L=3000, n_pairs=PLUMB_PAIRS, base="cyp", del_frac=0.08,
                                      n_groups=40, core_vars=70, pool_private=1200)
    ol = O.OracleLocus(*args)
    ref = O.type_locus(ol, sam, simulation=False)
    want = O.locus_abundance(ol, ref, True)
    t = LocusTables(*args)
    batch = TC.Batch([t], TC.make_params(), True)
    for _ in range(n_units):
        batch.add_unit(0, sam)
    L, c = _lib.lib(), _lib.ctx()
    L.hgt_profile_enable(c, 1)
    L.hgt_profile_reset(c)
    batch.run()
    ms, launches = (ctypes.c_double * 8)(), (ctypes.c_int64 * 8)()
    h2d, d2h = ctypes.c_int64(0), ctypes.c_int64(0)
    L.hgt_profile_read(c, ms, launches, ctypes.byref(h2d), ctypes.byref(d2h))
    L.hgt_profile_enable(c, 0)
    C = batch.unit_summary(0)["n_classes"][0]
    assert C == len(ref["tables"]["gene"].cmpt_items(ol))
    assert 256 << 10 < C * t.wp * 8 <= 4 << 20
    f = _lib.em_form(C, t.A, t.wp, False, 1, t.A, n_units)
    assert f.form == STREAM and bool(f.batch_coop) == (n_units <= 6)
    print("EMFORM typing batch of %d units: C=%d A=%d -> %s, first-level EM launches %d" % (
        n_units, C, t.A, "coop" if n_units <= 6 else "batched stream", launches[4]))
    assert launches[4] == (n_units if n_units <= 6 else 1)
    for u in range(n_units):
        for got in (batch.unit_em(u, 0), batch.unit_calls(u)):
            assert [a for a, _ in got] == [a for a, _ in want]
            for (_, x), (_, y) in zip(got, want):
                assert x == pytest.approx(y, rel=REL, abs=ABS)
    batch.close()
    t.close()

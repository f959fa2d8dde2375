"""GPU parity: EM kernel (csrc/em.cu) through the C ABI vs the oracle and the reference goldens."""
import numpy as np
import pytest

from conftest import GOLDEN_NAMES, load_golden

pytestmark = pytest.mark.gpu

REL = 1e-6  # tolerance stated by BASELINE.json north_star for EM abundances


def _check(res, ref):
    assert [a for a, _ in res] == [a for a, _ in ref]
    for (_, p), (_, q) in zip(res, ref):
        assert p == pytest.approx(q, rel=REL, abs=1e-12)


@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_em_matches_reference_goldens(name):
    from hisatgenotype_b200.typing_common import single_abundance
    g = load_golden(name)
    assert g["em_calls"]
    for call in g["em_calls"]:
        res = single_abundance(dict((k, c) for k, c in call["cmpt"]), call["remove_low"], call["lengths"])
        _check(res, call["result"])


def random_problem(rng, A, C, groups, dense_frac=0.05):
    """Class table shaped like Gene_cmpt: classes are subsets of one allele group (+ a few dense ones)."""
    names = ["A*%03d:%03d" % (i // 40 + 1, i % 40 + 1) for i in range(A)]
    gsize = max(1, A // groups)
    cmpt = {}
    truth = rng.choice(A, size=2, replace=False)
    while len(cmpt) < C:
        if rng.random() < dense_frac:
            mem = np.nonzero(rng.random(A) < 0.5)[0]
        else:
            t = truth[rng.integers(0, 2)] if rng.random() < 0.7 else rng.integers(0, A)
            g0 = (t // gsize) * gsize
            pool = np.arange(g0, min(A, g0 + gsize))
            mem = pool[rng.random(pool.size) < rng.uniform(0.05, 0.9)]
            mem = np.union1d(mem, [t])
        if mem.size == 0:
            continue
        key = "-".join(sorted(names[i] for i in mem))
        cmpt[key] = cmpt.get(key, 0) + int(rng.integers(1, 40))
    lengths = {n: int(3000 + rng.integers(0, 600)) for n in names}
    return cmpt, lengths


@pytest.mark.parametrize("A,C,groups,remove_low,use_len", [
    (50, 20, 5, False, False),
    (700, 84, 12, True, False),      # exon-table sized (BASELINE.md: C=84, A=702)
    (800, 300, 20, True, True),
    (2000, 500, 40, False, True),
    (4000, 1500, 60, True, True),
    (8000, 2000, 60, True, True),    # BASELINE.md "EM large"
    (8192, 6000, 64, True, False),   # multi-CTA cooperative path, streaming slabs
    (5000, 6000, 50, True, False),   # cooperative path, last warps without allele words
    (9000, 5000, 60, False, False),  # cooperative path, 16 slots per thread
])
def test_em_matches_c_oracle(A, C, groups, remove_low, use_len):
    import em_oracle
    from hisatgenotype_b200.typing_common import single_abundance
    rng = np.random.default_rng(A * 31 + C)
    cmpt, lengths = random_problem(rng, A, C, groups)
    ln = lengths if use_len else {}
    ref, _ = em_oracle.single_abundance(cmpt, remove_low, ln)
    res = single_abundance(cmpt, remove_low, ln)
    _check(res, ref)


def test_em_iteration_count_and_first_class():
    import em_oracle
    from hisatgenotype_b200 import _lib
    from hisatgenotype_b200.typing_common import _index_alleles, em_arrays
    rng = np.random.default_rng(5)
    cmpt, _ = random_problem(rng, 600, 150, 10)
    keys = list(cmpt)
    names, index = _index_alleles(keys)
    bits = _lib.pack_bits([[index[a] for a in k.split("-")] for k in keys], len(names))
    prob, inres, fk, iters = em_arrays(bits, [cmpt[k] for k in keys], len(names), None, False)
    ref, ref_iters = em_oracle.single_abundance(cmpt, False, {})
    assert iters == ref_iters
    assert int(inres.sum()) == len(ref)
    assert abs(prob.sum() - 1.0) < 1e-9


def test_em_empty_and_single_class():
    from hisatgenotype_b200.typing_common import single_abundance
    assert single_abundance({}) == []
    res = single_abundance({"A*01:01-A*01:02": 7})
    assert [a for a, _ in res] == ["A*01:01", "A*01:02"]
    assert res[0][1] == pytest.approx(0.5) and res[1][1] == pytest.approx(0.5)


def test_em_batch_matches_single():
    from hisatgenotype_b200 import _lib
    from hisatgenotype_b200.typing_common import _index_alleles, em_arrays
    rng = np.random.default_rng(11)
    probs = []
    for i in range(9):
        cmpt, lengths = random_problem(rng, 200 + 50 * i, 40 + 10 * i, 6)
        keys = list(cmpt)
        names, index = _index_alleles(keys)
        probs.append((cmpt, keys, names, index, lengths))
    Amax = max(len(p[2]) for p in probs)
    wp = _lib.row_pitch(Amax)
    bits = np.concatenate(
        [_lib.pack_bits([[p[3][a] for a in k.split("-")] for k in p[1]], len(p[2]), wp) for p in probs])
    cnt = np.concatenate([np.asarray([p[0][k] for k in p[1]], np.int64) for p in probs])
    coff = np.cumsum([0] + [len(p[1]) for p in probs]).astype(np.int64)
    aoff = np.cumsum([0] + [len(p[2]) for p in probs]).astype(np.int64)
    ln = np.concatenate([np.asarray([p[4][n] for n in p[2]], np.float64) for p in probs])
    rl = np.asarray([i % 2 for i in range(len(probs))], np.uint8)
    At = int(aoff[-1])
    prob = np.zeros(At)
    inres = np.zeros(At, np.uint8)
    fk = np.zeros(At, np.int32)
    iters = np.zeros(len(probs), np.int32)
    status = np.zeros(len(probs), np.int32)
    _lib.check(_lib.lib().hgt_em_batch(_lib.ctx(), len(probs), _lib.ptr(bits), _lib.ptr(cnt), _lib.ptr(coff),
                                       _lib.ptr(aoff), wp, _lib.ptr(ln), _lib.ptr(rl), _lib.ptr(prob),
                                       _lib.ptr(inres), _lib.ptr(fk), _lib.ptr(iters), _lib.ptr(status)))
    assert (status == 0).all()
    for i, p in enumerate(probs):
        b1 = _lib.pack_bits([[p[3][a] for a in k.split("-")] for k in p[1]], len(p[2]))
        pr, ir, f, it = em_arrays(b1, [p[0][k] for k in p[1]], len(p[2]), [p[4][n] for n in p[2]], bool(rl[i]))
        s = slice(int(aoff[i]), int(aoff[i + 1]))
        assert it == iters[i]
        np.testing.assert_array_equal(ir, inres[s])
        np.testing.assert_allclose(pr, prob[s], rtol=1e-12, atol=0)
        np.testing.assert_array_equal(f, fk[s])


@pytest.mark.parametrize("use_len", [False, True])
@pytest.mark.parametrize("A,C", [(200, 60), (3000, 400), (8192, 3000)])  # the last one runs on all SMs
def test_em_identical_columns_tie_exactly(A, C, use_len):
    """Alleles that are members of exactly the same classes have EXACTLY equal abundances in the reference (same
    arithmetic on the same numbers, common:1311-1336), and that tie decides their rank.  The kernel must keep the tie
    bit-exact wherever the two alleles sit (different 32-allele words, other alleles of the word present or not), with
    (no lengths) and without (lengths) the column merge, for any order of the class rows."""
    from hisatgenotype_b200 import _lib
    from hisatgenotype_b200.typing_common import em_arrays
    rng = np.random.default_rng(A * 7 + C + (1 if use_len else 0))
    member = rng.random((C, A)) < 0.08
    member[:, 0] = True  # no empty class
    twins = [(5, 150), (70, 71), (33, A - 1), (64, 129)]
    for a, b in twins:
        member[:, b] = member[:, a]
    cnt = rng.integers(1, 40, C).astype(np.int64)
    ln = np.full(A, 1000.0) if use_len else None  # equal lengths keep the twins tied
    first = None
    for trial in range(4):
        order = rng.permutation(C) if trial else np.arange(C)
        bits = _lib.pack_bits([np.nonzero(member[k])[0] for k in order], A)
        prob, inres, fk, iters = em_arrays(bits, cnt[order], A, ln, False)
        for a, b in twins:
            assert inres[a] == inres[b]
            assert prob[a] == prob[b], (trial, a, b, repr(prob[a]), repr(prob[b]))
            assert fk[a] == fk[b]
        if first is None:
            first = prob
        else:
            np.testing.assert_allclose(prob, first, rtol=1e-6, atol=1e-12)  # the row order only moves the last bits (tiny values: SQUAREM cancellation)


@pytest.mark.parametrize("A,C,remove_low,use_len,rel,abs_", [
    pytest.param(700, 300, True, False, 1e-9, 1e-15, id="700-300-True-False"),
    pytest.param(8192, 6000, True, False, 1e-9, 1e-15, id="8192-6000-True-False"),
    pytest.param(3000, 900, False, True, 1e-9, 1e-15, id="3000-900-False-True"),
    # hgt_em runs this shape and 700 x 300 in its one-CTA form, whose sums associate differently from the peer kernel's
    # cooperative sweep.  The pruned 700 x 300 still agrees to 1e-9; here (no pruning, lengths) SQUAREM carries the
    # difference to ~2e-9 relative, so this shape is held to the contract tolerance.
    pytest.param(2000, 500, False, True, REL, 1e-9, id="2000-500-False-True"),
])
def test_peer_kernel_single_rank_equals_hgt_em(A, C, remove_low, use_len, rel, abs_):
    """hgt_em_peer_dev with a world of ONE rank: the exchange step only reads the rank's own block, so the result must
    equal hgt_em (same loop) - iterations, keys, order and values.  The two-rank case needs two GPUs
    (tests/test_gpu_multi.py)."""
    import torch
    from hisatgenotype_b200 import _lib, em_dist
    from hisatgenotype_b200.typing_common import _index_alleles, em_arrays, rank_result
    rng = np.random.default_rng(A + C)
    cmpt, lengths = random_problem(rng, A, C, 30)
    keys = list(cmpt)
    names, index = _index_alleles(keys)
    n = len(names)
    wp = _lib.row_pitch(n)
    bits = _lib.pack_bits([[index[a] for a in k.split("-")] for k in keys], n)
    cnt = np.asarray([cmpt[k] for k in keys], np.int64)
    ln = [lengths[x] for x in names] if use_len else None
    prob, inres, fk, iters = em_arrays(bits, cnt, n, ln, remove_low)
    dev = torch.device("cuda", _lib.default_device())
    d_bits = torch.from_numpy(bits.view(np.int64).reshape(-1)).to(dev)
    d_cnt = torch.from_numpy(cnt).to(dev)
    for rep in range(2):  # the second call continues the block's sequence numbers
        p2, l2, f2, it2 = em_dist.single_abundance_peer(n, wp, d_bits.data_ptr(), d_cnt.data_ptr(), None, 0, len(keys), dev.index,
                                                        ln, remove_low)
        assert it2 == iters
        got = rank_result(names, p2.cpu().numpy(), l2.cpu().numpy().astype(np.uint8), f2.cpu().numpy())
        want = rank_result(names, prob, inres, fk)
        assert [a for a, _ in got] == [a for a, _ in want]
        for (_, x), (_, y) in zip(got, want):
            assert x == pytest.approx(y, rel=rel, abs=abs_)


@pytest.mark.parametrize("A,world", [(300, 2), (7000, 3)])
def test_class_merge_partitions_and_merges(A, world):
    """hgt_class_merge_dev for every rank of a world on the same gathered rows (duplicates inside and across the
    'shards'): the ranks' outputs are disjoint, their union is the merged table (counts added, smallest first index)."""
    import torch
    from hisatgenotype_b200 import _lib, em_dist
    rng = np.random.default_rng(A)
    wp = _lib.row_pitch(A)
    distinct = 500
    base = np.zeros((distinct, wp), np.uint64)
    for r in range(distinct):
        mem = rng.choice(A, size=int(rng.integers(1, 60)), replace=False)
        for a in mem:
            base[r, a >> 6] |= np.uint64(1) << np.uint64(a & 63)
    pick = rng.integers(0, distinct, size=1800)
    rows = base[pick]
    cnt = rng.integers(1, 50, size=pick.size).astype(np.int64)
    first = rng.permutation(pick.size).astype(np.int32)
    want = {}
    for k in range(pick.size):
        key = rows[k].tobytes()
        c, f = want.get(key, (0, 1 << 30))
        want[key] = (c + int(cnt[k]), min(f, int(first[k])))
    dev = torch.device("cuda", _lib.default_device())
    g_bits = torch.from_numpy(rows.view(np.int64).reshape(-1)).to(dev)
    g_cnt = torch.from_numpy(cnt).to(dev)
    g_first = torch.from_numpy(first).to(dev)
    got = {}
    for rank in range(world):
        o_bits, o_cnt, o_first, m = em_dist.merge_rows(g_bits, g_cnt, g_first, pick.size, A, wp, rank, world, dev.index)
        ob = o_bits.cpu().numpy().view(np.uint64).reshape(-1, wp)[:m]
        oc, of = o_cnt.cpu().numpy()[:m], o_first.cpu().numpy()[:m]
        assert m > 0
        for k in range(m):
            key = ob[k].tobytes()
            assert key not in got
            got[key] = (int(oc[k]), int(of[k]))
    assert got == want


def test_single_abundance_fractional_counts_and_unsorted_keys():
    """The reference does float(count) and breaks exact ties by dict insertion order = position inside the key string of the
    first class that holds the allele: fractional counts must not be truncated and keys need not be name-sorted."""
    import em_oracle
    from hisatgenotype_b200.typing_common import single_abundance
    rng = np.random.default_rng(77)
    cmpt, _ = random_problem(rng, 300, 90, 6)
    cmpt = {k: 0.25 * c + 0.5 for k, c in cmpt.items()}  # truncated to integers this would be a different problem
    ref, _ = em_oracle.single_abundance(cmpt, True, {})
    res = single_abundance(cmpt, True, {})
    _check(res, ref)
    trunc = single_abundance({k: int(c) for k, c in cmpt.items() if int(c) > 0}, True, {})
    assert any(abs(p - q) > 1e-4 for (_, p), (_, q) in zip(res, trunc)) or len(res) != len(trunc)
    tie = {"Z*09-A*01": 3}  # exact tie 0.5 / 0.5: the reference lists Z*09 first (it comes first in the key)
    ref, _ = em_oracle.single_abundance(tie, False, {})
    res = single_abundance(tie, False, {})
    assert [a for a, _ in ref] == ["Z*09", "A*01"]
    _check(res, ref)

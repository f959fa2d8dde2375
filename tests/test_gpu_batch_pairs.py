"""Batched diploid pair calls (Batch.pair_calls -> hgt_batch_pairs, csrc/pair_batch.cu) on the class tables a finished batch
keeps on the device, against the Python-3 restatement of the legacy joint_abundance (oracle/joint_oracle.py) and against the
host path typing_common.joint_abundance (hgt_pair_em) on the same dict: same ranked keys, same iterations, p within
1e-6 relative of the oracle and 1e-9 of the host path."""
import ctypes

import numpy as np
import pytest

import joint_oracle as J
from conftest import GOLDEN_NAMES, load_golden
from helpers import golden_db, product_locus, synthetic_case

pytestmark = pytest.mark.gpu


def same_as_host(got, cmpt):
    from hisatgenotype_b200.typing_common import joint_abundance
    g, git = got
    ref, it = joint_abundance(dict(cmpt), return_iters=True)
    if isinstance(ref, dict):
        assert g == ref == {}
    else:
        assert [k for k, _ in g] == [k for k, _ in ref]
        for (_, x), (_, y) in zip(g, ref):
            assert x == pytest.approx(y, rel=1e-9, abs=1e-15)
    assert git == it


def golden_batch(name):
    from hisatgenotype_b200 import typing_core as TC
    g = load_golden(name)
    p = g["params"]
    db = golden_db(g)
    genes = []
    for c in g["loci"]:
        if c["gene"] not in genes:
            genes.append(c["gene"])
    names = {c["gene"]: c["Gene_names"] for c in g["loci"]}
    loci = [product_locus(g, db, gene, names[gene]) for gene in genes]
    b = TC.Batch(loci, TC.make_params(p["num_editdist"], p["error_correction"], p["discordant"], p["simulation"]),
                 p["remove_low"])
    for c in g["loci"]:
        b.add_unit(genes.index(c["gene"]), c["sam"])
    b.run()
    return b, loci


@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_pair_calls_on_golden_units(name):
    b, loci = golden_batch(name)
    for table in (0, 1, 2) if loci[0].is_hla else (0,):
        calls = b.pair_calls(table, return_iters=True)
        for u in range(len(b.unit_locus)):
            cmpt = b.unit_gene_cmpt(u, table)
            got, it = calls[u]
            ref, it_ref = J.joint_abundance(dict(cmpt), None, True)
            if not cmpt:
                assert got == {} and it == 0
                continue
            assert [k for k, _ in got] == [k for k, _ in ref]
            for (_, x), (_, y) in zip(got, ref):
                assert x == pytest.approx(y, rel=1e-6, abs=1e-12)
            assert it == it_ref
            same_as_host(calls[u], cmpt)
            assert b.unit_pair_calls(u, table, return_iters=True) == calls[u]
    b.close()
    for t in loci:
        t.close()


def nested_names(n):
    """n sorted names, groups of four that contain each other: X*g:1 in X*g:10 in X*g:100 in X*g:100X*g:1."""
    out = []
    for g in range((n + 3) // 4):
        p = "X*%04d:" % g
        out += [p + "1", p + "10", p + "100", p + "100" + p + "1"]
    return sorted(out[:n])


_SYN = {}


def synthetic_batch():
    """4 loci (one of 2,100 alleles, one whose names contain each other), 40 samples: ragged depth, some empty units."""
    if "b" in _SYN:
        return _SYN["b"], _SYN["loci"], _SYN["units"]
    from hisatgenotype_b200 import synth
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.locus import LocusTables
    specs = [(41, 2100, 3000), (42, 300, 2500), (43, 160, 2000), (44, 120, 1800)]
    loci, sims = [], []
    for seed, A, L in specs:
        loc = synth.make_locus("A", seed, L=L, n_alleles=A, n_groups=12, core_vars=50, pool_private=300, del_frac=0.1)
        cont = synth.reference_containers([loc], "hla")
        loci.append(LocusTables("hla", "A", cont["refGenes"]["A"], cont["Genes"]["A"][cont["refGenes"]["A"]],
                                cont["Vars"]["A"], cont["Var_list"]["A"], cont["Links"], cont["Gene_names"]["A"],
                                cont["Gene_lengths"]["A"], cont["refGene_loci"]["A"][4], cont["refGene_loci"]["A"][5]))
        sims.append((loc, sorted(n for n in loc.alleles if loc.alleles[n])))
    t = loci[2]
    orig = list(t.names)
    t.names = nested_names(t.A)  # the pair model sees these names (unit_gene_cmpt writes its keys with them too)
    b = TC.Batch(loci, TC.make_params(), True)
    rng = np.random.default_rng(7)
    units = []
    # samples carrying two alleles of one nested group (X*g:1 and X*g:10): their pair contains X*g:1 twice
    live = set(sims[2][1])
    for g in range(len(orig) // 4):
        truth = [orig[4 * g], orig[4 * g + 1]]
        if all(a in live for a in truth):
            units.append(b.add_unit(2, synth.simulate_sam(sims[2][0], truth, n_pairs=300, rng=rng, err_rate=0.002)))
    for s in range(40):
        for li, (loc, names) in enumerate(sims):
            if (s + li) % 11 == 0:
                units.append(b.add_unit(li, b""))
                continue
            truth = [names[i] for i in rng.choice(len(names), 2, replace=False)]
            n_pairs = int(rng.integers(20, 400))
            units.append(b.add_unit(li, synth.simulate_sam(loc, truth, n_pairs=n_pairs, rng=rng, err_rate=0.004)))
    b.run()
    _SYN.update(b=b, loci=loci, units=units)
    return b, loci, units


def test_pair_calls_on_synthetic_batch():
    b, loci, units = synthetic_batch()
    assert len(units) >= 32 * 3 and max(t.A for t in loci) > 2048
    assert any(t.names[0] in t.names[1] for t in loci)
    calls = b.pair_calls(0, return_iters=True)
    n_empty = 0
    for u in units:
        cmpt = b.unit_gene_cmpt(u, 0)
        n_empty += not cmpt
        same_as_host(calls[u], cmpt)
    assert n_empty > 0
    # a pair whose two members contain the same name (the T[x] correction of the loop) is among the results
    t = loci[2]
    off, idx = t.name_subsets()
    sub = [set(idx[off[a]:off[a + 1]].tolist()) for a in range(t.A)]
    r = b.pair_arrays(0)
    shared = [(u, a, c) for u in units if b.unit_locus[u] == 2
              for a, c in zip(r["lo"][u, :r["n_total"][u]].tolist(), r["hi"][u, :r["n_total"][u]].tolist())
              if a != c and sub[a] & sub[c]]
    assert shared
    # the sizes of the loops: the host enumeration's pair count
    for u in units:
        cmpt = b.unit_gene_cmpt(u, 0)
        assert r["n_pairs"][u] == (pair_count(cmpt) if cmpt else 0)


def pair_count(cmpt):
    """pairs that survive the first pruning (the enumeration of typing_common.joint_abundance)"""
    names = sorted({a for k in cmpt for a in k.split("-")})
    index = {n: i for i, n in enumerate(names)}
    m = np.zeros(len(names))
    for k, c in cmpt.items():
        mem = k.split("-")
        for a in mem:
            m[index[a]] += float(c) / len(mem)
    ms = m[np.argsort(-m, kind="stable")]
    best = max(ms[0] + ms[1] if len(ms) >= 2 else ms[0], ms[0])
    return sum(int(not ((ms[i] + ms[j]) * 2 <= best)) for i in range(len(ms)) for j in range(i + 1, len(ms))) + \
        int(np.sum(~(ms * 2 <= best)))


def test_max_pairs_follows_the_host_rule(monkeypatch):
    """The limit is typing_common.joint_abundance's: it tests `total > MAX_PAIRS` after adding a candidate's partners, so
    the pairs (a, a) added after its last test do not count.  Limits just below the largest units' pair counts, where the
    two rules differ, give the same units an error on the device and on the host."""
    from hisatgenotype_b200 import _lib
    from hisatgenotype_b200 import typing_common
    b, loci, units = synthetic_batch()
    full = b.pair_calls(0, return_iters=True)
    q = b.pair_arrays(0)["n_pairs"]
    top = sorted({int(q[u]) for u in units}, reverse=True)[:3]
    limits = sorted({x - d for x in top for d in (1, 2, 3) if x - d >= 1})
    n_err = n_ok_above = 0
    for lim in limits:
        r = b.pair_arrays(0, max_pairs=lim)
        returned = b.pair_calls(0, return_iters=True, max_pairs=lim, errors="return")
        monkeypatch.setattr(typing_common, "MAX_PAIRS", lim)
        for u in units:
            if q[u] <= lim:  # neither rule can refuse the unit
                assert r["status"][u] == 0 and returned[u] == full[u]
                continue
            try:
                typing_common.joint_abundance(b.unit_gene_cmpt(u, 0))
                host_refuses = False
            except _lib.HgtError:
                host_refuses = True
            if host_refuses:
                n_err += 1
                assert r["status"][u] == _lib.HGT_ERR_UNSUPPORTED and r["n_total"][u] == 0
                assert isinstance(returned[u], _lib.HgtError) and returned[u].code == _lib.HGT_ERR_UNSUPPORTED
                with pytest.raises(_lib.HgtError) as e:
                    b.unit_pair_calls(u, 0, max_pairs=lim)
                assert e.value.code == _lib.HGT_ERR_UNSUPPORTED
            else:
                n_ok_above += 1
                assert r["status"][u] == 0 and returned[u] == full[u]
        monkeypatch.undo()
    assert n_err > 0
    with pytest.raises(_lib.HgtError):
        b.pair_calls(0, max_pairs=limits[0])


def test_larger_cap_reads_the_kept_result():
    """The library keeps the complete result: a call with a cap too small for some unit, then the call with a larger cap,
    launch nothing after the first computation."""
    from hisatgenotype_b200 import _lib
    from hisatgenotype_b200.locus import lib
    b, loci, units = synthetic_batch()
    table = max((0, 1), key=lambda t: int(b.pair_arrays(t)["n_total"].max()))
    full = b.pair_arrays(table)
    assert full["n_total"].max() > 1
    other = (1 << 22) - 1  # another key: the next call computes
    L, c = _lib.lib(), _lib.ctx()
    l0 = L.hgt_launch_count(c)
    first = b.pair_arrays(table, max_pairs=other)
    l1 = L.hgt_launch_count(c)
    assert l1 > l0
    nu = len(b.unit_locus)
    lo, hi = np.zeros((nu, 1), np.int32), np.zeros((nu, 1), np.int32)
    p = np.zeros((nu, 1), np.float64)
    n, it, st = (np.zeros(nu, np.int32) for _ in range(3))
    assert lib().hgt_batch_pairs(b.handle, table, other, 1, *[_lib.ptr(x) for x in (lo, hi, p, n, it, st)]) == 0
    assert np.array_equal(n, full["n_total"]) and np.array_equal(p[:, 0], full["prob"][:, 0])
    again = b.pair_arrays(table, max_pairs=other, cap=1)  # a second call with the needed cap
    assert L.hgt_launch_count(c) == l1
    for r in (first, again):
        for k in ("n_total", "iters", "status", "n_pairs"):
            assert np.array_equal(r[k], full[k])
        for u in range(nu):  # ([n_units][cap] arrays of different widths: the rows' filled part)
            m = int(full["n_total"][u])
            for k in ("lo", "hi", "prob"):
                assert np.array_equal(r[k][u, :m], full[k][u, :m])


def _dev_rows(b, u, table, wp):
    cudart = ctypes.CDLL("libcudart.so.12")
    bits, cnt, first, n = b.unit_table_dev(u, table)
    out = []
    for ptr, nb, dt in ((bits, n * wp * 8, np.uint64), (cnt, n * 8, np.uint64), (first, n * 4, np.int32)):
        a = np.zeros(max(nb, 8) // np.dtype(dt).itemsize, dt)
        if nb:
            assert cudart.cudaMemcpy(ctypes.c_void_p(a.ctypes.data), ctypes.c_void_p(ptr), ctypes.c_size_t(nb), 2) == 0
        out.append(a)
    return out


def test_repeatable_and_leaves_batch_unchanged():
    b, loci, units = synthetic_batch()
    some = units[::7]

    def snapshot():
        s = []
        for u in some:
            t = loci[b.unit_locus[u]]
            s.append((b.unit_calls(u), [x.tolist() for x in b.unit_table(u, 0)],
                      [x.tolist() for x in _dev_rows(b, u, 0, t.wp)]))
        return s

    before = snapshot()
    r1 = b.pair_arrays(0)
    r2 = b.pair_arrays(0)
    for k in ("lo", "hi", "prob", "n_total", "iters", "status"):
        assert np.array_equal(r1[k], r2[k])
    assert snapshot() == before


def test_bad_arguments():
    from hisatgenotype_b200 import _lib
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.locus import LocusTables, lib
    args, sam, _ = synthetic_case(5, 60, L=1500, n_pairs=200)
    t = LocusTables(*args)
    b = TC.Batch([t], TC.make_params(), True)
    b.add_unit(0, sam)
    nu = 1
    arr = [np.zeros(4, np.int32), np.zeros(4, np.int32), np.zeros(4, np.float64)] + [np.zeros(1, np.int32) for _ in range(3)]
    ptrs = [_lib.ptr(a) for a in arr]
    b.prepare()
    b.execute()
    assert lib().hgt_batch_pairs(b.handle, 0, 100, 4, *ptrs) == _lib.HGT_ERR_ARG  # not finished
    b.finish()
    assert lib().hgt_batch_pairs(b.handle, 0, 100, 4, *ptrs) == _lib.HGT_ERR_ARG  # no names on the locus
    t.ensure_names()
    assert lib().hgt_batch_pairs(b.handle, 3, 100, 4, *ptrs) == _lib.HGT_ERR_ARG  # the projected table
    assert lib().hgt_batch_pairs(b.handle, -1, 100, 4, *ptrs) == _lib.HGT_ERR_ARG
    assert lib().hgt_batch_pairs(b.handle, 0, 1 << 22, 4, *ptrs) == 0
    assert nu == 1 and arr[5][0] == 0
    b.close()
    t.close()

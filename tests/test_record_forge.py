"""Self-check of the record forge (tests/record_forge.py): error-free forged reads walk, in the oracle, to exactly the
allele's variants inside the read's window, whatever the read length, clips, Zs or insertions."""
import numpy as np
import pytest

import hgt_oracle as O
from record_forge import Forge, window_variants


def _locus(seed, ins_frac):
    from hisatgenotype_b200 import synth
    return synth.make_locus("A", seed, L=1500, n_alleles=40, n_groups=4, core_vars=40, pool_private=120,
                            del_frac=0.25, ins_frac=ins_frac)


@pytest.mark.parametrize("zs", [True, False])
@pytest.mark.parametrize("ins_frac", [0.0, 0.2])
def test_forged_reads_walk_to_their_allele(zs, ins_frac):
    from hisatgenotype_b200 import synth
    loc = _locus(7, ins_frac)
    cont = synth.reference_containers([loc], "hla")
    g = "A"
    ol = O.OracleLocus("hla", g, cont["refGenes"][g], cont["Genes"][g][cont["refGenes"][g]], cont["Vars"][g],
                       cont["Var_list"][g], cont["Links"], cont["Gene_names"][g], cont["Gene_lengths"][g],
                       cont["refGene_loci"][g][4], cont["refGene_loci"][g][5])
    fg = Forge(loc, zs=zs)
    rng = np.random.default_rng(1)
    names = sorted(n for n in loc.alleles if loc.alleles[n])
    L = len(loc.backbone)
    counts, nt_sets = [dict() for _ in range(L)], [[] for _ in range(L)]
    n_ins = n_clip = 0
    for k in range(300):
        a = names[int(rng.integers(0, len(names)))]
        length = int(rng.choice([50, 100, 129, 250]))
        toks = fg.tokens(a)
        nb = sum(1 for t in toks if t[0] != "D")
        while True:
            s = int(rng.integers(0, nb - length))
            cl, cr = int(rng.integers(0, 4)) * (k % 3 == 0), int(rng.integers(0, 4)) * (k % 5 == 0)
            try:
                line, part = fg.record("r%d" % k, a, s, length, flag=0, clip_left=cl, clip_right=cr)
            except AssertionError:
                continue
            break
        rec = O.parse_record(line, False, 0)
        cmp_list, right, ncorr, mis, seq = O.walk_record(ol, rec, counts, nt_sets, False)
        got = [e[3] for e in cmp_list if e[0] != O.MATCH]
        assert got == [loc.var_ids[v] for v in window_variants(part)], line
        assert right == part[-1][1] + (part[-1][2] if part[-1][0] == "D" else 1)
        assert rec.NM == 0 and not mis and len(seq) == length - cl - cr
        n_ins += any(t[0] == "I" for t in part)
        n_clip += cl + cr > 0
    assert n_clip > 0
    if ins_frac:
        assert n_ins > 20

"""Shared helpers for the parity tests."""
import numpy as np

import hgt_oracle as O
from hisatgenotype_b200 import dbio


def golden_db(g):
    return dbio.load_database_text(g["db"])


def oracle_locus(g, db, gene, names):
    locus = db["refGene_loci"][gene]
    return O.OracleLocus(g["params"]["base"], gene, db["refGenes"][gene], db["Genes"][gene][db["refGenes"][gene]],
                         db["Vars"][gene], db["Var_list"][gene], db["Links"], names, db["Gene_lengths"][gene],
                         locus[4], locus[5])


def product_locus(g, db, gene, names, host_only=False):
    from hisatgenotype_b200.locus import LocusTables
    locus = db["refGene_loci"][gene]
    return LocusTables(g["params"]["base"], gene, db["refGenes"][gene], db["Genes"][gene][db["refGenes"][gene]],
                       db["Vars"][gene], db["Var_list"][gene], db["Links"], names, db["Gene_lengths"][gene],
                       locus[4], locus[5], host_only=host_only)


def pileup_arrays(counts, nt_sets):
    """oracle pileup (list of dicts / lists) -> counts[L][6] (A,C,G,T,other,D), nt mask[L]"""
    L = len(counts)
    c = np.zeros((L, 6), np.uint32)
    m = np.zeros(L, np.uint8)
    code = {"A": 0, "C": 1, "G": 2, "T": 3, "D": 5}
    for i, d in enumerate(counts):
        for nt, k in d.items():
            c[i, code.get(nt, 4)] += k
        for nt in nt_sets[i]:
            m[i] |= 1 << "ACGT".index(nt)
    return c, m


def compat_from_rows(loc, left, right, rows, mask):
    """Set form of add_count (SURVEY.md appendix A.5) on integer rows, Python-int bitsets."""
    alleles = loc.all_mask
    own = set(int(r) for r in rows)
    for r in own:
        alleles &= loc.bits[r]
    neg = 0
    for r, (pos, vid) in enumerate(loc.var_list):
        if loc.bits[r] is None or r in own:
            continue
        vr = loc.var_right(vid)
        if left <= pos <= right or left <= vr <= right:
            neg |= loc.bits[r]
    return alleles & ~neg & mask


def tables_from_jobs(loc, walk, hla):
    """Gene_cmpt / Gene_counts from the flattened job lists of hgt_host_walk, in the reference's dict orders."""
    masks = [loc.all_mask, loc.exon_mask, loc.primary_mask]
    gn_order = [loc.index[n] for n in loc.table_names]
    out = []
    for tb in range(3):
        cmpt, counts = {}, {}
        if tb > 0 and (not hla or masks[tb] == 0):
            out.append(([], []))
            continue
        job_off, hl, hr, ro, rows = walk.tables_out[tb]
        for p in range(walk.num_pairs):
            level = [masks[tb]]
            for h in range(job_off[p], job_off[p + 1]):
                s = compat_from_rows(loc, int(hl[h]), int(hr[h]), rows[ro[h]:ro[h + 1]], masks[tb])
                level.append(0)
                for c in range(len(level) - 1, 0, -1):
                    level[c] |= level[c - 1] & s
            best = masks[tb]
            for c in range(len(level) - 1, 0, -1):
                if level[c]:
                    best = level[c]
                    break
            for i in gn_order:
                if (best >> i) & 1:
                    counts[i] = counts.get(i, 0) + 1
            cmpt[best] = cmpt.get(best, 0) + 1
        out.append(([["-".join(loc.names_of(b)), c] for b, c in cmpt.items()],
                    [[loc.names[i], c] for i, c in counts.items()]))
    return out


def synthetic_case(seed, A, L=2500, n_pairs=1000, base="hla", del_frac=0.1, alphabet="ACGT", n_groups=12, core_vars=60,
                   pool_private=300, err_rate=0.004, paired=True, read_len=100, frag_len=350):
    """Database + reads from hisatgenotype_b200.synth (sizes the reference-captured goldens do not reach): returns
    (LocusTables/OracleLocus constructor args, alignment lines, truth alleles)."""
    from hisatgenotype_b200 import synth
    loc = synth.make_locus("A", seed, L=L, n_alleles=A, n_groups=n_groups, core_vars=core_vars,
                           pool_private=pool_private, del_frac=del_frac, alphabet=alphabet)
    cont = synth.reference_containers([loc], base)
    g = "A"
    args = (base, g, cont["refGenes"][g], cont["Genes"][g][cont["refGenes"][g]], cont["Vars"][g], cont["Var_list"][g],
            cont["Links"], cont["Gene_names"][g], cont["Gene_lengths"][g], cont["refGene_loci"][g][4],
            cont["refGene_loci"][g][5])
    rng = np.random.default_rng(seed)
    names = sorted(n for n in loc.alleles if loc.alleles[n])
    truth = [names[i] for i in rng.choice(len(names), 2, replace=False)]
    sam = synth.simulate_sam(loc, truth, n_pairs=n_pairs, rng=rng, err_rate=err_rate, paired=paired, read_len=read_len,
                             frag_len=frag_len)
    return args, sam, truth


def assert_tables_equal_oracle(run_tables, ref, ol, hla):
    """run_tables(tb) -> (Gene_cmpt items, Gene_counts items) of the product; ref = hgt_oracle.type_locus result."""
    for tb, key in ((0, "gene"), (1, "exon"), (2, "primary")):
        if tb > 0 and not hla:
            continue
        cmpt, counts = run_tables(tb)
        assert cmpt == ref["tables"][key].cmpt_items(ol), "Gene_cmpt of table %s differs" % key
        assert counts == ref["tables"][key].count_items(ol), "Gene_counts of table %s differs" % key

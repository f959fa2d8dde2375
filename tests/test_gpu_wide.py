"""GPU parity of stage (a) at the shapes bench.py runs (VERDICT r01 "weak" 1): every words-per-lane instantiation of
the allele-set kernels (A = 2,100 -> 2 words per lane, 7,000 / 8,191 -> 4, 9,000 -> 8), hla (three tables + two-level
EM) and non-hla, and a deletion-rich locus whose pairs expand to >= 8 haplotypes (the 8-bit-plane class kernel).
The oracle (oracle/hgt_oracle.py, pinned by the reference-captured goldens) runs on the same lines."""
import numpy as np
import pytest

import hgt_oracle as O
from helpers import assert_tables_equal_oracle, synthetic_case

pytestmark = pytest.mark.gpu

WIDE = [  # (A, base, words per lane)
    (2100, "hla", 2), (2100, "cyp", 2), (7000, "hla", 4), (7000, "cyp", 4), (8191, "hla", 4), (8191, "cyp", 4),
    (9000, "hla", 8), (9000, "cyp", 8),
]


@pytest.mark.parametrize("A,base,wpl", WIDE)
def test_wide_tables_bit_exact(A, base, wpl):
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.locus import LocusTables
    args, sam, truth = synthetic_case(100 + A % 97, A, L=3000, n_pairs=700, base=base, del_frac=0.08,
                                      n_groups=40, core_vars=70, pool_private=1200)
    ol = O.OracleLocus(*args)
    t = LocusTables(*args)
    assert {1: 1, 2: 2, 3: 4, 4: 4}.get((t.wp + 31) // 32, 8) == wpl, (t.wp, wpl)
    hla = base == "hla"
    ref = O.type_locus(ol, sam, simulation=False)
    # single-unit entry point
    run = TC.type_locus(t, sam)
    assert run.num_reads == ref["num_reads"] and run.num_pairs == ref["num_pairs"]
    assert_tables_equal_oracle(lambda tb: (list(map(list, run.gene_cmpt(tb).items())), run.gene_counts(tb)), ref, ol, hla)
    run.close()
    # batch entry point, two units of the same locus (the second one = the first half of the reads)
    half = sam[:len(sam) // 2 // 2 * 2]
    ref2 = O.type_locus(ol, half, simulation=False)
    batch = TC.Batch([t], TC.make_params(), True)
    batch.add_unit(0, sam)
    batch.add_unit(0, half)
    batch.run()
    for u, r in ((0, ref), (1, ref2)):
        s = batch.unit_summary(u)
        assert s["num_reads"] == r["num_reads"] and s["num_pairs"] == r["num_pairs"]
        assert_tables_equal_oracle(lambda tb: (list(map(list, batch.unit_gene_cmpt(u, tb).items())),
                                               batch.unit_gene_counts(u, tb)), r, ol, hla)
        want = O.locus_abundance(ol, r, True)
        got = batch.unit_calls(u)
        assert [a for a, _ in got] == [a for a, _ in want]
        for (_, x), (_, y) in zip(got, want):
            assert x == pytest.approx(y, rel=1e-6, abs=1e-12)
    batch.close()
    t.close()


@pytest.mark.parametrize("A,base", [(300, "hla"), (2100, "hla"), (7000, "cyp")])
def test_many_haplotype_pairs(A, base):
    """Homopolymer-rich backbone + 70 % deletions: deletions have many equivalent placements (Alts_left/right), so
    pairs expand to >= 8 haplotypes and take the 8-bit-plane class kernel."""
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.locus import LocusTables
    args, sam, truth = synthetic_case(5, A, L=2500, n_pairs=600, base=base, del_frac=0.7, alphabet="AAAC", n_groups=8,
                                      core_vars=50, pool_private=200 if A <= 300 else 900)
    ol = O.OracleLocus(*args)
    t = LocusTables(*args)
    hla = base == "hla"
    ref = O.type_locus(ol, sam, simulation=False)
    batch = TC.Batch([t], TC.make_params(), True)
    batch.add_unit(0, sam)
    batch.run()
    stats = batch.job_stats()
    assert stats["max_haplotypes_per_job"] >= 8 and stats["n_big_jobs"] > 0, stats
    s = batch.unit_summary(0)
    assert s["num_reads"] == ref["num_reads"] and s["num_pairs"] == ref["num_pairs"]
    assert_tables_equal_oracle(lambda tb: (list(map(list, batch.unit_gene_cmpt(0, tb).items())),
                                           batch.unit_gene_counts(0, tb)), ref, ol, hla)
    batch.close()
    t.close()

"""Device half of the record-shape cases (tests/record_forge.py): the record stage on the GPU against the oracle on the
same lines - totals, pileup, the three tables in dict order, and every surviving record's haplotypes - for reads of
50-250 bases (the warp mask pass, its serial fall-back past 128 bases and three M segments), mask probes at each word of
the 128-bit error-correction mask, known / novel indels, a batch whose long lines overflow the shared-memory stage, every
capacity of the walk at its limit and one past it, and pair jobs of exactly 7 and 8 haplotypes (the 3- / 8-bit-plane
split of the class kernel)."""
import os
import subprocess
import sys

import numpy as np
import pytest

import record_forge as F
from test_record_shapes import LENGTHS, _params, m_segments, oracle_corrections, oracle_run

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def check_unit(batch, u, t, ol, ref, hts, hla):
    """Totals, tables (dict order, Gene_counts) and per-record haplotypes of unit u against the oracle."""
    from hisatgenotype_b200 import typing_core as TC
    s = batch.unit_summary(u)
    assert s["num_reads"] == ref["num_reads"] and s["num_pairs"] == ref["num_pairs"], (s, ref["num_reads"])
    for tb, key in ((TC.TABLE_GENE, "gene"), (TC.TABLE_EXON, "exon"), (TC.TABLE_PRIMARY, "primary")):
        if tb != TC.TABLE_GENE and not hla:
            continue
        assert list(map(list, batch.unit_gene_cmpt(u, tb).items())) == ref["tables"][key].cmpt_items(ol), key
        assert batch.unit_gene_counts(u, tb) == ref["tables"][key].count_items(ol), key
    got = batch.unit_read_haplotypes(u, t.var_ids)
    assert len(got) == len(hts) == ref["num_reads"]
    for (gl, gf, gh), (wl, wf, wh) in zip(got, hts):
        assert (gl, gf) == (wl, wf)
        assert sorted(gh) == wh, (wl, gh, wh)


def device_matches_oracle(args, lines, kw, pileup=True):
    """Single-unit batch and (for the pileup) the single-run entry point on the same lines."""
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.locus import LocusTables
    ol, ref, hts = oracle_run(args, lines, kw)
    t = LocusTables(*args)
    hla = args[0] == "hla"
    batch = TC.Batch([t], _params(kw), True)
    batch.add_unit(0, lines)
    batch.run()
    check_unit(batch, 0, t, ol, ref, hts, hla)
    batch.close()
    if pileup:
        run = TC.type_locus(t, lines, kw.get("num_editdist", 2), kw.get("error_correction", True),
                            kw.get("allow_discordant", False), False)
        counts, mask = run.pileup()
        from helpers import pileup_arrays
        c, m = pileup_arrays(ref["counts"], ref["nt_sets"])
        np.testing.assert_array_equal(counts, c)
        np.testing.assert_array_equal(mask, m)
        run.close()
    t.close()
    return ref, hts


@pytest.mark.parametrize("paired", [True, False])
@pytest.mark.parametrize("read_len", LENGTHS)
def test_lengths(read_len, paired):
    args, sam = F.length_case(read_len, paired)
    kw = dict(allow_discordant=not paired)
    ref, hts = device_matches_oracle(args, sam, kw)
    if read_len > 128:
        assert all(len(x.split("\t")[9]) > 128 for x in sam)
    if read_len >= 150:
        assert sum(m_segments(x) > 3 for x in sam) > 0
    assert sum(1 for s in ref["nt_sets"] if s) > 100
    assert oracle_corrections(args, sam, kw, ref) > 10


@pytest.mark.parametrize("read_len", [100, 250])
def test_lengths_cyp(read_len):
    args, sam = F.length_case(read_len, True, base="cyp")
    device_matches_oracle(args, sam, {})


def test_mask_probes():
    loc, lines, hit = F.probe_case()
    assert all(v > 0 for v in hit.values()), hit
    ref, hts = device_matches_oracle(F.locus_args(loc), lines, dict(allow_discordant=True))
    # every probe survived (one corrected error each); a missed correction drops its SNP id from the haplotype
    assert sum(lines[li][0] in "pq" for li, _, _ in hts) == sum(1 for x in lines if x[0] in "pq")


def test_indels():
    loc, lines = F.indel_case()
    ref, hts = device_matches_oracle(F.locus_args(loc), lines, {})
    strs = [h for _, _, hs in hts for h in hs]
    assert any("nvI" in h for h in strs) and any("nvD" in h for h in strs)


def _block_bytes(texts):
    """Bytes of every 128-line block of the batch arena (units one after the other) and the stage size the walk picks
    (the formula of reads_execute in typing.cu).  The arena also pads every unit to 16 bytes; that shifts a block by at
    most 15 bytes and the average by less than one, far inside the margins the test asserts."""
    lens = [len(x) + 1 for lines in texts for x in lines]
    n = len(lens)
    blocks = [sum(lens[i:i + 128]) for i in range(0, n, 128)]
    stage = min(160 << 10, max(16 << 10, (sum(lens) // n * 147 + 1023) // 1024 * 1024 + 1024))
    return blocks, stage


def test_staging_long_block_in_short_batch():
    """A large 100-base unit and a 250-base unit in one batch: the stage is sized from the average line, so the blocks of
    the long unit are read from global memory.  Each unit equals the oracle and the same unit typed alone."""
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.locus import LocusTables
    from helpers import synthetic_case
    args, short, _ = synthetic_case(12, 120, L=1500, n_pairs=2500, del_frac=0.3, n_groups=6, core_vars=40,
                                    pool_private=150, err_rate=0.01)
    _, long_, _ = synthetic_case(12, 120, L=1500, n_pairs=240, del_frac=0.3, n_groups=6, core_vars=40,
                                 pool_private=150, err_rate=0.01, read_len=250, frag_len=600)
    blocks, stage = _block_bytes([short, long_])
    n_short_blocks = len(short) // 128
    assert max(blocks[n_short_blocks + 1:]) > stage + 1024 and stage >= max(blocks[:n_short_blocks]) + 1024
    t = LocusTables(*args)
    batch = TC.Batch([t], TC.make_params(), True)
    for lines in (short, long_):
        batch.add_unit(0, lines)
    batch.run()
    for u, lines in enumerate((short, long_)):
        ol, ref, hts = oracle_run(args, lines, {})
        check_unit(batch, u, t, ol, ref, hts, True)
        b1 = TC.Batch([t], TC.make_params(), True)
        b1.add_unit(0, lines)
        b1.run()
        assert b1.unit_read_haplotypes(0) == batch.unit_read_haplotypes(u)
        assert b1.unit_calls(0) == batch.unit_calls(u)
        b1.close()
    batch.close()
    t.close()


@pytest.mark.parametrize("env", ["HGT_STAGE_KB=16"])
def test_stage_switches(env):
    """The length, probe and staging cases with a 16 KB stage (every block of 128 lines overflows it).  The switch is
    read once per process, hence the child interpreter."""
    k, v = env.split("=")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(ROOT, "tests", "test_gpu_record_shapes.py"), "-x", "-q",
                        "-m", "gpu", "-k", "test_lengths or test_mask_probes or test_staging_long",
                        "-p", "no:cacheprovider"], env=dict(os.environ, **{k: v}), cwd=ROOT, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]


@pytest.mark.parametrize("kind", sorted(F.CAP_MESSAGES))
def test_capacity_at_limit(kind):
    loc, base, lines, kw = F.cap_case(kind, False)
    ref, hts = device_matches_oracle(F.locus_args(loc, base), lines, kw)
    assert 0 in [li for li, _, _ in hts]  # the record at the limit survived the walk


@pytest.mark.parametrize("kind", sorted(F.CAP_MESSAGES))
def test_capacity_past_limit_refused(kind):
    """One past the limit: the whole batch (a good unit with it) is refused with the walk's message, never typed."""
    from hisatgenotype_b200 import _lib
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.locus import LocusTables
    loc, base, good, kw = F.cap_case(kind, False)
    _, _, bad, _ = F.cap_case(kind, True)
    t = LocusTables(*F.locus_args(loc, base))
    batch = TC.Batch([t], _params(kw), True)
    batch.add_unit(0, good)
    batch.add_unit(0, bad)
    with pytest.raises(_lib.HgtError) as e:
        batch.run()
    assert e.value.code == _lib.HGT_ERR_UNSUPPORTED
    assert F.CAP_MESSAGES[kind] in str(e.value)
    batch.close()
    t.close()


def test_job_split_7_and_8():
    """Exon-table jobs of exactly 7 haplotypes (3 bit planes) and exactly 8 (8 bit planes), winning counts 7 and 8; plus
    the pair of 255 haplotypes (the largest count) of the capacity case."""
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.locus import LocusTables
    loc, lines, n8 = F.job_split_case()
    args = F.locus_args(loc)
    ol, ref, hts = oracle_run(args, lines, {})
    t = LocusTables(*args)
    batch = TC.Batch([t], TC.make_params(), True)
    batch.add_unit(0, lines)
    batch.run()
    st = batch.job_stats()
    assert st["max_haplotypes_per_job"] == 8 and st["n_big_jobs"] == n8, st
    assert st["n_jobs"] == 3 * ref["num_pairs"]
    check_unit(batch, 0, t, ol, ref, hts, True)
    batch.close()
    t.close()
    loc, base, lines, kw = F.cap_case("pair_hts", False)
    args = F.locus_args(loc, base)
    ol, ref, hts = oracle_run(args, lines, kw)
    t = LocusTables(*args)
    batch = TC.Batch([t], _params(kw), True)
    batch.add_unit(0, lines)
    batch.run()
    assert batch.job_stats()["max_haplotypes_per_job"] == 255
    check_unit(batch, 0, t, ol, ref, hts, True)
    batch.close()
    t.close()

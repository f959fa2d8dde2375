"""Host half of the record-shape cases (tests/record_forge.py): the record walk's __host__ __device__ rules, run by
hgt_host_walk, against the oracle on reads of 50-250 bases, error-correction probes at the mask word boundaries, known
and novel indels, and every capacity of the walk at its limit (typed as the oracle types it) and one past it
(refused with HGT_ERR_UNSUPPORTED)."""
import numpy as np
import pytest

import hgt_oracle as O
import record_forge as F
from helpers import pileup_arrays, tables_from_jobs

LENGTHS = [50, 96, 100, 101, 127, 128, 129, 150, 250]


def _params(kw):
    from hisatgenotype_b200.typing_core import make_params
    return make_params(kw.get("num_editdist", 2), kw.get("error_correction", True), kw.get("allow_discordant", False))


def oracle_run(args, lines, kw):
    ol = O.OracleLocus(*args)
    hts = []
    ref = O.type_locus(ol, lines, False, kw.get("num_editdist", 2), kw.get("error_correction", True),
                       kw.get("allow_discordant", False), collect_hts=hts)
    return ol, ref, hts


def host_walk(args, lines, kw, ref):
    from hisatgenotype_b200.locus import LocusTables
    from hisatgenotype_b200.typing_core import HostWalk
    t = LocusTables(*args, host_only=True)
    c, m = pileup_arrays(ref["counts"], ref["nt_sets"])
    try:
        return HostWalk(t, lines, _params(kw), c, m)
    finally:
        t.close()


def assert_host_matches_oracle(args, lines, kw):
    ol, ref, hts = oracle_run(args, lines, kw)
    walk = host_walk(args, lines, kw, ref)
    assert walk.num_reads == ref["num_reads"] and walk.num_pairs == ref["num_pairs"]
    res = tables_from_jobs(ol, walk, args[0] == "hla")
    for tb, key in ((0, "gene"), (1, "exon"), (2, "primary")):
        if tb > 0 and args[0] != "hla":
            continue
        assert res[tb][0] == ref["tables"][key].cmpt_items(ol), key
        assert res[tb][1] == ref["tables"][key].count_items(ol), key
    return ref, hts


def m_segments(line):
    return line.split("\t")[5].count("M")


def oracle_corrections(args, lines, kw, ref):
    """Records the oracle's error correction changed to the reference (ncorr > 0) - corrections to a known SNP do not
    count there - among those that pass the filters in front of the walk."""
    ol = O.OracleLocus(*args)
    n = 0
    for line in lines:
        rec = O.parse_record(line, False, 0)
        if rec.flag & 0x4 or rec.NM > kw.get("num_editdist", 2) or (not kw.get("allow_discordant") and not rec.flag & 2):
            continue
        n += O.walk_record(ol, rec, ref["counts"], ref["nt_sets"], True)[2] > 0
    return n


@pytest.mark.parametrize("paired", [True, False])
@pytest.mark.parametrize("read_len", LENGTHS)
def test_read_lengths(read_len, paired):
    args, sam = F.length_case(read_len, paired)
    kw = dict(allow_discordant=not paired)
    ref, hts = assert_host_matches_oracle(args, sam, kw)
    assert ref["num_reads"] > 0.5 * len(sam)
    if read_len >= 150:
        assert sum(m_segments(x) > 3 for x in sam) > 0
    # error correction fired: positions carry an nt_set and the oracle corrected reads to the reference
    assert sum(1 for s in ref["nt_sets"] if s) > 100
    assert oracle_corrections(args, sam, kw, ref) > 10


def test_mask_probes():
    loc, lines, hit = F.probe_case()
    assert all(v > 0 for v in hit.values()), hit
    assert_host_matches_oracle(F.locus_args(loc), lines, dict(allow_discordant=True))


def test_indels():
    loc, lines = F.indel_case()
    ref, hts = assert_host_matches_oracle(F.locus_args(loc), lines, {})
    strs = [h for _, _, hs in hts for h in hs]
    assert any("nvI" in h for h in strs) and any("nvD" in h for h in strs)
    assert sum("I" in x.split("\t")[5] for x in lines) > 50 and sum("Zs:Z:" in x for x in lines) > 50


@pytest.mark.parametrize("kind", sorted(F.CAP_MESSAGES))
def test_capacity_at_limit_types_like_oracle(kind):
    loc, base, lines, kw = F.cap_case(kind, False)
    ref, hts = assert_host_matches_oracle(F.locus_args(loc, base), lines, kw)
    assert 0 in [li for li, _, _ in hts]  # the record at the limit survived the walk


@pytest.mark.parametrize("kind", sorted(F.CAP_MESSAGES))
def test_capacity_past_limit_refused(kind):
    from hisatgenotype_b200 import _lib
    loc, base, lines, kw = F.cap_case(kind, True)
    args = F.locus_args(loc, base)
    ol, ref, hts = oracle_run(args, lines, kw)
    with pytest.raises(_lib.HgtError) as e:
        host_walk(args, lines, kw, ref)
    assert e.value.code == _lib.HGT_ERR_UNSUPPORTED
    assert F.CAP_MESSAGES[kind] in str(e.value)


def test_job_split_counts():
    loc, lines, n8 = F.job_split_case()
    args = F.locus_args(loc)
    ref, hts = assert_host_matches_oracle(args, lines, {})
    walk = host_walk(args, lines, {}, ref)
    job_off = walk.tables_out[1][0]
    sizes = np.diff(job_off)
    assert sorted(set(sizes.tolist())) == [7, 8] and int((sizes == 8).sum()) == n8

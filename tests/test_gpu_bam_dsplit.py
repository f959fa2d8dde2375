"""The device split (sam_intake.split_bam_device, csrc/bam_dsplit.cu): BGZF-compressed BAM files split by backbone on the
GPU, each bucket rendered into the text arena from HBM.  Every bucket's text must equal the host split's
(split_bam(..., text=True)), its errors the host split's, and everything downstream the packed BamUnit path."""
import ctypes
import random
import re
import struct

import numpy as np
import pytest

from bam_writer import bam_header, bam_stream, bgzf, encode_record, write_bam
from conftest import GOLDEN_NAMES, load_golden
from helpers import golden_db, product_locus
from test_bam_intake import _hdr, _one
from test_gpu_bam_intake import _unit_results
from test_gpu_bgzf_inflate import _counters, _samples
from test_sam_split import coordinate_sorted

pytestmark = pytest.mark.gpu


def _text(split, s, ref):
    """Bucket (s, ref) rendered by a batch of one unit."""
    from hisatgenotype_b200 import synth
    from hisatgenotype_b200 import typing_core as TC
    global _TINY
    if "_TINY" not in globals():
        loc = synth.make_locus("A", 40, L=3000, n_alleles=120, n_groups=8, core_vars=50, pool_private=200, del_frac=0.08)
        _TINY = _tables([loc])[0]
    b = TC.Batch([_TINY], TC.make_params())
    u = b.add_unit_bam_dsplit(0, split.unit(s, ref))
    b.prepare()
    t = b.unit_text(u)
    b.close()
    return t


def _tables(locs):
    from hisatgenotype_b200 import synth
    from hisatgenotype_b200.locus import LocusTables
    cont = synth.reference_containers(locs, "hla")
    return [LocusTables("hla", l.gene, cont["refGenes"][l.gene], cont["Genes"][l.gene][cont["refGenes"][l.gene]],
                        cont["Vars"][l.gene], cont["Var_list"][l.gene], cont["Links"], cont["Gene_names"][l.gene],
                        cont["Gene_lengths"][l.gene], cont["refGene_loci"][l.gene][4], cont["refGene_loci"][l.gene][5])
            for l in locs]


def _same_as_host(files, refs, drop_qual=False):
    """Every bucket of one device split equals split_bam's text of its file."""
    from hisatgenotype_b200.sam_intake import split_bam, split_bam_device
    with split_bam_device(files, refs, drop_qual=drop_qual) as sp:
        rec, size = sp.sizes()
        for s, f in enumerate(files):
            host = split_bam(f, refs, n_threads=2, drop_qual=drop_qual, text=True)
            for r, name in enumerate(refs):
                if name in refs[r + 1:]:
                    continue  # split_bam's dict holds the last bucket of a repeated name; the others are empty
                assert size[s, r] == len(host[name]) and rec[s, r] == host[name].count(b"\n"), (s, name)
                assert _text(sp, s, r) == host[name], (s, name)


@pytest.mark.parametrize("name", GOLDEN_NAMES)
@pytest.mark.parametrize("block", [65280, 1024, 100])
@pytest.mark.parametrize("drop_qual", [False, True])
def test_goldens_render_the_host_text_and_type_like_bam_units(name, block, drop_qual):
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.sam_intake import split_bam, split_bam_device
    g = load_golden(name)
    p = g["params"]
    db = golden_db(g)
    caps = g["loci"][:len(p["loci"])]
    refs = [c["ref_allele"] for c in caps]
    bam = write_bam(coordinate_sorted(caps), [(r, 100000) for r in refs], block=block)
    host = split_bam(bam, refs, n_threads=2, drop_qual=drop_qual, text=True)
    blobs = split_bam(bam, refs, n_threads=2, drop_qual=drop_qual)
    genes = []
    for c in caps:
        if c["gene"] not in genes:
            genes.append(c["gene"])
    names = {c["gene"]: c["Gene_names"] for c in caps}
    loci = [product_locus(g, db, gn, names[gn]) for gn in genes]
    with split_bam_device([bam], refs, drop_qual=drop_qual) as sp:
        batch = TC.Batch(loci, TC.make_params(p["num_editdist"], p["error_correction"], p["discordant"], p["simulation"]),
                         p["remove_low"])
        pairs = []
        for c in caps:
            li = genes.index(c["gene"])
            pairs.append((batch.add_unit_bam_dsplit(li, sp.unit(0, c["ref_allele"])), batch.add_unit_bam(li, blobs[c["ref_allele"]]), c))
        batch.prepare()
    for ud, ub, c in pairs:
        r = c["ref_allele"]
        assert batch.unit_text(ud) == host[r] == batch.unit_text(ub)
        if not drop_qual:
            assert host[r] == ("\n".join(c["sam"]) + "\n").encode()
    batch.execute()
    batch.finish()
    for ud, ub, c in pairs:
        assert _unit_results(batch, ud) == _unit_results(batch, ub)
    batch.close()
    for t in loci:
        t.close()


def _line(name, pos, flag=0, ref="X", rnext="*", tags=""):
    return "%s\t%d\t%s\t%d\t60\t1M\t%s\t0\t0\tA\tI%s" % (name, flag, ref, pos, rnext, tags)


def test_order_adversaries_in_one_call():
    rng = random.Random(17)
    hdr = [("X", 1000), ("Y", 1000), ("Z", 1000)]
    files = []
    # names sharing prefixes of 0 .. 253 bytes, names that are prefixes of others, bytes >= 0x80 (Latin-1 in the SAM line)
    lines = []
    for i in range(3000):
        k = rng.randrange(248)
        stem = "p" * k
        tail = "".join(rng.choice("ab\xe9\xff~") for _ in range(rng.randrange(0, min(3, 254 - k) + 1)))
        lines.append(_line((stem + tail)[:254] or "q", rng.randrange(-1, 3) + 1, ref=rng.choice(["X", "Y", "*"])))
    files.append(lines)
    # equal name and POS with different FLAGs (input order), POS -1 (0 in SAM), refID -1, other references, RNEXT elsewhere
    lines = []
    for i in range(2000):
        nm = "r%d" % rng.randrange(50)
        lines.append(_line(nm, rng.choice([0, 1, 2]), flag=rng.choice([0, 16, 99, 147, 4]),
                           ref=rng.choice(["X", "Y", "Z", "*"]), rnext=rng.choice(["*", "=", "Y", "Z"])))
    files.append(lines)
    enc = []
    for lines in files:
        raw = bam_stream(lines[:0], hdr)
        idx = {n: i for i, (n, _) in enumerate(hdr)}
        enc.append(bgzf(raw + b"".join(encode_record(l, idx) for l in lines), 4096))
    # a header listing one backbone twice, records on both entries
    hdr2 = [("X", 1000), ("Y", 500), ("X", 1000)]
    recs = []
    for i in range(500):
        rec = bytearray(encode_record(_line("d%d" % rng.randrange(60), rng.randrange(1, 9), rnext="="), {"X": 0}))
        k = rng.choice([0, 2])
        struct.pack_into("<ii", rec, 4, k, struct.unpack_from("<i", rec, 8)[0])
        struct.pack_into("<i", rec, 24, rng.choice([-1, 0, 1, 2]))
        recs.append(bytes(rec))
    enc.append(bgzf(bam_header(hdr2) + b"".join(recs), 1000))
    # thousands of header references, and a header longer than the 64 KB read-back window
    many = [("c%05d_%s" % (i, "x" * 20), 100) for i in range(4000)] + [("X", 1000)]
    idx = {n: i for i, (n, _) in enumerate(many)}
    enc.append(bgzf(bam_header(many) + b"".join(encode_record(_line("m%d" % (i % 97), i % 7 + 1, ref=rng.choice(["X", "c00007_" + "x" * 20])), idx)
                                                for i in range(3000)), 65280))
    big_text = "@CO\t" + "y" * 100000 + "\n"
    enc.append(bgzf(bam_header(hdr, text=big_text) + b"".join(encode_record(_line("t%d" % i, i + 1), {"X": 0}) for i in range(100)), 65280))
    _same_as_host(enc, ["X", "Y", "Z", "c00007_" + "x" * 20])
    _same_as_host(enc, ["X", "Y", "X"])


def _message(e):
    """The library's message, without the "libhgt error <code>: " that HgtError puts in front."""
    return re.sub(r"^libhgt error -?\d+: ", "", str(e.value))


def test_rejections_equal_the_host_split_and_the_context_stays_usable():
    from hisatgenotype_b200 import _lib
    from hisatgenotype_b200.sam_intake import split_bam, split_bam_device
    good = _hdr() + _one("\tNM:i:0")
    cases = [b"BAX\1" + good[4:], good[:-3]]
    rec = bytearray(_one())
    struct.pack_into("<i", rec, 20, 1000)
    cases.append(_hdr() + bytes(rec))
    cases += [_hdr() + _one(raw_tags=b"XZZab"), _hdr() + _one(raw_tags=b"XQq\x01")]
    rec = bytearray(_one())
    struct.pack_into("<i", rec, 4, 5)
    cases.append(_hdr() + bytes(rec))
    cases += [_hdr() + _one(t) for t in ("\tXF:f:1.5", "\tXB:B:f,1.5", "\tCG:B:I,1600")]
    recs = [encode_record("a%05d\t0\tX\t5\t60\t1M\t*\t0\t0\tA\tI" % i, {"X": 0}) for i in range(20000)]
    recs.insert(10000, encode_record("bad1\t0\tX\t5\t60\t1M\t*\t0\t0\tA\tI", {"X": 0}, raw_tags=b"XQq\x01"))
    recs.append(encode_record("bad2\t0\tX\t5\t60\t1M\t*\t0\t0\tA\tI", {"X": 0}, raw_tags=b"XQq\x01"))
    cases.append(_hdr() + b"".join(recs))
    fine = bgzf(good)
    for raw in cases:
        with pytest.raises((AssertionError, _lib.HgtError)) as host:
            split_bam(raw, ["X"])
        for at in (0, 1):  # as the first stream, and behind a good one
            files = [bgzf(raw, 700)] if at == 0 else [fine, bgzf(raw, 700)]
            with pytest.raises(host.type) as dev:
                split_bam_device(files, ["X"])
            assert _message(dev) == "stream %d: " % at + _message(host).split(": ", 1)[1], raw[:40]
            if host.type is _lib.HgtError:
                assert dev.value.code == host.value.code == _lib.HGT_ERR_UNSUPPORTED
    assert "bad1" in str(dev.value)
    # a corrupt block: inflate_bgzf's message
    z = bytearray(bgzf(good))
    z[struct.unpack_from("<H", z, 16)[0] + 1 - 8] ^= 1
    with pytest.raises(AssertionError, match=re.escape("stream 1: BGZF block at byte 0: CRC32 mismatch")):
        split_bam_device([fine, bytes(z)], ["X"])
    # a header-only file, a file without the EOF block
    hdr = bam_stream([], [("X", 1000), ("Y", 10)], text="@HD\tVN:1.6\n")
    with split_bam_device([bgzf(hdr)], ["X", "Y", "Z"]) as sp:
        assert sp.sizes()[0].tolist() == [[0, 0, 0]]
        assert _text(sp, 0, 0) == b""
    lines = ["q%d\t0\tX\t%d\t60\t1M\t*\t0\t0\tA\tI" % (i, i + 1) for i in range(50)]
    with pytest.warns(UserWarning, match="EOF"):
        with split_bam_device([write_bam(lines, [("X", 1000)], block=512, eof=False)], ["X"]) as sp:
            assert _text(sp, 0, "X").decode().splitlines() == sorted(lines)
    with split_bam_device([fine], ["X"]) as sp:  # the context still works
        assert _text(sp, 0, "X") == split_bam(good, ["X"], text=True)["X"]


def test_scale_counters_mixed_units_and_two_batches():
    from hisatgenotype_b200 import _lib, synth
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.sam_intake import read_bgzf, split_bam, split_bam_device
    bams, refs = _samples()
    L = _lib.lib()
    ctx = _lib.ctx(None)
    n_blocks = 0
    for b in bams:
        arr = np.frombuffer(b, np.uint8)
        h = ctypes.c_void_p()
        _lib.check(L.hgt_bgzf_open(1, (ctypes.c_void_p * 1)(arr.ctypes.data), (ctypes.c_size_t * 1)(arr.size), ctypes.byref(h)))
        nb = ctypes.c_int64(0)
        _lib.check(L.hgt_bgzf_sizes(h, None, ctypes.byref(nb), None))
        L.hgt_bgzf_free(h)
        n_blocks += nb.value
    raws = [read_bgzf(b) for b in bams]
    S, R = len(bams), len(refs)
    names = sum(len(r.encode()) for r in refs)  # every file's header lists the refs
    a8 = lambda x: (x + 7) & ~7
    L.hgt_profile_reset(ctx)
    _, h0, d0 = _counters(ctx)
    sp = split_bam_device(bams, refs)
    _, h1, d1 = _counters(ctx)
    assert h1 - h0 == sum(len(b) for b in bams) + 16 * (n_blocks + 1) + 8 * (S + 1) + 48 * (S + 1) \
        + S * a8(8 * R + 4 + names) + 4 * S * R
    assert d1 - d0 == 56 * S + 16 * (S * R + 2) + sum(min(len(r), 65536) for r in raws)
    assert d1 - d0 < sum(len(r) for r in raws) / 10
    locs = [synth.make_locus(gene, 40 + i, L=3000, n_alleles=120, n_groups=8, core_vars=50, pool_private=200, del_frac=0.08)
            for i, gene in enumerate(("A", "B", "C"))]
    tables = _tables(locs)
    for run in range(2):  # one handle feeds two batches
        batch = TC.Batch(tables, TC.make_params(n_threads=3), True)
        trip = []
        for s in range(S):
            text = split_bam(bams[s], refs, n_threads=2, text=True)
            blobs = split_bam(bams[s], refs, n_threads=2)
            for li, r in enumerate(refs):
                trip.append((batch.add_unit_bam_dsplit(li, sp.unit(s, r)), batch.add_unit(li, text[r]),
                             batch.add_unit_bam(li, blobs[r]), text[r]))
        batch.prepare()
        for ud, ut, ub, t in trip:
            assert batch.unit_text(ud) == t == batch.unit_text(ub)
        batch.execute()
        batch.finish()
        for ud, ut, ub, _ in trip:
            rd = _unit_results(batch, ud)
            assert rd == _unit_results(batch, ut) == _unit_results(batch, ub)
        batch.close()
    sp.close()
    for t in tables:
        t.close()


@pytest.mark.parametrize("name", ["hla_pair_err", "cyp_pair"])
def test_reports_from_device_units(name):
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.sam_intake import split_bam_device
    g = load_golden(name)
    p = g["params"]
    db = golden_db(g)
    n_loci = len(p["loci"])
    reports = [g["reports"][k] for k in sorted(g["reports"], key=lambda s: int(s.split("test-")[1].split(".")[0]))]
    tables = {}
    for t_i, ref_text in enumerate(reports):
        caps = g["loci"][t_i * n_loci:(t_i + 1) * n_loci]
        for cap in caps:
            if cap["gene"] not in tables:
                tables[cap["gene"]] = product_locus(g, db, cap["gene"], cap["Gene_names"])
        refs = [c["ref_allele"] for c in caps]
        bam = write_bam(coordinate_sorted(caps), [(r, 100000) for r in refs], block=4096)
        with split_bam_device([bam], refs) as sp:
            body, _ = TC.typing_from_alignments(
                p["base"], tables, [cap["test_Gene_names"] for cap in caps],
                {cap["gene"]: sp.unit(0, cap["ref_allele"]) for cap in caps}, p["simulation"], p["num_editdist"],
                p["error_correction"], p["discordant"], p["remove_low"], p["best_alleles"], p["output_allele_counts"])
        marker = "\n\t\thisat2 graph\n"
        assert body == ref_text[ref_text.index(marker):]
    for t in tables.values():
        t.close()

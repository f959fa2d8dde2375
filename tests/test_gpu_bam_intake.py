"""Native BAM intake on the GPU: packed BAM units (sam_intake.split_bam) rendered into the text arena by
bam_text_len_kernel / bam_render_kernel (csrc/typing.cu, formatter csrc/bam_dev.cuh) must give the bytes `samtools view`
printed (tests/golden) and everything downstream must equal the text path, unit for unit."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from bam_writer import write_bam
from conftest import GOLDEN_NAMES, ROOT, load_golden
from helpers import golden_db, product_locus
from test_sam_split import coordinate_sorted

pytestmark = pytest.mark.gpu


def _outcome(f, *a):
    try:
        return ("ok", f(*a))
    except Exception as e:  # the reference's exceptions (KeyError, ZeroDivisionError, TypeError) must match too
        return (type(e).__name__, str(e))


def _unit_results(batch, u):
    out = {"summary": batch.unit_summary(u), "counts": _outcome(batch.unit_gene_counts, u)}
    for tb in range(4):
        r = _outcome(batch.unit_table, u, tb)
        out["table%d" % tb] = (r[0], [np.asarray(x).tobytes() for x in r[1]]) if r[0] == "ok" else r
    for level in (0, 1):
        out["em%d" % level] = _outcome(batch.unit_em, u, level)
    out["calls"] = _outcome(batch.unit_calls, u)
    return out


@pytest.mark.parametrize("name", GOLDEN_NAMES)
@pytest.mark.parametrize("drop_qual", [False, True])
def test_bam_unit_renders_samtools_text_and_types_like_text(name, drop_qual):
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.sam_intake import split_bam, split_sam
    g = load_golden(name)
    p = g["params"]
    db = golden_db(g)
    caps = g["loci"][:len(p["loci"])]
    refs = [c["ref_allele"] for c in caps]
    lines = coordinate_sorted(caps)
    bam = write_bam(lines, [(r, 100000) for r in refs], block=4096)
    blobs = split_bam(bam, refs, n_threads=2, drop_qual=drop_qual)
    host = split_bam(bam, refs, n_threads=2, drop_qual=drop_qual, text=True)
    sam = split_sam(("\n".join(lines) + "\n").encode(), refs, n_threads=2, drop_qual=drop_qual)
    genes = []
    for c in caps:
        if c["gene"] not in genes:
            genes.append(c["gene"])
    names = {c["gene"]: c["Gene_names"] for c in caps}
    loci = [product_locus(g, db, gene, names[gene]) for gene in genes]
    batch = TC.Batch(loci, TC.make_params(p["num_editdist"], p["error_correction"], p["discordant"], p["simulation"]),
                     p["remove_low"])
    pairs = []
    for c in caps:
        li = genes.index(c["gene"])
        pairs.append((batch.add_unit_bam(li, blobs[c["ref_allele"]]), batch.add_unit(li, sam[c["ref_allele"]]), c))
    batch.prepare()
    for ub, ut, c in pairs:
        r = c["ref_allele"]
        assert batch.unit_text(ub) == host[r] == sam[r]
        assert batch.unit_text(ut) == sam[r]
        if not drop_qual:
            assert host[r] == ("\n".join(c["sam"]) + "\n").encode()
    batch.execute()
    batch.finish()
    for ub, ut, c in pairs:
        rb, rt = _unit_results(batch, ub), _unit_results(batch, ut)
        assert rb == rt
        assert rb["summary"]["num_reads"] == c["num_reads"] and rb["summary"]["num_pairs"] == c["num_pairs"]
    batch.close()
    for t in loci:
        t.close()


def test_synthetic_multi_locus_batch_pinned_and_pageable():
    """~50 k records over 3 loci and 6 samples, several units per locus, units without records, blobs in page-locked and
    in pageable memory, text units between them: the device-rendered arena equals split_sam's text for every unit, and
    each BAM unit types like its text twin."""
    from hisatgenotype_b200 import _lib, synth
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.locus import LocusTables
    from hisatgenotype_b200.sam_intake import split_bam, split_sam
    locs = [synth.make_locus(gene, 40 + i, L=3000, n_alleles=120, n_groups=8, core_vars=50, pool_private=200, del_frac=0.08)
            for i, gene in enumerate(("A", "B", "C"))]
    cont = synth.reference_containers(locs, "hla")
    refs = [cont["refGenes"][l.gene] for l in locs]
    tables = [LocusTables("hla", l.gene, cont["refGenes"][l.gene], cont["Genes"][l.gene][cont["refGenes"][l.gene]],
                          cont["Vars"][l.gene], cont["Var_list"][l.gene], cont["Links"], cont["Gene_names"][l.gene],
                          cont["Gene_lengths"][l.gene], cont["refGene_loci"][l.gene][4], cont["refGene_loci"][l.gene][5])
              for l in locs]
    sims = [synth.ReadSimulator(l) for l in locs]
    samples = []
    n_rec = 0
    for s in range(6):
        rng = np.random.default_rng(100 + s)
        text = b""
        for li, l in enumerate(locs):
            if (s + li) % 4 == 0:
                continue  # this sample has no reads on this locus: an empty unit
            names = sorted(n for n in l.alleles if l.alleles[n])
            truth = [names[i] for i in rng.choice(len(names), 2, replace=False)]
            text += sims[li].generate(truth, 1800, seed=s * 8 + li + 1, err_rate=0.005, read_len=100, frag_len=350,
                                      paired=True, prefix="s%d_" % s)
        lines = text.decode().splitlines()
        n_rec += len(lines)
        samples.append((lines, text))
    assert 40000 <= n_rec <= 70000
    pinned = _lib.PinnedText(64 << 20)
    batch = TC.Batch(tables, TC.make_params(n_threads=3), True)
    expect = []
    for s, (lines, text) in enumerate(samples):
        bam = write_bam(lines, [(r, 100000) for r in refs], block=65280)
        sam = split_sam(text, refs, n_threads=2)
        if s % 2 == 0:
            at = split_bam(bam, refs, n_threads=2, pinned=pinned)
            for li, r in enumerate(refs):
                expect.append((batch.add_unit_bam_ptr(li, *at[r]), sam[r], li))
        else:
            blobs = split_bam(bam, refs, n_threads=2)
            for li, r in enumerate(refs):
                expect.append((batch.add_unit_bam(li, blobs[r]), sam[r], li))
        for li, r in enumerate(refs):
            expect.append((batch.add_unit(li, sam[r]), sam[r], li))
    assert any(len(t) == 0 for _, t, _ in expect)
    batch.prepare()
    for u, text, _ in expect:
        assert batch.unit_text(u) == text, u
    batch.execute()
    batch.finish()
    n_units = len(refs)
    for s in range(len(samples)):
        base = s * 2 * n_units
        for li in range(n_units):
            assert _unit_results(batch, base + li) == _unit_results(batch, base + n_units + li)
    batch.close()
    pinned.close()
    for t in tables:
        t.close()


def test_add_unit_bam_rejects_bad_blobs():
    import struct
    from hisatgenotype_b200 import _lib
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.sam_intake import split_bam
    g = load_golden("hla_basic")
    db = golden_db(g)
    c = g["loci"][0]
    blob = bytes(split_bam(write_bam(c["sam"], [(c["ref_allele"], 100000)]), [c["ref_allele"]])[c["ref_allele"]])
    magic, flags, n_rec, n_names, names_bytes = struct.unpack_from("<IIqII", blob)
    o_recs = (24 + 4 * (n_names + 1) + names_bytes + 7) & ~7
    p = g["params"]
    t = product_locus(g, db, c["gene"], c["Gene_names"])
    batch = TC.Batch([t], TC.make_params(p["num_editdist"], p["error_correction"], p["discordant"], p["simulation"]),
                     p["remove_low"])
    bad = []
    past = bytearray(blob)  # the last record ends past the blob
    struct.pack_into("<Q", past, o_recs + 8 * n_rec, len(blob) + 8)
    bad.append(bytes(past))
    back = bytearray(blob)  # offsets not monotone
    struct.pack_into("<Q", back, o_recs + 8, struct.unpack_from("<Q", blob, o_recs)[0] - 4)
    bad.append(bytes(back))
    bad.append(blob[:o_recs + 8])  # offset table cut
    bad.append(b"XXXX" + blob[4:])  # magic
    more = bytearray(blob)  # more records than the table holds
    struct.pack_into("<q", more, 8, 1 << 40)
    bad.append(bytes(more))
    for b in bad:
        with pytest.raises(_lib.HgtError) as e:
            batch.add_unit_bam(0, b)
        assert e.value.code == _lib.HGT_ERR_ARG
    u = batch.add_unit_bam(0, blob)  # the batch is still usable
    batch.run()
    assert batch.unit_summary(u)["num_reads"] == c["num_reads"]
    batch.close()
    t.close()


@pytest.mark.parametrize("name", ["hla_pair_err", "hla_indel", "cyp_pair"])
def test_typing_drop_in_with_bam_file(name, tmp_path):
    """HGT_NATIVE_INTAKE=1 with a BAM alignment file: no samtools (the stand-in exits 97), the reference's report."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "shim_bam_driver.py"), name, str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    line = [x for x in r.stdout.splitlines() if x.startswith("SHIM_RESULT ")][-1]
    res = json.loads(line[len("SHIM_RESULT "):])
    assert all(res["checks"].values()), res["checks"]
    g = load_golden(name)
    assert set(res["reports"]) == set(g["reports"])
    assert r.stdout.splitlines()[-1] == "BAM_FILES %d" % len(g["reports"])  # every test was typed from a BAM file
    for k, text in g["reports"].items():
        assert res["reports"][k] == text, k

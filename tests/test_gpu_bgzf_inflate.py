"""BGZF inflate on the GPU (sam_intake.inflate_bgzf, hgt_bgzf_inflate: bgzf_inflate_kernel, one warp per block): the bytes
read_bgzf (zlib) gives for every stream of the corpus and for a large multi-sample BAM set, the documented copies and one
launch per call, every malformed block refused with its rule while the context stays usable, and the native BAM intake of
typing() fed from it."""
import json
import os
import re
import subprocess
import sys
import warnings

import numpy as np
import pytest

from bam_writer import EOF_BLOCK, write_bam
from bgzf_corpus import bad_blocks, corpus, deflate, member, stream
from conftest import GOLDEN_NAMES, ROOT, load_golden
from test_sam_split import coordinate_sorted

pytestmark = pytest.mark.gpu


def _zlib(data):
    from hisatgenotype_b200.sam_intake import read_bgzf
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return read_bgzf(data)


def _counters(ctx):
    import ctypes
    from hisatgenotype_b200 import _lib
    L = _lib.lib()
    h2d, d2h = ctypes.c_int64(0), ctypes.c_int64(0)
    L.hgt_profile_read(ctx, None, None, ctypes.byref(h2d), ctypes.byref(d2h))
    return L.hgt_launch_count(ctx), h2d.value, d2h.value


def test_corpus_one_call_and_stream_by_stream():
    from hisatgenotype_b200.sam_intake import inflate_bgzf
    streams = corpus()
    want = [_zlib(d) for _, d in streams]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        got = inflate_bgzf([d for _, d in streams])
        assert [bytes(g) for g in got] == want
        for (name, d), w in zip(streams, want):
            assert bytes(inflate_bgzf([d])[0]) == w, name


def _samples():
    """~50 k records over 3 loci and 6 samples (the generator of test_synthetic_multi_locus_batch_pinned_and_pageable),
    one BAM file per sample."""
    from hisatgenotype_b200 import synth
    locs = [synth.make_locus(gene, 40 + i, L=3000, n_alleles=120, n_groups=8, core_vars=50, pool_private=200, del_frac=0.08)
            for i, gene in enumerate(("A", "B", "C"))]
    cont = synth.reference_containers(locs, "hla")
    refs = [cont["refGenes"][l.gene] for l in locs]
    sims = [synth.ReadSimulator(l) for l in locs]
    bams, n_rec = [], 0
    for s in range(6):
        rng = np.random.default_rng(100 + s)
        text = b""
        for li, l in enumerate(locs):
            names = sorted(n for n in l.alleles if l.alleles[n])
            truth = [names[i] for i in rng.choice(len(names), 2, replace=False)]
            text += sims[li].generate(truth, 1800, seed=s * 8 + li + 1, err_rate=0.005, read_len=100, frag_len=350,
                                      paired=True, prefix="s%d_" % s)
        lines = text.decode().splitlines()
        n_rec += len(lines)
        bams.append(write_bam(lines, [(r, 100000) for r in refs], block=65280))
    assert 40000 <= n_rec <= 80000
    return bams, refs


def test_large_call_pageable_and_pinned_copies_and_launches():
    import ctypes
    from hisatgenotype_b200 import _lib
    from hisatgenotype_b200.sam_intake import inflate_bgzf
    bams, _ = _samples()
    want = [_zlib(b) for b in bams]
    L = _lib.lib()
    ctx = _lib.ctx()
    n_blocks = 0
    for b in bams:
        arr = np.frombuffer(b, np.uint8)
        h = ctypes.c_void_p()
        _lib.check(L.hgt_bgzf_open(1, (ctypes.c_void_p * 1)(arr.ctypes.data), (ctypes.c_size_t * 1)(arr.size),
                                   ctypes.byref(h)))
        nb = ctypes.c_int64(0)
        _lib.check(L.hgt_bgzf_sizes(h, None, ctypes.byref(nb), None))
        L.hgt_bgzf_free(h)
        n_blocks += nb.value
    pinned = _lib.PinnedText(sum(len(b) + 16 for b in bams))
    pinned_in = [pinned.view(*pinned.add(b)) for b in bams]
    for inputs in (bams, pinned_in):
        L.hgt_profile_reset(ctx)
        k0, _, _ = _counters(ctx)
        got = inflate_bgzf(inputs)
        k1, h2d, d2h = _counters(ctx)
        assert [bytes(g) for g in got] == want
        assert k1 - k0 == 1  # one kernel per call (hgt.h)
        assert h2d == sum(len(b) for b in bams) + 16 * (n_blocks + 1)
        assert d2h == sum(len(w) for w in want) + 8
    pinned.close()


def test_rejections_report_the_rule_and_the_context_stays_usable():
    from hisatgenotype_b200.sam_intake import inflate_bgzf
    fine = stream(b"fine" * 1000)
    first = member(deflate(b"ok"), b"ok")
    for name, block, rule in bad_blocks():
        with pytest.raises(AssertionError, match="^stream 1: BGZF block at byte %d: %s" % (len(first), re.escape(rule))):
            inflate_bgzf([fine, first + block + EOF_BLOCK])
    assert bytes(inflate_bgzf([fine])[0]) == b"fine" * 1000


@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_split_bam_on_gpu_inflate_equals_host_inflate(name):
    from hisatgenotype_b200.sam_intake import inflate_bgzf, read_bgzf, split_bam
    g = load_golden(name)
    caps = g["loci"][:len(g["params"]["loci"])]
    refs = [c["ref_allele"] for c in caps]
    bam = write_bam(coordinate_sorted(caps), [(r, 100000) for r in refs], block=1024)
    raw = inflate_bgzf([bam])[0]
    for text in (False, True):
        assert split_bam(raw, refs, n_threads=2, text=text) == split_bam(read_bgzf(bam), refs, n_threads=2, text=text)


@pytest.mark.parametrize("name", ["hla_pair_err", "cyp_pair"])
def test_typing_drop_in_inflates_bam_on_the_gpu(name, tmp_path):
    """HGT_NATIVE_INTAKE=1 with BAM files: the reference's reports, every file inflated by the kernel."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "shim_bgzf_driver.py"), name, str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    out = r.stdout.splitlines()
    res = json.loads([x for x in out if x.startswith("SHIM_RESULT ")][-1][len("SHIM_RESULT "):])
    assert all(res["checks"].values()), res["checks"]
    g = load_golden(name)
    assert res["reports"] == g["reports"]
    n_files = len(g["reports"])
    assert out[-2] == "BAM_FILES %d" % n_files
    assert out[-1] == "INFLATE_CALLS %d %d" % (n_files, n_files)

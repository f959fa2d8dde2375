"""BGZF inflate of the native BAM intake, host emulation (hgt_bgzf_inflate_host: the functions of csrc/bgzf_dev.cuh the
device runs, on host threads): byte for byte what read_bgzf (zlib) gives on every DEFLATE shape, the same accept / reject
decision on every malformed block, with a message naming the stream, the byte offset and the rule."""
import random
import re
import struct
import warnings
import zlib

import pytest

from bam_writer import EOF_BLOCK
from bgzf_corpus import bad_blocks, corpus, deflate, header_bad, member, stream

CORPUS = corpus()


@pytest.mark.parametrize("name", [n for n, _ in CORPUS])
def test_host_inflate_equals_zlib(name):
    from hisatgenotype_b200.sam_intake import inflate_bgzf_host, read_bgzf
    data = dict(CORPUS)[name]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        want = read_bgzf(data)
    for nt in (1, 3):
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            got = inflate_bgzf_host([data], nt)
        assert len(got) == 1 and bytes(got[0]) == want
        assert len(w) == (0 if data.endswith(EOF_BLOCK) else 1)


def test_host_inflate_many_streams_in_one_call():
    from hisatgenotype_b200.sam_intake import inflate_bgzf_host, read_bgzf
    streams = [d for _, d in CORPUS]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        got = inflate_bgzf_host(streams, 4)
        assert [bytes(g) for g in got] == [read_bgzf(d) for d in streams]


def test_sizes_and_eof():
    import ctypes
    import numpy as np
    from hisatgenotype_b200 import _lib
    L = _lib.lib()
    streams = [stream(b"x" * 100000), stream(b"y" * 10, eof=False), b"", EOF_BLOCK]
    arrs = [np.frombuffer(s, np.uint8) for s in streams]
    h = ctypes.c_void_p()
    ptrs = (ctypes.c_void_p * 4)(*[a.ctypes.data if a.size else None for a in arrs])
    _lib.check(L.hgt_bgzf_open(4, ptrs, (ctypes.c_size_t * 4)(*[a.size for a in arrs]), ctypes.byref(h)))
    out, nb, eof = (ctypes.c_size_t * 4)(), (ctypes.c_int64 * 4)(), (ctypes.c_int32 * 4)()
    _lib.check(L.hgt_bgzf_sizes(h, out, nb, eof))
    L.hgt_bgzf_free(h)
    assert list(out) == [100000, 10, 0, 0] and list(nb) == [3, 1, 0, 1] and list(eof) == [1, 0, 0, 1]


@pytest.mark.parametrize("case", bad_blocks(), ids=lambda c: c[0])
def test_host_rejects_each_rule_like_zlib(case):
    """One hand-made block per rule: read_bgzf refuses it, and so does the emulation, naming stream 1 and the block's
    offset (it follows a valid block) with the rule."""
    from hisatgenotype_b200.sam_intake import inflate_bgzf_host, read_bgzf
    _, block, rule = case
    first = member(deflate(b"ok"), b"ok")
    bad = first + block + EOF_BLOCK
    with pytest.raises(Exception):
        read_bgzf(bad)
    with pytest.raises(AssertionError, match="^stream 1: BGZF block at byte %d: %s" % (len(first), re.escape(rule))):
        inflate_bgzf_host([stream(b"fine" * 1000), bad], 2)


@pytest.mark.parametrize("case", header_bad(), ids=lambda c: c[0])
def test_host_header_errors_read_bgzf_wording(case):
    from hisatgenotype_b200.sam_intake import inflate_bgzf_host, read_bgzf
    _, data, msg = case
    with pytest.raises(AssertionError, match=re.escape(msg)):
        read_bgzf(data)
    with pytest.raises(AssertionError, match="^stream 0: .*" + re.escape(msg)):
        inflate_bgzf_host([data])


def test_isize_above_64k_refused():
    """The one input read_bgzf accepts and this path refuses: a block that claims more than 64 KiB."""
    from hisatgenotype_b200.sam_intake import inflate_bgzf_host, read_bgzf
    raw = bytes(70000)
    data = member(deflate(raw), raw) + EOF_BLOCK
    assert read_bgzf(data) == raw
    with pytest.raises(AssertionError, match="stream 0: BGZF block at byte 0: ISIZE 70000 > 65536"):
        inflate_bgzf_host([data])


def _fuzz_inputs():
    rng = random.Random(2024)
    base = []
    for level, strat in ((0, zlib.Z_DEFAULT_STRATEGY), (1, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_DEFAULT_STRATEGY),
                         (9, zlib.Z_FIXED), (6, zlib.Z_RLE), (6, zlib.Z_HUFFMAN_ONLY)):
        raw = b"".join(b"r%d\tACGTTGCA%s\n" % (rng.randrange(50), bytes(rng.choice(b"ACGT") for _ in range(rng.randrange(60))))
                       for _ in range(40))
        blk = stream(raw, level=level, strategy=strat, eof=False)
        base.append(blk)
    cases = []
    for i in range(3000):
        blk = bytearray(rng.choice(base))
        head = 18
        kind = rng.randrange(4)
        if kind < 2:  # bit flips inside the DEFLATE data
            for _ in range(1 + rng.randrange(3)):
                p = head + rng.randrange(len(blk) - head - 8)
                blk[p] ^= 1 << rng.randrange(8)
        elif kind == 2:  # bit flips anywhere in the block, header and trailer included
            p = rng.randrange(len(blk))
            blk[p] ^= 1 << rng.randrange(8)
        else:  # DEFLATE data cut short, the header's BSIZE following
            cut = 1 + rng.randrange(min(40, len(blk) - head - 8))
            blk = blk[:len(blk) - 8 - cut] + blk[len(blk) - 8:]
            struct.pack_into("<H", blk, 16, len(blk) - 1)
        cases.append(bytes(blk) + EOF_BLOCK)
    return cases


def test_fuzz_host_decoder_decides_like_read_bgzf():
    """A seeded few thousand bit-flipped and truncated blocks: the host decoder always returns, refuses exactly what
    read_bgzf refuses, and otherwise gives read_bgzf's bytes."""
    from hisatgenotype_b200.sam_intake import inflate_bgzf_host, read_bgzf
    n_rejected = 0
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for data in _fuzz_inputs():
            try:
                want = read_bgzf(data)
            except Exception:
                want = None
            try:
                got = bytes(inflate_bgzf_host([data], 1)[0])
            except AssertionError:
                got = None
            assert (want is None) == (got is None), data.hex()
            if want is None:
                n_rejected += 1
            else:
                assert got == want
    assert 1000 < n_rejected < 3000  # both outcomes occur often

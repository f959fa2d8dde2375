"""The record index of the device split, run by its host emulation (sam_intake.bam_index_host: the chunk guess, walk, fix-up
passes and serial resolve of csrc/bam_dsplit.cu on host threads) against the serial block_size chain of the host split, on
streams built to mislead the guesses."""
import random
import struct

import pytest

from bam_writer import bam_stream, encode_record
from conftest import GOLDEN_NAMES, load_golden
from test_sam_split import coordinate_sorted

CHUNKS = [64, 100, 1000, 4096, 65536]


def _serial(raw):
    """Record offsets by the host split's chain rule, or (byte, records) of the break."""
    l_text = struct.unpack_from("<i", raw, 4)[0]
    o = 8 + l_text
    n_ref = struct.unpack_from("<i", raw, o)[0]
    o += 4
    for _ in range(n_ref):
        o += 4 + struct.unpack_from("<i", raw, o)[0] + 4
    offs = []
    while o < len(raw):
        if len(raw) - o < 4:
            break
        bs = struct.unpack_from("<i", raw, o)[0]
        if bs < 32 or bs > len(raw) - o - 4:
            break
        offs.append(o)
        o += 4 + bs
    if o != len(raw):
        return None, (o, len(offs))
    return offs, None


def _check(raw, chunks=CHUNKS):
    from hisatgenotype_b200.sam_intake import bam_index_host, split_bam
    want, brk = _serial(raw)
    for chunk in chunks:
        for nt in (1, 4):
            if brk is None:
                assert bam_index_host(raw, chunk, nt).tolist() == want, chunk
            else:
                msg = "truncated or malformed record at byte %d of the BAM stream (after %d records)" % brk
                with pytest.raises(AssertionError) as e:
                    bam_index_host(raw, chunk, nt)
                assert str(e.value) == "hgt_bam_index_host: " + msg
    if brk is not None:  # the host split reports the same break
        with pytest.raises(AssertionError) as e:
            split_bam(raw, ["X"])
        assert str(e.value) == "hgt_bam_split_create: " + msg


@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_goldens(name):
    g = load_golden(name)
    caps = g["loci"][:len(g["params"]["loci"])]
    _check(bam_stream(coordinate_sorted(caps), [(c["ref_allele"], 100000) for c in caps]))


def _decoy(rng):
    """A record that passes the plausibility test, as bytes to hide inside another record."""
    line = "d%d\t0\tX\t%d\t60\t4M\t*\t0\t0\tACGT\tIIII" % (rng.randrange(1000), rng.randrange(1, 100))
    return encode_record(line, {"X": 0})


def test_false_starts_in_tags_and_qual():
    """Whole valid-looking records embedded in B:C tag arrays and in QUAL, and block_size-like bytes in Z tags."""
    rng = random.Random(7)
    recs = []
    for i in range(3000):
        k = rng.randrange(4)
        if k == 0:  # a decoy record inside a B:C array (no NUL constraint)
            d = _decoy(rng)
            raw = b"XBBC" + struct.pack("<I", len(d)) + d
            recs.append(encode_record("r%d\t0\tX\t5\t60\t4M\t*\t0\t0\tACGT\tIIII" % i, {"X": 0}, raw_tags=raw))
        elif k == 1:  # a decoy as QUAL bytes (QUAL is raw bytes in BAM)
            d = _decoy(rng)
            seq = "A" * len(d)
            rec = bytearray(encode_record("r%d\t0\tX\t5\t60\t%dM\t*\t0\t0\t%s\t%s" % (i, len(d), seq, "I" * len(d)), {"X": 0}))
            q = len(rec) - len(d)
            rec[q:q + len(d)] = d
            recs.append(bytes(rec))
        elif k == 2:  # block_size-like integers inside a Z tag
            z = "".join(chr(rng.choice([32, 33, 36, 40, 48, 64, 65])) for _ in range(rng.randrange(1, 300)))
            recs.append(encode_record("r%d\t0\tX\t5\t60\t4M\t*\t0\t0\tACGT\tIIII\tXZ:Z:%s" % (i, z), {"X": 0}))
        else:
            recs.append(encode_record("r%d\t0\tX\t5\t60\t4M\t*\t0\t0\tACGT\tIIII" % i, {"X": 0}))
    _check(bam_stream([], [("X", 1000)]) + b"".join(recs))


def test_records_longer_than_a_chunk_and_minimum_records():
    """~60 KB tags (the exit skips whole chunks), mixed with 36-byte records (block_size 32, the least the chain takes)."""
    rng = random.Random(11)
    recs = []
    for i in range(200):
        k = rng.randrange(3)
        if k == 0:
            big = rng.randrange(1000, 60000)
            raw = b"XBBC" + struct.pack("<I", big) + bytes(rng.randrange(256) for _ in range(big))
            recs.append(encode_record("b%d\t0\tX\t5\t60\t4M\t*\t0\t0\tACGT\tIIII" % i, {"X": 0}, raw_tags=raw))
        elif k == 1:
            rec = bytearray(36)
            struct.pack_into("<iiiBBHHHiiii", rec, 0, 32, 0, 4, 1, 0, 4680, 0, 4, 0, -1, -1, 0)
            recs.append(bytes(rec))  # name "" + NUL is not there: the chain takes it, the check would not
        else:
            recs.append(_decoy(rng))
    _check(bam_stream([], [("X", 1000)]) + b"".join(recs))


def test_chain_breaks():
    rng = random.Random(5)
    good = [encode_record("r%d\t0\tX\t5\t60\t4M\t*\t0\t0\tACGT\tIIII" % i, {"X": 0}) for i in range(2000)]
    hdr = bam_stream([], [("X", 1000)])
    body = b"".join(good)
    _check(hdr + body[:-3])                                     # cut short
    for at in (0, 17, 999, 1999):
        bad = list(good)
        rec = bytearray(bad[at])
        struct.pack_into("<i", rec, 0, rng.choice([31, 0, -5, 1 << 30]))  # block_size below 32 or past the end
        bad[at] = bytes(rec)
        _check(hdr + b"".join(bad))
    _check(hdr + body + b"\x01\x02")                            # two stray bytes
    _check(hdr)                                                 # header only

"""Native BAM intake on the host (sam_intake.read_bgzf / split_bam, csrc/bam_split.cpp, the formatter of csrc/bam_dev.cuh
through its host render): the text of a BAM unit is what `samtools view` printed for the captured alignments (tests/golden),
and the same per-reference text split_sam gives for the SAM form of the same records."""
import random
import struct

import pytest

from bam_writer import bam_stream, bgzf, encode_record, write_bam
from conftest import GOLDEN_NAMES, load_golden
from test_sam_split import coordinate_sorted


def _golden_refs(caps):
    return [(c["ref_allele"], 100000) for c in caps]


@pytest.mark.parametrize("name", GOLDEN_NAMES)
@pytest.mark.parametrize("block", [65280, 1024])
def test_split_bam_text_is_samtools_view(name, block):
    from hisatgenotype_b200.sam_intake import BamUnit, split_bam
    g = load_golden(name)
    caps = g["loci"][:len(g["params"]["loci"])]
    refs = [c["ref_allele"] for c in caps]
    bam = write_bam(coordinate_sorted(caps), _golden_refs(caps), block=block)
    for nt in (1, 3):
        out = split_bam(bam, refs, n_threads=nt, text=True)
        for c in caps:
            assert out[c["ref_allele"]].decode().splitlines() == c["sam"]
        blobs = split_bam(bam, refs, n_threads=nt)
        assert all(isinstance(b, BamUnit) for b in blobs.values())


def test_split_bam_equals_split_sam_any_order_and_threads():
    """The generator of test_split_order_rule_any_input_order_and_threads, through BAM: same per-reference text; records
    of refID -1 and of other references are dropped."""
    from hisatgenotype_b200.sam_intake import split_bam, split_sam
    rng = random.Random(3)
    recs = []
    for i in range(3000):
        nm = "r%d%s" % (rng.randrange(400), rng.choice(["", "|x", "A", "_2"]))
        ref = rng.choice(["L1*BACKBONE", "L2*BACKBONE", "other", "*"])
        recs.append("%s\t%d\t%s\t%d\t60\t100M\t=\t1\t0\tACGT\tIIII\tNM:i:0\tMD:Z:100\tNH:i:1" % (nm, 99, ref, rng.randrange(1, 50)))
    refs = ["L1*BACKBONE", "L2*BACKBONE"]
    hdr = [("L1*BACKBONE", 1000), ("other", 1000), ("L2*BACKBONE", 1000)]
    want = split_sam("\n".join(recs).encode(), refs, n_threads=2)
    assert all(want[r] for r in refs)
    for nt in (1, 2, 7):
        got = split_bam(write_bam(recs, hdr, block=4096), refs, n_threads=nt, text=True)
        assert got == want


FORMAT_LINES = [
    "r00\t4\tX\t0\t0\t*\t*\t0\t0\tACGT\tIIII",                                # unmapped, * CIGAR, POS 0, RNEXT *
    "r01\t99\tX\t10\t60\t4M\t=\t20\t14\tACGT\tABCD\tNM:i:0",                   # RNEXT =
    "r02\t65\tX\t11\t3\t2S2M\tY\t7\t0\tACGT\t#+5?",                            # RNEXT another reference
    "r03\t147\tX\t12\t60\t3M1I2D1M\t=\t5\t-361\tACGTA\tIIIII",                 # negative TLEN, I/D ops
    "r04\t4\tX\t13\t0\t*\t*\t0\t0\t*\t*",                                     # l_seq 0
    "r05\t0\tX\t14\t60\t4M\t*\t0\t0\tACGT\t*",                                # QUAL 0xff
    "r06\t0\tX\t15\t60\t16M\t*\t0\t0\t=ACMGRSVTWYHKDBN\t" + "I" * 16,         # = / N / IUPAC bases
    "r07\t0\tX\t16\t60\t5M\t*\t0\t0\tNNNNN\t!!!!!",                            # odd l_seq, QUAL 0
    "r08\t0\tX\t17\t60\t1M1N1P1=1X1H\t*\t0\t0\tACGT\tIIII",                    # other CIGAR ops
    "r09\t0\tX\t18\t0\t*\t*\t0\t0\tA\tI\tXA:i:-128\tXB:i:255\tXC:i:-32768\tXD:i:65535\tXE:i:-2147483648\tXF:i:4294967295",
    "r10\t0\tX\t19\t0\t*\t*\t0\t0\tA\tI\tXA:i:-129\tXB:i:256\tXC:i:-32769\tXD:i:65536\tXE:i:0\tXF:i:-1\tXG:i:127",
    "r11\t0\tX\t20\t0\t*\t*\t0\t0\tA\tI\tXA:A:q\tXZ:Z:hello world|1,2\tXH:H:1AE301\tXE:Z:",
    "r12\t0\tX\t21\t0\t*\t*\t0\t0\tA\tI\tBa:B:c,-128,0,127\tBb:B:C,0,255\tBc:B:s,-32768,32767\tBd:B:S,0,65535"
    "\tBe:B:i,-2147483648,2147483647\tBf:B:I,0,4294967295\tBg:B:c",
    "r13\t0\tX\t2147483647\t255\t4M\tY\t2147483647\t-2147483647\tACGT\tIIII",  # large POS / PNEXT / TLEN
    "n" * 254 + "\t0\tX\t22\t60\t1M\t*\t0\t0\tA\tI",                           # 254-byte name
]


def test_formatting_rules():
    """Each rule of htslib's sam_format1 against the SAM line the record was written from."""
    from hisatgenotype_b200.sam_intake import split_bam, split_sam
    hdr = [("X", 3000000000 // 2), ("Y", 1000)]
    raw = bam_stream(FORMAT_LINES, hdr)
    for data in (raw, bgzf(raw, 100)):
        out = split_bam(data, ["X", "Y"], n_threads=2, text=True)
        assert out["Y"] == b""
        assert out["X"].decode().split("\n")[:-1] == sorted(FORMAT_LINES, key=lambda l: l.split("\t")[0].encode())
    # the same text as the SAM split of the source lines (which takes POS up to 2e9)
    lines = [l for l in FORMAT_LINES if not l.startswith("r13")]
    assert split_bam(bam_stream(lines, hdr), ["X"], text=True)["X"] == split_sam("\n".join(lines).encode(), ["X"])["X"]


@pytest.mark.parametrize("name", GOLDEN_NAMES[:3])
def test_split_bam_drop_qual(name):
    """drop_qual: QUAL becomes '*', every other column is identical, and the blob is smaller."""
    from hisatgenotype_b200.sam_intake import split_bam
    g = load_golden(name)
    caps = g["loci"][:len(g["params"]["loci"])]
    refs = [c["ref_allele"] for c in caps]
    bam = write_bam(coordinate_sorted(caps), _golden_refs(caps), block=2048)
    full = split_bam(bam, refs, n_threads=2)
    dropped = split_bam(bam, refs, n_threads=2, drop_qual=True)
    text = split_bam(bam, refs, n_threads=2, drop_qual=True, text=True)
    for c in caps:
        r = c["ref_allele"]
        assert len(dropped[r]) < len(full[r])
        got = text[r].decode().splitlines()
        assert len(got) == len(c["sam"])
        for a, b in zip(got, c["sam"]):
            ca, cb = a.split("\t"), b.split("\t")
            assert ca[:10] == cb[:10] and ca[11:] == cb[11:] and ca[10] == "*"


def _one(tags="", raw_tags=b"", line=None):
    line = line or "q1\t0\tX\t5\t60\t4M\t*\t0\t0\tACGT\tIIII" + tags
    return encode_record(line, {"X": 0}, raw_tags)


def _hdr():
    return bam_stream([], [("X", 1000)])


def test_rejections():
    from hisatgenotype_b200 import _lib
    from hisatgenotype_b200.sam_intake import read_bgzf, split_bam
    good = _hdr() + _one("\tNM:i:0")
    assert split_bam(good, ["X"], text=True)["X"].startswith(b"q1\t0\tX\t5\t")
    # bad magic
    with pytest.raises(AssertionError, match="magic"):
        split_bam(b"BAX\1" + good[4:], ["X"])
    # truncated block, bad CRC
    z = bgzf(good)
    with pytest.raises(AssertionError, match="truncated"):
        split_bam(z[:30], ["X"])
    bad_crc = bytearray(z)
    n0 = struct.unpack_from("<H", z, 16)[0] + 1  # first block's size
    bad_crc[n0 - 8] ^= 1
    with pytest.raises(AssertionError, match="CRC"):
        read_bgzf(bytes(bad_crc))
    # block_size inconsistent with its fields (l_seq larger than the record holds)
    rec = bytearray(_one())
    struct.pack_into("<i", rec, 20, 1000)
    with pytest.raises(AssertionError, match="q1.*block_size"):
        split_bam(_hdr() + bytes(rec), ["X"])
    # a record cut short (the block_size chain leaves the stream)
    with pytest.raises(AssertionError, match="truncated"):
        split_bam(good[:-3], ["X"])
    # an aux tag past the record end (Z without NUL), an unknown tag type
    with pytest.raises(AssertionError, match="q1.*XZ.*past the record end"):
        split_bam(_hdr() + _one(raw_tags=b"XZZab"), ["X"])
    with pytest.raises(AssertionError, match="q1.*XQ.*unknown type"):
        split_bam(_hdr() + _one(raw_tags=b"XQq\x01"), ["X"])
    # a refID outside the header
    rec = bytearray(_one())
    struct.pack_into("<i", rec, 4, 5)
    with pytest.raises(AssertionError, match="refID"):
        split_bam(_hdr() + bytes(rec), ["X"])
    # float tags and the long-CIGAR placeholder: unsupported, naming the read and the tag
    for tags, tag in (("\tXF:f:1.5", "XF"), ("\tXB:B:f,1.5", "XB"), ("\tCG:B:I,1600", "CG")):
        with pytest.raises(_lib.HgtError, match="q1.*" + tag) as e:
            split_bam(_hdr() + _one(tags), ["X"])
        assert e.value.code == _lib.HGT_ERR_UNSUPPORTED
    # the first bad record in input order is the one reported, whatever the thread count
    recs = [encode_record("a%05d\t0\tX\t5\t60\t1M\t*\t0\t0\tA\tI" % i, {"X": 0}) for i in range(20000)]
    recs.insert(10000, encode_record("bad1\t0\tX\t5\t60\t1M\t*\t0\t0\tA\tI", {"X": 0}, raw_tags=b"XQq\x01"))
    recs.append(encode_record("bad2\t0\tX\t5\t60\t1M\t*\t0\t0\tA\tI", {"X": 0}, raw_tags=b"XQq\x01"))
    for nt in (1, 8):
        with pytest.raises(AssertionError, match="bad1"):
            split_bam(_hdr() + b"".join(recs), ["X"], n_threads=nt)


def test_header_only_and_missing_eof():
    from hisatgenotype_b200.sam_intake import BamUnit, split_bam
    hdr = bam_stream([], [("X", 1000), ("Y", 10)], text="@HD\tVN:1.6\n")
    out = split_bam(bgzf(hdr), ["X", "Y", "Z"])
    assert set(out) == {"X", "Y", "Z"}
    for blob in out.values():
        assert isinstance(blob, BamUnit)
        magic, flags, n_records = struct.unpack_from("<IIq", blob)
        assert magic == 0x31424748 and n_records == 0
    assert split_bam(bgzf(hdr), ["X"], text=True) == {"X": b""}
    lines = ["q%d\t0\tX\t%d\t60\t1M\t*\t0\t0\tA\tI" % (i, i + 1) for i in range(50)]
    with pytest.warns(UserWarning, match="EOF"):
        got = split_bam(write_bam(lines, [("X", 1000)], block=512, eof=False), ["X"], text=True)
    assert got["X"].decode().splitlines() == sorted(lines)


def test_read_alignment_kinds(tmp_path):
    """The native typing() path: SAM text and BAM are read natively; CRAM and BGZF that is not BAM stay with samtools."""
    from hisatgenotype_b200.sam_intake import read_alignment
    sam = b"q1\t0\tX\t5\t60\t1M\t*\t0\t0\tA\tI\n"
    p = tmp_path / "a"
    p.write_bytes(sam)
    assert read_alignment(str(p)) == ("sam", sam)
    raw = bam_stream(["q1\t0\tX\t5\t60\t1M\t*\t0\t0\tA\tI"], [("X", 10)])
    p.write_bytes(bgzf(raw))
    assert read_alignment(str(p)) == ("bam", raw)
    p.write_bytes(b"CRAM\3\0" + b"\0" * 30)
    assert read_alignment(str(p)) == (None, None)
    p.write_bytes(bgzf(b"##fileformat=VCFv4.2\n"))
    assert read_alignment(str(p)) == (None, None)

"""BGZF test inputs shared by tests/test_bgzf_inflate.py (host emulation) and tests/test_gpu_bgzf_inflate.py (device):
a corpus of valid streams covering every DEFLATE shape zlib writes plus three it never writes (from a small raw-DEFLATE
bit writer), and one malformed block per rule of csrc/bgzf_dev.cuh with the message it must give."""
import random
import struct
import zlib

from bam_writer import EOF_BLOCK, bgzf, write_bam
from conftest import GOLDEN_NAMES, load_golden
from test_sam_split import coordinate_sorted


def member(cdata, raw, crc=None, isize=None, bc=True):
    """One BGZF block around raw DEFLATE bytes; the trailer holds raw's CRC32 and length unless given.  bc=False: the
    extra field holds another subfield instead of BC."""
    bsize = 12 + 6 + len(cdata) + 8
    extra = b"BC\x02\x00" + struct.pack("<H", bsize - 1) if bc else b"XY\x02\x00\x00\x00"
    return (b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\x00" + extra + cdata +
            struct.pack("<II", zlib.crc32(raw) if crc is None else crc, len(raw) if isize is None else isize))


def deflate(raw, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, flush_every=0):
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    if not flush_every:
        return c.compress(raw) + c.flush()
    out = b""
    for o in range(0, len(raw), flush_every):
        out += c.compress(raw[o:o + flush_every]) + c.flush(zlib.Z_FULL_FLUSH)  # ends in an empty stored block
    return out + c.flush()


def stream(data, block=65280, eof=True, **kw):
    """BGZF of data with the given zlib settings."""
    blocks = [member(deflate(data[o:o + block], **kw), data[o:o + block]) for o in range(0, len(data), block)]
    return b"".join(blocks) + (EOF_BLOCK if eof else b"")


class BitWriter:
    """Raw DEFLATE, LSB-first; Huffman codes MSB-first."""

    def __init__(self):
        self.acc, self.n, self.out = 0, 0, bytearray()

    def bits(self, v, k):
        self.acc |= v << self.n
        self.n += k
        while self.n >= 8:
            self.out.append(self.acc & 255)
            self.acc >>= 8
            self.n -= 8

    def code(self, c, k):
        for i in range(k - 1, -1, -1):
            self.bits((c >> i) & 1, 1)

    def done(self):
        if self.n:
            self.out.append(self.acc & 255)
        self.acc, self.n = 0, 0
        return bytes(self.out)


def canonical(lens):
    """{symbol: length} -> {symbol: (code, length)} (RFC 1951 3.2.2)."""
    bl = [0] * 16
    for v in lens.values():
        bl[v] += 1
    code, nxt = 0, [0] * 16
    for b in range(1, 16):
        code = (code + bl[b - 1]) << 1
        nxt[b] = code
    out = {}
    for s in sorted(lens):
        if lens[s]:
            out[s] = (nxt[lens[s]], lens[s])
            nxt[lens[s]] += 1
    return out


def _len_code(n):
    for s in range(29):
        ext = 0 if s < 8 or s == 28 else (s >> 2) - 1
        base = 3 + s if s < 8 else 258 if s == 28 else ((4 + (s & 3)) << ext) + 3
        if base <= n < base + (1 << ext) and not (s == 27 and n == 258):
            return 257 + s, ext, n - base


def _dist_code(d):
    for s in range(30):
        ext = 0 if s < 4 else (s >> 1) - 1
        base = s + 1 if s < 4 else ((2 + (s & 1)) << ext) + 1
        if base <= d < base + (1 << ext):
            return s, ext, d - base


CL_LENS = {0: 2, 1: 3, 2: 3, 3: 4, 4: 4, 17: 4, 18: 4, 5: 5, 6: 5, 7: 5, 8: 5, 9: 6, 10: 6, 11: 6, 12: 6, 13: 6, 14: 6, 15: 6,
           16: 6}  # a complete code-length code (Kraft sum 1)
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]


def dynamic_block(w, lit_lens, dist_lens, nlen, ndist, items, final=True, cl_lens=CL_LENS, raw_lengths=None):
    """One dynamic block into BitWriter w.  items: ("lit", byte) / ("match", length, distance); EOB is added.
    raw_lengths: CL symbols to write instead of the lengths ([(sym, extra bits, extra value)])."""
    w.bits(1 if final else 0, 1)
    w.bits(2, 2)
    w.bits(nlen - 257, 5)
    w.bits(ndist - 1, 5)
    w.bits(19 - 4, 4)
    for s in CL_ORDER:
        w.bits(cl_lens.get(s, 0), 3)
    clc = canonical(cl_lens)
    seq = raw_lengths
    if seq is None:
        lens = [lit_lens.get(s, 0) for s in range(nlen)] + [dist_lens.get(s, 0) for s in range(ndist)]
        seq, i = [], 0
        while i < len(lens):
            j = i
            while j < len(lens) and lens[j] == lens[i]:
                j += 1
            run = j - i
            if lens[i] == 0 and run >= 11:
                k = min(run, 138)
                seq.append((18, 7, k - 11))
            elif lens[i] == 0 and run >= 3:
                k = min(run, 10)
                seq.append((17, 3, k - 3))
            else:
                k = 1
                seq.append((lens[i], 0, 0))
            i += k
    for sym, ext, val in seq:
        w.code(*clc[sym])
        if ext:
            w.bits(val, ext)
    lc, dc = canonical(lit_lens), canonical(dist_lens)
    for it in items:
        if it[0] == "lit":
            w.code(*lc[it[1]])
        else:
            s, ext, val = _len_code(it[1])
            w.code(*lc[s])
            w.bits(val, ext)
            s, ext, val = _dist_code(it[2])
            w.code(*dc[s])
            w.bits(val, ext)
    w.code(*lc[256])


def fixed_block(w, syms, final=True):
    """A fixed-Huffman block of raw symbols: ("lit", s) for any literal/length symbol 0..287 (286/287 included),
    ("dist", d) for any distance code 0..31 with extra ("bits", v, k)."""
    w.bits(1 if final else 0, 1)
    w.bits(1, 2)
    for it in syms:
        if it[0] == "lit":
            s = it[1]
            if s < 144:
                w.code(0x30 + s, 8)
            elif s < 256:
                w.code(0x190 + s - 144, 9)
            elif s < 280:
                w.code(s - 256, 7)
            else:
                w.code(0xC0 + s - 280, 8)
        elif it[0] == "dist":
            w.code(it[1], 5)
        else:
            w.bits(it[1], it[2])


def _unusual():
    """The three shapes zlib never writes, as (deflate bytes, inflated bytes)."""
    out = []
    # a single distance code of length 1 (incomplete: legal), matches of distance 1 and 3
    w = BitWriter()
    lit = {97: 2, 98: 2, 256: 2, 258: 3, 259: 3}
    dynamic_block(w, lit, {0: 1}, 260, 1, [("lit", 97), ("match", 4, 1), ("lit", 98), ("match", 5, 1)])
    out.append((w.done(), b"a" * 5 + b"b" * 6))
    w = BitWriter()
    dynamic_block(w, lit, {2: 1}, 260, 3, [("lit", 97), ("lit", 98), ("lit", 97), ("match", 4, 3)])
    out.append((w.done(), b"abaaba" + b"a"))
    # no distance codes at all (one distance length of 0): literals only
    w = BitWriter()
    dynamic_block(w, {97: 1, 256: 2, 98: 2}, {}, 257, 1, [("lit", 97), ("lit", 98)] * 40)
    out.append((w.done(), b"ab" * 40))
    # literal/length codes of length 15 (lengths 1..14, 15, 15: complete)
    syms = list(range(65, 79)) + [256, 79]
    lens = {s: min(i + 1, 15) for i, s in enumerate(syms)}
    w = BitWriter()
    data = bytes([79, 65, 78, 79, 70] * 7)
    dynamic_block(w, lens, {}, 257, 1, [("lit", b) for b in data])
    out.append((w.done(), data))
    return out


def corpus():
    """[(name, BGZF bytes)] of valid streams."""
    out = []
    for name in GOLDEN_NAMES:
        g = load_golden(name)
        caps = g["loci"][:len(g["params"]["loci"])]
        for block in (65280, 1024):
            out.append(("%s_%d" % (name, block), write_bam(coordinate_sorted(caps), [(c["ref_allele"], 100000) for c in caps],
                                                           block=block)))
    rng = random.Random(7)
    text = b"".join(b"r%d\t99\tA*01:01\t%d\t60\t100M\t=\t%d\t350\t%s\n" % (
        i, rng.randrange(1, 3000), rng.randrange(1, 3000), bytes(rng.choice(b"ACGT") for _ in range(100)))
        for i in range(1500))
    for level in (0, 1, 6, 9):
        out.append(("level%d" % level, stream(text, level=level)))
    for sname in ("Z_FIXED", "Z_HUFFMAN_ONLY", "Z_RLE", "Z_FILTERED"):
        out.append((sname, stream(text, strategy=getattr(zlib, sname))))
    out.append(("full_flush", stream(text, flush_every=5000)))
    out.append(("full_flush_stored", stream(text[:30000], level=0, flush_every=7000)))
    noise = bytes(rng.randrange(256) for _ in range(3 * 65536))
    out.append(("incompressible", stream(noise, block=65280)))
    halves = [noise[:40000], noise[40000:65280]]  # two stored blocks in the largest member BGZF holds
    stored = b"".join(bytes([last]) + struct.pack("<HH", len(h), len(h) ^ 0xffff) + h for last, h in zip((0, 1), halves))
    out.append(("two_stored_64k", member(stored, noise[:65280]) + EOF_BLOCK))
    unit = bytes(rng.randrange(256) for _ in range(32768))
    out.append(("repetitive", stream(unit * 6, level=9)))
    out.append(("runs", stream(b"".join(bytes([rng.randrange(4) + 65]) * rng.randrange(1, 600) for _ in range(800)),
                               strategy=zlib.Z_RLE)))
    out.append(("isize0_blocks", bgzf(text[:5000], 2500)[:-28] + member(deflate(b""), b"") + bgzf(text[5000:9000], 4000)))
    out.append(("eof_only", EOF_BLOCK))
    out.append(("empty", b""))
    out.append(("unusual", b"".join(member(c, r) for c, r in _unusual()) + EOF_BLOCK))
    return out


def _fixed(syms):
    w = BitWriter()
    fixed_block(w, syms)
    return w.done()


def _dyn_header(nlen, ndist, cl_lens):
    w = BitWriter()
    w.bits(1, 1)
    w.bits(2, 2)
    w.bits(nlen - 257, 5)
    w.bits(ndist - 1, 5)
    w.bits(19 - 4, 4)
    for s in CL_ORDER:
        w.bits(cl_lens.get(s, 0), 3)
    return w


def bad_blocks():
    """[(name, block bytes, message regex)]: one malformed block per rule; each needs the zlib / read_bgzf refusal too."""
    good_raw = b"hello hello hello"
    good = deflate(good_raw)
    out = [
        ("btype3", member(b"\x07\0\0\0", b"x"), "invalid block type"),
        ("stored_len", member(b"\x01\x05\x00\x00\x00hello", b"hello"), "invalid stored block lengths"),
        ("hlit", member(_dyn_header(287, 1, CL_LENS).done() + b"\0" * 8, b"x"), "too many length or distance symbols"),
        ("hdist", member(_dyn_header(257, 31, CL_LENS).done() + b"\0" * 8, b"x"), "too many length or distance symbols"),
        ("cl_over", member(_dyn_header(257, 1, {0: 1, 1: 1, 2: 1}).done() + b"\0" * 8, b"x"), "invalid code lengths set"),
        ("cl_incomplete", member(_dyn_header(257, 1, {0: 2, 1: 2}).done() + b"\0" * 8, b"x"), "invalid code lengths set"),
        ("repeat_first", member(_raw_dyn([(16, 2, 0)], 258, 1), b"x"), "invalid bit length repeat"),
        ("repeat_past", member(_raw_dyn([(18, 7, 127), (18, 7, 127)], 258, 1), b"x"), "invalid bit length repeat"),
        ("no_eob", member(_raw_dyn([(0, 0, 0)] * 97 + [(1, 0, 0)] * 2 + [(18, 7, 127)] + [(0, 0, 0)] * 21 + [(1, 0, 0)],
                                   258, 1), b"x"), "invalid code -- missing end-of-block"),
        ("lit_over", member(_dyn_lens([(97, 1), (98, 1), (256, 1)], 257, [1]), b"x"), "invalid literal/lengths set"),
        ("lit_incomplete", member(_dyn_lens([(97, 2), (256, 2)], 257, [1]), b"x"), "invalid literal/lengths set"),
        ("dist_over", member(_dyn_lens([(97, 1), (256, 1)], 257, [1, 1, 1]), b"x"), "invalid distances set"),
        ("dist_incomplete", member(_dyn_lens([(97, 1), (256, 1)], 257, [2]), b"x"), "invalid distances set"),
        ("no_dist_code", member(_no_dist_match(), b"aaaa"), "invalid distance code"),
        ("lit286", member(_fixed([("lit", 97), ("lit", 286), ("lit", 256)]), b"a"), "invalid literal/length code"),
        ("dist30", member(_fixed([("lit", 97), ("lit", 257), ("dist", 30), ("lit", 256)]), b"aaaa"), "invalid distance code"),
        ("too_far", member(_fixed([("lit", 97), ("lit", 257), ("dist", 1), ("lit", 256)]), b"aaaa"),
         "invalid distance too far back"),
        ("isize_over", member(good, good_raw, isize=len(good_raw) - 1), "ISIZE %d, inflated more than" % (len(good_raw) - 1)),
        ("isize_under", member(good, good_raw, isize=len(good_raw) + 1),
         "ISIZE %d, inflated %d bytes" % (len(good_raw) + 1, len(good_raw))),
        ("trailing", member(good + b"\0", good_raw), "deflate stream does not end with the block"),
        ("overrun", member(good[:-2], good_raw), "deflate stream runs past the end of the block"),
        ("crc", member(good, good_raw, crc=zlib.crc32(good_raw) ^ 1), "CRC32 mismatch"),
    ]
    return out


def _dyn_lens(lit_pairs, nlen, dist_list):
    """A dynamic header with these literal/length and distance lengths, then zero padding (the set check comes first)."""
    lens = [0] * nlen
    for s, l in lit_pairs:
        lens[s] = l
    return _raw_dyn([(l, 0, 0) for l in lens + dist_list], nlen, len(dist_list))


def _raw_dyn(seq, nlen, ndist):
    w = _dyn_header(nlen, ndist, CL_LENS)
    clc = canonical(CL_LENS)
    for sym, ext, val in seq:
        w.code(*clc[sym])
        if ext:
            w.bits(val, ext)
    return w.done() + b"\0" * 8


def _no_dist_match():
    """A block without distance codes that decodes a length symbol and then needs a distance."""
    lens = [0] * 258
    lens[97], lens[256], lens[257] = 1, 2, 2
    seq = [(l, 0, 0) for l in lens] + [(0, 0, 0)]
    w = _dyn_header(258, 1, CL_LENS)
    clc = canonical(CL_LENS)
    for sym, ext, val in seq:
        w.code(*clc[sym])
    lc = canonical({97: 1, 256: 2, 257: 2})
    w.code(*lc[97])
    w.code(*lc[257])
    return w.done() + b"\0" * 4


def header_bad():
    """[(name, stream bytes, read_bgzf's message)]: header rules of the open walk."""
    good = member(deflate(b"abc"), b"abc")
    return [
        ("not_gzip", b"\x1f\x8c" + good[2:], "not a BGZF block at byte 0"),
        ("no_fextra", good[:3] + b"\0" + good[4:], "not a BGZF block at byte 0"),
        ("no_bc", member(deflate(b"abc"), b"abc", bc=False), "without the BGZF BC field at byte 0"),
        ("short_header", good[:10], "truncated BGZF block header at byte 0"),
        ("truncated", good + good[:-1], "truncated BGZF block at byte %d" % len(good)),
    ]

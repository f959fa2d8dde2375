"""Test-side BAM writer: SAM lines -> BAM records (the encoding samtools picks) -> BGZF blocks of a chosen uncompressed
size, with the EOF block.  Small block sizes put records across block boundaries."""
import struct
import zlib

EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
_CIGAR_OPS = "MIDNSHP=X"
_NT16 = {c: i for i, c in enumerate("=ACMGRSVTWYHKDBN")}


def reg2bin(beg, end):
    """BAM bin of the 0-based, end-exclusive interval [beg, end) (SAM spec 5.3)."""
    end -= 1
    if beg >> 14 == end >> 14:
        return ((1 << 15) - 1) // 7 + (beg >> 14)
    if beg >> 17 == end >> 17:
        return ((1 << 12) - 1) // 7 + (beg >> 17)
    if beg >> 20 == end >> 20:
        return ((1 << 9) - 1) // 7 + (beg >> 20)
    if beg >> 23 == end >> 23:
        return ((1 << 6) - 1) // 7 + (beg >> 23)
    if beg >> 26 == end >> 26:
        return ((1 << 3) - 1) // 7 + (beg >> 26)
    return 0


def int_tag_type(v):
    """The smallest integer type for v, as samtools stores an `XX:i:v` tag."""
    if v < 0:
        return "c" if v >= -128 else "s" if v >= -32768 else "i"
    return "C" if v <= 255 else "S" if v <= 65535 else "I"


def encode_tag(field):
    tag, ty, val = field.split(":", 2)
    out = tag.encode()
    if ty == "i":
        t = int_tag_type(int(val))
        return out + t.encode() + struct.pack("<" + t.replace("C", "B").replace("c", "b").replace("S", "H").replace("s", "h"),
                                                int(val))
    if ty == "A":
        return out + b"A" + val.encode()
    if ty in "ZH":
        return out + ty.encode() + val.encode() + b"\0"
    if ty == "B":
        sub, *vals = val.split(",")
        fmt = {"c": "b", "C": "B", "s": "h", "S": "H", "i": "i", "I": "I", "f": "f"}[sub]
        conv = float if sub == "f" else int
        return out + b"B" + sub.encode() + struct.pack("<I", len(vals)) + b"".join(struct.pack("<" + fmt, conv(x)) for x in vals)
    if ty == "f":
        return out + b"f" + struct.pack("<f", float(val))
    raise ValueError(field)


def encode_record(line, ref_index, raw_tags=b""):
    """One SAM line -> one BAM record (block_size first).  raw_tags: bytes appended to the encoded tags as they are."""
    f = line.rstrip("\n").split("\t")
    qname, flag, rname, pos, mapq, cigar, rnext, pnext, tlen, seq, qual = f[:11]
    ref = -1 if rname == "*" else ref_index[rname]
    pos0 = int(pos) - 1
    ops = []
    if cigar != "*":
        n = ""
        for c in cigar:
            if c.isdigit():
                n += c
            else:
                ops.append(int(n) << 4 | _CIGAR_OPS.index(c))
                n = ""
    rlen = sum(o >> 4 for o in ops if (o & 15) in (0, 2, 3, 7, 8))
    bin_ = reg2bin(pos0, pos0 + (rlen or 1)) if pos0 >= 0 else 4680
    next_ref = -1 if rnext == "*" else ref if rnext == "=" else ref_index[rnext]
    if seq == "*":
        seq_b, l_seq = b"", 0
    else:
        l_seq = len(seq)
        codes = [_NT16[c] for c in seq.upper()] + [0]
        seq_b = bytes(codes[i] << 4 | codes[i + 1] for i in range(0, l_seq, 2))
    if l_seq == 0:
        qual_b = b""
    elif qual == "*":
        qual_b = b"\xff" * l_seq
    else:
        qual_b = bytes(ord(c) - 33 for c in qual)
    name = qname.encode() + b"\0"
    body = struct.pack("<iiBBHHHiiii", ref, pos0, len(name), int(mapq), bin_, len(ops), int(flag), l_seq, next_ref,
                       int(pnext) - 1, int(tlen))
    body += name + b"".join(struct.pack("<I", o) for o in ops) + seq_b + qual_b
    body += b"".join(encode_tag(t) for t in f[11:]) + raw_tags
    return struct.pack("<i", len(body)) + body


def bam_header(refs, text=""):
    """refs: [(name, length)]"""
    t = text.encode()
    out = b"BAM\1" + struct.pack("<i", len(t)) + t + struct.pack("<i", len(refs))
    for name, ln in refs:
        nm = name.encode() + b"\0"
        out += struct.pack("<i", len(nm)) + nm + struct.pack("<i", ln)
    return out


def bgzf(data, block=65280, eof=True, level=6):
    """BGZF blocks of at most `block` uncompressed bytes each, plus the EOF block."""
    out = []
    for o in range(0, len(data), block):
        chunk = data[o:o + block]
        c = zlib.compressobj(level, zlib.DEFLATED, -15)
        cdata = c.compress(chunk) + c.flush()
        bsize = 18 + len(cdata) + 8
        out.append(b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", bsize - 1) + cdata +
                   struct.pack("<II", zlib.crc32(chunk), len(chunk)))
    if eof:
        out.append(EOF_BLOCK)
    return b"".join(out)


def bam_stream(lines, refs, text=""):
    """Decompressed BAM: header + one record per SAM line.  refs: [(name, length)]"""
    idx = {name: i for i, (name, _) in enumerate(refs)}
    return bam_header(refs, text) + b"".join(encode_record(l, idx) for l in lines)


def write_bam(lines, refs, block=65280, eof=True):
    return bgzf(bam_stream(lines, refs), block, eof)

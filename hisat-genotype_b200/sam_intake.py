"""Native SAM / BAM intake: the aligner's SAM text or a BAM file -> per-locus, name-grouped alignment units, without
samtools.

Replaces `samtools view <bam> <backbone> | sort -k1,1 -s` (reference hisatgenotype_typing_core.py:436-468) and the BAM
round trip in front of it (hisatgenotype_typing_common.py:1038-1054) for every locus of a sample in one pass (libhgt
hgt_sam_split_* / hgt_bam_split_*, host threads).  A BAM unit travels to the GPU as packed records and is rendered into
alignment text there (hgt_batch_add_unit_bam)."""
from __future__ import annotations

import ctypes
import os
import struct
import zlib

import numpy as np

from . import _lib


def split_sam(sam_text, ref_names, n_threads=0, pinned=None, drop_qual=False):
    """sam_text: bytes of SAM (headers allowed, any record order).  ref_names: backbone names (RNAME), e.g. "A*BACKBONE".
    Returns {ref_name: bytes}, or with pinned=_lib.PinnedText {ref_name: (address, n_bytes)} written into it.
    drop_qual: write '*' for the QUAL column (never read by typing; 27 % fewer bytes to copy to the GPU for 2x100 bp records)."""
    if isinstance(sam_text, str):
        sam_text = sam_text.encode()
    L = _lib.lib()
    n = len(ref_names)
    enc = [r.encode() for r in ref_names]
    arr = (ctypes.c_char_p * n)(*enc)
    h = ctypes.c_void_p()
    L.hgt_sam_split_create_opts.restype = ctypes.c_int
    L.hgt_sam_split_create_opts.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int32, ctypes.POINTER(ctypes.c_char_p),
                                            ctypes.c_int32, ctypes.c_int32, ctypes.POINTER(ctypes.c_void_p)]
    rc = L.hgt_sam_split_create_opts(sam_text, len(sam_text), n, arr, int(n_threads), 1 if drop_qual else 0, ctypes.byref(h))
    if rc == _lib.HGT_ERR_PARSE:
        raise AssertionError(_lib.last_error())
    _lib.check(rc)
    try:
        sizes = (ctypes.c_size_t * n)()
        lines = (ctypes.c_int64 * n)()
        _lib.check(L.hgt_sam_split_sizes(h, sizes, lines))
        out = {}
        for r, name in enumerate(ref_names):
            if pinned is not None:
                addr, nb = pinned.reserve(sizes[r])
                _lib.check(L.hgt_sam_split_write(h, r, ctypes.c_void_p(addr)))
                out[name] = (addr, nb)
            else:
                buf = np.empty(max(int(sizes[r]), 1), np.uint8)
                _lib.check(L.hgt_sam_split_write(h, r, buf.ctypes.data_as(ctypes.c_void_p)))
                out[name] = buf[:sizes[r]].tobytes()
        return out
    finally:
        L.hgt_sam_split_free(h)


class BamUnit(bytes):
    """A packed BAM unit (hgt_bam_split_write_records; layout in csrc/bam_dev.cuh): what split_bam returns per reference, and
    what Batch.add_unit_bam / typing_from_alignments take in place of alignment text."""


_BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def _bgzf_blocks(data):
    """(start, end) of every BGZF block: gzip members whose extra field carries BC with BSIZE = block size - 1."""
    blocks = []
    o, n = 0, len(data)
    while o < n:
        assert n - o >= 18, "truncated BGZF block header at byte %d" % o
        assert data[o] == 31 and data[o + 1] == 139 and data[o + 2] == 8 and data[o + 3] & 4, \
            "not a BGZF block at byte %d" % o
        xlen = struct.unpack_from("<H", data, o + 10)[0]
        assert o + 12 + xlen <= n, "truncated BGZF block header at byte %d" % o
        x, bsize = o + 12, None
        while x + 4 <= o + 12 + xlen:
            si1, si2, slen = data[x], data[x + 1], struct.unpack_from("<H", data, x + 2)[0]
            if si1 == 66 and si2 == 67 and slen == 2:
                bsize = struct.unpack_from("<H", data, x + 4)[0]
            x += 4 + slen
        assert bsize is not None, "gzip member without the BGZF BC field at byte %d" % o
        end = o + bsize + 1
        assert 12 + xlen + 8 <= bsize + 1 and end <= n, "truncated BGZF block at byte %d" % o
        blocks.append((o, end, 12 + xlen))
        o = end
    return blocks


def _inflate_blocks(data, blocks):
    out = []
    for o, end, head in blocks:
        crc, isize = struct.unpack_from("<II", data, end - 8)
        d = zlib.decompressobj(-15)
        try:
            raw = d.decompress(bytes(data[o + head:end - 8]))
        except zlib.error as e:
            raise AssertionError("corrupt BGZF block at byte %d: %s" % (o, e))
        assert d.eof and not d.unused_data, "corrupt BGZF block at byte %d (deflate stream does not end with the block)" % o
        assert len(raw) == isize, "BGZF block at byte %d: ISIZE %d, inflated %d bytes" % (o, isize, len(raw))
        assert zlib.crc32(raw) == crc, "BGZF block at byte %d: CRC32 mismatch" % o
        out.append(raw)
    return b"".join(out)


def read_bgzf(data, n_threads=0):
    """Inflate a BGZF file (BAM's compression) to its uncompressed bytes: blocks inflate in parallel on a thread pool
    (zlib releases the GIL), every block's CRC32 and ISIZE are checked.  A missing EOF marker block is accepted, as
    samtools accepts it (with a warning); a truncated or corrupt block raises AssertionError."""
    import os
    from concurrent.futures import ThreadPoolExecutor
    data = memoryview(data)
    blocks = _bgzf_blocks(data)
    if not bytes(data[-len(_BGZF_EOF):]) == _BGZF_EOF:
        import warnings
        warnings.warn("BGZF input has no EOF marker block; it may be truncated")
    n_threads = int(n_threads) or os.cpu_count() or 1
    if n_threads <= 1 or len(blocks) < 64:
        return _inflate_blocks(data, blocks)
    per = max(16, (len(blocks) + 4 * n_threads - 1) // (4 * n_threads))
    chunks = [blocks[i:i + per] for i in range(0, len(blocks), per)]
    with ThreadPoolExecutor(n_threads) as pool:
        return b"".join(pool.map(lambda c: _inflate_blocks(data, c), chunks))


def _bgzf_run(streams, inflate, pinned):
    """hgt_bgzf_open on the streams (any buffers), then inflate(handle, dst) into page-locked memory (pinned: True for a
    new arena, or a _lib.PinnedText to take it from) or into ordinary memory (False): one buffer per stream.  Header
    errors and rejected blocks raise AssertionError (HGT_ERR_PARSE)."""
    L = _lib.lib()
    arrs = [np.frombuffer(s, np.uint8) for s in streams]
    n = len(arrs)
    ptrs = (ctypes.c_void_p * max(n, 1))(*[a.ctypes.data if a.size else None for a in arrs])
    sizes = (ctypes.c_size_t * max(n, 1))(*[a.size for a in arrs])
    h = ctypes.c_void_p()
    rc = L.hgt_bgzf_open(n, ptrs, sizes, ctypes.byref(h))
    if rc == _lib.HGT_ERR_PARSE:
        raise AssertionError(_lib.last_error())
    _lib.check(rc)
    try:
        out_n = (ctypes.c_size_t * max(n, 1))()
        eof = (ctypes.c_int32 * max(n, 1))()
        _lib.check(L.hgt_bgzf_sizes(h, out_n, None, eof))
        for i in range(n):
            if not eof[i]:
                import warnings
                warnings.warn("BGZF input has no EOF marker block; it may be truncated")
        if pinned:
            arena = pinned if isinstance(pinned, _lib.PinnedText) else _lib.PinnedText(sum(out_n[:n]) + 16 * n + 16)
            addrs = [arena.reserve(out_n[i])[0] for i in range(n)]
            outs = [arena.view(a, out_n[i]) for i, a in enumerate(addrs)]
        else:
            outs = [np.empty(out_n[i], np.uint8) for i in range(n)]
            addrs = [o.ctypes.data for o in outs]
            outs = [memoryview(o) for o in outs]
        rc = inflate(h, (ctypes.c_void_p * max(n, 1))(*addrs))
        if rc == _lib.HGT_ERR_PARSE:
            raise AssertionError(_lib.last_error())
        _lib.check(rc)
        return outs
    finally:
        L.hgt_bgzf_free(h)


def inflate_bgzf(streams, device=None, pinned=None):
    """Inflate BGZF streams (a list of buffers, e.g. BAM files) on the GPU in one call: one warp per block, every block's
    CRC32 and ISIZE checked on the device (hgt_bgzf_inflate).  Returns one buffer per stream, backed by page-locked memory,
    whose bytes() equal read_bgzf's.  A missing EOF block warns as read_bgzf does; a malformed or corrupt block raises
    AssertionError naming the stream and byte offset.  A block of ISIZE > 65536 (which no BGZF writer produces) is refused
    here, and read_bgzf accepts it.  pinned: a _lib.PinnedText to take the output from instead of a new allocation."""
    L = _lib.lib()
    ctx = _lib.ctx(device)
    return _bgzf_run(streams, lambda h, dst: L.hgt_bgzf_inflate(ctx, h, dst), pinned if pinned is not None else True)


def inflate_bgzf_host(streams, n_threads=0):
    """The host emulation of inflate_bgzf (hgt_bgzf_inflate_host: the device decoder's code on host threads) - test
    infrastructure, not on the typing path; the buffers are in ordinary memory."""
    L = _lib.lib()
    return _bgzf_run(streams, lambda h, dst: L.hgt_bgzf_inflate_host(h, int(n_threads), dst), False)


def split_bam(bam_bytes, ref_names, n_threads=0, pinned=None, drop_qual=False, text=False):
    """bam_bytes: a BAM file (BGZF, inflated first by read_bgzf) or its decompressed stream (any buffer, e.g. what
    inflate_bgzf returns; it is read in place).  ref_names: backbone names.
    Returns {ref_name: BamUnit} (packed records for Batch.add_unit_bam), with text=True {ref_name: bytes} (the SAM text
    `samtools view` prints for the same records, in the same order as split_sam), or with pinned=_lib.PinnedText
    {ref_name: (address, n_bytes)} of either written into it.  Records are bucketed and ordered as split_sam does.
    drop_qual: the QUAL bytes are left out ('*' in the text).  Malformed input raises AssertionError; float tags and the
    CG long-CIGAR tag raise HgtError (HGT_ERR_UNSUPPORTED)."""
    if bytes(bam_bytes[:2]) == b"\x1f\x8b":
        bam_bytes = read_bgzf(bam_bytes, n_threads)
    stream = np.frombuffer(bam_bytes, np.uint8)  # no copy: the split reads the caller's buffer (alive until the handle is freed)
    L = _lib.lib()
    n = len(ref_names)
    enc = [r.encode() for r in ref_names]
    arr = (ctypes.c_char_p * n)(*enc)
    h = ctypes.c_void_p()
    rc = L.hgt_bam_split_create(stream.ctypes.data_as(ctypes.c_void_p), stream.size, n, arr, int(n_threads),
                                1 if drop_qual else 0, ctypes.byref(h))
    if rc == _lib.HGT_ERR_PARSE:
        raise AssertionError(_lib.last_error())
    _lib.check(rc)
    try:
        sizes = (ctypes.c_size_t * n)()
        if text:
            _lib.check(L.hgt_bam_split_sizes(h, None, sizes, None))
            write = L.hgt_bam_split_write_text
        else:
            _lib.check(L.hgt_bam_split_sizes(h, sizes, None, None))
            write = L.hgt_bam_split_write_records
        out = {}
        for r, name in enumerate(ref_names):
            if pinned is not None:  # PinnedText hands out 16-byte aligned slices
                addr, nb = pinned.reserve(sizes[r])
                _lib.check(write(h, r, ctypes.c_void_p(addr)))
                out[name] = (addr, nb)
            else:
                buf = np.empty(max(int(sizes[r]), 8) // 8 + 1, np.uint64)  # 8-byte aligned
                _lib.check(write(h, r, buf.ctypes.data_as(ctypes.c_void_p)))
                data = buf.view(np.uint8)[:sizes[r]].tobytes()
                out[name] = data if text else BamUnit(data)
        return out
    finally:
        L.hgt_bam_split_free(h)


def hisat2_command(simulation, index_name, base_fname, read_fname, fastq, threads):
    """The command line of the reference's align_reads() for aligner == "hisat2" on a graph index
    (hisatgenotype_typing_common.py:995-1024), without the samtools stages behind it."""
    cmd = ["hisat2", "--mm"]
    if not simulation:
        cmd += ["--no-unal"]
    cmd += ["--no-spliced-alignment", "-X", "1000", "--max-altstried", "64", "--haplotype"]
    if base_fname == "codis":
        cmd += ["--enable-codis", "--no-softclip"]
    cmd += ["-x", index_name]
    assert len(read_fname) in (1, 2)
    cmd += ["-p", str(threads)]
    if not fastq:
        cmd += ["-f"]
    if len(read_fname) == 1:
        cmd += ["-U", read_fname[0]]
    else:
        cmd += ["-1", "%s" % read_fname[0], "-2", "%s" % read_fname[1]]
    return cmd


def align_to_sam(simulation, index_name, base_fname, read_fname, fastq, threads, verbose=0):
    """HISAT2's SAM text straight from its stdout: no `samtools view -bS`, `sort`, `index` (common:1033-1056)."""
    import subprocess
    import sys
    cmd = hisat2_command(simulation, index_name, base_fname, read_fname, fastq, threads)
    if verbose >= 1:
        print(" ".join(cmd), file=sys.stderr)
    proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL)
    return proc.stdout


def read_alignment(path, n_threads=0, device=None):
    """The alignment file as the native intake takes it: ("sam", text), ("bam", decompressed BAM stream), or (None, None)
    for what stays with samtools, like the reference: CRAM, and BGZF that is not BAM.  With a device, a BGZF file is read
    into page-locked memory and inflated on that GPU (inflate_bgzf); the BAM stream is then a page-locked buffer."""
    with open(path, "rb") as f:
        head = f.read(4)
        if device is not None and head[:2] == b"\x1f\x8b" and head[3:4] and head[3] & 4:
            n = os.fstat(f.fileno()).st_size
            pinned = _lib.PinnedText(n)
            data = pinned.view(pinned.reserve(n)[0], n)
            f.seek(0)
            got = 0
            while got < n:
                k = f.readinto(data[got:])
                if not k:
                    break
                got += k
            raw = inflate_bgzf([data[:got]], device)[0]
            return ("bam", raw) if bytes(raw[:4]) == b"BAM\1" else (None, None)
        f.seek(0)
        data = f.read()
    if data[:4] == b"CRAM":
        return None, None
    if data[:2] == b"\x1f\x8b":
        raw = read_bgzf(data, n_threads) if data[3:4] and data[3] & 4 else b""
        if raw[:4] != b"BAM\1":
            return None, None
        return "bam", raw
    return "sam", data

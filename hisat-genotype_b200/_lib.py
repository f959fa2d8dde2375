"""ctypes binding of libhgt.so (C ABI in include/hgt.h).  There is no CPU fallback: if the CUDA library is
missing or no B200 is visible, every entry point raises."""
from __future__ import annotations

import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhgt.so")

HGT_OK, HGT_ERR_CUDA, HGT_ERR_KEY, HGT_ERR_ZERODIV, HGT_ERR_ARG = 0, -1, -2, -3, -4
HGT_ERR_UNSUPPORTED, HGT_ERR_PARSE, HGT_ERR_AMBIGUITY, HGT_ERR_NOMEM, HGT_ERR_PEER = -5, -6, -7, -8, -9

c_void_p, c_int, c_i32, c_i64, c_size_t = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int32, ctypes.c_int64,
                                           ctypes.c_size_t)
P = ctypes.POINTER


class HgtError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libhgt error %d: %s" % (code, msg))
        self.code = code


EM_FORM_COMPACT, EM_FORM_STREAM, EM_FORM_COOP = 0, 1, 2
EM_FORM_NAMES = {EM_FORM_COMPACT: "compact", EM_FORM_STREAM: "stream", EM_FORM_COOP: "coop"}


class EmForm(ctypes.Structure):
    """hgt_em_form_info (include/hgt.h)."""
    _fields_ = [("form", ctypes.c_int32), ("grid", ctypes.c_int32), ("na", ctypes.c_int32), ("slab_rows", ctypes.c_int32),
                ("slab_bytes", ctypes.c_int64), ("merge", ctypes.c_int32), ("collapse", ctypes.c_int32),
                ("batch_coop", ctypes.c_int32)]


_lib = None
_ctx = {}


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "libhgt.so not built (%s): run `python -c 'import __graft_entry__ as g; g.build()'` or "
                "`make -C hisat-genotype_b200/csrc`; this package has no CPU fallback" % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        L.hgt_last_error.restype = ctypes.c_char_p
        L.hgt_abi_version.restype = c_int
        L.hgt_row_pitch.restype = c_int
        L.hgt_row_pitch.argtypes = [c_int]
        L.hgt_init.restype = c_int
        L.hgt_init.argtypes = [c_int, P(c_void_p)]
        L.hgt_free.restype = None
        L.hgt_free.argtypes = [c_void_p]
        L.hgt_launch_count.restype = c_i64
        L.hgt_launch_count.argtypes = [c_void_p]
        L.hgt_sm_count.restype = c_int
        L.hgt_sm_count.argtypes = [c_void_p]
        L.hgt_em.restype = c_int
        L.hgt_em.argtypes = [c_void_p, c_void_p, c_void_p, c_i32, c_i32, c_i32, c_void_p, c_i32, c_void_p, c_void_p,
                             c_void_p, P(c_i32)]
        L.hgt_em_f64.restype = c_int
        L.hgt_em_f64.argtypes = L.hgt_em.argtypes
        L.hgt_em_batch.restype = c_int
        L.hgt_em_batch.argtypes = [c_void_p, c_i32, c_void_p, c_void_p, c_void_p, c_void_p, c_i32, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
        L.hgt_em_workspace_bytes.restype = c_size_t
        L.hgt_em_workspace_bytes.argtypes = [c_void_p, c_i32, c_i32]
        L.hgt_em_dev.restype = c_int
        L.hgt_em_dev.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_i32, c_i32, c_i32, c_void_p, c_i32, c_i32,
                                 c_i32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
        L.hgt_em_form.restype = c_int
        L.hgt_em_form.argtypes = [c_void_p, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, P(EmForm)]
        L.hgt_batch_add_units.restype = c_i64
        L.hgt_batch_add_units.argtypes = [c_void_p, c_i64, c_void_p, c_void_p, c_void_p]
        L.hgt_batch_abundances.restype = c_int
        L.hgt_batch_abundances.argtypes = [c_void_p, c_i32, c_void_p, c_void_p, c_void_p, c_void_p]
        L.hgt_sam_split_create.restype = c_int
        L.hgt_sam_split_create.argtypes = [ctypes.c_char_p, c_size_t, c_i32, c_void_p, c_i32, P(c_void_p)]
        L.hgt_sam_split_sizes.restype = c_int
        L.hgt_sam_split_sizes.argtypes = [c_void_p, c_void_p, c_void_p]
        L.hgt_sam_split_write.restype = c_int
        L.hgt_sam_split_write.argtypes = [c_void_p, c_i32, c_void_p]
        L.hgt_sam_split_free.restype = None
        L.hgt_sam_split_free.argtypes = [c_void_p]
        L.hgt_bam_split_create.restype = c_int
        L.hgt_bam_split_create.argtypes = [c_void_p, c_size_t, c_i32, c_void_p, c_i32, c_i32, P(c_void_p)]
        L.hgt_bam_split_sizes.restype = c_int
        L.hgt_bam_split_sizes.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p]
        L.hgt_bam_split_write_records.restype = c_int
        L.hgt_bam_split_write_records.argtypes = [c_void_p, c_i32, c_void_p]
        L.hgt_bam_split_write_text.restype = c_int
        L.hgt_bam_split_write_text.argtypes = [c_void_p, c_i32, c_void_p]
        L.hgt_bam_split_free.restype = None
        L.hgt_bam_split_free.argtypes = [c_void_p]
        L.hgt_bgzf_open.restype = c_int
        L.hgt_bgzf_open.argtypes = [c_i32, c_void_p, c_void_p, P(c_void_p)]
        L.hgt_bgzf_sizes.restype = c_int
        L.hgt_bgzf_sizes.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p]
        L.hgt_bgzf_inflate.restype = c_int
        L.hgt_bgzf_inflate.argtypes = [c_void_p, c_void_p, c_void_p]
        L.hgt_bgzf_inflate_host.restype = c_int
        L.hgt_bgzf_inflate_host.argtypes = [c_void_p, c_i32, c_void_p]
        L.hgt_bgzf_free.restype = None
        L.hgt_bgzf_free.argtypes = [c_void_p]
        L.hgt_batch_add_unit_bam.restype = c_i64
        L.hgt_batch_add_unit_bam.argtypes = [c_void_p, c_i32, c_void_p, c_size_t]
        L.hgt_bam_dsplit_create.restype = c_int
        L.hgt_bam_dsplit_create.argtypes = [c_void_p, c_void_p, c_i32, c_void_p, c_i32, P(c_void_p)]
        L.hgt_bam_dsplit_sizes.restype = c_int
        L.hgt_bam_dsplit_sizes.argtypes = [c_void_p, c_void_p, c_void_p]
        L.hgt_bam_dsplit_free.restype = None
        L.hgt_bam_dsplit_free.argtypes = [c_void_p]
        L.hgt_batch_add_unit_bam_dsplit.restype = c_i64
        L.hgt_batch_add_unit_bam_dsplit.argtypes = [c_void_p, c_i32, c_void_p, c_i32, c_i32]
        L.hgt_bam_index_host.restype = c_int
        L.hgt_bam_index_host.argtypes = [c_void_p, c_size_t, c_i64, c_i32, c_i64, c_void_p, P(c_i64)]
        L.hgt_batch_unit_text.restype = c_int
        L.hgt_batch_unit_text.argtypes = [c_void_p, c_i64, c_void_p, P(c_size_t)]
        L.hgt_batch_unit_reads.restype = c_int
        L.hgt_batch_unit_reads.argtypes = [c_void_p, c_i64] + [c_void_p] * 10
        L.hgt_pair_em.restype = c_int
        L.hgt_pair_em.argtypes = [c_void_p, c_void_p, c_void_p, c_i32, c_i32, c_void_p, c_i32, c_void_p, c_void_p, P(c_i32)]
        L.hgt_host_alloc.restype = c_int
        L.hgt_host_alloc.argtypes = [c_size_t, P(c_void_p)]
        L.hgt_host_free.restype = None
        L.hgt_host_free.argtypes = [c_void_p]
        L.hgt_profile_enable.restype = None
        L.hgt_profile_enable.argtypes = [c_void_p, c_int]
        L.hgt_profile_reset.restype = None
        L.hgt_profile_reset.argtypes = [c_void_p]
        L.hgt_profile_read.restype = None
        L.hgt_profile_read.argtypes = [c_void_p, c_void_p, c_void_p, P(c_i64), P(c_i64)]
        L.hgt_profile_host.restype = None
        L.hgt_profile_host.argtypes = [c_void_p, c_void_p]
        _lib = L
    return _lib


def last_error():
    return lib().hgt_last_error().decode("utf-8", "replace")


def check(rc):
    if rc != HGT_OK:
        raise HgtError(rc, last_error())


def default_device():
    for k in ("HGT_DEVICE", "LOCAL_RANK"):
        if os.environ.get(k, "") != "":
            return int(os.environ[k])
    return 0


def ctx(device=None):
    """Lazily created per (process, device) context — safe under multiprocessing fork because nothing touches
    CUDA before the first call in the worker (the reference runs typing in Pool workers, hisatgenotype:613)."""
    dev = default_device() if device is None else device
    key = (os.getpid(), dev)
    if key not in _ctx:
        h = c_void_p()
        check(lib().hgt_init(dev, ctypes.byref(h)))
        _ctx[key] = h
    return _ctx[key]


def new_ctx(device=None):
    """An additional context on the device (own stream, own buffer pool, own counters): batches on different contexts may
    run from different host threads at the same time (typing_core.BatchPipeline).  Loci may be shared between them."""
    dev = default_device() if device is None else device
    h = c_void_p()
    check(lib().hgt_init(dev, ctypes.byref(h)))
    return h


class PinnedText:
    """Alignment text of many units in ONE page-locked allocation (hgt_host_alloc): the copy engine reads it directly.
    add(bytes) -> (address, length) to hand to Batch.add_unit_ptr()."""

    def __init__(self, capacity):
        self.cap = int(capacity)
        self.used = 0
        self.base = c_void_p()
        check(lib().hgt_host_alloc(self.cap, ctypes.byref(self.base)))

    def add(self, data):
        n = len(data)
        if self.used + n > self.cap:
            raise MemoryError("PinnedText: capacity %d exceeded" % self.cap)
        addr = self.base.value + self.used
        ctypes.memmove(addr, data, n)
        self.used += (n + 15) & ~15
        return addr, n

    def reserve(self, n):
        """n bytes of the arena for the caller to fill: (address, n)."""
        n = int(n)
        if self.used + n > self.cap:
            raise MemoryError("PinnedText: capacity %d exceeded" % self.cap)
        addr = self.base.value + self.used
        self.used += (n + 15) & ~15
        return addr, n

    def reset(self):
        """Hand the whole arena out again; earlier slices are no longer the caller's."""
        self.used = 0

    def view(self, addr, n):
        """A writable buffer (memoryview of unsigned bytes) over [addr, addr + n) of the arena; it keeps the arena alive."""
        arr = (ctypes.c_ubyte * int(n)).from_address(addr)
        arr._owner = self
        return memoryview(np.ctypeslib.as_array(arr)) if n else memoryview(b"")

    def close(self):
        if self.base is not None and self.base.value:
            lib().hgt_host_free(self.base)
            self.base = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def em_form(n_classes, n_alleles, wp=None, has_lengths=False, n_ctas=0, a_live_max=0, n_problems=1, device=None):
    """The form hgt_em_dev runs a problem of this size in (hgt_em_form): EmForm."""
    out = EmForm()
    check(lib().hgt_em_form(ctx(device), int(n_classes), int(n_alleles), int(wp or row_pitch(n_alleles)),
                            1 if has_lengths else 0, int(n_ctas), int(a_live_max), int(n_problems), ctypes.byref(out)))
    return out


def ptr(a):
    return None if a is None else a.ctypes.data_as(c_void_p)


def row_pitch(n_alleles):
    return lib().hgt_row_pitch(int(n_alleles))


def pack_bits(index_lists, n_alleles, wp=None):
    """[[allele index,...],...] -> uint64 [n][wp] bit matrix."""
    wp = wp or row_pitch(n_alleles)
    out = np.zeros((len(index_lists), wp), np.uint64)
    for k, idx in enumerate(index_lists):
        idx = np.asarray(idx, np.int64)
        if idx.size:
            np.bitwise_or.at(out[k], idx >> 6, np.uint64(1) << (idx & 63).astype(np.uint64))
    return out


def unpack_bits(row, n_alleles):
    """uint64 row -> sorted allele indices."""
    b = np.unpackbits(np.ascontiguousarray(row).view(np.uint8), bitorder="little")[:n_alleles]
    return np.nonzero(b)[0]

"""EM abundance for ONE locus whose reads (hence class tables) are sharded over several GPUs (SURVEY.md 8e).

Every rank holds the Gene_cmpt classes of its own reads; a class can occur on several ranks.  The pieces, in the order
Batch.sharded_abundance uses them:
    pileup_allreduce_hook   sums the raw pileup counts over the ranks before the representative-base sets are derived
                            (the reference uses the pileup of ALL reads, common:1124-1134)
    merge_class_tables      gathers every rank's class table (gather_class_tables: NCCL all_gather, once per call) and
                            keeps the rows this rank owns, duplicates merged (CUDA: hgt_class_merge_dev, csrc/typing.cu),
                            so that every class lives on exactly one rank
    single_abundance_peer   the reference loop (common:1282-1410) as ONE cooperative kernel per rank that sums the
                            per-allele accumulators of every sweep over the ranks through NVLink peer memory
                            (CUDA: hgt_em_peer_dev, csrc/em.cu; exchange blocks mapped with CUDA IPC by PeerGroup)
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib

FK_NONE = 0x7FFFFFFF


class _DevAlias:
    """A raw device pointer as a __cuda_array_interface__ object (torch.as_tensor makes a zero-copy view of it)."""

    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"data": (int(ptr), False), "shape": (int(n),), "typestr": typestr, "version": 2}


def _alias(ptr, n, typestr, device):
    return torch.as_tensor(_DevAlias(ptr, n, typestr), device=device)


class PeerGroup:
    """Exchange blocks of all ranks for the peer-memory EM (hgt_em_peer_dev): every rank cudaMallocs one block, the
    64-byte CUDA IPC handles travel through one all_gather and every rank maps the others' blocks.  Creation is a
    collective call; instances are cached per (device, allele count, group)."""
    _cache = {}

    def __init__(self, n_alleles, dev_index, group=None):
        import torch.distributed as dist
        self.L = _lib.lib()
        self.ctx = _lib.ctx(dev_index)
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        L = self.L
        L.hgt_em_peer_alloc.restype = ctypes.c_int
        L.hgt_em_peer_alloc.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.POINTER(ctypes.c_void_p), ctypes.c_char_p]
        L.hgt_em_peer_open.restype = ctypes.c_int
        L.hgt_em_peer_open.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.POINTER(ctypes.c_void_p)]
        L.hgt_em_peer_close.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.hgt_em_peer_free.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        own = ctypes.c_void_p()
        handle = ctypes.create_string_buffer(64)
        _lib.check(L.hgt_em_peer_alloc(self.ctx, int(n_alleles), ctypes.byref(own), handle))
        self.own = own.value
        self.blocks = (ctypes.c_void_p * self.world)()
        self.blocks[self.rank] = self.own
        if self.world > 1:
            dev = torch.device("cuda", dev_index)
            mine = torch.frombuffer(bytearray(handle.raw), dtype=torch.uint8).to(dev)
            every = torch.empty(self.world * 64, dtype=torch.uint8, device=dev)
            dist.all_gather_into_tensor(every, mine, group=group)
            every = every.cpu().numpy().tobytes()
            for r in range(self.world):
                if r == self.rank:
                    continue
                p = ctypes.c_void_p()
                _lib.check(L.hgt_em_peer_open(self.ctx, every[64 * r:64 * r + 64], ctypes.byref(p)))
                self.blocks[r] = p.value
            dist.barrier(group=group)  # nobody launches before every block is mapped everywhere

    @classmethod
    def get(cls, n_alleles, dev_index, group=None):
        key = (dev_index, int(n_alleles), id(group))
        if key not in cls._cache:
            cls._cache[key] = cls(n_alleles, dev_index, group)
        return cls._cache[key]


def gather_class_tables(bits, cnt, first, wp, group=None):
    """All ranks' class tables, concatenated in rank order: (rows int64 [n_total * wp], count int64 [n_total], first int32
    [n_total], n_total).  Inputs are torch tensors of this rank (any device the group's backend serves: CUDA under NCCL, CPU
    under gloo - tests/test_dist_em.py); tables may have different lengths, also zero."""
    import torch.distributed as dist
    dev = bits.device
    world = dist.get_world_size(group)
    n = int(cnt.numel())
    n_t = torch.tensor([n], dtype=torch.int64, device=dev)
    n_all = [torch.zeros_like(n_t) for _ in range(world)]
    dist.all_gather(n_all, n_t, group=group)
    n_all = [int(x) for x in n_all]
    n_max = max(max(n_all), 1)
    p_bits = torch.zeros(n_max * wp, dtype=torch.int64, device=dev)
    p_cnt = torch.zeros(n_max, dtype=torch.int64, device=dev)
    p_first = torch.zeros(n_max, dtype=torch.int32, device=dev)
    if n > 0:
        p_bits[:n * wp] = bits.reshape(-1)
        p_cnt[:n] = cnt
        p_first[:n] = first
    g_bits = [torch.empty_like(p_bits) for _ in range(world)]
    g_cnt = [torch.empty_like(p_cnt) for _ in range(world)]
    g_first = [torch.empty_like(p_first) for _ in range(world)]
    dist.all_gather(g_bits, p_bits, group=group)
    dist.all_gather(g_cnt, p_cnt, group=group)
    dist.all_gather(g_first, p_first, group=group)
    # drop the padding rows
    return (torch.cat([g_bits[r][:n_all[r] * wp] for r in range(world)]), torch.cat([g_cnt[r][:n_all[r]] for r in range(world)]),
            torch.cat([g_first[r][:n_all[r]] for r in range(world)]), sum(n_all))


def merge_class_tables(A, wp, bits_ptr, cnt_ptr, first_ptr, n, key_offset, dev_index, group=None):
    """All ranks' class tables -> the rows this rank owns, duplicates merged (hgt_class_merge_dev).  Returns torch
    tensors (rows int64 [m * wp], count int64 [m], first int32 [m]) and m.  The tables travel once per call with NCCL
    all_gather (bulk transfer: what NCCL is for); the latency-critical per-sweep exchange of the EM is the peer kernel."""
    import torch.distributed as dist
    dev = torch.device("cuda", dev_index)
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    n = int(n)
    if n > 0:
        bits = _alias(bits_ptr, n * wp, "<i8", dev)
        cnt = _alias(cnt_ptr, n, "<i8", dev)
        first = _alias(first_ptr, n, "<i4", dev) + int(key_offset)  # global pair indices
    else:
        bits = torch.zeros(0, dtype=torch.int64, device=dev)
        cnt = torch.zeros(0, dtype=torch.int64, device=dev)
        first = torch.zeros(0, dtype=torch.int32, device=dev)
    g_bits, g_cnt, g_first, n_in = gather_class_tables(bits, cnt, first, wp, group)
    o_bits, o_cnt, o_first, m = merge_rows(g_bits, g_cnt, g_first, n_in, A, wp, rank, world, dev_index)
    # rows in the order of their first pair (unique, = the reference's dict order): the kernel hands rows out in warp-scheduling
    # order, and the row order decides the floating-point association of the EM sums - sorted, a run repeats bit for bit
    order = torch.argsort(o_first[:m])
    return (o_bits.view(-1, wp)[:m][order].contiguous().view(-1), o_cnt[:m][order].contiguous(), o_first[:m][order].contiguous(), m)


def merge_rows(g_bits, g_cnt, g_first, n_in, A, wp, rank, world, dev_index):
    """hgt_class_merge_dev on gathered rows (torch tensors on the device): the rows rank `rank` of `world` owns."""
    dev = torch.device("cuda", dev_index)
    L = _lib.lib()
    L.hgt_class_merge_workspace_bytes.restype = ctypes.c_size_t
    L.hgt_class_merge_workspace_bytes.argtypes = [ctypes.c_int64]
    L.hgt_class_merge_dev.restype = ctypes.c_int
    L.hgt_class_merge_dev.argtypes = [ctypes.c_void_p] * 5 + [ctypes.c_int64] + [ctypes.c_int32] * 4 + [ctypes.c_void_p] * 5
    ws = torch.empty(L.hgt_class_merge_workspace_bytes(n_in), dtype=torch.uint8, device=dev)
    o_bits = torch.empty(max(n_in, 1) * wp, dtype=torch.int64, device=dev)
    o_cnt = torch.empty(max(n_in, 1), dtype=torch.int64, device=dev)
    o_first = torch.empty(max(n_in, 1), dtype=torch.int32, device=dev)
    o_n = torch.zeros(1, dtype=torch.int32, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    _lib.check(L.hgt_class_merge_dev(_lib.ctx(dev_index), st, g_bits.data_ptr(), g_cnt.data_ptr(), g_first.data_ptr(), n_in, A, wp,
                                     rank, world, o_bits.data_ptr(), o_cnt.data_ptr(), o_first.data_ptr(), o_n.data_ptr(),
                                     ws.data_ptr()))
    m = int(o_n.item())
    return o_bits, o_cnt, o_first, m


def single_abundance_peer(A, wp, bits_ptr, cnt_u64_ptr, key_ptr, key_offset, n_classes, dev_index, allele_len=None,
                          remove_low=False, group=None, keep=()):
    """single_abundance over class rows spread over the ranks as ONE cooperative kernel per rank that sums the per-allele
    accumulators through NVLink peer memory (hgt_em_peer_dev).  Returns (prob, in_result, first_key, iters) as torch
    tensors on the device; identical on every rank."""
    dev = torch.device("cuda", dev_index)
    L = _lib.lib()
    pg = PeerGroup.get(A, dev_index, group)
    L.hgt_em_workspace_bytes.restype = ctypes.c_size_t
    L.hgt_em_workspace_bytes.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32]
    L.hgt_em_peer_dev.restype = ctypes.c_int
    L.hgt_em_peer_dev.argtypes = ([ctypes.c_void_p] * 6 + [ctypes.c_int32] * 4 + [ctypes.c_void_p] + [ctypes.c_int32] * 3 +
                                  [ctypes.c_void_p] * 6)
    ctx = _lib.ctx(dev_index)
    ws = torch.empty(L.hgt_em_workspace_bytes(ctx, int(n_classes), A), dtype=torch.uint8, device=dev)
    prob = torch.zeros(A, dtype=torch.float64, device=dev)
    inres = torch.zeros(A, dtype=torch.uint8, device=dev)
    fk = torch.full((A,), FK_NONE, dtype=torch.int32, device=dev)
    ist = torch.zeros(3, dtype=torch.int32, device=dev)
    ln = None if allele_len is None else torch.as_tensor(np.asarray(allele_len, np.float64), device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    _lib.check(L.hgt_em_peer_dev(ctx, st, bits_ptr, None, cnt_u64_ptr, key_ptr, int(key_offset), int(n_classes), A, wp,
                                 None if ln is None else ln.data_ptr(), 1 if remove_low else 0, pg.rank, pg.world, pg.blocks,
                                 prob.data_ptr(), inres.data_ptr(), fk.data_ptr(), ist.data_ptr(), ws.data_ptr()))
    iters, status, _ = ist.tolist()
    if status == _lib.HGT_ERR_KEY:
        raise KeyError("allele vanished from next_prob output during SQUAREM step")
    if status == _lib.HGT_ERR_ZERODIV:
        raise ZeroDivisionError("float division by zero")
    if status != 0:
        raise _lib.HgtError("hgt_em_peer_dev: status %d (-9 = a rank did not reach an exchange in time)" % status)
    return prob, inres != 0, fk, iters


def pileup_allreduce_hook(group=None):
    """ctypes callback for hgt_batch_set_pileup_hook: sums the raw base counts of a read-sharded locus over the ranks
    (the reference derives nt_set from the pileup of ALL reads, common:1124-1134)."""
    import torch.distributed as dist

    @ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p)
    def hook(_arg, dev_counts, n_u32, _stream):
        try:
            t = _alias(dev_counts, n_u32, "<i4", torch.device("cuda"))
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)  # int32 wrap-around == uint32 sum
            torch.cuda.synchronize()
            return 0
        except Exception:  # never unwind through the C frame
            import traceback
            traceback.print_exc()
            return 1

    return hook

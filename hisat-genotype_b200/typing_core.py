"""Host-side mirror of the reference's hisatgenotype_typing_core API for the typing hot path.

  type_locus()   stage (a) for one (sample, locus): alignment lines in, Gene_cmpt / Gene_counts out — the
                 per-read loop of typing() (reference hisatgenotype_typing_core.py:598-1596) on the GPU.
  locus_abundance()   the EM driver of typing() (core:1679-1789) on device-resident tables.
  typing() / genotyping_locus()   drop-in entry points with the reference's signatures and .report format
                 (core:249-286, 2278-2309); see report.py.
There is no CPU fallback: everything below needs libhgt.so and a B200.
"""
from __future__ import annotations

import ctypes
import os
import time

import numpy as np

from . import _lib
from .locus import LocusTables, Params, lib
from .typing_common import rank_result

TABLE_GENE, TABLE_EXON, TABLE_PRIMARY = 0, 1, 2


def make_params(num_editdist=2, error_correction=True, allow_discordant=False, simulation=False, base_locus=0,
                n_threads=0, chunk_bytes=0):
    return Params(int(num_editdist), 1 if error_correction else 0, 1 if allow_discordant else 0,
                  1 if simulation else 0, int(base_locus), int(n_threads), int(chunk_bytes))


def _sam_bytes(sam):
    if isinstance(sam, bytes):
        return sam
    if isinstance(sam, str):
        return sam.encode()
    return ("\n".join(sam) + "\n").encode()


class TypingRun:
    """Result of stage (a) for one (sample, locus); tables stay on the device until asked for."""

    def __init__(self, tables: LocusTables, sam, params: Params):
        self.tables = tables
        self.handle = ctypes.c_void_p()
        buf = _sam_bytes(sam)
        rc = lib().hgt_typing_run(_lib.ctx(tables.device), tables.handle, buf, len(buf), ctypes.byref(params),
                                  ctypes.byref(self.handle))
        if rc == _lib.HGT_ERR_AMBIGUITY:
            raise SystemExit("Error: %s" % _lib.last_error())
        if rc == _lib.HGT_ERR_PARSE:
            raise AssertionError(_lib.last_error())
        _lib.check(rc)
        nr, npairs = ctypes.c_int64(0), ctypes.c_int64(0)
        ncls = (ctypes.c_int32 * 3)()
        _lib.check(lib().hgt_typing_summary(self.handle, ctypes.byref(nr), ctypes.byref(npairs), ctypes.byref(ncls)))
        self.num_reads, self.num_pairs = nr.value, npairs.value
        self.n_classes = [ncls[0], ncls[1], ncls[2]]
        self._cache = {}

    def close(self):
        if self.handle is not None and self.handle.value:
            lib().hgt_typing_free(self.handle)
            self.handle = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def table_arrays(self, table):
        """(class_bits[C][wp], class_count[C], class_first[C], allele_count[A], allele_first[A])"""
        if table not in self._cache:
            t = self.tables
            C = self.n_classes[table]
            bits = np.zeros((max(C, 1), t.wp), np.uint64)
            cnt = np.zeros(max(C, 1), np.int64)
            first = np.zeros(max(C, 1), np.int64)
            acount = np.zeros(t.A, np.int64)
            afirst = np.zeros(t.A, np.int64)
            _lib.check(lib().hgt_typing_table(self.handle, table, _lib.ptr(bits), _lib.ptr(cnt), _lib.ptr(first),
                                              _lib.ptr(acount), _lib.ptr(afirst)))
            self._cache[table] = (bits[:C], cnt[:C], first[:C], acount, afirst)
        return self._cache[table]

    def gene_cmpt(self, table=TABLE_GENE):
        """Gene_cmpt of the table as an insertion-ordered dict (core:1229-1234)."""
        bits, cnt, _, _, _ = self.table_arrays(table)
        return {self.tables.key_of(bits[k]): int(cnt[k]) for k in range(len(cnt))}

    def gene_counts(self, table=TABLE_GENE):
        """Gene_counts in dict order: alleles enter at the first pair that counts them, in Gene_names order
        within one pair (core:1179-1190)."""
        _, _, _, acount, afirst = self.table_arrays(table)
        t = self.tables
        idx = np.nonzero(acount > 0)[0]
        order = sorted(idx.tolist(), key=lambda a: (int(afirst[a]), int(t.gn_rank[a])))
        return [[t.names[a], int(acount[a])] for a in order]

    def pileup(self):
        t = self.tables
        counts = np.zeros((len(t.ref_seq), 6), np.uint32)
        mask = np.zeros(len(t.ref_seq), np.uint8)
        _lib.check(lib().hgt_typing_pileup(self.handle, _lib.ptr(counts), _lib.ptr(mask)))
        return counts, mask

    def abundance(self, table, keep_alleles=None, lengths=None, remove_low=False):
        """single_abundance on a device-resident table; keep_alleles projects the classes first (core:1753-1766)."""
        t = self.tables
        keep = t.mask_of(keep_alleles) if keep_alleles is not None else None
        ln = None
        if lengths:
            ln = np.asarray([lengths[n] for n in t.names], np.float64)
        prob = np.zeros(t.A, np.float64)
        inres = np.zeros(t.A, np.uint8)
        fk = np.zeros(t.A, np.int32)
        iters = ctypes.c_int32(0)
        rc = lib().hgt_typing_em(_lib.ctx(t.device), self.handle, table, _lib.ptr(keep), _lib.ptr(ln),
                                 1 if remove_low else 0, _lib.ptr(prob), _lib.ptr(inres), _lib.ptr(fk),
                                 ctypes.byref(iters))
        if rc == _lib.HGT_ERR_KEY:
            raise KeyError(_lib.last_error())
        if rc == _lib.HGT_ERR_ZERODIV:
            raise ZeroDivisionError("float division by zero")
        _lib.check(rc)
        return rank_result(t.names, prob, inres, fk)


def type_locus(tables, sam, num_editdist=2, error_correction=True, allow_discordant=False, simulation=False,
               base_locus=0):
    return TypingRun(tables, sam, make_params(num_editdist, error_correction, allow_discordant, simulation,
                                              base_locus))


def locus_abundance(run: TypingRun, remove_low_abundance_alleles=True):
    """Gene_prob for one locus: the EM driver of typing() (core:1679-1789)."""
    t = run.tables
    if t.is_hla:
        exon_prob = run.abundance(TABLE_EXON, None, None, remove_low_abundance_alleles)
        gene_prob = exon_prob
        exon_alleles, exon_prob_sum = set(), 0.0
        for i, (allele, prob) in enumerate(exon_prob):
            if i >= 10 and prob < 0.03:
                break
            group = t.allele_rep_groups[allele]
            if len(group) <= 1:
                continue
            exon_prob_sum += prob
            exon_alleles |= set(group)
        if len(exon_alleles) > 0:
            full = run.abundance(TABLE_GENE, exon_alleles, t.gene_lengths, True)
            combined = {}
            for allele, prob in exon_prob:
                if allele not in exon_alleles:
                    combined[allele] = prob
            for allele, prob in full:
                combined[allele] = prob * exon_prob_sum
            gene_prob = sorted(([a, p] for a, p in combined.items()), key=lambda x: x[1], reverse=True)
        return gene_prob
    if run.n_classes[TABLE_GENE] <= 1:
        if run.n_classes[TABLE_GENE] == 1:
            # the reference evaluates Gene_cmpt.keys()[0] here, a TypeError on Python 3 (core:1787)
            raise TypeError("'dict_keys' object is not subscriptable")
        return []
    return run.abundance(TABLE_GENE, None, None, False)


class Batch:
    """Many (sample, locus) units through the GPU together (hgt_batch_* in include/hgt.h)."""

    def __init__(self, loci, params=None, remove_low_abundance_alleles=True, device=None, ctx=None):
        self.loci = list(loci)
        self.params = params or make_params()
        self.device = device
        arr = (ctypes.c_void_p * len(self.loci))(*[t.handle for t in self.loci])
        self.handle = ctypes.c_void_p()
        _lib.check(lib().hgt_batch_create(ctx or _lib.ctx(device), len(self.loci), arr, ctypes.byref(self.params),
                                          1 if remove_low_abundance_alleles else 0, ctypes.byref(self.handle)))
        self._texts = []
        self.unit_locus = []

    def add_unit(self, locus_index, sam):
        buf = _sam_bytes(sam)
        self._texts.append(buf)  # must outlive prepare()
        u = lib().hgt_batch_add_unit(self.handle, locus_index, ctypes.cast(ctypes.c_char_p(buf), ctypes.c_void_p),
                                     len(buf))
        if u < 0:
            _lib.check(int(u))
        self.unit_locus.append(locus_index)
        return int(u)

    def add_unit_ptr(self, locus_index, address, n_bytes):
        """Alignment text that already lives in (ideally page-locked, _lib.PinnedText) host memory; the caller keeps it
        valid until prepare() returns."""
        u = lib().hgt_batch_add_unit(self.handle, locus_index, ctypes.c_void_p(address), n_bytes)
        if u < 0:
            _lib.check(int(u))
        self.unit_locus.append(locus_index)
        return int(u)

    def add_unit_bam(self, locus_index, blob):
        """A packed BAM unit (sam_intake.split_bam): prepare() renders its records into alignment text on the GPU."""
        buf = np.frombuffer(blob, np.uint8)
        if buf.ctypes.data % 8:
            buf = np.frombuffer(np.frombuffer(blob + b"\0" * (-len(blob) % 8), np.uint64).copy(), np.uint8)[:len(blob)]
        self._texts.append(buf)  # must outlive prepare()
        return self.add_unit_bam_ptr(locus_index, buf.ctypes.data, len(blob))

    def add_unit_bam_ptr(self, locus_index, address, n_bytes):
        """A packed BAM unit already in (ideally page-locked, _lib.PinnedText) host memory, 8-byte aligned; the caller keeps
        it valid until prepare() returns."""
        u = lib().hgt_batch_add_unit_bam(self.handle, locus_index, ctypes.c_void_p(address), n_bytes)
        if u < 0:
            _lib.check(int(u))
        self.unit_locus.append(locus_index)
        return int(u)

    def add_unit_bam_dsplit(self, locus_index, unit):
        """A sam_intake.DeviceBamUnit: prepare() renders the bucket into alignment text straight from the split's device
        memory.  The split must stay open until prepare() returns."""
        u = lib().hgt_batch_add_unit_bam_dsplit(self.handle, locus_index, unit.split.handle, unit.stream, unit.ref)
        if u < 0:
            _lib.check(int(u))
        self._texts.append(unit.split)  # kept alive until prepare()
        self.unit_locus.append(locus_index)
        return int(u)

    def unit_text(self, u):
        """After prepare(): the unit's alignment text as it sits in the device arena (rendered on the GPU for a BAM unit)."""
        n = ctypes.c_size_t(0)
        _lib.check(lib().hgt_batch_unit_text(self.handle, u, None, ctypes.byref(n)))
        buf = np.empty(max(n.value, 1), np.uint8)
        _lib.check(lib().hgt_batch_unit_text(self.handle, u, buf.ctypes.data_as(ctypes.c_void_p), ctypes.byref(n)))
        return buf[:n.value].tobytes()

    def _call(self, rc):
        if rc == _lib.HGT_ERR_AMBIGUITY:
            raise SystemExit("Error: %s" % _lib.last_error())
        if rc == _lib.HGT_ERR_PARSE:
            raise AssertionError(_lib.last_error())
        _lib.check(rc)

    def prepare(self):
        self._call(lib().hgt_batch_prepare(self.handle))
        self._texts = []

    def execute(self, stream=None):
        self._call(lib().hgt_batch_execute(self.handle, stream))

    def finish(self, stream=None):
        self._call(lib().hgt_batch_finish(self.handle, stream))

    def run(self):
        self.prepare()
        self.execute()
        self.finish()

    def totals(self):
        v = [ctypes.c_int64(0) for _ in range(6)]
        _lib.check(lib().hgt_batch_totals(self.handle, *[ctypes.byref(x) for x in v]))
        keys = ("n_units", "num_reads", "num_pairs", "n_haplotypes", "n_rows", "algorithmic_bytes")
        return dict(zip(keys, (x.value for x in v)))

    def job_stats(self):
        v = (ctypes.c_int64 * 4)()
        _lib.check(lib().hgt_batch_job_stats(self.handle, ctypes.byref(v)))
        return dict(n_jobs=v[0], n_big_jobs=v[1], max_haplotypes_per_job=v[2], n_haplotypes=v[3])

    def unit_summary(self, u):
        nr, npairs = ctypes.c_int64(0), ctypes.c_int64(0)
        nc, it, stt = (ctypes.c_int32 * 4)(), (ctypes.c_int32 * 2)(), (ctypes.c_int32 * 2)()
        _lib.check(lib().hgt_batch_unit_summary(self.handle, u, ctypes.byref(nr), ctypes.byref(npairs),
                                                ctypes.byref(nc), ctypes.byref(it), ctypes.byref(stt)))
        return dict(num_reads=nr.value, num_pairs=npairs.value, n_classes=list(nc), em_iters=list(it),
                    em_status=list(stt))

    def unit_table(self, u, table):
        t = self.loci[self.unit_locus[u]]
        C = self.unit_summary(u)["n_classes"][table]
        bits = np.zeros((max(C, 1), t.wp), np.uint64)
        cnt = np.zeros(max(C, 1), np.int64)
        first = np.zeros(max(C, 1), np.int64)
        acount = np.zeros(t.A, np.int64)
        afirst = np.zeros(t.A, np.int64)
        _lib.check(lib().hgt_batch_unit_table(self.handle, u, table, _lib.ptr(bits), _lib.ptr(cnt), _lib.ptr(first),
                                              _lib.ptr(acount), _lib.ptr(afirst)))
        return bits[:C], cnt[:C], first[:C], acount, afirst

    def unit_gene_cmpt(self, u, table=TABLE_GENE):
        t = self.loci[self.unit_locus[u]]
        bits, cnt, _, _, _ = self.unit_table(u, table)
        return {t.key_of(bits[k]): int(cnt[k]) for k in range(len(cnt))}

    def unit_gene_counts(self, u, table=TABLE_GENE):
        t = self.loci[self.unit_locus[u]]
        _, _, _, acount, afirst = self.unit_table(u, table)
        idx = np.nonzero(acount > 0)[0]
        order = sorted(idx.tolist(), key=lambda a: (int(afirst[a]), int(t.gn_rank[a])))
        return [[t.names[a], int(acount[a])] for a in order]

    def unit_em(self, u, level):
        """Ranked [[allele, prob]] of the first- (level 0) or second-level (1) EM; None if level 1 did not run."""
        t = self.loci[self.unit_locus[u]]
        prob = np.zeros(t.A, np.float64)
        inres = np.zeros(t.A, np.uint8)
        fk = np.zeros(t.A, np.int32)
        it, stt = ctypes.c_int32(0), ctypes.c_int32(0)
        _lib.check(lib().hgt_batch_unit_em(self.handle, u, level, _lib.ptr(prob), _lib.ptr(inres), _lib.ptr(fk),
                                           ctypes.byref(it), ctypes.byref(stt)))
        if stt.value == 1:
            return None
        if stt.value == _lib.HGT_ERR_KEY:
            raise KeyError("allele vanished from next_prob output during SQUAREM step")
        if stt.value == _lib.HGT_ERR_ZERODIV:
            raise ZeroDivisionError("float division by zero")
        return rank_result(t.names, prob, inres, fk)

    def unit_abundance(self, u):
        """Gene_prob of the unit: the combination rule of core:1771-1782 (hla) or the plain EM (core:1789)."""
        t = self.loci[self.unit_locus[u]]
        first = self.unit_em(u, 0)
        if not t.is_hla:
            nc = self.unit_summary(u)["n_classes"][TABLE_GENE]
            if nc <= 1:
                if nc == 1:
                    raise TypeError("'dict_keys' object is not subscriptable")  # core:1787 on Python 3
                return []
            return first
        second = self.unit_em(u, 1)
        if second is None:
            return first
        exon_alleles, exon_prob_sum = set(), 0.0
        for i, (allele, prob) in enumerate(first):
            if i >= 10 and prob < 0.03:
                break
            group = t.allele_rep_groups[allele]
            if len(group) <= 1:
                continue
            exon_prob_sum += prob
            exon_alleles |= set(group)
        combined = {}
        for allele, prob in first:
            if allele not in exon_alleles:
                combined[allele] = prob
        for allele, prob in second:
            combined[allele] = prob * exon_prob_sum
        return sorted(([a, p] for a, p in combined.items()), key=lambda x: x[1], reverse=True)

    # ---- read-sharded locus (several ranks hold disjoint reads of the same unit, SURVEY.md 8e) ---------------------
    def set_pileup_allreduce(self, group=None):
        """Sum the raw pileup counts over the ranks before nt_set is derived (needs torch.distributed initialised)."""
        from . import em_dist
        self._hook = em_dist.pileup_allreduce_hook(group)  # keep the callback alive
        _lib.check(lib().hgt_batch_set_pileup_hook(self.handle, ctypes.cast(self._hook, ctypes.c_void_p), None))

    def set_skip_em(self, skip=True):
        _lib.check(lib().hgt_batch_set_skip_em(self.handle, 1 if skip else 0))

    def unit_table_dev(self, u, table):
        """(bits_ptr, count_u64_ptr, first_ptr, n_classes) of a device-resident table."""
        b, c, f = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_void_p()
        n = ctypes.c_int32(0)
        _lib.check(lib().hgt_batch_unit_table_dev(self.handle, u, table, ctypes.byref(b), ctypes.byref(c), ctypes.byref(f),
                                                  ctypes.byref(n)))
        return b.value, c.value, f.value, n.value

    def sharded_abundance(self, u, table=TABLE_GENE, lengths=None, remove_low=False, group=None, max_n=None):
        """single_abundance over the union of every rank's classes of unit u (read-sharded locus, SURVEY.md 8e).
        Returns (ranked [[allele, prob]] (the first max_n entries when given), iterations); identical on every rank.
        The ranks' tables are merged so that every class lives on exactly one rank (em_dist.merge_class_tables), then ONE
        cooperative kernel per rank runs the whole loop and sums the per-allele accumulators through NVLink peer memory
        (em_dist.single_abundance_peer)."""
        import torch
        import torch.distributed as dist
        from . import em_dist
        import time
        t0 = time.perf_counter()
        t = self.loci[self.unit_locus[u]]
        bits, cnt, first, n = self.unit_table_dev(u, table)
        offset = 0
        multi = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
        dev_index = self.device if self.device is not None else _lib.default_device()
        if multi:
            dev = torch.device("cuda", dev_index)
            mine = torch.tensor([self.unit_summary(u)["num_pairs"]], dtype=torch.int64, device=dev)
            every = [torch.zeros_like(mine) for _ in range(dist.get_world_size(group))]
            dist.all_gather(every, mine, group=group)
            offset = int(sum(int(x) for x in every[:dist.get_rank(group)]))
        ln = None if not lengths else np.asarray([lengths[x] for x in t.names], np.float64)
        keep = ()
        if multi:
            m_bits, m_cnt, m_first, n = em_dist.merge_class_tables(t.A, t.wp, bits, cnt, first, n, offset, dev_index, group)
            keep = (m_bits, m_cnt, m_first)
            bits, cnt, first, offset = m_bits.data_ptr(), m_cnt.data_ptr(), m_first.data_ptr(), 0
        t1 = time.perf_counter()
        prob, live, fk, iters = em_dist.single_abundance_peer(t.A, t.wp, bits, cnt, first, offset, n, dev_index, ln,
                                                              remove_low, group, keep)
        self.shard_classes = int(n)
        prob, live, fk = prob.cpu().numpy(), live.cpu().numpy().astype(np.uint8), fk.cpu().numpy()
        t2 = time.perf_counter()
        ranked = rank_result(t.names, prob, live, fk, max_n)
        t3 = time.perf_counter()
        # wall-clock split of the call, read by bench.py: set-up (offsets, table merge), EM loop incl. the final copy, ranking
        self.shard_ms = {"setup": (t1 - t0) * 1e3, "em_loop": (t2 - t1) * 1e3, "rank": (t3 - t2) * 1e3,
                         "em": "peer", "classes": self.shard_classes}
        return ranked, iters

    def unit_calls(self, u, max_n=None):
        """Gene_prob of the unit ranked natively (same result as unit_abundance); max_n limits the list length."""
        t = self.loci[self.unit_locus[u]]
        if not t.is_hla:
            nc = self.unit_summary(u)["n_classes"][TABLE_GENE]
            if nc <= 1:
                if nc == 1:
                    raise TypeError("'dict_keys' object is not subscriptable")  # core:1787 on Python 3
                return []
        cap = t.A if max_n is None else int(max_n)
        idx = np.zeros(max(cap, 1), np.int32)
        prob = np.zeros(max(cap, 1), np.float64)
        n = ctypes.c_int32(0)
        rc = lib().hgt_batch_unit_abundance(self.handle, u, cap, _lib.ptr(idx), _lib.ptr(prob), ctypes.byref(n))
        if rc == _lib.HGT_ERR_KEY:
            raise KeyError("allele vanished from next_prob output during SQUAREM step")
        if rc == _lib.HGT_ERR_ZERODIV:
            raise ZeroDivisionError("float division by zero")
        _lib.check(rc)
        k = min(cap, n.value)
        return [[t.names[int(idx[i])], float(prob[i])] for i in range(k)]

    def unit_read_haplotypes(self, u, var_ids=None):
        """Per surviving alignment record of unit u, in text order: (line index in the unit's text, FLAG, [haplotype, ...]) -
        the left_positive_hts / right_positive_hts the reference's typing() holds when it builds the assembly nodes
        (core:1386-1406 -> 1408-1540; SURVEY.md 8f-4).  A haplotype is the reference's string "left-id-...-right" when
        var_ids (variant ids in Var_list order, LocusTables.var_ids) is given, else (left, [rows], right).  A novel indel
        (no id in the database; the reference numbers those in encounter order, core:404-431) appears as
        "nvI<pos>_<len>" / "nvD<pos>_<len>"."""
        n = [ctypes.c_int64(0) for _ in range(3)]
        _lib.check(lib().hgt_batch_unit_reads(self.handle, u, ctypes.byref(n[0]), ctypes.byref(n[1]), ctypes.byref(n[2]),
                                              None, None, None, None, None, None, None))
        nr, nh, ni = (x.value for x in n)
        line = np.zeros(max(nr, 1), np.int64)
        flag = np.zeros(max(nr, 1), np.int32)
        hoff = np.zeros(nr + 1, np.int64)
        hl = np.zeros(max(nh, 1), np.int32)
        hr = np.zeros(max(nh, 1), np.int32)
        ioff = np.zeros(nh + 1, np.int64)
        ids = np.zeros(max(ni, 1), np.int32)
        _lib.check(lib().hgt_batch_unit_reads(self.handle, u, ctypes.byref(n[0]), ctypes.byref(n[1]), ctypes.byref(n[2]),
                                              _lib.ptr(line), _lib.ptr(flag), _lib.ptr(hoff), _lib.ptr(hl), _lib.ptr(hr),
                                              _lib.ptr(ioff), _lib.ptr(ids)))

        def name(i):
            if i >= 0:
                return var_ids[i]
            c = -2 - i
            return "nv%s%d_%d" % ("I" if (c >> 29) & 1 else "D", (c >> 10) & 0x7ffff, c & 0x3ff)

        out = []
        for r in range(nr):
            haps = []
            for h in range(hoff[r], hoff[r + 1]):
                rows = ids[ioff[h]:ioff[h + 1]].tolist()
                if var_ids is None:
                    haps.append((int(hl[h]), rows, int(hr[h])))
                else:
                    haps.append("-".join([str(int(hl[h]))] + [name(i) for i in rows] + [str(int(hr[h]))]))
            out.append((int(line[r]), int(flag[r]), haps))
        return out

    def top_calls(self, max_n=2):
        """unit_calls(u, max_n) of every unit, through one library call (hgt_batch_abundances)."""
        nu, cap = len(self.unit_locus), int(max_n)
        idx = np.zeros((max(nu, 1), max(cap, 1)), np.int32)
        prob = np.zeros((max(nu, 1), max(cap, 1)), np.float64)
        n = np.zeros(max(nu, 1), np.int32)
        st = np.zeros(max(nu, 1), np.int32)
        _lib.check(lib().hgt_batch_abundances(self.handle, cap, _lib.ptr(idx), _lib.ptr(prob), _lib.ptr(n), _lib.ptr(st)))
        out = []
        idx_l, prob_l, n_l, st_l = idx.tolist(), prob.tolist(), n.tolist(), st.tolist()
        for u in range(nu):
            t = self.loci[self.unit_locus[u]]
            if st_l[u] != 0 or not t.is_hla:
                out.append(self.unit_calls(u, max_n))  # raises what the reference raises / the single-class rule
                continue
            k = min(cap, n_l[u])
            names = t.names
            out.append([[names[idx_l[u][i]], prob_l[u][i]] for i in range(k)])
        return out

    def add_units_ptr(self, units):
        """[(locus_index, address, n_bytes), ...] in one library call."""
        n = len(units)
        li = (ctypes.c_int32 * n)(*[u[0] for u in units])
        ad = (ctypes.c_void_p * n)(*[u[1] for u in units])
        nb = (ctypes.c_size_t * n)(*[u[2] for u in units])
        first = lib().hgt_batch_add_units(self.handle, n, li, ad, nb)
        if first < 0:
            _lib.check(int(first))
        self.unit_locus.extend(u[0] for u in units)
        return int(first)

    def close(self):
        if self.handle is not None and self.handle.value:
            lib().hgt_batch_free(self.handle)
            self.handle = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BatchPipeline:
    """A stream of batches with `depth` of them in flight.  Each lane is a host thread with its own library context (own
    CUDA stream, own buffer pool), so the host-to-device copy of batch k+1 runs on the copy engine while the kernels of
    batch k run, and the host work of one batch (result read-back, Python) overlaps the GPU work of the other.  The loci
    (device tables) are shared.  Results come back in submission order.

        pipe = BatchPipeline(tables, params, depth=2)
        for calls in pipe.map(batches, lambda batch: batch.top_calls(2)):   # batches: iterables of (locus, addr, n) or (locus, text)
            ...
    """

    def __init__(self, loci, params=None, remove_low_abundance_alleles=True, device=None, depth=3):
        import threading
        self.loci, self.params, self.remove_low, self.device = list(loci), params or make_params(), remove_low_abundance_alleles, device
        self.depth = max(1, int(depth))
        self._local = threading.local()
        self.trace = None  # set to a list: [t_start, t_prepared, t_executed, t_finished, t_results] of every batch
        self._ctxs = []
        self._lock = threading.Lock()
        self._copy_turn = threading.Lock()

    def contexts(self):
        return list(self._ctxs)

    def _ctx(self):
        c = getattr(self._local, "ctx", None)
        if c is None:
            c = _lib.new_ctx(self.device)
            self._local.ctx = c
            with self._lock:
                self._ctxs.append(c)
        return c

    def _one(self, units, fn):
        b = Batch(self.loci, self.params, self.remove_low, device=self.device, ctx=self._ctx())
        try:
            t = [time.perf_counter()]
            if units and all(len(unit) == 3 for unit in units):
                b.add_units_ptr(units)
            else:
                for unit in units:
                    if len(unit) == 3:
                        b.add_unit_ptr(*unit)
                    else:
                        b.add_unit(*unit)
            with self._copy_turn:  # one bulk host-to-device transfer at a time: the lanes fall out of step, so the
                b.prepare()        # transfer of one batch runs under the kernels of the others
            t.append(time.perf_counter())
            b.execute()
            t.append(time.perf_counter())
            b.finish()
            t.append(time.perf_counter())
            out = fn(b)
            t.append(time.perf_counter())
            if self.trace is not None:
                self.trace.append(t)
            return out
        finally:
            b.close()

    def map(self, batches, fn):
        from collections import deque
        from concurrent.futures import ThreadPoolExecutor
        pool = getattr(self, "_pool", None)
        if pool is None:
            pool = self._pool = ThreadPoolExecutor(self.depth)
        pending = deque()
        for units in batches:
            pending.append(pool.submit(self._one, units, fn))
            if len(pending) >= self.depth:
                yield pending.popleft().result()
        while pending:
            yield pending.popleft().result()

    def close(self):
        pool = getattr(self, "_pool", None)
        if pool is not None:
            pool.shutdown(wait=True)
            self._pool = None
        for c in self._ctxs:
            lib().hgt_free(c)
        self._ctxs = []


def typing_from_alignments(base_fname, locus_tables, locus_list, alignments, simulation, num_editdist=2,
                           error_correction=True, allow_discordant=False, remove_low_abundance_alleles=True,
                           best_alleles=False, output_allele_counts=False, aligner="hisat2", index_type="graph",
                           base_locus=0, device=None):
    """The part of typing() between the alignment files and the report, for index_type == "graph"
    (reference hisatgenotype_typing_core.py:336-343, 370-2142 minus assembly).

    locus_tables  {gene: LocusTables}
    locus_list    as typing() receives it: gene names, or in simulation mode the lists of truth alleles
                  (gene = names[0].split('*')[0], core:380-383)
    alignments    {gene: alignment lines in `samtools view <bam> <backbone> | sort -k1,1 -s` order (core:458-468), or a
                  sam_intake.BamUnit of split_bam or a sam_intake.DeviceBamUnit of split_bam_device, rendered into those
                  lines on the GPU}
    Returns (report body text starting at the aligner line, test_passed dict of the simulation mode)."""
    from . import report
    from .sam_intake import BamUnit, DeviceBamUnit
    assert index_type == "graph", "the linear-index branch (core:1597-1648) stays on the reference path"
    genes, truths = [], []
    for entry in locus_list:
        if simulation:
            genes.append(entry[0].split("*")[0])
            truths.append(list(entry))
        else:
            genes.append(entry)
            truths.append([])
    uniq = []
    for g in genes:
        if g not in uniq:
            uniq.append(g)
    batch = Batch([locus_tables[g] for g in uniq],
                  make_params(num_editdist, error_correction, allow_discordant, simulation, base_locus),
                  remove_low_abundance_alleles, device=device)
    try:
        for g in genes:
            if isinstance(alignments[g], BamUnit):
                batch.add_unit_bam(uniq.index(g), alignments[g])
            elif isinstance(alignments[g], DeviceBamUnit):
                batch.add_unit_bam_dsplit(uniq.index(g), alignments[g])
            else:
                batch.add_unit(uniq.index(g), alignments[g])
        batch.run()
        text = [report.aligner_line(aligner, index_type)]
        test_passed = {}
        for u, g in enumerate(genes):
            summ = batch.unit_summary(u)
            if summ["num_reads"] <= 0:
                continue
            block, success = report.locus_block(summ["num_reads"], summ["num_pairs"], batch.unit_gene_counts(u, TABLE_GENE),
                                                batch.unit_calls(u), simulation, truths[u], output_allele_counts,
                                                best_alleles)
            text.append(block)
            for ok in success:
                if ok:
                    key = "%s %s" % (aligner, index_type)
                    test_passed[key] = test_passed.get(key, 0) + 1
    finally:
        batch.close()
    return "".join(text), test_passed


_TYPING_PARAMS = ("simulation", "full_path_base_fname", "locus_list", "genotype_genome", "partial", "partial_alleles",
                  "refGenes", "Genes", "Gene_names", "Gene_lengths", "refGene_loci", "Vars", "Var_list", "Links", "aligners",
                  "num_editdist", "assembly", "output_base", "error_correction", "keep_alignment", "allow_discordant",
                  "type_primary_exons", "remove_low_abundance_alleles", "display_alleles", "fastq", "read_fname",
                  "alignment_fname", "num_frag_list", "read_len", "fragment_len", "threads", "best_alleles", "verbose",
                  "assembly_verbose", "out_dir", "dbversion", "output_allele_counts", "test_i")  # core:249-286


def is_contracted_call(a):
    """Is this typing() call on the path this package implements?  The other branches of the reference's typing() stay on
    the reference (SURVEY.md 8a): --assembly (core:1408-1540, 1791-2074), genotype-genome typing (core:372-377, 627-630),
    CODIS pair distances (core:451-456, 680-716), linear indexes / bowtie2 (core:1597-1648), and the debug prints of
    verbose >= 2 (core:609, 820, 1195)."""
    base_fname = a["full_path_base_fname"].split("/")[-1]
    return (not a["assembly"] and a["genotype_genome"] == "" and base_fname != "codis" and (a["verbose"] or 0) < 2
            and len(a["aligners"]) > 0 and all(index_type == "graph" and aligner == "hisat2" for aligner, index_type in a["aligners"]))


def typing_dispatch(reference_module, reference_typing, *args, **kwargs):
    """What the drop-in module installs as typing(): the contracted path on the GPU, everything else to the reference's own
    typing() (same positional / keyword arguments, same return value)."""
    if len(args) > len(_TYPING_PARAMS):
        raise TypeError("typing() takes %d positional arguments but %d were given" % (len(_TYPING_PARAMS), len(args)))
    a = dict(zip(_TYPING_PARAMS, args))
    for k, v in kwargs.items():
        if k not in _TYPING_PARAMS or k in a:
            raise TypeError("typing() got an unexpected or repeated argument '%s'" % k)
        a[k] = v
    a.setdefault("test_i", 0)
    missing = [k for k in _TYPING_PARAMS if k not in a]
    if missing:
        raise TypeError("typing() missing required arguments: %s" % ", ".join(missing))
    if not is_contracted_call(a):
        return reference_typing(*args, **kwargs)
    return typing(*[a[k] for k in _TYPING_PARAMS], _reference=reference_module)


def genotyping_locus(*args, **kwargs):
    """The reference's genotyping_locus (core:2278-2309: database loading, simulation harness, one typing() call per sample
    or test) with typing() and single_abundance() replaced: a pass-through to the drop-in module, which must be first on
    sys.path together with the reference's hisatgenotype_modules (shim/_hgt_shim.py)."""
    import hisatgenotype_typing_core as drop_in
    if not hasattr(drop_in, "_product"):
        raise ImportError("hisatgenotype_typing_core on sys.path is not the drop-in module of hisat-genotype_b200/shim "
                          "(or HGT_DISABLE is set)")
    return drop_in.genotyping_locus(*args, **kwargs)


def typing(simulation, full_path_base_fname, locus_list, genotype_genome, partial, partial_alleles, refGenes, Genes,
           Gene_names, Gene_lengths, refGene_loci, Vars, Var_list, Links, aligners, num_editdist, assembly, output_base,
           error_correction, keep_alignment, allow_discordant, type_primary_exons, remove_low_abundance_alleles,
           display_alleles, fastq, read_fname, alignment_fname, num_frag_list, read_len, fragment_len, threads,
           best_alleles, verbose, assembly_verbose, out_dir, dbversion, output_allele_counts, test_i=0, _reference=None):
    """Drop-in for the reference's typing() (core:249-2171) on the contracted path (is_contracted_call): same arguments,
    same `.report` file, same return value (test_passed in simulation mode, else None).  Alignment itself stays on the
    reference path (its align_reads + samtools); everything between the alignment file and the report runs through libhgt
    on the GPU.  _reference = the reference's hisatgenotype_typing_core module (given by the drop-in module; found on
    sys.path otherwise): its align_reads is used and its VERSION files are printed in the header (core:309-325)."""
    import os
    import subprocess
    import sys

    from . import report
    a = dict(zip(_TYPING_PARAMS, (simulation, full_path_base_fname, locus_list, genotype_genome, partial, partial_alleles,
                                  refGenes, Genes, Gene_names, Gene_lengths, refGene_loci, Vars, Var_list, Links, aligners,
                                  num_editdist, assembly, output_base, error_correction, keep_alignment, allow_discordant,
                                  type_primary_exons, remove_low_abundance_alleles, display_alleles, fastq, read_fname,
                                  alignment_fname, num_frag_list, read_len, fragment_len, threads, best_alleles, verbose,
                                  assembly_verbose, out_dir, dbversion, output_allele_counts, test_i)))
    if _reference is None:
        import hisatgenotype_typing_core as mod
        _reference = getattr(mod, "_reference", mod)
    if not is_contracted_call(a):
        return _reference.typing(*[a[k] for k in _TYPING_PARAMS])
    ref_common = _reference.typing_common  # the module the reference's typing() calls align_reads through (core:358)
    from . import sam_intake
    # HGT_NATIVE_INTAKE=1: a SAM or BAM alignment file is read and split natively (SURVEY.md 8f-3) instead of through
    # samtools pipes (CRAM and BGZF that is not BAM stay with samtools)
    native = os.environ.get("HGT_NATIVE_INTAKE", "") not in ("", "0")
    base_fname = full_path_base_fname.split("/")[-1]
    report_base = "%s/%s-%s." % (out_dir, output_base, base_fname)
    if simulation:
        core_fid = str(test_i + 1)
        report_base += "test-"
    else:
        core_fid = "_".join(read_fname[0].split("/")[-1].split(".")[:-1])
    report_base += core_fid
    version_dir = "/".join(os.path.dirname(_reference.__file__).split("/")[:-1])  # core:310-312
    hg_version = open(version_dir + "/VERSION").read()
    h2_version = open(version_dir + "/hisat2/VERSION").read()
    out = [report.header(h2_version, hg_version, dbversion, " ".join(sys.argv))]
    test_passed = {}
    tables = {}
    try:
        for aligner, index_type in aligners:
            remove_alignment_file = False
            aln = alignment_fname
            native_text = native_bam = None
            if aln == "":
                if native:  # HISAT2's SAM stream straight into the native intake: no samtools view -bS / sort / index
                    native_text = sam_intake.align_to_sam(simulation, full_path_base_fname + "." + index_type, base_fname,
                                                          read_fname, fastq, threads, verbose)
                else:
                    remove_alignment_file = True
                    aln = "%s_output.bam" % base_fname if simulation else "%s.bam" % core_fid
                    ref_common.align_reads(aligner, simulation, full_path_base_fname + "." + index_type, index_type, base_fname,
                                           read_fname, fastq, threads, aln, verbose)
            elif native:
                kind, data = sam_intake.read_alignment(aln, threads, device=_lib.default_device())  # BGZF inflates on the GPU
                if kind == "bam":
                    native_bam = data
                elif kind == "sam":
                    native_text = data
            genes_here = []
            for entry in locus_list:
                gene = entry[0].split("*")[0] if simulation else entry
                if gene in genes_here:
                    continue
                genes_here.append(gene)
                if gene not in tables:
                    ref_allele = refGenes[gene]
                    loc = refGene_loci[gene]
                    tables[gene] = LocusTables(base_fname, gene, ref_allele, Genes[gene][ref_allele], Vars[gene], Var_list[gene],
                                               Links, Gene_names[gene], Gene_lengths[gene], loc[-2], loc[-1])
            alignments = None
            if native_text is not None:
                # native intake (sam_intake.py): one pass over the SAM text instead of `samtools view | sort -k1,1 -s` per locus
                by_ref = sam_intake.split_sam(native_text, [refGenes[g] for g in genes_here], threads)
                alignments = {g: by_ref[refGenes[g]] for g in genes_here}
            elif native_bam is not None:
                # BAM: the host splits the records, the GPU renders them into alignment text (packed units)
                by_ref = sam_intake.split_bam(native_bam, [refGenes[g] for g in genes_here], threads)
                alignments = {g: by_ref[refGenes[g]] for g in genes_here}
            else:
                alignments = {}
                for gene in genes_here:
                    if not os.path.exists(aln + ".bai"):
                        os.system("samtools index %s" % aln)
                    view = subprocess.Popen(["samtools", "view", aln, refGenes[gene]], stdout=subprocess.PIPE,
                                            stderr=subprocess.DEVNULL)
                    srt = subprocess.Popen(["sort", "-k", "1,1", "-s"], stdin=view.stdout, stdout=subprocess.PIPE,
                                           stderr=subprocess.DEVNULL)
                    alignments[gene] = srt.communicate()[0]
            body, passed = typing_from_alignments(base_fname, tables, locus_list, alignments, simulation, num_editdist,
                                                  error_correction, allow_discordant, remove_low_abundance_alleles,
                                                  best_alleles, output_allele_counts, aligner, index_type)
            out.append(body)
            for k, v in passed.items():
                test_passed[k] = test_passed.get(k, 0) + v
            if not keep_alignment and remove_alignment_file:
                os.system("rm %s*" % aln)
    finally:
        for t in tables.values():
            t.close()
    text = "".join(out)
    with open("%s.report" % report_base, "w") as f:
        f.write(text)
    if verbose or assembly_verbose or simulation:
        sys.stderr.write(text)
    if simulation:
        return test_passed


def smoke_check(device=None):
    """One small stage (a) + (b) run on the GPU checked against the oracle: a 2,100-allele synthetic hla locus (two
    words per lane in the allele-set kernels), 300 read pairs, three tables bit-exact and the ranked calls identical.
    Called by __graft_entry__.smoke(); the oracle is the checker only (tests / smoke / bench cpu_baseline)."""
    import hgt_oracle as O  # oracle/ is on sys.path only inside smoke() and the tests
    from . import synth
    loc = synth.make_locus("A", 17, L=2500, n_alleles=2100, n_groups=30, core_vars=60, pool_private=700, del_frac=0.1)
    cont = synth.reference_containers([loc], "hla")
    g = "A"
    args = ("hla", g, cont["refGenes"][g], cont["Genes"][g][cont["refGenes"][g]], cont["Vars"][g], cont["Var_list"][g],
            cont["Links"], cont["Gene_names"][g], cont["Gene_lengths"][g], cont["refGene_loci"][g][4],
            cont["refGene_loci"][g][5])
    rng = np.random.default_rng(17)
    names = sorted(n for n in loc.alleles if loc.alleles[n])
    truth = [names[i] for i in rng.choice(len(names), 2, replace=False)]
    sam = synth.simulate_sam(loc, truth, n_pairs=300, rng=rng, err_rate=0.004)
    ol = O.OracleLocus(*args)
    ref = O.type_locus(ol, sam, simulation=False)
    t = LocusTables(*args, device=device)
    batch = Batch([t], make_params(), True, device=device)
    try:
        batch.add_unit(0, sam)
        batch.run()
        s = batch.unit_summary(0)
        assert (s["num_reads"], s["num_pairs"]) == (ref["num_reads"], ref["num_pairs"]), (s, ref["num_reads"])
        for tb, key in ((TABLE_GENE, "gene"), (TABLE_EXON, "exon"), (TABLE_PRIMARY, "primary")):
            assert list(map(list, batch.unit_gene_cmpt(0, tb).items())) == ref["tables"][key].cmpt_items(ol), key
            assert batch.unit_gene_counts(0, tb) == ref["tables"][key].count_items(ol), key
        calls = batch.unit_calls(0, 4)
        assert len(calls) >= 1
    finally:
        batch.close()
        t.close()
    return {"reads": ref["num_reads"], "pairs": ref["num_pairs"], "top": calls[:2], "truth": truth}


class HostWalk:
    """Host half of stage (a) with a caller-supplied pileup (no GPU): used by the CPU-side tests."""

    def __init__(self, tables: LocusTables, sam, params: Params, counts, nt_mask):
        buf = _sam_bytes(sam)
        counts = np.ascontiguousarray(counts, np.uint32)
        nt_mask = np.ascontiguousarray(nt_mask, np.uint8)
        h = ctypes.c_void_p()
        rc = lib().hgt_host_walk(tables.handle, buf, len(buf), ctypes.byref(params), _lib.ptr(counts),
                                 _lib.ptr(nt_mask), ctypes.byref(h))
        _lib.check(rc)
        nr, npairs = ctypes.c_int64(0), ctypes.c_int64(0)
        nh, nrows = (ctypes.c_int64 * 3)(), (ctypes.c_int64 * 3)()
        _lib.check(lib().hgt_walk_summary(h, ctypes.byref(nr), ctypes.byref(npairs), ctypes.byref(nh),
                                          ctypes.byref(nrows)))
        self.num_reads, self.num_pairs = nr.value, npairs.value
        self.tables_out = []
        for tb in range(3):
            job_off = np.zeros(self.num_pairs + 1, np.int64)
            hl = np.zeros(max(nh[tb], 1), np.int32)
            hr = np.zeros(max(nh[tb], 1), np.int32)
            ro = np.zeros(nh[tb] + 1, np.int64)
            rows = np.zeros(max(nrows[tb], 1), np.int32)
            _lib.check(lib().hgt_walk_table(h, tb, _lib.ptr(job_off), _lib.ptr(hl), _lib.ptr(hr), _lib.ptr(ro),
                                            _lib.ptr(rows)))
            self.tables_out.append((job_off, hl[:nh[tb]], hr[:nh[tb]], ro, rows[:nrows[tb]]))
        lib().hgt_walk_free(h)

"""Per-locus tables for the GPU typing path, derived from the reference's containers.

Mirrors the per-locus set-up typing() performs before its read loop
(reference hisatgenotype_modules/hisatgenotype_typing_core.py:385-596):
  allele index space (sorted names, backbone excluded; key order of core:1229-1230)
  variant rows in Var_list order, Links as CSR allele lists (core:476-487)
  exonic variants and representative alleles (get_exonic_vars core:67-78, get_rep_alleles core:86-115)
  alternative haplotypes around deletions (get_alternatives, hisatgenotype_typing_common.py:1424-1657)
and hands them to libhgt as an hgt_locus_desc (include/hgt.h).
"""
from __future__ import annotations

import bisect
import ctypes
import threading

import numpy as np

from . import _lib

_TYPE_CODE = {"single": 0, "deletion": 1, "insertion": 2}
_NAMES_LOCK = threading.Lock()  # loci are shared by batches on several threads (typing_core.BatchPipeline)


class LocusDesc(ctypes.Structure):
    _fields_ = [
        ("n_alleles", ctypes.c_int32), ("n_vars", ctypes.c_int32), ("ref_len", ctypes.c_int32),
        ("ref_seq", ctypes.c_char_p),
        ("var_pos", ctypes.c_void_p), ("var_len", ctypes.c_void_p), ("var_type", ctypes.c_void_p),
        ("var_base", ctypes.c_void_p), ("var_flags", ctypes.c_void_p), ("var_ids", ctypes.c_char_p),
        ("link_off", ctypes.c_void_p), ("link_allele", ctypes.c_void_p),
        ("n_exons", ctypes.c_int32), ("exons", ctypes.c_void_p),
        ("n_primary_exons", ctypes.c_int32), ("primary_exons", ctypes.c_void_p),
        ("exon_rep_mask", ctypes.c_void_p), ("primary_rep_mask", ctypes.c_void_p),
        ("gene_names_rank", ctypes.c_void_p), ("is_hla", ctypes.c_int32), ("alts_text", ctypes.c_char_p),
        ("group_off", ctypes.c_void_p), ("group_member", ctypes.c_void_p), ("allele_len", ctypes.c_void_p),
    ]


class Params(ctypes.Structure):
    _fields_ = [("num_editdist", ctypes.c_int32), ("error_correction", ctypes.c_int32),
                ("allow_discordant", ctypes.c_int32), ("simulation", ctypes.c_int32),
                ("base_locus", ctypes.c_int32), ("n_threads", ctypes.c_int32), ("chunk_bytes", ctypes.c_int32)]


def _bind(L):
    if getattr(L, "_hgt_typing_bound", False):
        return L
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64
    P = ctypes.POINTER
    L.hgt_locus_create.restype = ctypes.c_int
    L.hgt_locus_create.argtypes = [vp, P(LocusDesc), P(vp)]
    L.hgt_locus_free.restype = None
    L.hgt_locus_free.argtypes = [vp]
    L.hgt_typing_run.restype = ctypes.c_int
    L.hgt_typing_run.argtypes = [vp, vp, ctypes.c_char_p, ctypes.c_size_t, P(Params), P(vp)]
    L.hgt_typing_free.restype = None
    L.hgt_typing_free.argtypes = [vp]
    L.hgt_typing_summary.restype = ctypes.c_int
    L.hgt_typing_summary.argtypes = [vp, P(i64), P(i64), P(i32 * 3)]
    L.hgt_typing_table.restype = ctypes.c_int
    L.hgt_typing_table.argtypes = [vp, i32, vp, vp, vp, vp, vp]
    L.hgt_typing_pileup.restype = ctypes.c_int
    L.hgt_typing_pileup.argtypes = [vp, vp, vp]
    L.hgt_typing_em.restype = ctypes.c_int
    L.hgt_typing_em.argtypes = [vp, vp, i32, vp, vp, i32, vp, vp, vp, P(i32)]
    L.hgt_batch_create.restype = ctypes.c_int
    L.hgt_batch_create.argtypes = [vp, i32, P(vp), P(Params), i32, P(vp)]
    L.hgt_batch_free.restype = None
    L.hgt_batch_free.argtypes = [vp]
    L.hgt_batch_add_unit.restype = i64
    L.hgt_batch_add_unit.argtypes = [vp, i32, vp, ctypes.c_size_t]
    for fn in ("hgt_batch_prepare", "hgt_batch_run"):
        getattr(L, fn).restype = ctypes.c_int
        getattr(L, fn).argtypes = [vp]
    for fn in ("hgt_batch_execute", "hgt_batch_finish"):
        getattr(L, fn).restype = ctypes.c_int
        getattr(L, fn).argtypes = [vp, vp]
    L.hgt_batch_totals.restype = ctypes.c_int
    L.hgt_batch_totals.argtypes = [vp] + [P(i64)] * 6
    L.hgt_batch_job_stats.restype = ctypes.c_int
    L.hgt_batch_job_stats.argtypes = [vp, P(i64 * 4)]
    L.hgt_batch_unit_summary.restype = ctypes.c_int
    L.hgt_batch_unit_summary.argtypes = [vp, i64, P(i64), P(i64), P(i32 * 4), P(i32 * 2), P(i32 * 2)]
    L.hgt_batch_unit_table.restype = ctypes.c_int
    L.hgt_batch_unit_table.argtypes = [vp, i64, i32, vp, vp, vp, vp, vp]
    L.hgt_batch_unit_em.restype = ctypes.c_int
    L.hgt_batch_unit_em.argtypes = [vp, i64, i32, vp, vp, vp, P(i32), P(i32)]
    L.hgt_batch_unit_abundance.restype = ctypes.c_int
    L.hgt_batch_unit_abundance.argtypes = [vp, i64, i32, vp, vp, P(i32)]
    L.hgt_batch_set_skip_em.restype = ctypes.c_int
    L.hgt_batch_set_skip_em.argtypes = [vp, i32]
    L.hgt_batch_set_pileup_hook.restype = ctypes.c_int
    L.hgt_batch_set_pileup_hook.argtypes = [vp, vp, vp]
    L.hgt_batch_unit_table_dev.restype = ctypes.c_int
    L.hgt_batch_unit_table_dev.argtypes = [vp, i64, i32, P(vp), P(vp), P(vp), P(i32)]
    L.hgt_host_walk.restype = ctypes.c_int
    L.hgt_host_walk.argtypes = [vp, ctypes.c_char_p, ctypes.c_size_t, P(Params), vp, vp, P(vp)]
    L.hgt_walk_summary.restype = ctypes.c_int
    L.hgt_walk_summary.argtypes = [vp, P(i64), P(i64), P(i64 * 3), P(i64 * 3)]
    L.hgt_walk_table.restype = ctypes.c_int
    L.hgt_walk_table.argtypes = [vp, i32, vp, vp, vp, vp, vp]
    L.hgt_walk_free.restype = None
    L.hgt_walk_free.argtypes = [vp]
    L.hgt_locus_set_names.restype = ctypes.c_int
    L.hgt_locus_set_names.argtypes = [vp, i32, P(ctypes.c_char_p)]
    L.hgt_locus_name_subsets.restype = ctypes.c_int
    L.hgt_locus_name_subsets.argtypes = [vp, vp, vp, P(i64)]
    L.hgt_batch_pairs.restype = ctypes.c_int
    L.hgt_batch_pairs.argtypes = [vp, i32, i64, i32, vp, vp, vp, vp, vp, vp]
    L.hgt_batch_pair_sizes.restype = ctypes.c_int
    L.hgt_batch_pair_sizes.argtypes = [vp, vp]
    L._hgt_typing_bound = True
    return L


def lib():
    return _bind(_lib.lib())


def get_exonic_vars(gene_vars, exons):
    out = set()
    for var_id, (t, pos, data) in gene_vars.items():
        right = pos + int(data) - 1 if t == "deletion" else pos
        for el, er in exons:
            if pos >= el and right <= er:
                out.add(var_id)
    return out


def get_rep_alleles(links, exon_vars, in_alleles=None):
    """Alleles sharing the same set of exonic variants form a group; its first member (in the order alleles are
    met while walking Links) represents it.  Alleles without exonic variants belong to no group."""
    allele_vars, order = {}, []
    for var_id, alleles in links.items():
        if var_id not in exon_vars:
            continue
        for allele in alleles:
            if in_alleles is not None and allele not in in_alleles:
                continue
            if allele not in allele_vars:
                allele_vars[allele] = set()
                order.append(allele)
            allele_vars[allele].add(var_id)
    groups = {}
    for allele in order:
        groups.setdefault(frozenset(allele_vars[allele]), []).append(allele)
    reps, rep_groups = {}, {}
    for members in groups.values():
        rep_groups[members[0]] = members
        for m in members:
            reps[m] = members[0]
    return reps, rep_groups


def get_alternatives(ref_seq, allele_vars, gene_vars, var_list):
    """Alternative haplotypes with identical sequence to the left / right of each deletion.

    Returns (alts_left, alts_right): {haplotype string: set of haplotype strings}, the containers the reference
    calls Alts_left / Alts_right.  Walks outwards from every deletion one base at a time, on both the haplotype
    that carries the deletion and the one that does not, following only variant successions seen in some allele.
    """
    n_ref = len(ref_seq)
    adjacent = set()
    for ids in allele_vars.values():
        adjacent.update(zip(ids[:-1], ids[1:]))
    right_sorted = []
    for _, vid in var_list:
        t, pos, data = gene_vars[vid]
        if t == "deletion":
            pos = pos + int(data) - 1
        elif t == "insertion":
            pos += 1
        right_sorted.append((pos, vid))
    right_sorted.sort(key=lambda x: x[0])
    right_keys = [p for p, _ in right_sorted]
    left_keys = [p for p, _ in var_list]
    tables = {True: {}, False: {}}

    def grow(ht, to_left, skip):
        pos = ht[0] - 1 if to_left else ht[-1] + 1
        if not 0 <= pos < n_ref:
            return []
        if to_left:
            found = [([pos] + ht[1:], ref_seq[pos])]
            neighbour = ht[1] if len(ht) > 2 else None
            j = bisect.bisect_left(right_keys, pos + 1) - 1
            while j >= 0:
                vid = right_sorted[j][1]
                j -= 1
                t, vpos, data = gene_vars[vid]
                if t == "deletion":
                    if vpos == 0:
                        continue
                    vpos = vpos + int(data) - 1
                if vpos > pos:
                    continue
                if vpos < pos:
                    break
                if vid == skip or (neighbour is not None and (vid, neighbour) not in adjacent):
                    continue
                if t == "single":
                    found.append(([vpos, vid] + ht[1:], data))
                elif t == "deletion":
                    found += grow([vpos - int(data) + 1, vid] + ht[1:], to_left, skip)
        else:
            found = [(ht[:-1] + [pos], ref_seq[pos])]
            neighbour = ht[-2] if len(ht) > 2 else None
            j = bisect.bisect_left(left_keys, pos)
            while j < len(var_list):
                vid = var_list[j][1]
                j += 1
                t, vpos, data = gene_vars[vid]
                if vpos < pos:
                    continue
                if vpos > pos:
                    break
                if vid == skip or (neighbour is not None and (neighbour, vid) not in adjacent):
                    continue
                if t == "single":
                    found.append((ht[:-1] + [vid, vpos], data))
                elif t == "deletion":
                    found += grow(ht[:-1] + [vid, vpos + int(data) - 1], to_left, skip)
        return found

    def explore(origin, ht, alt, to_left, depth):
        extended = False
        alt_next = grow(alt, to_left, origin)
        for ht2, base in grow(ht, to_left, None):
            for alt2, base2 in alt_next:
                if base != base2:
                    continue
                if (ht2[0] == alt2[0]) if to_left else (ht2[-1] == alt2[-1]):
                    continue
                extended = True
                explore(origin, ht2, alt2, to_left, depth + 1)
        if depth > 0 and not extended:
            a = "-".join(str(x) for x in ht)
            b = "-".join(str(x) for x in alt)
            tables[to_left].setdefault(a, set()).add(b)
            tables[to_left].setdefault(b, set()).add(a)

    for _, vid in var_list:
        t, pos, data = gene_vars[vid]
        if pos == 0 or t != "deletion":
            continue
        n = int(data)
        if pos + n >= n_ref:
            continue
        explore(vid, [pos, vid, pos + n - 1], [pos + n, pos + n - 1], True, 0)
        explore(vid, [pos, vid, pos + n - 1], [pos, pos - 1], False, 0)
    return tables[True], tables[False]


class LocusTables:
    """One locus, ready for the GPU.  Arguments are the reference's own containers for the locus."""

    def __init__(self, base_fname, gene, ref_allele, ref_seq, gene_vars, var_list, links, gene_names,
                 gene_lengths, exons, primary_exons, device=None, host_only=False):
        self.base_fname, self.gene, self.ref_allele, self.ref_seq = base_fname, gene, ref_allele, ref_seq
        self.gene_names = list(gene_names)
        self.gene_lengths = gene_lengths
        self.is_hla = base_fname == "hla"
        table_names = [n for n in self.gene_names if n.find("BACKBONE") == -1]
        self.names = sorted(table_names)
        self.index = {n: i for i, n in enumerate(self.names)}
        self.A = len(self.names)
        self.wp = _lib.row_pitch(self.A)
        self.V = len(var_list)
        self.exons = [list(e) for e in exons]
        self.primary_exons = [list(e) for e in primary_exons]
        # --- variants -----------------------------------------------------------------------------------
        self.var_ids = [vid for _, vid in var_list]
        var_pos = np.zeros(max(self.V, 1), np.int32)
        var_len = np.ones(max(self.V, 1), np.int32)
        var_type = np.zeros(max(self.V, 1), np.uint8)
        var_base = np.zeros(max(self.V, 1), np.uint8)
        var_flags = np.zeros(max(self.V, 1), np.uint8)
        link_off = np.zeros(self.V + 1, np.int64)
        link_allele = []
        allele_vars = {}
        for r, (pos, vid) in enumerate(var_list):
            t, p, data = gene_vars[vid]
            var_pos[r] = p
            var_type[r] = _TYPE_CODE[t]
            if t == "deletion":
                var_len[r] = int(data)
            elif t == "insertion":
                var_len[r] = len(data)
            else:
                var_base[r] = ord(data[0]) if len(data) == 1 else 0
            flags = 2 if vid.startswith("hv") else 0
            if vid in links:
                flags |= 1
                for allele in links[vid]:
                    i = self.index.get(allele)
                    if i is not None:
                        link_allele.append(i)
                    if allele in self.index or allele == ref_allele:
                        allele_vars.setdefault(allele, []).append(vid)
            var_flags[r] = flags
            link_off[r + 1] = len(link_allele)
        self.allele_vars = allele_vars
        # --- representative alleles -----------------------------------------------------------------------
        self.exon_vars = get_exonic_vars(gene_vars, self.exons)
        self.primary_exon_vars = get_exonic_vars(gene_vars, self.primary_exons)
        self.allele_reps, self.allele_rep_groups = get_rep_alleles(links, self.exon_vars)
        self.allele_rep_set = set(self.allele_reps.values())
        self.primary_reps, self.primary_rep_groups = get_rep_alleles(links, self.primary_exon_vars,
                                                                     self.allele_rep_set)
        self.primary_rep_set = set(self.primary_reps.values())
        for a in self.primary_reps:  # check_repset_inclusion (validation_check.py:344-355)
            if a not in self.allele_rep_set:
                raise SystemExit("Error: %s not in Rep set!" % a)
        self.exon_mask = self.mask_of(self.allele_rep_set)
        self.primary_mask = self.mask_of(self.primary_rep_set)
        gn_rank = np.zeros(self.A, np.int32)
        for rank, n in enumerate(table_names):
            gn_rank[self.index[n]] = rank
        self.gn_rank = gn_rank
        # --- alternative haplotypes -------------------------------------------------------------------------
        self.alts_left, self.alts_right = get_alternatives(ref_seq, allele_vars, gene_vars, var_list)
        lines = []
        for tag, tab in (("L", self.alts_left), ("R", self.alts_right)):
            for key, alts in tab.items():
                lines.append("%s\t%s\t%s\n" % (tag, key, ",".join(sorted(alts))))
        # --- native handle ------------------------------------------------------------------------------------
        self._keep = dict(var_pos=var_pos, var_len=var_len, var_type=var_type, var_base=var_base,
                          var_flags=var_flags, link_off=link_off,
                          link_allele=np.asarray(link_allele if link_allele else [0], np.int32),
                          exons=np.asarray(self.exons if self.exons else [[0, 0]], np.int32).ravel(),
                          primary=np.asarray(self.primary_exons if self.primary_exons else [[0, 0]], np.int32).ravel(),
                          ids=b"".join(v.encode() + b"\0" for v in self.var_ids) + b"\0",
                          alts="".join(lines).encode(), ref=ref_seq.encode())
        k = self._keep
        d = LocusDesc()
        d.n_alleles, d.n_vars, d.ref_len = self.A, self.V, len(ref_seq)
        d.ref_seq = k["ref"]
        d.var_pos, d.var_len, d.var_type = _lib.ptr(var_pos), _lib.ptr(var_len), _lib.ptr(var_type)
        d.var_base, d.var_flags, d.var_ids = _lib.ptr(var_base), _lib.ptr(var_flags), k["ids"]
        d.link_off, d.link_allele = _lib.ptr(link_off), _lib.ptr(k["link_allele"])
        d.n_exons, d.exons = len(self.exons), _lib.ptr(k["exons"])
        d.n_primary_exons, d.primary_exons = len(self.primary_exons), _lib.ptr(k["primary"])
        d.exon_rep_mask, d.primary_rep_mask = _lib.ptr(self.exon_mask), _lib.ptr(self.primary_mask)
        d.gene_names_rank = _lib.ptr(gn_rank)
        d.is_hla = 1 if self.is_hla else 0
        d.alts_text = k["alts"]
        # exon groups (allele_rep_groups) as CSR over representative alleles, and allele lengths
        group_off = np.zeros(self.A + 1, np.int64)
        members = []
        for a, name in enumerate(self.names):
            grp = self.allele_rep_groups.get(name)
            if grp:
                members.extend(self.index[m] for m in grp if m in self.index)
            group_off[a + 1] = len(members)
        k["group_off"] = group_off
        k["group_member"] = np.asarray(members if members else [0], np.int32)
        k["allele_len"] = np.asarray([float(gene_lengths.get(n, len(ref_seq))) for n in self.names], np.float64)
        d.group_off, d.group_member = _lib.ptr(k["group_off"]), _lib.ptr(k["group_member"])
        d.allele_len = _lib.ptr(k["allele_len"])
        self._desc = d
        self.handle = ctypes.c_void_p()
        self.device = device
        ctx = None if host_only else _lib.ctx(device)
        _lib.check(lib().hgt_locus_create(ctx, ctypes.byref(d), ctypes.byref(self.handle)))

    def ensure_names(self):
        """Hand the allele names to the library (once): the batched pair model needs which names occur inside which."""
        if getattr(self, "_names_set", False):
            return
        with _NAMES_LOCK:
            if not getattr(self, "_names_set", False):
                arr = (ctypes.c_char_p * self.A)(*[n.encode() for n in self.names])
                _lib.check(lib().hgt_locus_set_names(self.handle, self.A, arr))
                self._names_set = True

    def name_subsets(self):
        """(off[A + 1], idx): for allele a, idx[off[a]:off[a + 1]] = the alleles whose name is a substring of a's name."""
        self.ensure_names()
        n = ctypes.c_int64(0)
        _lib.check(lib().hgt_locus_name_subsets(self.handle, None, None, ctypes.byref(n)))
        off = np.zeros(self.A + 1, np.int64)
        while True:  # (the names may be replaced by another thread between the size query and the read)
            idx = np.zeros(max(n.value, 1), np.int32)
            n.value = idx.size
            rc = lib().hgt_locus_name_subsets(self.handle, _lib.ptr(off), _lib.ptr(idx), ctypes.byref(n))
            if rc != _lib.HGT_ERR_ARG or n.value <= idx.size:
                _lib.check(rc)
                return off, idx[:n.value]

    def mask_of(self, names):
        m = np.zeros(self.wp, np.uint64)
        for n in names:
            i = self.index.get(n)
            if i is not None:
                m[i >> 6] |= np.uint64(1) << np.uint64(i & 63)
        return m

    def key_of(self, row):
        return "-".join(self.names[i] for i in _lib.unpack_bits(row, self.A))

    def close(self):
        if getattr(self, "handle", None) is not None and self.handle.value:
            lib().hgt_locus_free(self.handle)
            self.handle = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

"""Synthetic HLA-like allele/variant databases in the on-disk format the typing path consumes.

There is no network in the build/bench environment, so the IMGT-derived database that
``hisatgenotype_typing_process.extract_vars`` (reference
hisatgenotype_modules/hisatgenotype_typing_process.py:313-1255) would write is replaced by a
deterministic generator that emits the *same nine files* with the same column layout:

  <base>_backbone.fa, <base>_sequences.fa   60-column FASTA (process:1225-1232)
  <base>.locus        name chr left right len exon_str strand (process:1055-1063, common:279-309)
  <base>.snp / .index.snp   id \t single|deletion|insertion \t backbone \t pos \t data (process:1088-1102)
  <base>.link         id \t allele allele ...            (process:1105-1106)
  <base>.haplotype    htN \t backbone \t left \t right \t id,id   (process:1215-1220)
  <base>.allele / .partial   one allele name per line    (process:1233-1236)

Constraints honoured (SURVEY.md appendix C): ids are hv<N> in .snp order; variants sorted by
(pos, type I<M<D, data) like key_varKey (process:275-295); within one allele variants never
overlap (core:2220 asserts monotone positions); deletions never start at 0 nor touch the
backbone end (common:1622-1628); <base>_sequences.fa equals backbone+variants.
"""
from __future__ import annotations

import os
from dataclasses import dataclass, field

import numpy as np

NT = "ACGT"


@dataclass
class Locus:
    gene: str
    backbone: str
    # variants in .snp order: (type, pos, data) with data str (base / del length / inserted seq)
    variants: list = field(default_factory=list)
    var_ids: list = field(default_factory=list)  # "hv<N>"
    alleles: dict = field(default_factory=dict)  # allele name -> sorted list of variant indices
    exons: list = field(default_factory=list)  # [(left, right, primary)]
    chrom: str = "chr6"
    strand: str = "+"

    @property
    def backbone_name(self):
        return "%s*BACKBONE" % self.gene

    def allele_seq(self, name):
        """backbone + variants, the rule of read_Gene_alleles_from_vars (core:2215-2234)."""
        seq, prev = [], 0
        bb = self.backbone
        for vi in self.alleles[name]:
            t, pos, data = self.variants[vi]
            assert prev <= pos
            if pos > prev:
                seq.append(bb[prev:pos])
            if t == "single":
                seq.append(data)
                prev = pos + 1
            elif t == "deletion":
                prev = pos + int(data)
            else:
                seq.append(data)
                prev = pos
        if prev < len(bb):
            seq.append(bb[prev:])
        return "".join(seq)


_TYPE_ORD = {"insertion": 0, "single": 1, "deletion": 2}


def _pat2num(s):
    n = 0
    for c in s:
        n = 4 * n + NT.index(c)
    return n


def _var_key(v):
    t, pos, data = v
    last = int(data) if t == "deletion" else _pat2num(data)
    return (pos, _TYPE_ORD[t], last)


def _compatible_subset(cands, variants):
    """Keep a maximal prefix-greedy subset of candidate variant indices that can coexist in one allele."""
    out, prev = [], 0
    last_ins_pos = -1
    for vi in sorted(cands, key=lambda i: _var_key(variants[i])):
        t, pos, data = variants[vi]
        if pos < prev:
            continue
        if t == "insertion":
            if pos == last_ins_pos:
                continue
            last_ins_pos = pos
            prev = pos
        elif t == "single":
            prev = pos + 1
        else:
            prev = pos + int(data)
        out.append(vi)
    return out


def make_locus(gene, seed, L=3500, n_alleles=200, n_groups=12, core_vars=60, pool_private=400,
               private_per_allele=3, del_frac=0.06, ins_frac=0.0, exons=None, chrom="chr6",
               backbone_allele=True, alphabet=NT):
    """One locus: alleles come in groups sharing a core variant set, plus a few toggles each.  A short `alphabet`
    (e.g. "AC") makes the backbone repetitive, so deletions get many equivalent placements (Alts_left/right)."""
    rng = np.random.default_rng(seed)
    bb = "".join(alphabet[i] for i in rng.integers(0, len(alphabet), size=L))
    if exons is None:
        # three exons, first two primary (the ".locus" example of SURVEY appendix C, scaled to L)
        e = [(int(L * 0.09), int(L * 0.17), True), (int(L * 0.29), int(L * 0.37), True),
             (int(L * 0.51), int(L * 0.60), False)]
    else:
        e = exons
    # ---- variant pool ----------------------------------------------------------------
    pool = {}

    def new_variant():
        for _ in range(100):
            r = rng.random()
            pos = int(rng.integers(1, L - 12))
            if r < del_frac:
                v = ("deletion", pos, str(int(rng.integers(1, 7))))
            elif r < del_frac + ins_frac:
                n = int(rng.integers(1, 4))
                v = ("insertion", pos, "".join(NT[i] for i in rng.integers(0, 4, size=n)))
            else:
                alt = NT[(NT.index(bb[pos]) + int(rng.integers(1, 4))) % 4]
                v = ("single", pos, alt)
            if v not in pool:
                pool[v] = len(pool)
                return v
        raise RuntimeError("variant pool exhausted")

    n_core_pool = n_groups * core_vars
    core_pool = [new_variant() for _ in range(max(1, int(n_core_pool * 0.7)))]
    private_pool = [new_variant() for _ in range(pool_private)]
    variants = list(pool.keys())
    variants.sort(key=_var_key)
    index = {v: i for i, v in enumerate(variants)}
    core_idx = [index[v] for v in core_pool]
    priv_idx = [index[v] for v in private_pool]
    # make sure every exon carries variants (alleles without exonic variants cannot be called on
    # the hla path: get_rep_alleles core:86-115)
    groups = []
    for g in range(n_groups):
        k = min(core_vars, len(core_idx))
        groups.append(list(rng.choice(core_idx, size=k, replace=False)))
    alleles = {}
    per_group = [n_alleles // n_groups + (1 if g < n_alleles % n_groups else 0) for g in range(n_groups)]
    seen = set()
    for g in range(n_groups):
        made = 0
        tries = 0
        while made < per_group[g] and tries < per_group[g] * 50:
            tries += 1
            cand = set(groups[g])
            if made > 0:
                drop = rng.integers(0, 3)
                for vi in rng.choice(groups[g], size=min(int(drop), len(groups[g])), replace=False):
                    cand.discard(int(vi))
                add = rng.integers(1, private_per_allele + 1)
                for vi in rng.choice(priv_idx, size=int(add), replace=False):
                    cand.add(int(vi))
            vs = tuple(_compatible_subset([int(c) for c in cand], variants))
            if len(vs) == 0 or vs in seen:
                continue
            seen.add(vs)
            made += 1
            alleles["%s*%02d:%02d" % (gene, g + 1, made)] = list(vs)
    # drop unused variants, renumber
    used = sorted({vi for vs in alleles.values() for vi in vs})
    remap = {old: new for new, old in enumerate(used)}
    variants = [variants[i] for i in used]
    for name in alleles:
        alleles[name] = [remap[i] for i in alleles[name]]
    if backbone_allele:
        alleles["%s*%02d:%02d" % (gene, n_groups + 1, 1)] = []
    loc = Locus(gene=gene, backbone=bb, variants=variants, var_ids=[], alleles=alleles, exons=e, chrom=chrom)
    return loc


def write_database(loci, base, ix_dir, id_prefix="hv", partial_names=()):
    """Write the nine database files for a list of loci; variant ids are numbered across loci."""
    os.makedirs(ix_dir, exist_ok=True)
    full = os.path.join(ix_dir, base)
    f = {ext: open(full + ext, "w") for ext in
         ["_backbone.fa", "_sequences.fa", ".locus", ".snp", ".index.snp", ".haplotype", ".link", ".allele",
          ".partial"]}
    num_vars = 0
    num_ht = 0
    for loc in loci:
        bb, L = loc.backbone, len(loc.backbone)
        print(">%s" % loc.backbone_name, file=f["_backbone.fa"])
        for s in range(0, L, 60):
            print(bb[s:s + 60], file=f["_backbone.fa"])
        exon_str = ",".join("%d-%d%s" % (l, r, "p" if p else "") for l, r, p in loc.exons)
        print("%s\t%s\t%d\t%d\t%d\t%s\t%s" % (loc.backbone_name, loc.chrom, 0, L - 1, L, exon_str, loc.strand),
              file=f[".locus"])
        loc.var_ids = ["%s%d" % (id_prefix, num_vars + i) for i in range(len(loc.variants))]
        num_vars += len(loc.variants)
        links = [[] for _ in loc.variants]
        for name in sorted(loc.alleles):
            for vi in loc.alleles[name]:
                links[vi].append(name)
        for vi, (t, pos, data) in enumerate(loc.variants):
            line = "%s\t%s\t%s\t%d\t%s" % (loc.var_ids[vi], t, loc.backbone_name, pos, data)
            print(line, file=f[".snp"])
            print(line, file=f[".index.snp"])
            print("%s\t%s" % (loc.var_ids[vi], " ".join(links[vi])), file=f[".link"])
        # haplotypes: chains of variants closer than inter_gap=30 (process:1131-1149), one row per distinct
        # allele-specific combination inside the chain
        order = list(range(len(loc.variants)))

        def right_of(vi):
            t, pos, data = loc.variants[vi]
            return pos + int(data) - 1 if t == "deletion" else pos

        i = 0
        allele_sets = {n: set(v) for n, v in loc.alleles.items()}
        while i < len(order):
            j = i + 1
            prev = right_of(order[i])
            while j < len(order) and loc.variants[order[j]][1] <= prev + 30:
                prev = max(prev, right_of(order[j]))
                j += 1
            chain = order[i:j]
            combos = set()
            cs = set(chain)
            for name, vs in allele_sets.items():
                c = tuple(sorted(cs & vs))
                if c:
                    combos.add(c)
            for c in sorted(combos):
                left = loc.variants[c[0]][1]
                right = max(right_of(v) for v in c)
                print("ht%d\t%s\t%d\t%d\t%s" % (num_ht, loc.backbone_name, left, right,
                                                ",".join(loc.var_ids[v] for v in c)), file=f[".haplotype"])
                num_ht += 1
            i = j
        for name in sorted(loc.alleles):
            seq = loc.allele_seq(name)
            print(">%s" % name, file=f["_sequences.fa"])
            for s in range(0, len(seq), 60):
                print(seq[s:s + 60], file=f["_sequences.fa"])
            print(name, file=f[".allele"])
            if name in partial_names:
                print(name, file=f[".partial"])
    for fh in f.values():
        fh.close()
    return full


# ----------------------------------------------------------------------------------------------------------------
# In-memory reference containers and synthetic alignment records (bench / large parity cases)
# ----------------------------------------------------------------------------------------------------------------
def reference_containers(loci, base="hla", id_prefix="hv"):
    """The containers genotyping_locus() builds from the database files (core:2417-2485), straight from Locus
    objects: refGenes, refGene_loci, Vars, Var_list, Links, Gene_names, Gene_lengths, Genes (backbone only)."""
    refGenes, refGene_loci, Vars, Var_list, Links, Genes, Gene_names, Gene_lengths = {}, {}, {}, {}, {}, {}, {}, {}
    num = 0
    for loc in loci:
        g = loc.gene
        L = len(loc.backbone)
        refGenes[g] = loc.backbone_name
        refGene_loci[g] = [loc.backbone_name, loc.chrom, 0, L - 1, [[l, r] for l, r, _ in loc.exons],
                           [[l, r] for l, r, p in loc.exons if p]]
        loc.var_ids = ["%s%d" % (id_prefix, num + i) for i in range(len(loc.variants))]
        num += len(loc.variants)
        Vars[g] = {loc.var_ids[i]: [t, pos, data] for i, (t, pos, data) in enumerate(loc.variants)}
        Var_list[g] = [[pos, loc.var_ids[i]] for i, (t, pos, data) in enumerate(loc.variants)]
        links = [[] for _ in loc.variants]
        lengths = {loc.backbone_name: L}
        for name in sorted(loc.alleles):
            n = L
            for vi in loc.alleles[name]:
                links[vi].append(name)
                t, pos, data = loc.variants[vi]
                if t == "deletion":
                    n -= int(data)
                elif t == "insertion":
                    n += len(data)
            lengths[name] = n
        for vi, names in enumerate(links):
            Links[loc.var_ids[vi]] = names
        # Gene_names order: backbone, alleles in order of first appearance along Var_list/Links, then alleles
        # identical to the backbone (core:2199-2237, 2462-2467)
        order, seen = [loc.backbone_name], {loc.backbone_name}
        for vi in range(len(loc.variants)):
            for name in links[vi]:
                if name not in seen:
                    seen.add(name)
                    order.append(name)
        for name in sorted(loc.alleles):
            if name not in seen:
                seen.add(name)
                order.append(name)
        Gene_names[g] = order
        Gene_lengths[g] = lengths
        Genes[g] = {loc.backbone_name: loc.backbone}
    return dict(refGenes=refGenes, refGene_loci=refGene_loci, Vars=Vars, Var_list=Var_list, Links=Links, Genes=Genes,
                Gene_names=Gene_names, Gene_lengths=Gene_lengths)


_sim = None


def _simlib():
    global _sim
    if _sim is None:
        import atexit
        import ctypes
        import shutil
        import subprocess
        import tempfile
        tools = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools")
        so = os.path.join(tools, "libhgtsim.so")
        if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(os.path.join(tools, "simgen.cpp")):
            # not built by __graft_entry__.build() or older than its source: compile a private copy, because the
            # source tree may be read-only
            tmp = tempfile.mkdtemp(prefix="hgtsim-")
            atexit.register(shutil.rmtree, tmp, True)
            so = os.path.join(tmp, "libhgtsim.so")
            subprocess.check_call(["make", "-s", "-C", tools, "OUT=" + so])
        L = ctypes.CDLL(so)
        L.hgtsim_locus_create.restype = ctypes.c_void_p
        L.hgtsim_locus_create.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_char_p, ctypes.c_int] + \
            [ctypes.c_void_p] * 3 + [ctypes.c_char_p, ctypes.c_char_p]
        L.hgtsim_add_allele.restype = ctypes.c_int
        L.hgtsim_add_allele.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_char_p]
        L.hgtsim_locus_free.argtypes = [ctypes.c_void_p]
        L.hgtsim_generate.restype = ctypes.c_longlong
        L.hgtsim_generate.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int,
                                      ctypes.c_int, ctypes.c_double, ctypes.c_uint64, ctypes.c_int, ctypes.c_longlong,
                                      ctypes.c_char_p, ctypes.c_char_p, ctypes.c_longlong]
        _sim = L
    return _sim


class ReadSimulator:
    """Draws reads from alleles of one Locus and formats them as HISAT2-style alignment lines (tools/simgen.cpp)."""

    def __init__(self, loc):
        import ctypes
        self.loc = loc
        if not loc.var_ids:
            loc.var_ids = ["hv%d" % i for i in range(len(loc.variants))]
        n = len(loc.variants)
        tcode = {"single": 0, "deletion": 1, "insertion": 2}
        self._pos = np.asarray([v[1] for v in loc.variants] or [0], np.int32)
        self._len = np.asarray([int(v[2]) if v[0] == "deletion" else (len(v[2]) if v[0] == "insertion" else 1)
                                for v in loc.variants] or [1], np.int32)
        self._type = np.asarray([tcode[v[0]] for v in loc.variants] or [0], np.uint8)
        self._base = bytes((ord(v[2][0]) if v[0] == "single" else 0) for v in loc.variants) + b"\0"
        ids = b"".join(i.encode() + b"\0" for i in loc.var_ids) + b"\0"
        L = _simlib()
        self.h = L.hgtsim_locus_create(loc.backbone.encode(), len(loc.backbone), loc.backbone_name.encode(), n,
                                       self._pos.ctypes.data_as(ctypes.c_void_p),
                                       self._len.ctypes.data_as(ctypes.c_void_p),
                                       self._type.ctypes.data_as(ctypes.c_void_p), self._base, ids)
        self.slots = {}

    def slot(self, allele):
        import ctypes
        if allele not in self.slots:
            vs = np.asarray(self.loc.alleles[allele] or [0], np.int32)
            s = _simlib().hgtsim_add_allele(self.h, len(self.loc.alleles[allele]),
                                            vs.ctypes.data_as(ctypes.c_void_p), self._base)
            if s < 0:
                raise ValueError("allele %s carries an insertion; the simulator handles SNPs and deletions" % allele)
            self.slots[allele] = s
        return self.slots[allele]

    def generate(self, alleles, n_pairs, seed, err_rate=0.0, read_len=100, frag_len=350, paired=True, id_start=0,
                 prefix="r"):
        """bytes of SAM text: n_pairs pairs (2 lines each) or n_pairs single reads, name-sorted."""
        import ctypes
        slots = np.asarray([self.slot(a) for a in alleles], np.int32)
        cap = int(n_pairs) * (2 if paired else 1) * (330 + 2 * read_len) + 4096
        while True:
            buf = ctypes.create_string_buffer(cap)
            n = _simlib().hgtsim_generate(self.h, len(slots), slots.ctypes.data_as(ctypes.c_void_p), int(n_pairs),
                                          read_len, frag_len, float(err_rate), int(seed), 1 if paired else 0,
                                          int(id_start), prefix.encode(), buf, cap)
            if n >= 0:
                return buf.raw[:n]
            cap = -n + 4096

    def close(self):
        if self.h:
            _simlib().hgtsim_locus_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def simulate_sam(loc, alleles, n_pairs, rng=None, err_rate=0.0, seed=None, **kw):
    """Convenience wrapper: list of alignment lines for reads drawn from `alleles`."""
    sim = ReadSimulator(loc)
    if seed is None:
        seed = int(rng.integers(1, 2 ** 31)) if rng is not None else 1
    text = sim.generate(alleles, n_pairs, seed, err_rate, **kw)
    sim.close()
    return text.decode().splitlines()

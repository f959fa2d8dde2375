"""Hand-made alignment records over a synth.Locus, for tests that need record shapes the read simulator does not make:
any read length, sequencing errors at chosen read offsets, soft clips, known and novel insertions and deletions, N inside
an inserted sequence, and Zs present or absent.

A record is cut from an allele laid out as tokens along the backbone:
  ("M", bpos, base, var)   one aligned base (var = index of the known SNP it carries, else None)
  ("I", bpos, base, var)   one inserted base, placed in front of backbone position bpos
  ("D", bpos, length, var) a deletion of backbone [bpos, bpos + length)
and written in the format tools/simgen.cpp writes (HISAT2's): CIGAR of M / I / D / S, MD:Z, NM:i, NH:i:1 and
Zs:Z items "off|S|id", "off|D|id", "off|I|id" with offsets relative to the previous item, counted on the read without
its left clip."""
import re

import numpy as np

NT = "ACGT"


def allele_tokens(loc, allele):
    """Token list of an allele (backbone + its variants, the rule of synth.Locus.allele_seq)."""
    bb = loc.backbone
    out, prev = [], 0
    for vi in loc.alleles[allele]:
        t, pos, data = loc.variants[vi]
        out.extend(("M", b, bb[b], None) for b in range(prev, pos))
        if t == "single":
            out.append(("M", pos, data, vi))
            prev = pos + 1
        elif t == "deletion":
            out.append(("D", pos, int(data), vi))
            prev = pos + int(data)
        else:
            out.extend(("I", pos, c, vi) for c in data)
            prev = pos
    out.extend(("M", b, bb[b], None) for b in range(prev, len(bb)))
    return out


def _read_index(tokens):
    """Token index of every read base (M or I token) of the allele."""
    return [k for k, t in enumerate(tokens) if t[0] != "D"]


def known_alts(loc):
    """{backbone position: set of alt bases of known SNPs there}"""
    alts = {}
    for t, pos, data in loc.variants:
        if t == "single":
            alts.setdefault(pos, set()).add(data)
    return alts


class Forge:
    def __init__(self, loc, zs=True):
        self.loc = loc
        self.zs = zs
        if not loc.var_ids:
            loc.var_ids = ["hv%d" % i for i in range(len(loc.variants))]
        self._tok = {}
        self._alts = known_alts(loc)

    def tokens(self, allele):
        if allele not in self._tok:
            self._tok[allele] = allele_tokens(self.loc, allele)
        return self._tok[allele]

    def read_tokens(self, allele, start, length, novel_ins=None, novel_del=None):
        """Tokens of read bases [start, start + length) of the allele (start counts read bases, i.e. M and I tokens),
        with the deletions between them.  novel_ins = (k, seq): seq inserted in front of read base k (0 < k < length);
        novel_del = (k, n): the n backbone bases in front of read base k are deleted (read base k-1 and the next n must be
        plain backbone bases of the allele).  Positions past the last read base are shifted by n."""
        toks = self.tokens(allele)
        idx = _read_index(toks)
        if novel_del is not None:
            k, n = novel_del
            a = idx[start + k]
            run = toks[a:a + n]
            assert len(run) == n and all(t[0] == "M" and t[3] is None for t in run), "novel deletion over a variant"
            assert all(run[j][1] == run[0][1] + j for j in range(n))
            toks = toks[:a] + [("D", run[0][1], n, None)] + toks[a + n:]
            idx = _read_index(toks)
        assert start + length <= len(idx), "read runs past the allele end"
        lo, hi = idx[start], idx[start + length - 1]
        sel = list(toks[lo:hi + 1])
        if novel_ins is not None:
            k, seq = novel_ins
            assert 0 < k < length
            rk = _read_index(sel)[k]
            sel = sel[:rk] + [("I", sel[rk][1], c, None) for c in seq] + sel[rk:]
        return sel

    def record(self, name, allele, start, length, flag=0, errors=(), clip_left=0, clip_right=0, novel_ins=None,
               novel_del=None, zs=None, nm=None, pad=0, rng=None, pnext=0, tlen=0):
        """One alignment line.  errors: read offsets (of the aligned part, before clips) whose base is replaced by one
        that is neither the allele's base, nor the backbone's, nor a known SNP there (so it stays an unknown mismatch; in
        an inserted sequence the letter 'N' gives N inside an insertion).  clip_left / clip_right: bases of the aligned
        part turned into soft clips (the clipped bases stay in SEQ).  pad: bytes of an extra XP:Z tag the typing ignores.
        Returns (line, tokens of the aligned part)."""
        zs = self.zs if zs is None else zs
        sel = self.read_tokens(allele, start, length, novel_ins, novel_del)
        bb = self.loc.backbone
        read = [t for t in sel if t[0] != "D"]
        bases = [t[2] for t in read]
        err = set()
        for e in errors:
            if isinstance(e, tuple):  # (offset, letter)
                k, c = e
            else:
                k, c = e, None
            t = read[k]
            if c is None:
                avoid = {t[2]} | ({bb[t[1]]} | self._alts.get(t[1], set()) if t[0] == "M" else set())
                c = [x for x in NT if x not in avoid][0] if rng is None else \
                    rng.choice([x for x in NT if x not in avoid])
            bases[k] = c
            err.add(k)
        # soft clips: the first / last aligned read bases become S; the walk starts after the clip
        assert clip_left + clip_right < len(read)
        ridx = _read_index(sel)
        part = sel[ridx[clip_left]:ridx[len(read) - clip_right - 1] + 1]
        assert part[0][0] == "M" and part[-1][0] == "M", "an aligned part must start and end with a matched base"
        cigar, md, zs_items, nm_n = [], [], [], 0
        pos1 = part[0][1] + 1
        op_run, op = 0, None
        md_run = 0
        prev_type, prev_pos = None, 0
        r = clip_left  # read offset (with the left clip)

        def push(o, n):
            nonlocal op, op_run
            if o == op:
                op_run += n
            else:
                if op is not None:
                    cigar.append("%d%s" % (op_run, op))
                op, op_run = o, n

        def zs_item(kind, rpos, v):
            nonlocal prev_type, prev_pos
            rp = rpos - clip_left
            off = rp - (prev_pos + 1) if prev_type == "S" else (rp - prev_pos if prev_type is not None else rp)
            zs_items.append("%d|%s|%s" % (off, kind, self.loc.var_ids[v]))
            prev_type, prev_pos = kind, rp

        for t in part:
            if t[0] == "M":
                push("M", 1)
                b = bases[r]
                if b == bb[t[1]]:
                    md_run += 1
                else:
                    md.append("%d%s" % (md_run, bb[t[1]]))
                    md_run = 0
                    if r not in err and t[3] is not None:
                        zs_item("S", r, t[3])
                    else:
                        nm_n += 1
                r += 1
            elif t[0] == "I":
                if op != "I" and t[3] is not None:
                    zs_item("I", r, t[3])
                push("I", 1)
                nm_n += t[3] is None or r in err
                r += 1
            else:
                if op == "D":  # one D op would stand for both, with a length no variant has
                    raise ValueError("adjacent deletions in the read window")
                push("D", t[2])
                md.append("%d^%s" % (md_run, bb[t[1]:t[1] + t[2]]))
                md_run = 0
                if t[3] is not None:
                    zs_item("D", r, t[3])
                else:
                    nm_n += t[2]
        push(None, 0)
        md.append("%d" % md_run)
        if clip_left:
            cigar.insert(0, "%dS" % clip_left)
        if clip_right:
            cigar.append("%dS" % clip_right)
        seq = "".join(bases)
        fields = [name, str(flag), self.loc.backbone_name, str(pos1), "60", "".join(cigar),
                  "=" if flag & 1 else "*", str(pnext), str(tlen), seq, "I" * len(seq),
                  "AS:i:0", "NM:i:%d" % (nm_n if nm is None else nm), "MD:Z:" + "".join(md), "NH:i:1"]
        if zs and zs_items:
            fields.append("Zs:Z:" + ",".join(zs_items))
        if pad:
            fields.append("XP:Z:" + "A" * pad)
        return "\t".join(fields), part

    def pair(self, name, allele, start, length, frag_len, mate_len=None, errors1=(), errors2=(), **kw):
        """Two name-grouped lines, flags 99 / 147: the second mate ends frag_len read bases after the first begins (moved
        right by up to 10 bases when that would put one of its ends on an inserted base).  Novel indels, clips, nm and pad
        apply to the first mate."""
        mate_len = length if mate_len is None else mate_len
        only1 = {k: kw.pop(k) for k in ("novel_ins", "novel_del", "clip_left", "clip_right", "nm", "pad") if k in kw}
        toks = self.tokens(allele)
        idx = _read_index(toks)
        s2 = start + frag_len - mate_len
        for _ in range(10):
            if _fits(toks, idx, s2, mate_len):
                break
            s2 += 1
        l1, p1 = self.record(name, allele, start, length, flag=99, errors=errors1, **only1, **kw)
        l2, p2 = self.record(name, allele, s2, mate_len, flag=147, errors=errors2, **kw)
        a, b = int(l1.split("\t")[3]), int(l2.split("\t")[3])
        l1 = _set_mate(l1, b, b - a + mate_len)
        l2 = _set_mate(l2, a, -(b - a + mate_len))
        return [l1, l2]

    def sample(self, alleles, n, read_len, frag_len=None, err_rate=0.0, rng=None, prefix="f", zs=None):
        """n pairs (frag_len given) or n single-end reads drawn uniformly from the alleles' read-base ranges, name-grouped."""
        rng = rng or np.random.default_rng(0)
        out = []
        span = frag_len or read_len
        for p in range(n):
            a = alleles[int(rng.integers(0, len(alleles)))]
            toks = self.tokens(a)
            idx = _read_index(toks)
            while True:
                s = int(rng.integers(0, len(idx) - span + 1))
                ends = (s, s + read_len - 1) + ((s + span - read_len, s + span - 1) if frag_len else ())
                ok = all(toks[idx[x]][0] == "M" for x in ends)
                if ok:
                    break
            errs = [k for k in range(read_len) if err_rate and rng.random() < err_rate]
            name = "%s%07d" % (prefix, p)
            if frag_len:
                errs2 = [k for k in range(read_len) if err_rate and rng.random() < err_rate]
                out += self.pair(name, a, s, read_len, frag_len, errors1=errs, errors2=errs2, zs=zs, rng=rng)
            else:
                out.append(self.record(name, a, s, read_len, errors=errs, zs=zs, rng=rng)[0])
        return out


def _set_mate(line, pnext, tlen):
    f = line.split("\t")
    f[7], f[8] = str(pnext), str(tlen)
    return "\t".join(f)


def window_variants(part):
    """Known variant indices carried by the aligned part, in read order (an insertion counts once)."""
    out = []
    for t in part:
        if t[3] is not None and (not out or out[-1] != t[3]):
            out.append(t[3])
    return out


# ---- cases shared by the host (test_record_shapes.py) and device (test_gpu_record_shapes.py) tests ---------------------------
def locus_args(loc, base="hla"):
    """(LocusTables / OracleLocus constructor args) of one synth.Locus."""
    from hisatgenotype_b200 import synth
    cont = synth.reference_containers([loc], base)
    g = loc.gene
    return (base, g, cont["refGenes"][g], cont["Genes"][g][cont["refGenes"][g]], cont["Vars"][g], cont["Var_list"][g],
            cont["Links"], cont["Gene_names"][g], cont["Gene_lengths"][g], cont["refGene_loci"][g][4],
            cont["refGene_loci"][g][5])


def random_backbone(rng, L):
    return "".join(NT[i] for i in rng.integers(0, 4, size=L))


def length_case(read_len, paired, base="hla", seed=11):
    """Simulated reads of read_len bases on a deletion-rich locus, error rate high enough for error correction to fire
    (coverage ~40 so that the pileup sets nt_set)."""
    from helpers import synthetic_case
    L = 1500
    n = max(60, 40 * L // read_len // (2 if paired else 1))
    args, sam, truth = synthetic_case(seed, 120, L=L, n_pairs=n, base=base, del_frac=0.3, n_groups=6, core_vars=40,
                                      pool_private=150, err_rate=0.01, paired=paired, read_len=read_len,
                                      frag_len=max(350, 2 * read_len + 40))
    return args, sam


def dense_snp_locus(spacing=3, n_snp=60, L=700, seed=3):
    """A backbone with a SNP every `spacing` bases from position 100 and one allele carrying all of them: a read of n bases
    from position 100 has (n + spacing - 1) // spacing variant ids.  No deletions, so no Alts entries: every record
    stays in the first walk pass."""
    from hisatgenotype_b200 import synth
    rng = np.random.default_rng(seed)
    bb = random_backbone(rng, L)
    variants = []
    for k in range(n_snp):
        p = 100 + spacing * k
        variants.append(("single", p, NT[(NT.index(bb[p]) + 1) % 4]))
    alleles = {"A*01:01": list(range(n_snp)), "A*01:02": list(range(0, n_snp, 2)), "A*02:01": []}
    return synth.Locus(gene="A", backbone=bb, variants=variants, alleles=alleles,
                       exons=[(80, 300, True), (400, 600, False)])


def exon_cluster_locus(cluster=(7, 8), L=1200, seed=5):
    """Exons of 10 bases, 12 apart, in clusters of the given sizes (one cluster per 300 bases from position 100), and a few
    SNPs inside them: a read over a cluster of k exons has k exon haplotypes, each compatible with its allele."""
    from hisatgenotype_b200 import synth
    rng = np.random.default_rng(seed)
    bb = random_backbone(rng, L)
    exons, variants = [], []
    for c, k in enumerate(cluster):
        for e in range(k):
            left = 100 + 300 * c + 12 * e
            exons.append((left, left + 9, e < 2))
            p = left + 4
            variants.append(("single", p, NT[(NT.index(bb[p]) + 1) % 4]))
    nv = len(variants)
    alleles = {"A*01:01": list(range(nv)), "A*01:02": list(range(0, nv, 2)), "A*01:03": list(range(1, nv, 2)),
               "A*02:01": []}
    return synth.Locus(gene="A", backbone=bb, variants=variants, alleles=alleles, exons=exons)


def single_base_exon_locus(n_exons=300, L=800, seed=6):
    """n_exons adjacent exons of one base each from position 100: a read of n bases inside them has n exon haplotypes."""
    from hisatgenotype_b200 import synth
    rng = np.random.default_rng(seed)
    bb = random_backbone(rng, L)
    variants = [("single", p, NT[(NT.index(bb[p]) + 1) % 4]) for p in range(105, 100 + n_exons, 37)]
    nv = len(variants)
    alleles = {"A*01:01": list(range(nv)), "A*01:02": list(range(0, nv, 2)), "A*02:01": []}
    return synth.Locus(gene="A", backbone=bb, variants=variants, alleles=alleles,
                       exons=[(p, p, p < 110) for p in range(100, 100 + n_exons)])


def plain_locus(L=3000, seed=8):
    """A backbone with a few SNPs only near its ends (room for reads with long novel deletions in between)."""
    from hisatgenotype_b200 import synth
    rng = np.random.default_rng(seed)
    bb = random_backbone(rng, L)
    variants = [("single", p, NT[(NT.index(bb[p]) + 1) % 4]) for p in (20, 40, L - 40, L - 20)]
    alleles = {"A*01:01": [0, 1, 2, 3], "A*01:02": [0, 2], "A*02:01": []}
    return synth.Locus(gene="A", backbone=bb, variants=variants, alleles=alleles,
                       exons=[(10, 60, True), (L - 60, L - 10, False)])


def _fits(toks, idx, s, n, c=0):
    return s >= 0 and s + n <= len(idx) and toks[idx[s + c]][0] == "M" and toks[idx[s + n - 1]][0] == "M"


def _fit_start(toks, idx, s, n):
    """s, or the nearest start to its left whose window begins and ends on a matched base."""
    while not _fits(toks, idx, s, n):
        s -= 1
    return s


def probe_case(seed=21):
    """Error-correction probes of 128 bases on a deletion-rich locus, single-end.  Clean reads of one allele give every
    position an nt_set; each probe carries one error on a SNP of that allele (the correction turns it back into the
    SNP's id, a missed correction leaves an unknown mismatch and the id drops out of the haplotype), at read offset
    t in {0, 31, 32, 63, 64, 95, 96, 127}, after a left clip of c bases so that the M segment starts at r0 = c (word
    r0 // 32 = 0..3 of the mask, bit shift r0 % 32 != 0).  Probes whose window spans 3 and 4 deletions (4 and 5 M
    segments) with an error in the last segment, and reads that run past the backbone end, close the case.
    Returns (locus, lines, {kind: count})."""
    from hisatgenotype_b200 import synth
    loc = synth.make_locus("A", seed, L=1500, n_alleles=60, n_groups=4, core_vars=60, pool_private=150, del_frac=0.3)
    fg = Forge(loc)
    names = sorted(n for n in loc.alleles if loc.alleles[n])
    a = max(names, key=lambda n: sum(loc.variants[v][0] == "deletion" for v in loc.alleles[n]))
    toks = fg.tokens(a)
    idx = _read_index(toks)
    snps = [r for r, k in enumerate(idx) if toks[k][0] == "M" and toks[k][3] is not None]
    rng = np.random.default_rng(seed)
    lines = fg.sample([a], 1500 * 45 // 128, 128, rng=rng, prefix="c")
    hit = {"ws%d" % w: 0 for w in range(4)}
    hit.update(after_del=0, seg4=0, seg5=0, past_end=0)

    def deletions(s, a_, b_):  # read offsets k in [a_, b_] with a deletion right in front of read base k
        return [k for k in range(a_, b_ + 1) if toks[idx[s + k] - 1][0] == "D"]

    n = 0
    # (segment start r0, how): a left clip of r0 bases, or a deletion in front of read base r0 (no deletion between r0
    # and the end, so the segment runs from r0 to the read end)
    for r0 in (0, 5, 37, 70, 100):
        for how in ("clip", "del") if r0 else ("clip",):
            for t in (0, 31, 32, 63, 64, 95, 96, 127):
                if t < r0:
                    continue
                for j in range(len(snps)):
                    s = snps[(j + 7 * n) % len(snps)] - t
                    if not _fits(toks, idx, s, 128, r0 if how == "clip" else 0):
                        continue
                    if how == "clip" and not deletions(s, r0 + 1, 127):
                        break
                    if how == "del" and deletions(s, r0, 127) == [r0]:
                        break
                else:
                    continue
                lines.append(fg.record("p%04d" % n, a, s, 128, errors=[t], clip_left=r0 if how == "clip" else 0)[0])
                hit["ws%d" % (r0 // 32)] += 1
                hit["after_del"] += how == "del"
                n += 1
    # 4 and 5 M segments: windows over 3 / 4 deletions of the allele, error on the last SNP of the window
    for want, key in ((3, "seg4"), (4, "seg5")):
        got = 0
        for s in range(0, len(idx) - 128):
            if not _fits(toks, idx, s, 128):
                continue
            seg = toks[idx[s]:idx[s + 127] + 1]
            if sum(1 for x in seg if x[0] == "D") != want:
                continue
            last = [r - s for r in snps if s <= r < s + 128]
            if not last:
                continue
            lines.append(fg.record("q%04d" % n, a, s, 128, errors=[last[-1]])[0])
            n += 1
            got += 1
            if got == 6:
                break
        hit[key] = got
    # M past the backbone end: the last read of the allele, extended by 5 bases (the walk drops it, the pileup counts it)
    for k in range(3):
        line, part = fg.record("z%04d" % k, a, len(idx) - 100, 100)
        f = line.split("\t")
        ext = 5 + k
        f[5] = re.sub(r"(\d+)M$", lambda m: "%dM" % (int(m.group(1)) + ext), f[5])
        f[9] += "ACGTACGT"[:ext]
        f[10] += "I" * ext
        md = [j for j, x in enumerate(f) if x.startswith("MD:Z:")][0]
        f[md] = re.sub(r"(\d+)$", lambda m: str(int(m.group(1)) + ext), f[md])
        lines.append("\t".join(f))
        hit["past_end"] += 1
    return loc, lines, hit


def indel_case(seed=31):
    """Paired 100 + 100 base reads (fragment 300) from two alleles of a locus with known insertions and deletions, half
    with Zs and half without; plus novel insertions, novel deletions (repeated until the deletion carries the pileup, so
    the artificial-deletion rule of hla keeps them), an N inside an insertion, and soft clips at both ends.
    Returns (locus, lines)."""
    from hisatgenotype_b200 import synth
    loc = synth.make_locus("A", seed, L=1600, n_alleles=60, n_groups=4, core_vars=50, pool_private=150, del_frac=0.2,
                           ins_frac=0.2)
    fg = Forge(loc)
    rng = np.random.default_rng(seed)
    names = sorted(n for n in loc.alleles if loc.alleles[n])
    ins = [n for n in names if any(loc.variants[v][0] == "insertion" for v in loc.alleles[n])]
    truth = [ins[0], ins[len(ins) // 2]]
    lines = fg.sample(truth, 250, 100, frag_len=300, err_rate=0.004, rng=rng, prefix="a", zs=True)
    lines += fg.sample(truth, 250, 100, frag_len=300, err_rate=0.004, rng=rng, prefix="b", zs=False)
    a = truth[0]
    toks = fg.tokens(a)
    idx = _read_index(toks)
    plain = [r for r in range(60, len(idx) - 400) if all(toks[idx[r + j]][0] == "M" and toks[idx[r + j]][3] is None
                                                         and toks[idx[r + j]][1] == toks[idx[r]][1] + j
                                                         for j in range(8))]
    # novel insertion at one place, novel deletion (2 bases, NM 2) at another: 24 pairs each, the first mate carries it
    p_ins, p_del = plain[len(plain) // 4], plain[3 * len(plain) // 4]
    for j in range(24):
        s = _fit_start(toks, idx, p_ins - 30 - 3 * j, 100)
        lines += fg.pair("ni%03d" % j, a, s, 100, 300, novel_ins=(p_ins - s, "GA"))
        s = _fit_start(toks, idx, p_del - 30 - 3 * j, 100)
        lines += fg.pair("nd%03d" % j, a, s, 100, 300, novel_del=(p_del - s, 2))
    # N inside a novel insertion (misaligned, dropped), soft clips at both ends
    s = _fit_start(toks, idx, p_ins - 50, 100)
    lines += fg.pair("nn000", a, s, 100, 300, novel_ins=(p_ins - s, "ANC"))
    for j in range(8):
        s = _fit_start(toks, idx, plain[j * len(plain) // 8] - 40, 100)
        lines += fg.pair("sc%03d" % j, a, s, 100, 300, clip_left=3 + j, clip_right=9 - j)
    return loc, lines


# capacity cases: (locus, base, lines, make_params kwargs, refusal message one past the limit)
CAP_MESSAGES = {
    "ids": "more than 32 variants inside one read",
    "ids_amb": "more than 32 variants inside one read",
    "ids_slow": "more than 32 variants inside one read",
    "ends": "more than 16 alternative ends (or 16 variants in one) around a read",
    "cmp": "more than 96 differences in one alignment",
    "pair_hts": "a read pair expands to more than 255 haplotypes",
    "line": "alignment line longer than 65535 bytes",
    "novel": "novel indel outside the supported range (position < 2^19, length < 2^10)",
}


def homopolymer_locus(k, run=40, L=900, seed=4, snps_before=0, spacing=3):
    """A run of `run` A's at backbone 300 with k one-base deletions inside it (k equivalent placements, one allele each):
    a read ending in the run has up to k alternative ends on that side.  snps_before: a SNP every `spacing` bases
    in front of the run, carried by every deletion allele (the ids of a read that also has several ends)."""
    from hisatgenotype_b200 import synth
    rng = np.random.default_rng(seed)
    r0 = 300
    bb = random_backbone(rng, L)
    bb = bb[:r0 - 1] + "C" + "A" * run + "G" + bb[r0 + run + 1:]
    variants = [("deletion", r0 + 1 + j, "1") for j in range(k)]
    for j in range(snps_before):
        p = r0 - spacing * snps_before + spacing * j
        variants.append(("single", p, NT[(NT.index(bb[p]) + 1) % 4]))
    variants.sort(key=synth._var_key)
    dels = [i for i, v in enumerate(variants) if v[0] == "deletion"]
    snps = [i for i, v in enumerate(variants) if v[0] == "single"]
    alleles = {"A*%02d:01" % (j + 1): sorted([d] + snps) for j, d in enumerate(dels)}
    alleles["A*99:01"] = []
    return synth.Locus(gene="A", backbone=bb, variants=variants, alleles=alleles,
                       exons=[(100, 400, True), (500, 800, False)])


def oracle_ends(ol, line):
    """(left_alts, right_alts, middle ids) identify_ambigious_diffs gives the record, error correction off (sorted lists)."""
    import hgt_oracle as O
    L = len(ol.ref_seq)
    rec = O.parse_record(line, False, 0)
    cmp_list = O.walk_record(ol, rec, [dict() for _ in range(L)], [[] for _ in range(L)], False)[0]
    c2 = []
    for e in cmp_list:
        if e[0] == O.MATCH or (e[0] == O.MISMATCH and (e[3] == O.UNKNOWN or e[3].startswith("nv"))):
            ln = e[2] if e[0] == O.MATCH else 1
            if c2 and c2[-1][0] == O.MATCH:
                c2[-1][2] += ln
            else:
                c2.append([O.MATCH, e[1], ln])
        else:
            c2.append(list(e))
    l, r, la, ra = O.identify_ambiguous_diffs(ol, c2)
    return sorted(la), sorted(ra), [e[3] for e in c2[l:r + 1] if e[0] != O.MATCH]


def find_read(loc, allele, length, want, name="r0"):
    """The first read of `length` bases of the allele (by start) whose oracle ends satisfy want(la, ra, mid)."""
    import hgt_oracle as O
    ol = O.OracleLocus(*locus_args(loc))
    fg = Forge(loc)
    toks = fg.tokens(allele)
    idx = _read_index(toks)
    for s in range(len(idx) - length):
        if not _fits(toks, idx, s, length):
            continue
        line = fg.record(name, allele, s, length)[0]
        try:
            la, ra, mid = oracle_ends(ol, line)
        except O.AmbiguityError:
            continue
        if want(la, ra, mid):
            return line
    raise LookupError("no such read")


def _n_ids(la, ra, mid):
    return la[0].count("hv") + len(mid) + ra[0].count("hv")


def cap_case(kind, past):
    """The walk's capacity `kind` at its limit (past = False: must type exactly as the oracle does) or one past it.  The
    record at the limit is lines[0]."""
    if kind == "ends":  # 17 equivalent one-base deletions in a run of A's: a read with 16 / 17 alternative ends
        loc = homopolymer_locus(17)
        n = 17 if past else 16
        lines = [find_read(loc, "A*01:01", 100, lambda la, ra, mid: max(len(la), len(ra)) == n)]
        lines.append(Forge(loc).record("s0", "A*99:01", 600, 100)[0])
        return loc, "hla", lines, dict(allow_discordant=True)
    if kind in ("ids_amb", "ids_slow"):
        # ids_amb: ONE haplotype whose ends carry ids (the ambiguity pass counts end ids + middle ids): 32 / 33;
        # ids_slow: several haplotypes, 32 / 33 ids between the ends (the slow pass)
        loc = homopolymer_locus(3, snps_before=45)
        n = 33 if past else 32
        if kind == "ids_amb":
            def want(la, ra, mid):
                return len(la) == len(ra) == 1 and "hv" in la[0] + ra[0] and _n_ids(la, ra, mid) == n
        else:
            def want(la, ra, mid):
                return len(la) * len(ra) > 1 and len(mid) == n
        lines = [find_read(loc, "A*03:01" if kind == "ids_amb" else "A*01:01", 110, want)]
        lines.append(Forge(loc).record("s0", "A*99:01", 600, 100)[0])
        return loc, "hla", lines, dict(allow_discordant=True)
    if kind == "ids":  # 96 bases over a SNP every 3 bases: 32 ids; 97 bases: 33
        loc = dense_snp_locus()
        fg = Forge(loc)
        lines = [fg.record("r0", "A*01:01", 100, 97 if past else 96)[0],
                 fg.record("r1", "A*01:02", 400, 100)[0], fg.record("r2", "A*02:01", 20, 100)[0]]
        return loc, "hla", lines, dict(allow_discordant=True)
    if kind == "cmp":  # unknown mismatches at every other base, correction off: 96 / 97 entries (X M X ... M / M X ... M)
        loc = plain_locus()
        fg = Forge(loc)
        errs = list(range(1 if past else 0, 96, 2))
        lines = [fg.record("r0", "A*02:01", 1000, 100, errors=errs)[0], fg.record("r1", "A*01:01", 10, 100)[0]]
        return loc, "hla", lines, dict(allow_discordant=True, error_correction=False, num_editdist=1000)
    if kind == "pair_hts":  # one-base exons: mates over 128 and 127 (128) of them = 255 (256) exon haplotypes in one job
        loc = single_base_exon_locus()
        fg = Forge(loc)
        m2 = 128 if past else 127
        lines = fg.pair("r0", "A*01:01", 100, 128, 128 + m2, mate_len=m2) + fg.pair("r1", "A*01:02", 150, 60, 200)
        return loc, "hla", lines, {}
    if kind == "line":  # 65,535 / 65,536 bytes before the newline, padded with an XP:Z tag
        loc = plain_locus()
        fg = Forge(loc)
        base = fg.record("r0", "A*01:01", 700, 100)[0]
        pad = 65535 + past - len(base) - len("\tXP:Z:")
        lines = [fg.record("r0", "A*01:01", 700, 100, pad=pad)[0], fg.record("r1", "A*01:02", 10, 100)[0]]
        assert len(lines[0]) == 65535 + past
        return loc, "hla", lines, dict(allow_discordant=True)
    if kind == "novel":  # a novel deletion of 1,023 / 1,024 bases in 20 reads (all the reads over it)
        loc = plain_locus()
        fg = Forge(loc)
        n = 1024 if past else 1023
        lines = [fg.record("r%02d" % j, "A*02:01", 500 + j, 120, novel_del=(60 - j, n), nm=0)[0] for j in range(20)]
        lines.append(fg.record("s0", "A*01:01", 10, 100)[0])
        return loc, "hla", lines, dict(allow_discordant=True)
    raise KeyError(kind)


def job_split_case():
    """Pairs whose first mate covers a cluster of 7 exons, or of 8, and whose second mate lies outside every exon: exon-table
    jobs of exactly 7 and exactly 8 haplotypes, where the winning allele count is 7 and 8 (error-free reads).
    Returns (locus, lines, number of pairs over the 8-exon cluster)."""
    loc = exon_cluster_locus((7, 8))
    fg = Forge(loc)
    lines, n8 = [], 0
    for j in range(24):
        a = ("A*01:01", "A*01:02", "A*01:03")[j % 3]
        s = (95 if j % 2 == 0 else 395) - j % 5
        lines += fg.pair("j%03d" % j, a, s, 100, 800 - s)
        n8 += j % 2
    return loc, lines, n8

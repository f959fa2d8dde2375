"""Child process of tests/test_gpu_shim.py: the drop-in modules (hisat-genotype_b200/shim) in front of a STAND-IN reference
tree, typing() called the way genotyping_locus calls it, golden alignments as the "BAM" behind the rig's stand-in
samtools; prints the report files as JSON.

usage: shim_driver.py <golden name> <work dir> [native]"""
import json
import os
import stat
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, ROOT)

FAKE_COMMON = '''
import hisatgenotype_typing_process as typing_process
MARK = "reference common"
def single_abundance(Gene_cmpt, remove_low_abundance_allele=False, Gene_length={}):
    raise AssertionError("the reference's single_abundance must not run on the contracted path")
def align_reads(*args):
    raise AssertionError("align_reads must not run when an alignment file is given")
def _private_helper():
    return 7
'''
FAKE_PROCESS = '''
import hisatgenotype_typing_common as typing_common
'''
FAKE_CORE = '''
import hisatgenotype_typing_common as typing_common
CALLS = []
def typing(*args, **kwargs):
    CALLS.append((args, kwargs))
    return "reference typing"
def genotyping_locus(*args, **kwargs):
    return typing(*args, **kwargs)
'''


def write_stand_in_modules(mods):
    """The three reference modules the drop-in modules load, with the attributes their path touches."""
    os.makedirs(mods, exist_ok=True)
    for fn, text in (("hisatgenotype_typing_common.py", FAKE_COMMON), ("hisatgenotype_typing_process.py", FAKE_PROCESS),
                     ("hisatgenotype_typing_core.py", FAKE_CORE)):
        with open(os.path.join(mods, fn), "w") as f:
            f.write(text)


def main():
    name, work = sys.argv[1], sys.argv[2]
    native = len(sys.argv) > 3 and sys.argv[3] == "native"  # HGT_NATIVE_INTAKE=1 and NO samtools anywhere
    import _hgt_path
    _hgt_path.load()
    from conftest import load_golden
    from helpers import golden_db
    g = load_golden(name)
    p = g["params"]
    db = golden_db(g)
    ref = os.path.join(work, "reference")
    mods = os.path.join(ref, "hisatgenotype_modules")
    os.makedirs(os.path.join(ref, "hisat2"), exist_ok=True)
    write_stand_in_modules(mods)
    first = g["reports"][sorted(g["reports"])[0]].split("\n")
    open(os.path.join(ref, "hisat2", "VERSION"), "w").write(first[1][len("# HISAT2 - "):] + "\n")
    open(os.path.join(ref, "VERSION"), "w").write(first[3][len("# HISAT-genotype - "):] + "\n")
    bindir = os.path.join(work, "bin")
    os.makedirs(bindir, exist_ok=True)
    tool = os.path.join(bindir, "samtools")
    if native:
        os.environ["HGT_NATIVE_INTAKE"] = "1"
        open(tool, "w").write("#!/bin/sh\necho samtools must not run with the native intake >&2\nexit 97\n")
    else:
        open(tool, "w").write(open(os.path.join(ROOT, "oracle", "ref_rig", "samtools")).read().replace(
            "#!/usr/bin/env python3", "#!" + sys.executable, 1))
    os.chmod(tool, os.stat(tool).st_mode | stat.S_IXUSR)
    os.environ["PATH"] = bindir + os.pathsep + os.environ.get("PATH", "")
    os.environ["LC_ALL"] = "C"
    sys.path.insert(0, mods)
    sys.path.insert(0, os.path.join(ROOT, "hisat-genotype_b200", "shim"))
    import hisatgenotype_typing_common as common
    import hisatgenotype_typing_core as core
    checks = {
        "common_reexports": common.MARK == "reference common" and common._private_helper() == 7,
        "single_abundance_is_gpu": common.single_abundance.__module__ == "hisatgenotype_b200.typing_common",
        "typing_installed_in_reference": core._reference.typing is core.typing,
        "genotyping_locus_is_reference": core.genotyping_locus is core._reference.genotyping_locus,
    }
    cmd_line = first[first.index("# COMMAND:") + 1]
    sys.argv = cmd_line.split(" ")
    n_loci = len(p["loci"])
    rep_names = sorted(g["reports"], key=lambda s: int(s.split("test-")[1].split(".")[0]))
    out_dir = os.path.join(work, "out")
    os.makedirs(out_dir, exist_ok=True)
    reports, returned = {}, []
    gene_names = {}
    for cap in g["loci"]:
        gene_names[cap["gene"]] = cap["Gene_names"]
    for t_i, rep in enumerate(rep_names):
        caps = g["loci"][t_i * n_loci:(t_i + 1) * n_loci]
        aln = os.path.join(work, "test%d.bam" % t_i)
        with open(aln, "w") as f:
            for cap in caps:
                f.write("@SQ\tSN:%s\tLN:%d\n" % (cap["ref_allele"], len(db["Genes"][cap["gene"]][cap["ref_allele"]])))
            for cap in caps:
                for line in cap["sam"]:
                    f.write(line + "\n")
        args = (p["simulation"], os.path.join(work, "ix", p["base"]), [cap["test_Gene_names"] if p["simulation"] else cap["gene"] for cap in caps],
                "", True, set(), db["refGenes"], db["Genes"], gene_names, db["Gene_lengths"], db["refGene_loci"], db["Vars"],
                db["Var_list"], db["Links"], [["hisat2", "graph"]], p["num_editdist"], False, "assembly_graph",
                p["error_correction"], True, p["discordant"], False, p["remove_low"], [], False, p["read_fname"], aln, [],
                p["read_len"], p["frag_len"], 1, p["best_alleles"], 0, False, out_dir, "NONE", p["output_allele_counts"], t_i)
        # the way the reference's genotyping_locus reaches typing(): through the reference module's global
        returned.append(core.genotyping_locus(*args))
        reports[rep] = open(os.path.join(out_dir, rep)).read()
    checks["reference_typing_not_called"] = core._reference.CALLS == []
    # a call off the contracted path (--assembly) goes to the reference's typing() with the same arguments
    off = list(args)
    off[16] = True
    checks["assembly_delegated"] = core.typing(*off) == "reference typing" and core._reference.CALLS[-1] == (tuple(off), {})
    print("SHIM_RESULT " + json.dumps({"checks": checks, "reports": reports, "returned": returned}))


if __name__ == "__main__":
    main()

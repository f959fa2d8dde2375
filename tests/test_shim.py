"""CPU-side checks of the drop-in modules (hisat-genotype_b200/shim) in front of a reference tree.  No GPU call is made:
the checks are about names, dispatch and the unchanged CLI.  The tree is $HGT_REFERENCE when set (a hisat-genotype
checkout); otherwise a stand-in holding the modules of tests/shim_driver.py and an entry script that imports
genotyping_locus by name and parses its options, as the reference's `hisatgenotype` does (hisatgenotype:36).

What the stand-in can and cannot show: the dispatch, pass-through and re-export checks run on the shim's own code
either way, but "no name of the reference is missing" is then checked against the stand-in's few names, and the CLI
test then only shows that `from hisatgenotype_typing_core import genotyping_locus` resolves through the shim (the
stand-in script declares --locus-list itself).  Set $HGT_REFERENCE to a reference checkout for those two checks."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT
from shim_driver import write_stand_in_modules

SHIM = os.path.join(ROOT, "hisat-genotype_b200", "shim")

STAND_IN_CLI = r'''
import argparse
import hisatgenotype_typing_common as typing_common
from hisatgenotype_typing_core import genotyping_locus
parser = argparse.ArgumentParser(description="HISAT-genotype")
parser.add_argument("--base", default="hla")
parser.add_argument("--locus-list", default="")
args = parser.parse_args()
'''


@pytest.fixture(scope="module")
def mods(tmp_path_factory):
    """The reference tree's hisatgenotype_modules directory."""
    ref = os.environ.get("HGT_REFERENCE", "")
    if not ref:
        ref = str(tmp_path_factory.mktemp("reference"))
        write_stand_in_modules(os.path.join(ref, "hisatgenotype_modules"))
        with open(os.path.join(ref, "hisatgenotype"), "w") as f:
            f.write(STAND_IN_CLI)
    return os.path.join(ref, "hisatgenotype_modules")


CHILD = r'''
import json, sys, warnings
warnings.filterwarnings("ignore")
import hisatgenotype_typing_common as common
import hisatgenotype_typing_core as core
import _hgt_shim
ref_common = _hgt_shim.load_reference("hisatgenotype_typing_common")
ref_core = _hgt_shim.load_reference("hisatgenotype_typing_core")
def public(m):
    return sorted(k for k in vars(m) if not (k.startswith("__") and k.endswith("__")))
out = {
    "common_file": common.__file__, "core_file": core.__file__,
    "missing_common": [k for k in public(ref_common) if not hasattr(common, k)],
    "missing_core": [k for k in public(ref_core) if not hasattr(core, k)],
    "single_abundance_module": common.single_abundance.__module__,
    "typing_module": core.typing.__module__,
    "ref_global_typing_is_ours": ref_core.typing is core.typing,
    "genotyping_locus_is_reference": core.genotyping_locus is ref_core.genotyping_locus,
    "core_sees_shim_common": ref_core.typing_common is common,
    "process_sees_shim_common": ref_common.typing_process.typing_common is common,
    "other_names_identical": all(getattr(common, k) is getattr(ref_common, k) for k in public(ref_common) if k != "single_abundance")
                             and all(getattr(core, k) is getattr(ref_core, k) for k in public(ref_core) if k != "typing"),
}
if not _hgt_shim.disabled():
    calls = []
    core._reference_typing = lambda *a, **k: calls.append(("reference", a, k)) or "ref"
    core._product.typing = lambda *a, **k: calls.append(("product", a, k)) or "gpu"
    base = [True, "/ix/hla", [["A*01:01"]], "", True, set(), {}, {}, {}, {}, {}, {}, {}, {}, [["hisat2", "graph"]], 2, False,
            "assembly_graph", True, False, False, False, True, [], False, [], "", [], 100, 350, 1, False, 0, False, "out", "NONE", True]
    r = []
    r.append(core.typing(*base))                                   # contracted
    r.append(core.typing(*base, test_i=3))
    for idx, val in ((16, True), (3, "genotype_genome"), (1, "/ix/codis"), (14, [["hisat2", "linear"]]), (14, [["bowtie2", "linear"]]),
                     (14, [["hisat2", "graph"], ["hisat2", "linear"]]), (32, 2)):
        a = list(base); a[idx] = val
        r.append(core.typing(*a))
    out["dispatch"] = r
    out["dispatch_kinds"] = [c[0] for c in calls]
    out["product_got_reference"] = calls[0][2].get("_reference") is ref_core and calls[1][1][37] == 3
    out["reference_args_unchanged"] = calls[2][1][16] is True and len(calls[2][1]) == 37 and calls[2][2] == {}
    try:
        core.typing(*base[:5]); out["short_call"] = "no error"
    except TypeError as e:
        out["short_call"] = "TypeError"
print("CHILD " + json.dumps(out))
'''


def run_child(mods, disable):
    env = dict(os.environ, PYTHONPATH=SHIM + os.pathsep + mods, PYTHONHASHSEED="0")
    env.pop("HGT_DISABLE", None)
    if disable:
        env["HGT_DISABLE"] = "1"
    r = subprocess.run([sys.executable, "-W", "ignore", "-c", CHILD], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    return json.loads([x for x in r.stdout.splitlines() if x.startswith("CHILD ")][-1][6:])


def test_drop_in_modules_wrap_the_reference(mods):
    o = run_child(mods, False)
    assert o["common_file"].startswith(SHIM) and o["core_file"].startswith(SHIM)
    assert o["missing_common"] == [] and o["missing_core"] == []
    assert o["single_abundance_module"] == "hisatgenotype_b200.typing_common"
    assert o["typing_module"] == "hisatgenotype_typing_core"
    assert o["ref_global_typing_is_ours"] and o["genotyping_locus_is_reference"]
    assert o["core_sees_shim_common"] and o["process_sees_shim_common"] and o["other_names_identical"]
    assert o["dispatch"] == ["gpu", "gpu"] + ["ref"] * 7
    assert o["dispatch_kinds"] == ["product", "product"] + ["reference"] * 7
    assert o["product_got_reference"] and o["reference_args_unchanged"]
    assert o["short_call"] == "TypeError"


def test_hgt_disable_is_a_pure_pass_through(mods):
    o = run_child(mods, True)
    assert o["missing_common"] == [] and o["missing_core"] == []
    assert o["single_abundance_module"].startswith("_hgt_ref_")
    assert o["typing_module"].startswith("_hgt_ref_")
    assert o["other_names_identical"]


def test_reference_cli_starts_with_the_drop_in_modules_first(mods):
    """`hisatgenotype` imports genotyping_locus by name (hisatgenotype:36): with the shim directory first on PYTHONPATH the
    unchanged CLI must still come up (argument parser only; no database, no GPU)."""
    cli = os.path.join(os.path.dirname(mods), "hisatgenotype")
    env = dict(os.environ, PYTHONPATH=SHIM + os.pathsep + mods)
    r = subprocess.run([sys.executable, "-W", "ignore", cli, "--help"], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "--locus-list" in r.stdout

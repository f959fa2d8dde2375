"""Drop-in boundary on the GPU: hisat-genotype_b200/shim in front of a reference tree, typing() reached through the
reference's genotyping_locus -> module-global typing (core:2582, 2655), golden alignments as the alignment file, the
FULL `.report` (header included) equal to what the unmodified reference wrote (tests/golden).  The child process builds
a stand-in reference tree with the attributes the path touches (shim_driver.py); tests/test_shim.py checks names,
dispatch and the CLI on the CPU side, against a real reference tree when $HGT_REFERENCE names one."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT, load_golden

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name,mode", [("hla_pair_err", "samtools"), ("cyp_pair", "samtools"), ("hla_single_end", "samtools"),
                                       ("hla_pair_err", "native"), ("hla_indel", "native")])
def test_typing_through_drop_in_modules_writes_reference_report(name, mode, tmp_path):
    """mode "native": HGT_NATIVE_INTAKE=1 - the alignment file is read and split by libhgt (hgt_sam_split_*), any samtools
    call fails the run."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "shim_driver.py"), name, str(tmp_path), mode],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    line = [x for x in r.stdout.splitlines() if x.startswith("SHIM_RESULT ")][-1]
    res = json.loads(line[len("SHIM_RESULT "):])
    assert all(res["checks"].values()), res["checks"]
    g = load_golden(name)
    assert set(res["reports"]) == set(g["reports"])
    for k, text in g["reports"].items():
        assert res["reports"][k] == text, k
    if g["params"]["simulation"]:
        assert all(isinstance(x, dict) for x in res["returned"])  # test_passed (core:2170-2171)
    else:
        assert all(x is None for x in res["returned"])

"""bench.py end to end on a small database: --steps sets the number of timed steps and --dump-outputs writes what the
last of them computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


def test_bench_steps_and_dump_outputs(tmp_path):
    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1", "--samples", "2",
           "--scale", "0.05", "--oversized-sub-reads", "0", "--no-cpu-baseline", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, env=dict(os.environ, HGT_BENCH_NO_SMI="1"), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    line = json.loads([x for x in r.stdout.splitlines() if x.startswith("{")][-1])
    assert line["steps"] == 2 and len(line["step_ms_rank0"]) == 2
    got = {f[:-4]: np.load(str(out / f)) for f in os.listdir(str(out))}
    assert set(got) == {"unit_summary", "top_calls", "sample_units", "abundance", "allele_counts", "classes"}
    assert all(a.dtype == np.float64 and np.isfinite(a).all() for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    summary = got["unit_summary"]
    assert summary.shape == (12, 10)  # 2 samples x 6 loci
    assert summary[:, 0].sum() == line["reads_per_step"]
    assert got["sample_units"].tolist() == list(range(12))
    # the example call of the line comes from a separate batch of the same units: the same top two abundances
    assert got["top_calls"][0, :2, 1].tolist() == pytest.approx([p for _, p in line["example_call"]], rel=1e-12)
    assert (got["top_calls"][:, 0, 1] > 0).all()
    assert len(got["abundance"]) == len(got["allele_counts"])
    # one row per class of every table of every unit; a table's classes hold at most the unit's pairs
    n_cls = summary[:, 2:6].astype(int)
    assert len(got["classes"]) == n_cls.sum()
    rows = np.concatenate([[0], np.cumsum(n_cls.reshape(-1))])
    for u in range(12):
        gene = got["classes"][rows[4 * u]:rows[4 * u + 1]]
        assert len(gene) > 0 and 0 < gene[:, 0].sum() <= summary[u, 1]

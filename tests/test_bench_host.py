"""Host-side pieces of bench.py that need no GPU: the LPT packing of units onto ranks (SURVEY.md 8e), the
sub-record launcher's environment (children of a torchrun worker must not look for the agent's store) and the files
of --dump-outputs."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_lpt_pack_covers_and_balances():
    import bench
    rng = np.random.default_rng(3)
    costs = (rng.pareto(1.5, size=200) * 100 + 1).tolist()  # long tail, like reads x W over a panel of loci
    for n_bins in (1, 2, 4, 8):
        bins, loads = bench.lpt_pack(costs, n_bins)
        assert sorted(u for b in bins for u in b) == list(range(len(costs)))
        for b, load in zip(bins, loads):
            assert abs(sum(costs[u] for u in b) - load) < 1e-6 * max(load, 1.0)
        # LPT guarantee: the heaviest bin is within 4/3 of the optimum, itself >= max(mean load, largest unit)
        lower = max(sum(costs) / n_bins, max(costs))
        assert max(loads) <= 4.0 / 3.0 * lower + 1e-9
    bins, loads = bench.lpt_pack([], 4)
    assert bins == [[], [], [], []] and loads == [0.0] * 4


def test_subrecord_is_skipped_when_disabled():
    import argparse

    import bench
    args = argparse.Namespace(oversized_sub_reads=0)
    assert bench.oversized_subrecord(args, 0, 1) is None


def test_subrecord_child_environment(monkeypatch):
    """The child gets its own rendezvous port and none of the TORCHELASTIC_* variables (with them init_process_group would
    wait for the parent agent's store on the new port)."""
    import argparse
    import subprocess

    import bench
    seen = {}

    class Done:
        returncode = 0
        stdout = '{"value": 1.0, "config": {"workload": "w"}, "e2e": {"value": 2.0, "unit": "reads/s", "ms_per_step": 3.0}}\n'
        stderr = ""

    def fake_run(cmd, env=None, **kw):
        seen["cmd"], seen["env"] = cmd, env
        return Done()

    monkeypatch.setattr(subprocess, "run", fake_run)
    monkeypatch.setenv("MASTER_PORT", "29500")
    monkeypatch.setenv("TORCHELASTIC_USE_AGENT_STORE", "True")
    monkeypatch.setenv("TORCHELASTIC_RUN_ID", "x")
    sub = bench.oversized_subrecord(argparse.Namespace(oversized_sub_reads=1000), 0, 2)
    assert seen["env"]["MASTER_PORT"] == "29501"
    assert not any(k.startswith("TORCHELASTIC_") for k in seen["env"])
    assert "--workload" in seen["cmd"] and "oversized" in seen["cmd"] and "1000" in seen["cmd"]
    assert sub["value"] == 1.0 and sub["workload"] == "w" and sub["e2e"]["ms_per_step"] == 3.0
    # a rank other than 0 launches the child too (the job is collective) but reports nothing
    assert bench.oversized_subrecord(argparse.Namespace(oversized_sub_reads=1000), 1, 2) is None


class _FakeLocus:
    def __init__(self, n):
        self.A, self.wp = n, (n + 63) // 64
        self.names = ["L%d*%02d" % (n, i) for i in range(n)]


class _FakeBatch:
    """The Batch methods dump_outputs reads, on made-up results: unit u has u + 1 classes per table."""

    def __init__(self, loci, unit_locus):
        self.loci, self.unit_locus = loci, unit_locus

    def unit_summary(self, u):
        return dict(num_reads=10 * u, num_pairs=5 * u, n_classes=[u + 1] * 4, em_iters=[3, 0], em_status=[0, 1])

    def unit_calls(self, u, max_n=None):
        names = self.loci[self.unit_locus[u]].names
        calls = [[names[0], 0.75], [names[-1], 0.25]]
        return calls[:max_n]

    def top_calls(self, max_n):
        return [self.unit_calls(u, max_n) for u in range(len(self.unit_locus))]

    def unit_table(self, u, table):
        t = self.loci[self.unit_locus[u]]
        bits = np.full((u + 1, t.wp), 3, np.uint64)
        acount = np.arange(t.A, dtype=np.int64) + table
        return bits, np.full(u + 1, 7, np.int64), np.arange(u + 1, dtype=np.int64), acount, np.zeros(t.A, np.int64)


def test_dump_outputs_files(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_UNITS", 3)
    loci = [_FakeLocus(70), _FakeLocus(5)]
    batches = [_FakeBatch(loci, [0, 1, 1]), _FakeBatch(loci, [1, 0])]
    bench.dump_outputs(str(tmp_path), batches)
    got = {f[:-4]: np.load(os.path.join(str(tmp_path), f)) for f in os.listdir(str(tmp_path))}
    assert set(got) == {"unit_summary", "top_calls", "sample_units", "abundance", "allele_counts", "classes"}
    assert all(a.dtype == np.float64 and np.isfinite(a).all() for a in got.values())
    assert got["unit_summary"].shape == (5, 10)
    assert got["unit_summary"][4].tolist() == [10, 5, 2, 2, 2, 2, 3, 0, 0, 1]  # unit 1 of the second batch
    top = got["top_calls"]
    assert top.shape == (5, bench.DUMP_TOP, 2)
    assert top[0, 0].tolist() == [0, 0.75] and top[0, 1].tolist() == [69, 0.25] and (top[0, 2:] == [-1, 0]).all()
    pick = got["sample_units"].astype(int).tolist()
    assert len(pick) == 3 and pick == sorted(set(pick)) and all(0 <= k < 5 for k in pick)
    units = [(b, u) for b in batches for u in range(len(b.unit_locus))]
    n_alleles = [units[k][0].loci[units[k][0].unit_locus[units[k][1]]].A for k in pick]
    assert got["abundance"].shape == (sum(n_alleles),) and got["allele_counts"].shape == (sum(n_alleles), 4)
    assert got["abundance"][0] == 0.75 and got["abundance"][n_alleles[0] - 1] == 0.25
    assert got["abundance"].sum() == 3 * 1.0
    assert got["allele_counts"][1].tolist() == [1, 2, 3, 4]
    n_classes = [4 * (units[k][1] + 1) for k in pick]
    assert got["classes"].shape == (sum(n_classes), 4)
    w = units[pick[0]][0].loci[units[pick[0]][0].unit_locus[units[pick[0]][1]]].wp
    assert got["classes"][0, :3].tolist() == [7, 2 * w, 0]
    # the member hash tells classes of equal size apart and is the same for equal rows
    import hashlib
    row = np.full(w, 3, np.uint64).tobytes()
    assert got["classes"][0, 3] == int.from_bytes(hashlib.blake2b(row, digest_size=6).digest(), "little")
    assert got["classes"][0, 3] != int.from_bytes(hashlib.blake2b(np.full(w, 5, np.uint64).tobytes(), digest_size=6).digest(),
                                                  "little")
    # the same call writes the same sample
    bench.dump_outputs(str(tmp_path / "again"), batches)
    assert np.load(str(tmp_path / "again" / "sample_units.npy")).tolist() == got["sample_units"].tolist()

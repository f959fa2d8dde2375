#!/usr/bin/env python3
"""Benchmark of the typing hot path (stage a: per-read allele compatibility -> Gene_cmpt/Gene_counts, stage b: EM).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--samples S] [--impl reference] [--dump-outputs DIR]

Workload = BASELINE.json configs[1]: HLA-A/B/C/DQA1/DQB1/DRB1, paired-end 2x100 bp, 30x, synthetic database of the
named shape (SURVEY.md 8d) and reads drawn from a random diploid genotype per sample with 0.5 % sequencing
errors; alignment records are synthesised HISAT2-style from the true placement (tools/simgen.cpp).  One step =
one batch of S samples x 6 loci through the whole path.  Prints ONE JSON line (see DESIGN.md "Measurement").

  value  reads typed/s with the packed alignments already resident in HBM (execute+finish of a prepared batch)
  e2e    the same through the public batch call with HOST alignment text: intake, pileup, walk, H2D, kernels, D2H
  roofline      stage (a) kernels against the measured HBM copy bandwidth (MEASURED_PEAKS.json)
  cpu_baseline  the oracle port (oracle/hgt_oracle.py, oracle/em_oracle.c) on one host core, bounded sample
--impl reference: the oracle port on all host cores (multiprocessing over units, like hisatgenotype:613-665).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LOCI = [  # gene, backbone length, alleles, allele groups  (SURVEY.md 8d, config 2)
    ("A", 3500, 7000, 60), ("B", 3500, 8000, 64), ("C", 3500, 7000, 60),
    ("DQA1", 6000, 400, 10), ("DQB1", 7000, 2000, 30), ("DRB1", 11000, 3000, 40),
]
READ_LEN, FRAG_LEN, COVERAGE, ERR = 100, 350, 30, 0.005
DB_SEED = 7
# GPU stages bracketed with CUDA events (hgt_profile_read) and host stages (hgt_profile_host), see include/hgt.h
STAGES = ["records", "compat", "class", "counts", "em1", "project", "em2", "walk"]
HOST_STAGES = ["text_h2d_issue", "tables_linecount_wait", "", "", "", "alloc", "finish_host_and_em2", ""]


def build_database(scale=1.0):
    import _hgt_path
    _hgt_path.load()
    from hisatgenotype_b200 import synth
    loci = []
    for i, (gene, L, A, G) in enumerate(LOCI):
        A = max(40, int(A * scale))
        G = max(4, int(G * min(1.0, scale * 2)))
        loci.append(synth.make_locus(gene, DB_SEED + i, L=L, n_alleles=A, n_groups=G, core_vars=80,
                                     pool_private=max(100, int(1600 * min(1.0, A / 7000.0 + 0.2))), del_frac=0.06))
    cont = synth.reference_containers(loci, "hla")
    return loci, cont


def locus_args(cont, gene):
    return ("hla", gene, cont["refGenes"][gene], cont["Genes"][gene][cont["refGenes"][gene]], cont["Vars"][gene],
            cont["Var_list"][gene], cont["Links"], cont["Gene_names"][gene], cont["Gene_lengths"][gene],
            cont["refGene_loci"][gene][4], cont["refGene_loci"][gene][5])


def simulate_units(loci, sims, n_samples, sample0):
    """[(locus index, alignment text bytes)] for samples sample0 .. sample0+n_samples-1 (seeded per sample)."""
    import numpy as np
    units = []
    for s in range(sample0, sample0 + n_samples):
        rng = np.random.default_rng(1000 + s)
        for li, loc in enumerate(loci):
            names = sims[li]["names"]
            truth = [names[i] for i in rng.choice(len(names), 2, replace=False)]
            n_pairs = int(round(COVERAGE * len(loc.backbone) / (2.0 * READ_LEN)))
            text = sims[li]["sim"].generate(truth, n_pairs, seed=s * 64 + li + 1, err_rate=ERR, read_len=READ_LEN,
                                            frag_len=FRAG_LEN, paired=True, prefix="s%05d_" % s)
            units.append((li, text))
    return units


class ClockSampler:
    """nvidia-smi clocks / throttle reasons in a side process.  It is started BEFORE the warm-up steps (the first NVML
    query of a fresh nvidia-smi stalls kernel submission for tens of ms, which must not land in a timed step) and keeps
    sampling every 100 ms; the `with` block marks the timed region and summary() reports the samples taken inside it
    (all samples since start-up if the region was shorter than one interval, with "window" saying which)."""

    def __init__(self, device):
        self.rows, self.t0, self.t1 = [], None, None
        self.device = device
        self.proc = None
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            if os.environ.get("HGT_BENCH_NO_SMI"):
                raise OSError("sampling switched off")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, universal_newlines=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def wait_first(self, timeout=5.0):
        end = time.time() + timeout
        while self.proc and not self.rows and time.time() < end:
            time.sleep(0.02)

    def __enter__(self):
        self.t0 = time.time()
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def __exit__(self, *a):
        self.t1 = time.time()

    def close(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
            self.proc = None

    def summary(self):
        self.close()
        inside = [r for t, r in self.rows if self.t0 is not None and self.t0 <= t <= (self.t1 or t) + 0.1]
        window = "timed region"
        if not inside:
            inside, window = [r for _, r in self.rows], "warm-up + timed region (region shorter than the 100 ms interval)"
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in inside:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm), "window": window}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------------------
# oracle-port legs (CPU)
# ------------------------------------------------------------------------------------------------------------
_ORACLE = {}
ORACLE_DISCORDANT = [False]  # --discordant of the workload (single-end reads need it)


def _oracle_unit(job, keep=False):
    li, text = job
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import em_oracle
    import hgt_oracle as O
    ol = _ORACLE["loci"][li]
    t0 = time.perf_counter()
    res = O.type_locus(ol, text.decode().splitlines(), allow_discordant=ORACLE_DISCORDANT[0])
    ta = time.perf_counter() - t0
    t0 = time.perf_counter()
    iters = 0
    cm = res["tables"]["exon"].cmpt_items(ol)
    if cm:
        _, it = em_oracle.single_abundance(cm, True, None)
        iters += it
    tb = time.perf_counter() - t0
    if not keep:
        return res["num_reads"], ta, iters, tb
    # parity material (untimed): the three tables in dict order and the ranked calls of the EM driver
    tabs = {k: (res["tables"][k].cmpt_items(ol), res["tables"][k].count_items(ol)) for k in ("gene", "exon", "primary")}
    return res["num_reads"], ta, iters, tb, res["num_pairs"], tabs, O.locus_abundance(ol, res, True)


def build_oracle_loci(cont, loci):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import hgt_oracle as O
    _ORACLE["loci"] = [O.OracleLocus(*locus_args(cont, loc.gene)) for loc in loci]


def cpu_baseline(units, batch=None):
    """Oracle port on ONE core over a bounded sample of the same workload.  With `batch` (the GPU batch whose first
    units are these units) every table, count list and ranked call of the sample is compared with the GPU's: the bench
    checks what it times."""
    reads = ta = iters = tb = 0
    parity = {"units": 0, "tables": 0, "identical": True, "max_rel_abundance_err": 0.0, "first_difference": None}

    def differ(what):
        parity["identical"] = False
        if parity["first_difference"] is None:
            parity["first_difference"] = what

    for u, job in enumerate(units):
        out = _oracle_unit(job, keep=batch is not None)
        r, a, i, b = out[:4]
        reads += r
        ta += a
        iters += i
        tb += b
        if batch is None:
            continue
        pairs, tabs, calls = out[4:]
        s = batch.unit_summary(u)
        if (s["num_reads"], s["num_pairs"]) != (r, pairs):
            differ("unit %d: reads/pairs %s vs oracle %s" % (u, (s["num_reads"], s["num_pairs"]), (r, pairs)))
        for t_i, key in enumerate(("gene", "exon", "primary")):
            if list(map(list, batch.unit_gene_cmpt(u, t_i).items())) != tabs[key][0]:
                differ("unit %d: Gene_cmpt of table %s" % (u, key))
            if batch.unit_gene_counts(u, t_i) != tabs[key][1]:
                differ("unit %d: Gene_counts of table %s" % (u, key))
            parity["tables"] += 1
        got = batch.unit_calls(u)
        if [x for x, _ in got] != [x for x, _ in calls]:
            differ("unit %d: ranked alleles %s vs oracle %s" % (u, got[:3], calls[:3]))
        else:
            for (_, x), (_, y) in zip(got, calls):
                rel = abs(x - y) / max(abs(y), 1e-300)
                parity["max_rel_abundance_err"] = max(parity["max_rel_abundance_err"], rel)
                if rel > 1e-6 and abs(x - y) > 1e-12:
                    differ("unit %d: abundance %r vs oracle %r" % (u, x, y))
        parity["units"] += 1
    base = {"value": reads / ta if ta > 0 else None, "unit": "reads/s", "cores": 1, "kind": "port",
            "sample": "%d (sample, locus) units = %d reads of the same workload, oracle/hgt_oracle.py stage (a); "
                      "EM via oracle/em_oracle.c" % (len(units), reads),
            "em_iters_per_sec": iters / tb if tb > 0 else None, "seconds": ta + tb}
    return base, (parity if batch is not None else None)


def run_reference_arm(args):
    """--impl reference: the CPU implementation of the path (oracle port of the reference's Python) on all cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import multiprocessing as mp
    scale = args.scale
    loci, cont = build_database(scale)
    from hisatgenotype_b200 import synth
    sims = [{"sim": synth.ReadSimulator(l), "names": sorted(n for n in l.alleles if l.alleles[n])} for l in loci]
    build_oracle_loci(cont, loci)
    cores = os.cpu_count() or 1
    n_samples = max(1, args.ref_samples)
    ctx = mp.get_context("fork")
    times, reads_step = [], 0
    with ctx.Pool(cores) as pool:
        for step in range(args.warmup + args.steps):
            units = simulate_units(loci, sims, n_samples, 100000 + step * n_samples)
            t0 = time.perf_counter()
            out = pool.map(_oracle_unit, units, chunksize=1)
            dt = time.perf_counter() - t0
            if step >= args.warmup:
                times.append(dt)
                reads_step = sum(o[0] for o in out)
    ms = 1000.0 * sum(times) / len(times)
    value = reads_step / (ms / 1000.0)
    line = {
        "impl": "reference", "metric": "reads typed/sec", "value": value, "unit": "reads/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64 bitsets + f64 EM", "data": "synthetic",
        "config": workload_config(args, n_samples),
        "cpu_baseline": {"value": value, "unit": "reads/s", "cores": cores, "kind": "port",
                         "sample": "%d samples x 6 loci per step (%d reads), oracle port, multiprocessing over units"
                                   % (n_samples, reads_step)},
        "e2e": {"value": value, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


def workload_config(args, n_samples):
    return {"workload": "BASELINE configs[1]: HLA-A/B/C/DQA1/DQB1/DRB1 paired-end 2x100 30x, synthetic database "
                        "(A=7000/8000/7000/400/2000/3000 alleles, scale %.3g), batch of %d samples x 6 loci per step"
                        % (args.scale, n_samples),
            "samples_per_step": n_samples, "loci": [g for g, _, _, _ in LOCI], "coverage": COVERAGE,
            "read_len": READ_LEN, "error_rate": ERR, "db_seed": DB_SEED,
            "l2": "inputs per step exceed L2 and a 512 MiB buffer is rewritten between timed steps"}


# ------------------------------------------------------------------------------------------------------------
# BASELINE configs[3]: one oversized locus (A = 8192 alleles, W = 128 words per allele set), single-end reads
# ------------------------------------------------------------------------------------------------------------
def build_oversized():
    import _hgt_path
    _hgt_path.load()
    from hisatgenotype_b200 import synth
    loc = synth.make_locus("OV", 13, L=10000, n_alleles=8191, n_groups=64, core_vars=110, pool_private=3600,
                           del_frac=0.06)
    cont = synth.reference_containers([loc], "ov")
    return loc, cont


def run_oversized(args):
    import ctypes
    import numpy as np
    import torch
    import _hgt_path
    _hgt_path.load()
    from hisatgenotype_b200 import _lib, synth
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.locus import LocusTables

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        raise SystemExit("bench: --dump-outputs of the oversized workload needs one GPU (with more, the EM of the "
                         "read-sharded unit runs outside the batch)")
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    ctx = _lib.ctx(local)
    L = _lib.lib()
    loc, cont = build_oversized()
    a = list(locus_args(cont, "OV"))
    a[0] = "ov"
    table = LocusTables(*a, device=local)
    names = sorted(n for n in loc.alleles if loc.alleles[n])
    truth = [names[1000], names[5000]]
    n_reads = args.oversized_reads // world  # reads shard over the ranks (SURVEY.md 8e)
    sim = synth.ReadSimulator(loc)
    text = sim.generate(truth, n_reads, seed=77 + rank, err_rate=ERR, read_len=READ_LEN, frag_len=FRAG_LEN, paired=False,
                        prefix="k%02d_" % rank)
    # host threads of the intake / walk stages: the ranks of one box share its cores
    host_threads = max(1, (os.cpu_count() or 1) // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", world))))
    params = TC.make_params(allow_discordant=True, n_threads=host_threads)
    stream = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def new_batch():
        bt = TC.Batch([table], params, True, device=local)
        if world > 1:
            bt.set_pileup_allreduce()   # nt_set comes from the pileup of ALL reads: one all-reduce of the raw counts
            bt.set_skip_em(True)        # the EM runs sharded: partial sweeps + all-reduce (em_dist.py)
        bt.add_unit(0, text)
        return bt

    em_state = {"iters": 0, "calls": None}

    def run_gpu(bt):
        t0 = time.perf_counter()
        bt.execute(stream)
        t1 = time.perf_counter()
        bt.finish(stream)
        t2 = time.perf_counter()
        if world > 1:
            em_state["calls"], em_state["iters"] = bt.sharded_abundance(0, max_n=2)
            em_state["shard_ms"] = dict(bt.shard_ms, execute=(t1 - t0) * 1e3, finish=(t2 - t1) * 1e3,
                                        call=(time.perf_counter() - t2) * 1e3)

    batch = new_batch()
    batch.prepare()
    run_gpu(batch)
    tot = batch.totals()
    L.hgt_profile_enable(ctx, 1)
    # the database and the alignment text are millions of long-lived Python objects: park them in the permanent
    # generation so that a full collection (tens of ms) cannot fire inside a timed step
    import gc
    gc.collect()
    gc.freeze()
    sampler = ClockSampler(local)
    sampler.wait_first()
    for _ in range(args.warmup):
        run_gpu(batch)
    L.hgt_profile_reset(ctx)
    launches0 = L.hgt_launch_count(ctx)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    with sampler as clocks:
        for k in range(args.steps):
            flush.zero_()
            ev[k][0].record()
            run_gpu(batch)
            ev[k][1].record()
        barrier()
    dev_ms = float(sum(x.elapsed_time(y) for x, y in ev))
    em_trace_once(L, ctx, lambda: run_gpu(batch))
    launches = L.hgt_launch_count(ctx) - launches0
    stage_ms, stage_n = ctypes_array(8, "d"), ctypes_array(8, "q")
    h2d, d2h = ctypes.c_int64(0), ctypes.c_int64(0)
    L.hgt_profile_read(ctx, stage_ms, stage_n, ctypes.byref(h2d), ctypes.byref(d2h))
    stage = {n: stage_ms[i] / args.steps for i, n in enumerate(STAGES)}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [batch])
    summ = batch.unit_summary(0)
    C, it = summ["n_classes"][0], (em_state["iters"] if world > 1 else summ["em_iters"][0])
    em_bytes = it * (3 * C * (table.wp * 8 + 8) + 6 * table.A * 8)
    t_vec = torch.tensor([dev_ms, float(tot["num_reads"])], dtype=torch.float64, device="cuda")
    if world > 1:
        mx, sm = t_vec.clone(), t_vec.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        dev_ms_all, reads_all = float(mx[0]), float(sm[1])
    else:
        dev_ms_all, reads_all = dev_ms, float(tot["num_reads"])
    ms_per_step = dev_ms_all / args.steps
    value = reads_all / (ms_per_step / 1000.0)
    # e2e: alignment text in host memory -> ranked alleles
    L.hgt_profile_reset(ctx)
    e2e_ms = []
    for k in range(3):
        barrier()
        x, y = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if k == 1:
            L.hgt_profile_reset(ctx)
        x.record()
        bt = new_batch()
        bt.prepare()
        run_gpu(bt)
        calls = [em_state["calls"][:2]] if world > 1 else bt.top_calls(2)
        y.record()
        torch.cuda.synchronize()
        if k >= 1:
            e2e_ms.append(x.elapsed_time(y))
        bt.close()
    L.hgt_profile_read(ctx, stage_ms, stage_n, ctypes.byref(h2d), ctypes.byref(d2h))
    host_ms = ctypes_array(8, "d")
    L.hgt_profile_host(ctx, host_ms)
    e2e_vec = torch.tensor([sum(e2e_ms) / len(e2e_ms)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_vec, op=dist.ReduceOp.MAX)
    if rank == 0:
        peak, peak_src = measured_peak()
        a_ms = stage["compat"] + stage["class"]
        a_bytes = float(tot["algorithmic_bytes"])
        line = {
            "metric": "reads typed/sec", "value": value, "unit": "reads/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u64 bitsets + f64 EM", "data": "synthetic",
            "config": {"workload": "BASELINE configs[3]: one oversized locus, A=%d alleles (W=%d words), V=%d, L=%d, %d "
                                   "single-end 100 bp reads from a 2-allele genotype, 0.5 %% errors, reads sharded over %d "
                                   "GPU(s)" % (table.A, table.wp, table.V, len(loc.backbone), args.oversized_reads, world),
                       "l2": "per-step inputs (%.1f GB of allele-set rows) exceed L2; a 512 MiB buffer is rewritten between "
                             "timed steps" % (tot["num_pairs"] * table.wp * 8 / 1e9)},
            "reads_per_step": reads_all, "classes_rank0": C, "em_iters_rank0": it,
            "sharded_em_wall_ms_rank0": em_state.get("shard_ms"),
            "step_ms_rank0": [round(x.elapsed_time(y), 3) for x, y in ev],
            "stage_ms_per_step_rank0": stage,
            # N = 1: the cooperative EM launch is the dominant kernel; N > 1: the EM runs as partial sweeps + NCCL
            # all-reduce (em_dist.py) outside the stage timers and stage (a) is what the timers see
            "roofline": ({"bound": "hbm", "achieved": em_bytes / (stage["em1"] / 1000.0) / 1e9, "peak": peak, "unit": "GB/s",
                          "frac": em_bytes / (stage["em1"] / 1000.0) / 1e9 / peak,
                          "traffic": ncu_traffic("em_kernel", "oversized", args.oversized_reads),
                          "kernel": "em_kernel (cooperative, one problem on all SMs)", "peak_source": peak_src,
                          "launches_per_step": 1, "algorithmic_bytes_per_launch": float(em_bytes),
                          "avg_launch_ms": stage["em1"], "share_of_step": stage["em1"] / ms_per_step}
                         if world == 1 and stage["em1"] > 0 else
                         {"bound": "hbm", "achieved": a_bytes / (a_ms / 1000.0) / 1e9 if a_ms > 0 else None, "peak": peak,
                          "unit": "GB/s", "frac": a_bytes / (a_ms / 1000.0) / 1e9 / peak if a_ms > 0 else None,
                          "traffic": ncu_traffic("stage_a", "oversized", args.oversized_reads),
                          "kernel": "stage (a): compat_kernel + class_kernel", "peak_source": peak_src,
                          "algorithmic_bytes_per_step": a_bytes, "kernel_ms_per_step": a_ms}),
            "roofline_stage_a": {"bound": "hbm", "achieved": a_bytes / (a_ms / 1000.0) / 1e9 if a_ms > 0 else None,
                                 "peak": peak, "unit": "GB/s",
                                 "frac": a_bytes / (a_ms / 1000.0) / 1e9 / peak if a_ms > 0 else None,
                                 "traffic": ncu_traffic("stage_a", "oversized", args.oversized_reads, per="step"),
                                 "kernel": "stage (a): compat_kernel + class_kernel",
                                 "algorithmic_bytes_per_step": a_bytes, "kernel_ms_per_step": a_ms},
            "em_iters_per_sec_kernel_time": it / (stage["em1"] / 1000.0) if stage["em1"] > 0 else None,
            "e2e": {"value": reads_all / (float(e2e_vec[0]) / 1000.0), "unit": "reads/s",
                    "h2d_bytes_per_step": h2d.value / 2, "d2h_bytes_per_step": d2h.value / 2,
                    "ms_per_step": float(e2e_vec[0]), "input": "host alignment text, %d bytes on rank 0" % len(text),
                    "host_stage_ms_rank0": {n: host_ms[i] / 2 for i, n in enumerate(HOST_STAGES) if n},
                    "host_threads": host_threads, "host_cores": os.cpu_count()},
            "gpu_launches": int(launches), "clocks": clocks.summary(), "example_call": calls[0],
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0



# ------------------------------------------------------------------------------------------------------------
# BASELINE configs[0], [2], [4]: single locus (latency), full panel (LPT packing of units), 1,000-sample batch
# (strong scaling).  One JSON line each, same keys as the default line (value = device-resident, e2e = pipelined stream
# from page-locked host text).
# ------------------------------------------------------------------------------------------------------------
PANEL = [  # gene, backbone length, alleles, groups: 30 loci, sum of alleles ~ 25 k (SURVEY.md 8d config 3)
    ("A", 3500, 6000, 56), ("B", 3500, 7000, 60), ("C", 3500, 6000, 56), ("DRB1", 11000, 2000, 36), ("DQB1", 7000, 1500, 28),
    ("DPB1", 11000, 1200, 24), ("DQA1", 6000, 400, 10), ("E", 3500, 300, 8), ("DRB3", 11000, 300, 8), ("MICA", 11000, 250, 8),
    ("DPA1", 9000, 200, 6), ("MICB", 11000, 200, 6), ("DRB4", 11000, 150, 6), ("DRB5", 11000, 120, 5), ("G", 3500, 100, 5),
    ("F", 3500, 50, 4), ("H", 3500, 30, 4), ("DRA", 5000, 30, 4), ("J", 3500, 20, 4), ("K", 3500, 20, 4), ("DMA", 4500, 20, 4),
    ("DMB", 6000, 20, 4), ("DOA", 3500, 20, 4), ("DOB", 4500, 20, 4), ("TAP1", 9000, 20, 4), ("TAP2", 10000, 20, 4),
    ("L", 3500, 10, 4), ("V", 3000, 10, 4), ("Y", 3000, 10, 4), ("HFE", 10000, 10, 4),
]


def build_panel(scale=1.0):
    import _hgt_path
    _hgt_path.load()
    from hisatgenotype_b200 import synth
    loci = []
    for i, (gene, L, A, G) in enumerate(PANEL):
        A = max(10, int(A * scale))
        loci.append(synth.make_locus(gene, 11 + i, L=L, n_alleles=A, n_groups=max(2, min(G, A // 3)), core_vars=60,
                                     pool_private=max(40, int(1600 * min(1.0, A / 7000.0 + 0.05))), del_frac=0.06))
    return loci, synth.reference_containers(loci, "hla")


def lpt_pack(costs, n_bins):
    """Longest-processing-time-first packing: unit indices per bin and the bins' loads (SURVEY.md 8e)."""
    import heapq
    bins = [[] for _ in range(n_bins)]
    heap = [(0.0, b) for b in range(n_bins)]
    for u in sorted(range(len(costs)), key=lambda k: -costs[k]):
        load, b = heapq.heappop(heap)
        bins[b].append(u)
        heapq.heappush(heap, (load + costs[u], b))
    loads = [0.0] * n_bins
    for load, b in heap:
        loads[b] = load
    return bins, loads


def run_workload(args):
    import ctypes
    import gc
    import numpy as np
    import torch
    import _hgt_path
    _hgt_path.load()
    from hisatgenotype_b200 import _lib, synth
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.locus import LocusTables

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    os.environ["HGT_DEVICE"] = str(local)
    ctx = _lib.ctx(local)
    L = _lib.lib()
    wl = args.workload
    paired, scaling, extra = True, "strong", {}
    if wl == "single-locus":  # configs[0]: one HLA-A sample, ~10 k single-end reads: the latency of one typing call
        loci, cont = build_database(args.scale)
        loci = loci[:1]
        paired = False
        n_reads = 10000
        sims = [{"sim": synth.ReadSimulator(l), "names": sorted(n for n in l.alleles if l.alleles[n])} for l in loci]
        rng = np.random.default_rng(101)
        truth = [sims[0]["names"][i] for i in rng.choice(len(sims[0]["names"]), 2, replace=False)]
        steps_units = [[(0, sims[0]["sim"].generate(truth, n_reads, seed=101, err_rate=ERR, read_len=READ_LEN,
                                                    frag_len=FRAG_LEN, paired=False, prefix="q"))]]
        scaling = "weak"  # every rank types its own copy of the sample (replicas)
        desc = ("BASELINE configs[0]: HLA-A (A=%d alleles), one sample of %d single-end 100 bp reads per step, error rate %.3f"
                % (len(sims[0]["names"]), n_reads, ERR))
        discordant = True
    else:
        if wl == "panel":  # configs[2]
            loci, cont = build_panel(args.scale)
            n_samples = args.samples if args.samples != 128 else 32
            desc = ("BASELINE configs[2]: panel of %d loci, %d alleles in total, %d samples paired-end 2x100 30x; the (sample, "
                    "locus) units are packed onto the ranks longest-first by reads x words per allele set"
                    % (len(loci), sum(len(l.alleles) for l in loci), n_samples))
        else:  # batch1000, configs[4]
            loci, cont = build_database(args.scale)
            n_samples = args.batch_samples
            desc = ("BASELINE configs[4]: batch of %d samples x 6 loci (database of configs[1]), samples sharded over the ranks, "
                    "%d samples per step" % (n_samples, args.samples))
        sims = [{"sim": synth.ReadSimulator(l), "names": sorted(n for n in l.alleles if l.alleles[n])} for l in loci]
        discordant = False
        if wl == "panel":
            units = simulate_units(loci, sims, n_samples, 0)  # every rank simulates all, keeps its share
            wps = [_lib.row_pitch(len(l.alleles)) for l in loci]
            costs = [float(t.count(b"\n")) * wps[li] for li, t in units]
            bins, loads = lpt_pack(costs, world)
            mine = bins[rank]
            steps_units = [[units[u] for u in sorted(mine)]]
            extra["lpt"] = {"units": len(units), "units_rank0": len(bins[0]), "load_max_over_mean": max(loads) / (sum(loads) / world)}
            del units
        else:
            per_rank = (n_samples + world - 1) // world
            s0, s1 = rank * per_rank, min(n_samples, (rank + 1) * per_rank)
            steps_units = []
            for a in range(s0, s1, args.samples):
                steps_units.append(simulate_units(loci, sims, min(args.samples, s1 - a), a))
    tables = [LocusTables(*locus_args(cont, l.gene), device=local) for l in loci]
    host_threads = max(1, (os.cpu_count() or 1) // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", world))))
    params = TC.make_params(allow_discordant=discordant, n_threads=host_threads)
    stream = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    pinned = _lib.PinnedText(sum(len(t) + 16 for su in steps_units for _, t in su) + 16)
    step_ptrs = [[(li,) + pinned.add(text) for li, text in su] for su in steps_units]
    text_bytes = sum(len(t) for su in steps_units for _, t in su)
    first_units = steps_units[0][:args.cpu_baseline_units]
    steps_units = None
    gc.collect()
    gc.freeze()
    # ---- value: every step's text resident in HBM -> ranked alleles; K passes over the rank's whole share ------------------
    batches = []
    reads_rank = pairs_rank = 0
    for ptrs in step_ptrs:
        b = TC.Batch(tables, params, True, device=local)
        b.add_units_ptr(ptrs)
        b.prepare()
        b.execute(stream)
        b.finish(stream)
        t = b.totals()
        reads_rank += t["num_reads"]
        pairs_rank += t["num_pairs"]
        batches.append(b)
        if len(batches) * 4 > 24:  # bound the resident memory of a long job: keep at most six prepared batches
            break
    n_res = len(batches)
    reads_res = sum(b.totals()["num_reads"] for b in batches)
    L.hgt_profile_enable(ctx, 1)
    sampler = ClockSampler(local)
    sampler.wait_first()
    for _ in range(args.warmup):
        for b in batches:
            b.execute(stream)
            b.finish(stream)
    L.hgt_profile_reset(ctx)
    launches0 = L.hgt_launch_count(ctx)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    with sampler as clocks:
        for k in range(args.steps):
            flush.zero_()
            ev[k][0].record()
            for b in batches:
                b.execute(stream)
                b.finish(stream)
            ev[k][1].record()
        barrier()
    pass_ms = [a.elapsed_time(b) for a, b in ev]
    launches = L.hgt_launch_count(ctx) - launches0
    stage_ms, stage_n = ctypes_array(8, "d"), ctypes_array(8, "q")
    h2d, d2h = ctypes.c_int64(0), ctypes.c_int64(0)
    L.hgt_profile_read(ctx, stage_ms, stage_n, ctypes.byref(h2d), ctypes.byref(d2h))
    stage = {n: stage_ms[i] / args.steps for i, n in enumerate(STAGES)}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, batches)
    example = batches[0].top_calls(2)[0]
    parity_batch = batches[0]
    for b in batches[1:]:
        b.close()
    # ---- e2e: the rank's whole share as a stream of batches from page-locked host text ------------------------------------
    depth = args.pipeline_depth
    pipe = TC.BatchPipeline(tables, params, True, device=local, depth=depth)
    reps = max(1, (2 * depth + len(step_ptrs) - 1) // len(step_ptrs)) if wl != "batch1000" else 1
    for _ in pipe.map(step_ptrs[:depth] * (1 if len(step_ptrs) >= depth else depth), lambda bt: bt.top_calls(2)):
        pass
    for c in pipe.contexts():
        L.hgt_profile_reset(c)
    barrier()
    t0 = time.perf_counter()
    n_done = 0
    for _ in pipe.map(step_ptrs * reps, lambda bt: bt.top_calls(2)):
        n_done += 1
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / reps  # one pass over the rank's share
    pipe_h2d = pipe_d2h = 0
    for c in pipe.contexts():
        L.hgt_profile_read(c, stage_ms, stage_n, ctypes.byref(h2d), ctypes.byref(d2h))
        pipe_h2d += h2d.value
        pipe_d2h += d2h.value
    pipe.close()
    # latency of ONE batch alone (matters for configs[0]): prepare + execute + finish + calls, nothing else in flight
    lat = []
    for k in range(3):
        barrier()
        t1 = time.perf_counter()
        bt = TC.Batch(tables, params, True, device=local)
        bt.add_units_ptr(step_ptrs[0])
        bt.run()
        bt.top_calls(2)
        lat.append((time.perf_counter() - t1) * 1000.0)
        bt.close()
    # ---- reduce over ranks --------------------------------------------------------------------------------------------------
    dev_pass_s = (sum(pass_ms) / len(pass_ms)) / 1000.0 * (len(step_ptrs) / float(n_res))  # extrapolated to the whole share
    vec = torch.tensor([dev_pass_s, e2e_s, float(reads_rank if n_res == len(step_ptrs) else reads_res * len(step_ptrs) / n_res)],
                       dtype=torch.float64, device="cuda")
    if world > 1:
        mx = vec.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = vec.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        dev_s, e2e_all_s, reads_all = float(mx[0]), float(mx[1]), float(sm[2])
    else:
        dev_s, e2e_all_s, reads_all = float(vec[0]), float(vec[1]), float(vec[2])
    parity_failed = False
    if rank == 0:
        line = {
            "metric": "reads typed/sec", "value": reads_all / dev_s, "unit": "reads/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_s * 1000.0, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "u64 bitsets + f64 EM", "data": "synthetic",
            "config": {"workload": desc, "loci": [l.gene for l in loci], "coverage": COVERAGE if paired else None,
                       "read_len": READ_LEN, "error_rate": ERR, "paired": paired, "batches_per_pass_rank0": len(step_ptrs),
                       "l2": "a 512 MiB buffer is rewritten between timed passes"},
            "step": "one pass over the rank's share of the job (%d batch(es) on rank 0)" % len(step_ptrs),
            "reads_per_step": reads_all, "stage_ms_per_step_rank0": stage, "step_ms_rank0": [round(x, 3) for x in pass_ms],
            "e2e": {"value": reads_all / e2e_all_s, "unit": "reads/s", "ms_per_step": e2e_all_s * 1000.0,
                    "h2d_bytes_per_step": pipe_h2d / reps, "d2h_bytes_per_step": pipe_d2h / reps,
                    "input": "page-locked host alignment text, %d bytes on rank 0" % text_bytes,
                    "how": "typing_core.BatchPipeline, %d batches in flight, wall clock between device synchronisations, max "
                           "over ranks" % depth,
                    "single_batch_latency_ms_rank0": sorted(lat)[len(lat) // 2]},
            "gpu_launches": int(launches), "clocks": clocks.summary(), "example_call": example,
        }
        line.update(extra)
        if not args.no_cpu_baseline and world == 1:
            build_oracle_loci(cont, loci)
            ORACLE_DISCORDANT[0] = discordant
            line["cpu_baseline"], line["parity_checked"] = cpu_baseline(first_units, parity_batch)
            if line["parity_checked"] and not line["parity_checked"]["identical"]:
                sys.stderr.write("bench: GPU results differ from the oracle: %s\n" % line["parity_checked"]["first_difference"])
                parity_failed = True
        print(json.dumps(line))
    parity_batch.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 1 if parity_failed else 0

# ------------------------------------------------------------------------------------------------------------
def oversized_subrecord(args, rank, world):
    """BASELINE configs[3] (one oversized locus, reads sharded over the ranks, strong scaling) as a sub-record of the default
    line, so that `bench.py --gpus N` also reports the one workload with a data-path exchange (class-table merge + the
    peer-memory EM).  Every rank starts `bench.py --workload oversized` as a CHILD process with its own rendezvous port and
    a time limit: a failure there can cost the sub-record, never the main line."""
    import subprocess
    if args.oversized_sub_reads <= 0:
        return None
    env = {k: v for k, v in os.environ.items() if not k.startswith("TORCHELASTIC_")}  # (rank 0 of the children hosts their store)
    if world > 1:
        env["MASTER_PORT"] = str(int(os.environ.get("MASTER_PORT", "29500")) + 1)
    env["HGT_BENCH_NO_SMI"] = "1"
    cmd = [sys.executable, os.path.abspath(__file__), "--workload", "oversized", "--gpus", str(world), "--steps", "3", "--warmup", "3",
           "--no-cpu-baseline", "--oversized-reads", str(args.oversized_sub_reads)]
    t0 = time.perf_counter()
    try:
        out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=420)
    except subprocess.TimeoutExpired:
        return {"error": "timed out after 420 s"} if rank == 0 else None
    if rank != 0:
        return None
    rec = None
    for ln in out.stdout.splitlines():
        if ln.startswith("{"):
            try:
                rec = json.loads(ln)
            except ValueError:
                pass
    if rec is None:
        return {"error": "no line (exit %d): %s" % (out.returncode, out.stderr.strip().splitlines()[-1:] or "")}
    keep = ("metric", "value", "unit", "n_gpus", "ms_per_step", "scaling", "reads_per_step", "classes_rank0", "em_iters_rank0",
            "sharded_em_wall_ms_rank0", "stage_ms_per_step_rank0", "step_ms_rank0", "example_call")
    sub = {k: rec[k] for k in keep if k in rec}
    sub["workload"] = rec["config"]["workload"]
    sub["e2e"] = {k: rec["e2e"][k] for k in ("value", "unit", "ms_per_step") if k in rec.get("e2e", {})}
    sub["wall_s"] = round(time.perf_counter() - t0, 1)
    return sub


DUMP_LIMIT = 64 << 20  # bytes of all arrays --dump-outputs writes
DUMP_UNITS = 64  # units whose per-allele and per-class arrays are written (a seeded sample when the step has more)
DUMP_TOP = 5  # calls per unit in top_calls.npy


def dump_outputs(out_dir, batches):
    """--dump-outputs: what the timed path computed in its last step (the prepared batches after execute + finish), as
    float64 arrays out_dir/<name>.npy, so that two builds can be compared output for output on the same seeded inputs.
    Units are numbered in batch order.  For every unit:
      unit_summary   [U, 10]     reads, pairs, classes of the 4 tables, EM iterations (2 levels), EM status (2 levels)
      top_calls      [U, 5, 2]   allele index and abundance of the 5 best calls; -1 and 0 where the unit has fewer
    For a fixed sample of at most DUMP_UNITS units (sample_units: their numbers, ascending):
      abundance      [sum A]     Gene_prob of every allele of the unit's locus, 0 where the allele has none
      allele_counts  [sum A, 4]  Gene_counts of each table
      classes        [sum C, 4]  per class, table after table: read pairs, member alleles, first pair, and a 48-bit
                                 BLAKE2b hash of its member bitset (the packed words would exceed the size budget)"""
    import hashlib

    import numpy as np
    units = [(b, u) for b in batches for u in range(len(b.unit_locus))]
    index = {}

    def allele_index(t):
        if id(t) not in index:
            index[id(t)] = {n: i for i, n in enumerate(t.names)}
        return index[id(t)]

    summary = np.zeros((len(units), 10))
    top = np.zeros((len(units), DUMP_TOP, 2))
    top[:, :, 0] = -1
    k = 0
    for b in batches:
        for u, calls in enumerate(b.top_calls(DUMP_TOP)):
            s = b.unit_summary(u)
            summary[k] = [s["num_reads"], s["num_pairs"]] + s["n_classes"] + s["em_iters"] + s["em_status"]
            names = allele_index(b.loci[b.unit_locus[u]])
            for j, (allele, prob) in enumerate(calls):
                top[k, j] = names[allele], prob
            k += 1
    pick = np.sort(np.random.default_rng(0).choice(len(units), min(len(units), DUMP_UNITS), replace=False))
    abundance, counts, classes = [], [], []
    for k in pick:
        b, u = units[k]
        t = b.loci[b.unit_locus[u]]
        names = allele_index(t)
        prob = np.zeros(t.A)
        for allele, p in b.unit_calls(u):
            prob[names[allele]] = p
        abundance.append(prob)
        cnt = np.zeros((t.A, 4))
        for tb in range(4):
            bits, n_pairs, first, acount, _ = b.unit_table(u, tb)
            cnt[:, tb] = acount
            members = [int.from_bytes(hashlib.blake2b(row.tobytes(), digest_size=6).digest(), "little") for row in bits]
            classes.append(np.stack([n_pairs, np.bitwise_count(bits).sum(axis=1), first, np.asarray(members, np.float64)],
                                    axis=1))
        counts.append(cnt)
    out = {"unit_summary": summary, "top_calls": top, "sample_units": pick, "abundance": np.concatenate(abundance),
           "allele_counts": np.concatenate(counts), "classes": np.concatenate(classes)}
    out = {n: np.ascontiguousarray(a, np.float64) for n, a in out.items()}
    size = sum(a.nbytes for a in out.values())
    if size > DUMP_LIMIT:
        raise SystemExit("bench: --dump-outputs would write %d bytes, more than %d" % (size, DUMP_LIMIT))
    os.makedirs(out_dir, exist_ok=True)
    for n, a in out.items():
        np.save(os.path.join(out_dir, n + ".npy"), a)
    sys.stderr.write("bench: %d arrays, %d bytes, in %s\n" % (len(out), size, out_dir))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--samples", type=int, default=128, help="samples per step and GPU")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the database (tests only)")
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--ref-samples", type=int, default=4)
    ap.add_argument("--cpu-baseline-units", type=int, default=6)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="six-loci", choices=["six-loci", "oversized", "single-locus", "panel", "batch1000"])
    ap.add_argument("--batch-samples", type=int, default=1000, help="samples of the batch1000 workload (all ranks together)")
    ap.add_argument("--oversized-reads", type=int, default=1000000)
    ap.add_argument("--pipeline-depth", type=int, default=3, help="batches in flight in the end-to-end measurement")
    ap.add_argument("--oversized-sub-reads", type=int, default=10000000,
                    help="reads of the read-sharded oversized locus reported as the `oversized` sub-record of the default "
                         "line (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0's units) as DIR/<name>.npy; "
                         "the oversized workload on one GPU only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path, not of --impl reference")
    if args.impl == "reference":
        return run_reference_arm(args)
    if args.workload == "oversized":
        return run_oversized(args)
    if args.workload in ("single-locus", "panel", "batch1000"):
        return run_workload(args)

    import numpy as np
    import torch
    import _hgt_path
    _hgt_path.load()
    from hisatgenotype_b200 import _lib, synth
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.locus import LocusTables

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    os.environ["HGT_DEVICE"] = str(local)
    ctx = _lib.ctx(local)
    L = _lib.lib()

    loci, cont = build_database(args.scale)
    tables = [LocusTables(*locus_args(cont, l.gene), device=local) for l in loci]
    sims = [{"sim": synth.ReadSimulator(l), "names": sorted(n for n in l.alleles if l.alleles[n])} for l in loci]
    S = args.samples
    units = simulate_units(loci, sims, S, rank * S)  # loci/sample sharding: no communication (SURVEY.md 8e)
    # host threads of the intake / walk stages: the ranks of one box share its cores
    host_threads = max(1, (os.cpu_count() or 1) // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", world))))
    params = TC.make_params(n_threads=host_threads)
    stream = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # the step's input: every unit's alignment text in ONE page-locked host allocation (the e2e copies start there)
    pinned = _lib.PinnedText(sum(len(t) + 16 for _, t in units))
    unit_ptrs = [(li,) + pinned.add(text) for li, text in units]

    # ---- value: alignment text already resident in HBM -> ranked alleles ------------------------------------------------
    batch = TC.Batch(tables, params, True, device=local)
    for li, addr, n in unit_ptrs:
        batch.add_unit_ptr(li, addr, n)
    batch.prepare()
    batch.execute(stream)
    batch.finish(stream)
    tot = batch.totals()
    L.hgt_profile_enable(ctx, 1)
    # the database and the alignment text are millions of long-lived Python objects: park them in the permanent
    # generation so that a full collection (tens of ms) cannot fire inside a timed step
    import gc
    gc.collect()
    gc.freeze()
    sampler = ClockSampler(local)
    sampler.wait_first()
    for _ in range(args.warmup):
        batch.execute(stream)
        batch.finish(stream)
    L.hgt_profile_reset(ctx)
    launches0 = L.hgt_launch_count(ctx)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    with sampler as clocks:
        for k in range(args.steps):
            flush.zero_()
            ev[k][0].record()
            batch.execute(stream)
            batch.finish(stream)
            ev[k][1].record()
        barrier()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    dev_ms = float(sum(step_ms))
    em_trace_once(L, ctx, lambda: (batch.execute(stream), batch.finish(stream)))
    launches = L.hgt_launch_count(ctx) - launches0
    stage_ms = (ctypes_array(8, "d"))
    stage_n = (ctypes_array(8, "q"))
    import ctypes
    h2d, d2h = ctypes.c_int64(0), ctypes.c_int64(0)
    L.hgt_profile_read(ctx, stage_ms, stage_n, ctypes.byref(h2d), ctypes.byref(d2h))
    stage = {n: stage_ms[i] / args.steps for i, n in enumerate(STAGES)}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, [batch])
    # EM bookkeeping
    # SURVEY.md 8d: per loop iteration min(bit matrix, CSR) evaluated on the actual class tables:
    #   bit matrix 3 C (wp 8 + 8) + 6 A 8,   CSR 3 (4 nnz + 12 C) + 6 A 8   (nnz = members over all classes)
    em_iters = em_bytes = em_bytes_bitset = em_bytes_csr = 0
    for u in range(len(units)):
        s = batch.unit_summary(u)
        t = tables[batch.unit_locus[u]]
        for lvl, tb in ((0, 1), (1, 3)):
            it, C = s["em_iters"][lvl], s["n_classes"][tb]
            if it <= 0:
                continue
            nnz = int(np.bitwise_count(batch.unit_table(u, tb)[0]).sum())
            b_bits = 3 * C * (t.wp * 8 + 8) + 6 * t.A * 8
            b_csr = 3 * (4 * nnz + 12 * C) + 6 * t.A * 8
            em_iters += it
            em_bytes_bitset += it * b_bits
            em_bytes_csr += it * b_csr
            em_bytes += it * min(b_bits, b_csr)
    t_vec = torch.tensor([dev_ms, float(tot["num_reads"]), float(em_iters)], dtype=torch.float64, device="cuda")
    if world > 1:
        mx = t_vec.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = t_vec.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        dev_ms_all, reads_all, iters_all = float(mx[0]), float(sm[1]), float(sm[2])
    else:
        dev_ms_all, reads_all, iters_all = dev_ms, float(tot["num_reads"]), float(em_iters)
    ms_per_step = dev_ms_all / args.steps
    value = reads_all / (ms_per_step / 1000.0)

    # ---- e2e: host alignment text in, ranked alleles out ---------------------------------------------------------
    L.hgt_profile_reset(ctx)
    e2e_ms = []
    n_e2e = max(2, min(args.steps, 3))
    wall = {"add_units": 0.0, "prepare": 0.0, "execute": 0.0, "finish": 0.0, "results": 0.0}
    for k in range(1 + n_e2e):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if k == 1:
            L.hgt_profile_reset(ctx)
            wall = {n: 0.0 for n in wall}
        a.record()
        t0 = time.perf_counter()
        bt = TC.Batch(tables, params, True, device=local)
        for li, addr, n in unit_ptrs:
            bt.add_unit_ptr(li, addr, n)
        t1 = time.perf_counter()
        bt.prepare()
        t2 = time.perf_counter()
        bt.execute(stream)
        t3 = time.perf_counter()
        bt.finish(stream)
        t4 = time.perf_counter()
        calls = bt.top_calls(2)
        t5 = time.perf_counter()
        b.record()
        torch.cuda.synchronize()
        for n, dt in zip(("add_units", "prepare", "execute", "finish", "results"), (t1 - t0, t2 - t1, t3 - t2, t4 - t3, t5 - t4)):
            wall[n] += dt * 1000.0
        if k >= 1:
            e2e_ms.append(a.elapsed_time(b))
        bt.close()
    host_ms = ctypes_array(8, "d")
    L.hgt_profile_host(ctx, host_ms)
    e2e_host = {n: host_ms[i] / n_e2e for i, n in enumerate(HOST_STAGES) if n}
    e2e_wall = {n: v / n_e2e for n, v in wall.items()}
    L.hgt_profile_read(ctx, stage_ms, stage_n, ctypes.byref(h2d), ctypes.byref(d2h))
    serial_h2d, serial_d2h = h2d.value / n_e2e, d2h.value / n_e2e
    serial_ms = sum(e2e_ms) / len(e2e_ms)
    # the same steps as a STREAM of batches (typing_core.BatchPipeline): `depth` host threads, each with its own context
    # and CUDA stream, so the copy of step k+1 overlaps the kernels of step k.  Timed by the wall clock between two device
    # synchronisations (several streams are in flight; an event on one stream would not see the others).
    depth = args.pipeline_depth
    pipe = TC.BatchPipeline(tables, params, True, device=local, depth=depth)
    n_pipe = max(4 * depth, args.steps)
    calls = None
    for _ in pipe.map([unit_ptrs] * depth, lambda bt: bt.top_calls(2)):  # warm-up: every lane's pool and context
        pass
    for c in pipe.contexts():
        L.hgt_profile_reset(c)
    barrier()
    if os.environ.get("HGT_PIPE_TRACE"):
        pipe.trace = []
    t0 = time.perf_counter()
    for calls in pipe.map([unit_ptrs] * n_pipe, lambda bt: bt.top_calls(2)):
        pass
    torch.cuda.synchronize()
    pipe_ms = (time.perf_counter() - t0) * 1000.0 / n_pipe
    if pipe.trace:
        for t in sorted(pipe.trace):
            sys.stderr.write("pipe_trace start %7.2f prepared %7.2f executed %7.2f finished %7.2f results %7.2f ms\n"
                             % tuple((x - t0) * 1000.0 for x in t))
    pipe_h2d = pipe_d2h = 0
    for c in pipe.contexts():
        L.hgt_profile_read(c, stage_ms, stage_n, ctypes.byref(h2d), ctypes.byref(d2h))
        pipe_h2d += h2d.value
        pipe_d2h += d2h.value
    pipe.close()
    e2e_vec = torch.tensor([pipe_ms, serial_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_vec, op=dist.ReduceOp.MAX)
    e2e_value = reads_all / (float(e2e_vec[0]) / 1000.0)
    e2e_serial_value = reads_all / (float(e2e_vec[1]) / 1000.0)

    parity_failed = False
    text_bytes_step = sum(len(t) for _, t in units)
    barrier()
    over = oversized_subrecord(args, rank, world)  # (child processes; every rank takes part)
    barrier()
    if rank == 0:
        peak, peak_src = measured_peak()
        a_ms = stage["compat"] + stage["class"]
        a_bytes = float(tot["algorithmic_bytes"])
        achieved = a_bytes / (a_ms / 1000.0) / 1e9 if a_ms > 0 else None
        em_ms = stage["em1"] + stage["em2"]
        em_achieved = em_bytes / (em_ms / 1000.0) / 1e9 if em_ms > 0 else None
        line = {
            "metric": "reads typed/sec", "value": value, "unit": "reads/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64 bitsets + f64 EM", "data": "synthetic",
            "config": workload_config(args, S),
            "reads_per_step": reads_all, "pairs_per_step_rank0": tot["num_pairs"],
            "haplotypes_per_step_rank0": tot["n_haplotypes"], "variant_rows_per_step_rank0": tot["n_rows"],
            "em_iters_per_sec": iters_all / (ms_per_step / 1000.0) if ms_per_step else None,
            "em_iters_per_step": iters_all,
            "em_iters_per_sec_kernel_time": em_iters / (em_ms / 1000.0) if em_ms > 0 else None,
            "stage_ms_per_step_rank0": stage, "step_ms_rank0": [round(x, 3) for x in step_ms],
            # dominant kernel by GPU time: the batched EM (two launches per step: first level on the exon tables, second
            # level on the projected tables).  Its problems are shared-memory resident, so DRAM traffic is far below the
            # algorithmic bytes and the HBM fraction is a distance-to-roofline figure, not a saturation claim.
            "roofline": {"bound": "hbm", "achieved": em_achieved, "peak": peak, "unit": "GB/s",
                         "frac": em_achieved / peak if em_achieved else None,
                         "traffic": ncu_traffic("em_kernel", "six-loci", S),
                         # the problems live in shared memory: distance to the on-chip ceilings from the same ncu capture
                         "on_chip": ncu_traffic("em_kernel", "six-loci", S, per="on_chip"),
                         "kernel": "em_kernel (batched, one CTA per (sample, locus) problem)", "peak_source": peak_src,
                         "algorithmic_bytes_rule": "per problem and iteration min(bit matrix, CSR), SURVEY.md 8d",
                         "algorithmic_bytes_per_step_bit_matrix": float(em_bytes_bitset),
                         "algorithmic_bytes_per_step_csr": float(em_bytes_csr),
                         "launches_per_step": 2, "algorithmic_bytes_per_launch": float(em_bytes) / 2.0,
                         "avg_launch_ms": em_ms / 2.0, "algorithmic_bytes_per_step": float(em_bytes),
                         "kernel_ms_per_step": em_ms, "share_of_step": em_ms / ms_per_step if ms_per_step else None},
            "roofline_stage_a": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                                 "frac": achieved / peak if achieved else None,
                                 "traffic": ncu_traffic("stage_a", "six-loci", S, per="step"),
                                 "traffic_is": "DRAM bytes of all stage (a) launches of one step (like the algorithmic figure)",
                                 "kernel": "set stage: compat_kernel + class_kernel (+ class_sort_kernel), one launch each per locus",
                                 "algorithmic_bytes_per_step": a_bytes, "kernel_ms_per_step": a_ms,
                                 "share_of_step": a_ms / ms_per_step if ms_per_step else None},
            # the record stage (line index, parse, pileup, mate de-dup, walk, ambiguity passes, pair jobs) has to read the
            # alignment text: its algorithmic bytes are the text bytes of the step
            "roofline_records": {"bound": "hbm", "achieved": text_bytes_step / ((stage["records"] + stage["walk"]) / 1000.0) / 1e9,
                                 "peak": peak, "unit": "GB/s",
                                 "frac": text_bytes_step / ((stage["records"] + stage["walk"]) / 1000.0) / 1e9 / peak,
                                 "traffic": ncu_traffic("records", "six-loci", S, per="step"),
                                 "kernel": "record stage: index_lines, parse, pileup_text, head / candidate, walk (three passes), "
                                           "pair count / scans / fill",
                                 "algorithmic_bytes_per_step": float(text_bytes_step),
                                 "kernel_ms_per_step": stage["records"] + stage["walk"],
                                 "share_of_step": (stage["records"] + stage["walk"]) / ms_per_step if ms_per_step else None},
            "e2e": {"value": e2e_value, "unit": "reads/s", "h2d_bytes_per_step": pipe_h2d / n_pipe,
                    "d2h_bytes_per_step": pipe_d2h / n_pipe, "ms_per_step": float(e2e_vec[0]),
                    "input": "page-locked host alignment text, %d bytes per step on rank 0" % sum(len(t) for _, t in units),
                    "how": "typing_core.BatchPipeline: %d steps as a stream of batches, %d in flight (one host thread, library "
                           "context and CUDA stream each); every step copies its text host->device and reads its ranked "
                           "calls back; wall clock between device synchronisations, max over ranks" % (n_pipe, depth),
                    "steps": n_pipe, "in_flight": depth,
                    "serial": {"value": e2e_serial_value, "ms_per_step": float(e2e_vec[1]), "h2d_bytes_per_step": serial_h2d,
                               "d2h_bytes_per_step": serial_d2h, "wall_ms_rank0": e2e_wall, "host_stage_ms_rank0": e2e_host,
                               "how": "one batch at a time: prepare, execute, finish, results, on one stream"},
                    "host_threads": host_threads, "host_cores": os.cpu_count()},
            "gpu_launches": int(launches),
            "clocks": clocks.summary(),
            "example_call": calls[0],
        }
        if over is not None:
            line["oversized"] = over
        if not args.no_cpu_baseline and world == 1:  # the CPU baseline is timed on rank 0 at N = 1 only
            build_oracle_loci(cont, loci)
            line["cpu_baseline"], line["parity_checked"] = cpu_baseline(units[:args.cpu_baseline_units], batch)
        print(json.dumps(line))
        if line.get("parity_checked") and not line["parity_checked"]["identical"]:
            sys.stderr.write("bench: GPU results differ from the oracle: %s\n" % line["parity_checked"]["first_difference"])
            parity_failed = True
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 1 if parity_failed else 0


def ncu_traffic(kernel, workload, samples, per="launch"):
    """DRAM bytes (read + write) per launch - or per step - of `kernel` from the committed `ncu --set full` capture of this
    workload (profiles/traffic.json, written from the .ncu-rep by tools/ncu_traffic.py); None when no capture matches."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        e = t["%s:%s:%d" % (workload, kernel, samples)]
        if per == "on_chip":
            return e.get("on_chip")
        if per == "step":
            return e.get("dram_bytes_per_step", e["dram_bytes_per_launch"] * e["launches_captured"])
        return e["dram_bytes_per_launch"]
    except (OSError, KeyError, ValueError):
        return None


def em_trace_once(L, ctx, run):
    """HGT_EM_TRACE=1: one extra untimed step with the EM kernels' phase tracing on (hgt_em_trace); cycles of CTA 0 of
    every em_kernel launch go to stderr."""
    import ctypes
    if not os.environ.get("HGT_EM_TRACE"):
        return
    L.hgt_em_trace.restype = ctypes.c_int
    L.hgt_em_trace.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p]
    L.hgt_em_trace(ctx, 1, None)
    run()
    out = (ctypes.c_uint64 * 16)()
    L.hgt_em_trace(ctx, 0, out)
    names = ["stage_p", "phase1_sk", "phase2_acc", "coop_reduce", "normalise", "setup", "squarem_diff_prune", "compact64",
             "kernel_total", "sweeps", "launches", "all_cta_ns_sum", "all_cta_ns_max", "all_ctas",
             "dedup_signatures|coop_partials_sync1", "dedup_table|coop_slice_exchange"]
    sys.stderr.write("em_trace " + json.dumps({n: int(out[i]) for i, n in enumerate(names)}) + "\n")


def ctypes_array(n, code):
    import ctypes
    return ((ctypes.c_double if code == "d" else ctypes.c_int64) * n)()


if __name__ == "__main__":
    sys.exit(main())

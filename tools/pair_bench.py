"""Batched diploid pair calls (Batch.pair_calls -> hgt_batch_pairs, csrc/pair_batch.cu) on one BASELINE configs[1] step
(128 samples x HLA-A/B/C/DQA1/DQB1/DRB1, paired-end 2x100 bp, 30x, the seeded synthetic database and reads of bench.py).
The step is typed once (prepare / execute / finish); then, per table (0 = Gene, 1 = exon):
  - the wall time of Batch.pair_arrays (one library call for every unit, ending in its synchronisation), after warm-up
    calls, as min / median over --reps calls; every timed call has its own max_pairs (all far above any unit's pair
    count), so none is answered from the result the library keeps for a repeated call - that re-read is timed apart;
  - the distribution over units of the pairs after the first pruning (what a unit's loop works on), of the pairs in the
    result (p > 0) and of the loop iterations;
  - host typing_common.joint_abundance(unit_gene_cmpt(u, table)) on the first --host-units units, per unit, timed, and
    compared with the batch result (same keys in the same order, p within 1e-9 relative, same iterations).
Exit status 1 on any difference.  Prints one JSON line (GPU name and power limit included) and writes it to --out.

usage: python tools/pair_bench.py [--samples 128] [--reps 5] [--host-units 24] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    first = (r.stdout.strip().splitlines() or [""])[0]
    parts = [x.strip() for x in first.split(",")]
    return {"gpu": parts[0] if parts else "", "power_limit": parts[1] if len(parts) > 1 else ""}


def same(got, ref):
    if isinstance(ref, dict) or isinstance(got, dict):
        return got == ref
    if [k for k, _ in got] != [k for k, _ in ref]:
        return False
    return all(abs(x - y) <= 1e-9 * max(abs(y), 1e-300) for (_, x), (_, y) in zip(got, ref))


def dist(v):
    import numpy as np
    v = np.asarray(v, np.float64)
    if v.size == 0:
        return {}
    return {"min": float(v.min()), "p50": float(np.percentile(v, 50)), "p90": float(np.percentile(v, 90)),
            "max": float(v.max()), "mean": float(v.mean())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=128)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--host-units", type=int, default=24)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import numpy as np

    import bench
    import _hgt_path
    _hgt_path.load()
    from hisatgenotype_b200 import synth
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.locus import LocusTables
    from hisatgenotype_b200.typing_common import MAX_PAIRS, joint_abundance

    info = gpu_info()
    loci, cont = bench.build_database(1.0)
    tables = [LocusTables(*bench.locus_args(cont, l.gene)) for l in loci]
    sims = [{"sim": synth.ReadSimulator(l), "names": sorted(n for n in l.alleles if l.alleles[n])} for l in loci]
    units = bench.simulate_units(loci, sims, args.samples, 0)
    b = TC.Batch(tables, TC.make_params(), True)
    for li, text in units:
        b.add_unit(li, text)
    b.run()
    nu = len(units)
    out = dict(info, samples=args.samples, units=nu, loci=[l.gene for l in loci],
               alleles=[t.A for t in tables], reps=args.reps)
    ok = True
    for table in (0, 1):
        key = "table%d" % table
        b.pair_arrays(table, max_pairs=MAX_PAIRS - 1)  # warm-up (module load, names to the device)
        times = []
        for i in range(args.reps):
            t0 = time.perf_counter()
            r = b.pair_arrays(table, max_pairs=MAX_PAIRS - 2 - i)
            times.append((time.perf_counter() - t0) * 1e3)
        t0 = time.perf_counter()
        b.pair_arrays(table, max_pairs=MAX_PAIRS - 1 - args.reps)  # the kept result, read again
        kept_ms = (time.perf_counter() - t0) * 1e3
        r = b.pair_arrays(table)
        again = b.pair_arrays(table, max_pairs=MAX_PAIRS - 2 - args.reps)
        repeat_equal = all(np.array_equal(r[k], again[k]) for k in ("lo", "hi", "prob", "n_total", "iters", "status"))
        ok &= repeat_equal
        b._pairs = {(table, r["max_pairs"]): r}
        host_ms, mism = [], []
        for u in range(min(args.host_units, nu)):
            cm = b.unit_gene_cmpt(u, table)
            t0 = time.perf_counter()
            ref, it = joint_abundance(cm, return_iters=True)
            host_ms.append((time.perf_counter() - t0) * 1e3)
            got, git = b.unit_pair_calls(u, table, return_iters=True)
            if not same(got, ref) or git != it:
                mism.append(u)
        ok &= not mism
        out[key] = {"pair_calls_ms_min": min(times), "pair_calls_ms_p50": float(np.median(times)), "kept_result_ms": kept_ms,
                    "pairs_per_unit": dist(r["n_pairs"]), "survivors_per_unit": dist(r["n_total"]),
                    "iters_per_unit": dist(r["iters"]),
                    "pairs_x_iters_max": int((r["n_pairs"].astype(np.int64) * r["iters"]).max()),
                    "unsupported_units": int((r["status"] != 0).sum()),
                    "host_units": len(host_ms), "host_joint_abundance_ms_per_unit": dist(host_ms),
                    "host_joint_abundance_ms_sum": float(sum(host_ms)),
                    "parity": not mism, "mismatched_units": mism[:10], "repeat_bit_identical": repeat_equal}
    out["parity"] = bool(ok)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    b.close()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()

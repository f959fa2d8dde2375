"""Native BAM intake against the SAM intake on one GPU, for one BASELINE configs[1] step (128 samples x HLA-A/B/C/DQA1/DQB1/
DRB1, paired-end 2x100 bp, 30x, the seeded synthetic database and reads of bench.py), generated once as SAM text and as BAM
(one alignment file per sample).  Per step it times:
  - the host split of every sample: split_sam on the SAM text, split_bam on the BAM (BGZF inflate + record walk + sort +
    pack; inflate alone is reported too), with the host thread count;
  - prepare (copies + BAM render + line count, ending in a synchronise) for text / text without QUAL / BAM blobs / BAM blobs
    without QUAL, all from page-locked memory, with h2d_bytes from hgt_profile_read;
  - execute + finish.
  - BGZF inflate on the GPU (sam_intake.inflate_bgzf) from page-locked input to page-locked output, ending in a
    synchronise: the step's files in one call (bgzf_inflate_gpu_ms) and as one call per file, the shape typing() uses
    (bgzf_inflate_gpu_per_file_ms); the kernel alone from torch.profiler's device records (bgzf_inflate_kernel_ms); the
    compressed / inflated bytes and the call's h2d / d2h bytes; and split_bam fed from one-file inflate_bgzf calls
    (split_bam_gpu_inflate_ms, against split_bam_ms).
  - the device split (sam_intake.split_bam_device: inflate, record index, checks, bucketing and order on the GPU) of the
    step's files in one call from page-locked input, ending in its synchronisation (split_bam_device_ms), with the call's
    h2d / d2h bytes; and a bam_device variant of prepare / execute + finish whose units render from that split's HBM.
The calls of every variant must equal the text run's, and every file's GPU-inflated bytes read_bgzf's (exit status 1
otherwise).  Prints one JSON line (GPU name and power limit included) and writes it to --out when given.

usage: python tools/bam_intake_bench.py [--samples 128] [--steps 3] [--warmup 1] [--threads 0] [--out FILE]"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _encode_sample(job):
    from bam_writer import bam_stream, bgzf
    lines, refs = job
    return bgzf(bam_stream(lines, refs), 65280)


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    first = (r.stdout.strip().splitlines() or [""])[0]
    parts = [x.strip() for x in first.split(",")]
    return {"gpu": parts[0] if parts else "", "power_limit": parts[1] if len(parts) > 1 else ""}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=128)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--threads", type=int, default=0, help="host threads of the splits and BGZF inflate (0: all cores)")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import numpy as np
    import torch

    import bench
    import _hgt_path
    _hgt_path.load()
    from hisatgenotype_b200 import _lib, synth
    from hisatgenotype_b200 import typing_core as TC
    from hisatgenotype_b200.locus import LocusTables
    from hisatgenotype_b200.sam_intake import inflate_bgzf, read_bgzf, split_bam, split_bam_device, split_sam

    threads = args.threads or os.cpu_count() or 1
    info = gpu_info()
    loci, cont = bench.build_database(1.0)
    tables = [LocusTables(*bench.locus_args(cont, l.gene)) for l in loci]
    refs = [cont["refGenes"][l.gene] for l in loci]
    sims = [{"sim": synth.ReadSimulator(l), "names": sorted(n for n in l.alleles if l.alleles[n])} for l in loci]
    t0 = time.perf_counter()
    units = bench.simulate_units(loci, sims, args.samples, 0)
    per = len(loci)
    sams = [b"".join(t for _, t in units[s * per:(s + 1) * per]) for s in range(args.samples)]
    hdr = [(r, len(cont["Genes"][l.gene][r])) for r, l in zip(refs, loci)]
    from concurrent.futures import ProcessPoolExecutor
    with ProcessPoolExecutor(min(32, threads)) as pool:
        bams = list(pool.map(_encode_sample, [(s.decode().splitlines(), hdr) for s in sams], chunksize=1))
    gen_s = time.perf_counter() - t0
    n_records = sum(s.count(b"\n") for s in sams)

    L = _lib.lib()
    ctx = _lib.ctx()
    params = TC.make_params(n_threads=threads)

    def host_split(kind, drop_qual=False):
        out = []
        for s in range(args.samples):
            if kind == "sam":
                out.append(split_sam(sams[s], refs, threads, drop_qual=drop_qual))
            else:
                out.append(split_bam(bams[s], refs, threads, drop_qual=drop_qual))
        return out

    variants = {"text": ("sam", False), "text_noqual": ("sam", True), "bam": ("bam", False), "bam_noqual": ("bam", True)}
    pinned = {}
    for v, (kind, dq) in variants.items():
        parts = host_split(kind, dq)
        buf = _lib.PinnedText(sum(len(x) + 16 for p in parts for x in p.values()) + 16)
        pinned[v] = (buf, [[(li,) + buf.add(p[r]) for li, r in enumerate(refs)] for p in parts])

    def one_batch(v):
        b = TC.Batch(tables, params, True)
        if v == "bam_device":
            for s in range(args.samples):
                for li in range(len(refs)):
                    b.add_unit_bam_dsplit(li, dsplit.unit(s, li))
            return b
        kind = variants[v][0]
        for sample in pinned[v][1]:
            for li, addr, n in sample:
                if kind == "sam":
                    b.add_unit_ptr(li, addr, n)
                else:
                    b.add_unit_bam_ptr(li, addr, n)
        return b

    h2d = ctypes.c_int64(0)
    d2h = ctypes.c_int64(0)

    def run_step(v):
        b = one_batch(v)
        L.hgt_profile_reset(ctx)
        torch.cuda.synchronize()
        launches0 = L.hgt_launch_count(ctx)
        t = time.perf_counter()
        b.prepare()
        t_prep = time.perf_counter() - t
        prep_launches = L.hgt_launch_count(ctx) - launches0
        L.hgt_profile_read(ctx, None, None, ctypes.byref(h2d), ctypes.byref(d2h))
        prep_h2d = h2d.value
        t = time.perf_counter()
        b.execute()
        b.finish()
        torch.cuda.synchronize()
        t_exec = time.perf_counter() - t
        calls = b.top_calls(2)
        b.close()
        return t_prep, t_exec, prep_h2d, calls, prep_launches

    res = {"tool": "bam_intake_bench", **info, "samples": args.samples, "loci": len(loci), "records_per_step": n_records,
           "sam_bytes_per_step": sum(len(s) for s in sams), "bam_file_bytes_per_step": sum(len(b) for b in bams),
           "host_threads": threads, "steps": args.steps, "warmup": args.warmup, "generation_s": round(gen_s, 1),
           "variants": {}}
    # host splits (ms per step)
    for name, fn in (("split_sam_ms", lambda: host_split("sam")), ("split_bam_ms", lambda: host_split("bam")),
                     ("bgzf_inflate_ms", lambda: [read_bgzf(b, threads) for b in bams])):
        for _ in range(args.warmup):
            fn()
        ts = []
        for _ in range(args.steps):
            t = time.perf_counter()
            fn()
            ts.append((time.perf_counter() - t) * 1e3)
        res[name] = {"mean": round(float(np.mean(ts)), 2), "min": round(float(np.min(ts)), 2)}
    # BGZF inflate on the GPU: page-locked input, output into one reused page-locked arena
    inflated = [read_bgzf(b, threads) for b in bams]
    fin = _lib.PinnedText(sum(len(b) + 16 for b in bams) + 16)
    bams_pinned = [fin.view(*fin.add(b)) for b in bams]
    fout = _lib.PinnedText(sum(len(x) + 16 for x in inflated) + 16)

    def gpu_one_call():
        fout.reset()
        return inflate_bgzf(bams_pinned, pinned=fout)

    def gpu_per_file():
        fout.reset()
        return [inflate_bgzf([b], pinned=fout)[0] for b in bams_pinned]

    def split_gpu():
        fout.reset()
        return [split_bam(inflate_bgzf([b], pinned=fout)[0], refs, threads) for b in bams_pinned]

    inflate_ok = all(bytes(g) == w for g, w in zip(gpu_one_call(), inflated))
    inflate_ok = inflate_ok and all(bytes(g) == w for g, w in zip(gpu_per_file(), inflated))
    L.hgt_profile_reset(ctx)
    gpu_one_call()
    L.hgt_profile_read(ctx, None, None, ctypes.byref(h2d), ctypes.byref(d2h))
    res.update({"bgzf_compressed_bytes": sum(len(b) for b in bams), "bgzf_inflated_bytes": sum(len(x) for x in inflated),
                "bgzf_inflate_call_h2d_bytes": h2d.value, "bgzf_inflate_call_d2h_bytes": d2h.value})
    for name, fn in (("bgzf_inflate_gpu_ms", gpu_one_call), ("bgzf_inflate_gpu_per_file_ms", gpu_per_file),
                     ("split_bam_gpu_inflate_ms", split_gpu)):
        for _ in range(args.warmup):
            fn()
        ts = []
        for _ in range(args.steps):
            t = time.perf_counter()
            fn()
            ts.append((time.perf_counter() - t) * 1e3)
        res[name] = {"mean": round(float(np.mean(ts)), 2), "min": round(float(np.min(ts)), 2)}
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.steps):
            gpu_one_call()
    kern = [e for e in prof.key_averages() if "bgzf_inflate_kernel" in e.key]
    if kern:
        total_us = getattr(kern[0], "device_time_total", None) or getattr(kern[0], "cuda_time_total", 0)
        res["bgzf_inflate_kernel_ms"] = round(total_us / 1e3 / max(kern[0].count, 1), 3)
        res["bgzf_inflate_kernel_launches"] = kern[0].count
    else:
        res["bgzf_inflate_kernel_ms"] = None  # the profiler recorded no kernel of that name
    res["inflate_identical"] = inflate_ok
    # the device split: one call over the step's files, page-locked compressed input
    def dsplit_call():
        return split_bam_device(bams_pinned, refs)

    L.hgt_profile_reset(ctx)
    dsplit = dsplit_call()
    L.hgt_profile_read(ctx, None, None, ctypes.byref(h2d), ctypes.byref(d2h))
    res.update({"split_bam_device_h2d_bytes": h2d.value, "split_bam_device_d2h_bytes": d2h.value})
    for _ in range(args.warmup):
        dsplit_call().close()
    ts = []
    for _ in range(args.steps):
        t = time.perf_counter()
        sp = dsplit_call()
        ts.append((time.perf_counter() - t) * 1e3)
        sp.close()
    res["split_bam_device_ms"] = {"mean": round(float(np.mean(ts)), 2), "min": round(float(np.min(ts)), 2)}
    fin.close()
    fout.close()
    # prepare / execute + finish per variant, the variants alternating inside every step
    ref_calls = None
    ok = True
    run_variants = list(variants) + ["bam_device"]
    acc = {v: {"prepare_ms": [], "execute_finish_ms": [], "h2d_bytes": [], "launches": 0} for v in run_variants}
    for step in range(args.warmup + args.steps):
        for v in run_variants:
            t_prep, t_exec, hb, calls, acc[v]["launches"] = run_step(v)
            if v == "text":
                ref_calls = calls
            elif calls != ref_calls:
                ok = False
            if step >= args.warmup:
                acc[v]["prepare_ms"].append(t_prep * 1e3)
                acc[v]["execute_finish_ms"].append(t_exec * 1e3)
                acc[v]["h2d_bytes"].append(hb)
    for v, a in acc.items():
        res["variants"][v] = {"input_bytes": int(sum(n for s in pinned[v][1] for _, _, n in s)) if v in pinned else 0,
                              "prepare_ms": {"mean": round(float(np.mean(a["prepare_ms"])), 2),
                                             "min": round(float(np.min(a["prepare_ms"])), 2)},
                              "execute_finish_ms": {"mean": round(float(np.mean(a["execute_finish_ms"])), 2),
                                                    "min": round(float(np.min(a["execute_finish_ms"])), 2)},
                              "prepare_h2d_bytes": int(a["h2d_bytes"][-1]), "prepare_launches": int(a["launches"])}
    res["calls_identical"] = ok
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    dsplit.close()
    for buf, _ in pinned.values():
        buf.close()
    for t in tables:
        t.close()
    sys.exit(0 if ok and inflate_ok else 1)


if __name__ == "__main__":
    main()

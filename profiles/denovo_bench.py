"""Cost of the de novo adapter assembly (--adapter-denovo) on a B200.

1. k_end_kmers on the CLI's default sample: 2 x 100 000 rows x 150 bases at k = 12, split 69.  The 5' rows carry
   ADAPTER_LIB[8] with 10 % errors after a 0-30-base lead-in in 80 % of the rows (the 5' ends of the config[1] and
   config[2] workloads); the 3' rows are random.  Kernel device time from torch.profiler (two launches per call, one
   per half of the windows), and the whole tgsf_end_kmer_counts call (upload, table clears, kernels, 2 x 64 MB
   download) between CUDA events, both after warm-up.
2. `tgsfilter -x ont -A` wall time with and without --adapter-denovo on a config[2] FASTQ (synth.make_config(3, n)),
   the two arms alternated.  The library finds ADAPTER_LIB[8] at the 5' end there, so the assembly runs for the 3'
   end only.

    python profiles/denovo_bench.py [--reps 5] [--cli-reads 10000] [--out results.json]   # JSON on stdout
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tgsfilter_b200 import prepass, synth  # noqa: E402
from tgsfilter_b200.params import ADAPTER_LIB  # noqa: E402

ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], stdout=subprocess.PIPE,
                         text=True, check=True).stdout.strip().splitlines()[0]
    return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))


def sample_rows(n=100_000, c=150, seed=5):
    rng = np.random.default_rng(seed)
    e5 = ACGT[rng.integers(0, 4, (n, c), dtype=np.uint8)]
    e3 = ACGT[rng.integers(0, 4, (n, c), dtype=np.uint8)]
    for r in np.nonzero(rng.random(n) < 0.8)[0]:
        s = ACGT[rng.integers(0, 4, int(rng.integers(0, 31)))].tobytes() + synth.mutate(ADAPTER_LIB[8], 0.10, rng)
        e5[r, :len(s)] = np.frombuffer(s, dtype=np.uint8)
    return e5, e3


def kernel_timing(reps):
    import torch
    from torch.profiler import ProfilerActivity, profile
    e5, e3 = sample_rows()
    split = prepass.denovo_split(150)
    for rows in (e5, e3):  # warm-up: module load, first allocations
        prepass.device_end_kmers(rows, 12, split)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    call_ms = []
    for _ in range(reps):
        for rows in (e5, e3):
            start.record()
            prepass.device_end_kmers(rows, 12, split)
            stop.record()
            stop.synchronize()
            call_ms.append(start.elapsed_time(stop))
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            for rows in (e5, e3):
                prepass.device_end_kmers(rows, 12, split)
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if e.name.startswith("k_end_kmers") and e.device_type.name == "CUDA"]
    us = [e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total for e in ev]
    per_call = [us[i] + us[i + 1] for i in range(0, len(us) - 1, 2)]  # the two bands of one call
    return {"rows": "2 x 100000 x 150", "k": 12, "split": split, "launches": len(us),
            "kernel_ms_per_end_median": float(np.median(per_call)) / 1e3,
            "kernel_ms_per_end_max": float(np.max(per_call)) / 1e3,
            "call_ms_per_end_median": float(np.median(call_ms)), "call_ms_per_end_max": float(np.max(call_ms))}


def cli_timing(n_reads, reps):
    exe = os.path.join(ROOT, "src", "tgsfilter")
    d = tempfile.mkdtemp(prefix="denovo_bench_")
    try:
        batch = synth.make_config(3, n_reads, with_names=False)
        fq = os.path.join(d, "in.fq")
        synth.write_fastq(fq, batch.bases, batch.quals, batch.offsets)
        res = {"reads": n_reads, "bases": batch.n_bases}
        del batch
        times = {"without": [], "with_denovo": []}
        lines = {}
        for _ in range(reps):
            for name, extra in (("without", []), ("with_denovo", ["--adapter-denovo"])):
                t0 = time.perf_counter()
                pr = subprocess.run([exe, "-i", fq, "-x", "ont", "-A"] + extra, stdout=subprocess.DEVNULL,
                                    stderr=subprocess.PIPE, text=True, cwd=d)
                times[name].append(time.perf_counter() - t0)
                assert pr.returncode == 0, pr.stderr[-2000:]
                lines[name] = [ln for ln in pr.stderr.splitlines() if "adapter" in ln]
        for name, ts in times.items():
            res[name + "_s_median"] = float(np.median(ts))
            res[name + "_s_all"] = ts
            res[name + "_lines"] = lines[name]
        return res
    finally:
        shutil.rmtree(d, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cli-reads", type=int, default=10_000)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    res = {"gpu": gpu_info(), "count_kernel": kernel_timing(args.reps * 4),
           "cli_A_config2": cli_timing(args.cli_reads, args.reps)}
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

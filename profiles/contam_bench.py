"""Cost of the contaminant screen (tgsf_set_contaminants / --contam) on a B200.

Workload: config[1] of bench.py (synthetic ONT, 200 k reads, ~4.7 Gbases) generated on the GPU and kept resident
(tgsf_submit_device), -p 0 so that the `kmer` stage holds the screen alone.  Arms: no set, a 48.5 kb set (lambda-
sized: prefilter path, table in L2) and a 5 Mb set (no prefilter, 128 MB table, larger than L2); 1 % of the reads
are drawn from the set (4 % error) in every arm.  Per arm: the step device time (median of >= 5 steps after warm-up,
four sub-batches two in flight, max(end) - min(start) on the device clock like bench.py), the `kmer` stage time of
a pass with one batch in flight, and probes (= screened windows) per second of that stage.  Then the file-to-file
CLI time on a config[2] FASTQ with and without --contam.

    python profiles/contam_bench.py [--steps 7] [--out results.json]   # JSON on stdout without --out
"""
from __future__ import annotations

import argparse
import gzip
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from tgsfilter_b200 import _capi, synth  # noqa: E402
from tgsfilter_b200.engine import FilterEngine  # noqa: E402

K = 17


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], stdout=subprocess.PIPE,
                         text=True, check=True).stdout.strip().splitlines()[0]
    return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))


def plant(bases, offsets, genome, frac, seed):
    """Overwrite a fraction of the (device) reads with reads drawn from genome; returns their count."""
    import torch
    rng = np.random.default_rng(seed)
    sel = np.nonzero(rng.random(len(offsets) - 1) < frac)[0]
    for r in sel:
        s, e = int(offsets[r]), int(offsets[r + 1])
        bases[s:e] = torch.from_numpy(synth.contaminant_read(genome, e - s, 0.04, rng)).to(bases.device)
    return len(sel)


def run_arm(params, cset, subs, steps, warmup):
    """subs: [(bases, quals, d_off, offsets, total)] of separately generated sub-batches."""
    n_sub = len(subs)
    with FilterEngine(params) as eng:
        n_kmers = eng.set_contaminants(cset, k=K) if cset else 0

        def submit(j):
            b, q, o, offs, nb = subs[j]
            eng.submit_device(b.data_ptr(), q.data_ptr(), o.data_ptr(), len(offs) - 1, int(nb))

        # single-batch pass: kmer stage per sub-batch, screened windows and contaminant pieces
        kmer_ms, windows, n_contam = 0.0, 0, 0
        for j in range(n_sub):
            submit(j)
            _, pieces = eng.collect()
            kmer_ms += eng.last_stage_ms()["kmer"]
            scr = ((pieces["status"] == _capi.PIECE_EMIT) | (pieces["status"] == _capi.PIECE_CONTAM)) & (pieces["len"] >= K)
            windows += int((pieces["len"][scr].astype(np.int64) - K + 1).sum())
            n_contam += int((pieces["status"] == _capi.PIECE_CONTAM).sum())
        steps_ms = []
        for it in range(warmup + steps):
            spans = []
            for j in range(n_sub):
                submit(j)
                if j >= 1:
                    eng.collect(want_results=False)
                    spans.append(eng.last_span())
            eng.collect(want_results=False)
            spans.append(eng.last_span())
            if it >= warmup:
                steps_ms.append(max(e for _, e in spans) - min(s for s, _ in spans))
    return {"n_kmers": n_kmers, "step_ms_median": statistics.median(steps_ms), "step_ms": steps_ms,
            "kmer_stage_ms_single_batch": kmer_ms, "screened_windows": windows,
            "probes_per_s": (windows / (kmer_ms * 1e-3)) if cset else 0.0, "contam_pieces": n_contam}


def cli_f2f(genome, n_reads, reps=2):
    exe = os.path.join(ROOT, "src", "tgsfilter")
    d = tempfile.mkdtemp(prefix="contam_f2f_")
    batch = synth.make_config(3, n_reads, with_names=False)
    batch, planted, _ = synth.mix_contaminants(batch, genome, 0.01, 0.04)
    fq = os.path.join(d, "in.fq")
    with open(fq, "wb") as f:
        synth.write_fastq_to(f, batch.bases, batch.quals, batch.offsets)
    fa = os.path.join(d, "contam.fa.gz")
    with open(fa, "wb") as f:
        f.write(gzip.compress(b">c\n" + b"".join(genome[i:i + 80] + b"\n" for i in range(0, len(genome), 80))))
    res = {"reads": n_reads, "bases": batch.n_bases, "planted_reads": int(len(planted))}
    for name, extra in (("without", []), ("with_contam", ["--contam", fa])):
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            pr = subprocess.run([exe, "-i", fq, "-x", "ont", "-o", os.path.join(d, "out.fq")] + extra,
                                stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True)
            ts.append(time.perf_counter() - t0)
            assert pr.returncode == 0, pr.stderr[-2000:]
        res[name + "_s"] = min(ts)
        res[name + "_info"] = [ln for ln in pr.stderr.splitlines() if "contaminant" in ln or "-mers loaded" in ln]
    for f in os.listdir(d):
        os.remove(os.path.join(d, f))
    os.rmdir(d)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=200_000)
    ap.add_argument("--steps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--f2f-reads", type=int, default=5000)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    import torch
    dev = torch.device("cuda:0")
    info = gpu_info()
    small = synth.make_contaminant(48_502)
    large = synth.make_contaminant(5_000_000, seed=synth.SEED0 + 102)
    params = synth.config_params(2)
    params.n_slots = 2
    params.max_read_len = 4 << 20
    arms = {}
    for name, genome in (("none", small), ("small_48.5kb", small), ("large_5Mb", large)):
        subs, planted = [], 0
        for j in range(4):  # four sub-batches, each its own allocation (16-byte aligned streams)
            sub = bench.gen_workload_gpu(2, args.reads // 4, bench.batch_seed(2, 0, j), dev)
            planted += plant(sub[0], sub[3], genome, 0.01, seed=7 + j)
            subs.append(sub)
        torch.cuda.synchronize()
        arms[name] = run_arm(params, [genome] if name != "none" else None, subs, args.steps, args.warmup)
        arms[name]["planted_reads"] = planted
        arms[name]["bases"] = int(sum(int(s[4]) for s in subs))
        del subs
        torch.cuda.empty_cache()
        print(name, json.dumps({k: v for k, v in arms[name].items() if k != "step_ms"}), flush=True)
    f2f = cli_f2f(small, args.f2f_reads)
    print("f2f", json.dumps(f2f), flush=True)
    res = {"gpu": info, "workload": f"config[1] (bench.py config 2), {args.reads} reads resident, -p 0, k = {K}, "
           "min_frac 0.05, 1 % of reads planted from the arm's set (4 % error)",
           "arms": arms, "cli_f2f_config2": f2f}
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

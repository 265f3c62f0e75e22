"""Cost of the contaminant screen's per-record attribution (tgsf_set_contaminants_labelled / --contam-report) on a B200.

Workload: config[1] of bench.py (synthetic ONT, 200 k reads, ~4.7 Gbases) generated on the GPU and kept resident
(tgsf_submit_device), -p 0 so that the `kmer` stage holds the contaminant screen alone.  The set has three records:
lambda-sized (48.5 kb), plasmid-sized (6 kb) and 5 Mb (5.05 Mb in all: no prefilter, table larger than L2).  A
fraction of the reads (1 % or 20 %) is overwritten, on the device, with exact copies of a random record (either
strand, the record tiled to the read's length), so every window of a planted read is a hit: the attribution's worst
case per contaminated base.  Per fraction and install mode (plain tgsf_set_contaminants / labelled): the step device
time (median of the timed steps after warm-up, four sub-batches two in flight, max(end) - min(start) on the device
clock like bench.py), the `kmer` stage time of a pass with one batch in flight, the contaminant pieces and bases, and
the host wall time of installing the set (median of three).

    python profiles/contam_records_bench.py [--steps 5] [--out results.json]   # JSON on stdout without --out
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from tgsfilter_b200 import _capi, synth  # noqa: E402
from tgsfilter_b200.engine import FilterEngine  # noqa: E402
from tgsfilter_b200.params import rev_comp  # noqa: E402

K = 17


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], stdout=subprocess.PIPE,
                         text=True, check=True).stdout.strip().splitlines()[0]
    return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))


def plant(subs, cset, frac, seed, dev):
    """Overwrite a fraction of every sub-batch's device reads with copies of a random record; returns the count."""
    import torch
    rng = np.random.default_rng(seed)
    longest = max(int(np.diff(s[3]).max()) for s in subs)
    tiles = []
    for rec in cset:  # each record and its reverse complement, tiled past the longest read plus one record
        reps = (longest + len(rec)) // len(rec) + 1
        tiles.append([torch.from_numpy(np.frombuffer(r * reps, dtype=np.uint8).copy()).to(dev)
                      for r in (rec, rev_comp(rec))])
    n = 0
    for b, _, _, offs, _ in subs:
        sel = np.nonzero(rng.random(len(offs) - 1) < frac)[0]
        for r in sel:
            s, e = int(offs[r]), int(offs[r + 1])
            i = int(rng.integers(0, len(cset)))
            t = tiles[i][int(rng.integers(0, 2))]
            o = int(rng.integers(0, len(cset[i])))
            b[s:e] = t[o:o + (e - s)]
        n += len(sel)
    torch.cuda.synchronize()
    return n


def install(eng, cset, labelled):
    if labelled:
        return eng.set_contaminants_labelled(cset, k=K)[0]
    return eng.set_contaminants(cset, k=K)


def run_arm(params, cset, subs, steps, warmup, labelled):
    with FilterEngine(params) as eng:
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            n_kmers = install(eng, cset, labelled)
            ts.append(time.perf_counter() - t0)

        def submit(j):
            b, q, o, offs, nb = subs[j]
            eng.submit_device(b.data_ptr(), q.data_ptr(), o.data_ptr(), len(offs) - 1, int(nb))

        kmer_ms, n_contam, contam_bases = 0.0, 0, 0
        for j in range(len(subs)):
            submit(j)
            _, pieces = eng.collect()
            kmer_ms += eng.last_stage_ms()["kmer"]
            c = pieces["status"] == _capi.PIECE_CONTAM
            n_contam += int(c.sum())
            contam_bases += int(pieces["len"][c].astype(np.int64).sum())
        tally = None
        if labelled:
            reads, bases = eng.contam_record_stats()
            assert int(reads.sum()) == n_contam and int(bases.sum()) == contam_bases
            tally = {"reads": [int(x) for x in reads], "bases": [int(x) for x in bases]}
        steps_ms = []
        for it in range(warmup + steps):
            spans = []
            for j in range(len(subs)):
                submit(j)
                if j >= 1:
                    eng.collect(want_results=False)
                    spans.append(eng.last_span())
            eng.collect(want_results=False)
            spans.append(eng.last_span())
            if it >= warmup:
                steps_ms.append(max(e for _, e in spans) - min(s for s, _ in spans))
    return {"n_kmers": n_kmers, "install_s_median": statistics.median(ts), "install_s": ts,
            "step_ms_median": statistics.median(steps_ms), "step_ms": steps_ms,
            "kmer_stage_ms_single_batch": kmer_ms, "contam_pieces": n_contam, "contam_bases": contam_bases,
            "tally_single_batch_pass": tally}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=200_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    import torch
    dev = torch.device("cuda:0")
    res = {"gpu": gpu_info(), "k": K}
    cset = [synth.make_contaminant(48_502), synth.make_contaminant(6_000, seed=synth.SEED0 + 201),
            synth.make_contaminant(5_000_000, seed=synth.SEED0 + 102)]
    res["set_records"] = [len(r) for r in cset]
    cfg = 2  # config[1]
    params = synth.config_params(cfg)
    params.n_slots = 2
    params.max_read_len = 4 << 20
    for frac in (0.01, 0.20):
        subs = [bench.gen_workload_gpu(cfg, args.reads // 4, bench.batch_seed(cfg, 0, j), dev) for j in range(4)]
        planted = plant(subs, cset, frac, int(frac * 1000), dev)
        bases = int(sum(int(s[4]) for s in subs))
        arms = {}
        for arm in ("plain", "labelled", "plain_again", "labelled_again"):  # alternated: run-to-run spread
            arms[arm] = run_arm(params, cset, subs, args.steps, args.warmup, arm.startswith("labelled"))
            print(f"{frac:.0%}", arm, json.dumps({k: v for k, v in arms[arm].items()
                                                  if k not in ("step_ms", "install_s", "tally_single_batch_pass")}),
                  flush=True)
        res[f"planted_{frac:.2f}"] = {
            "reads": args.reads, "bases": bases, "planted_reads": planted, "arms": arms,
            "kmer_stage_delta_ms": arms["labelled"]["kmer_stage_ms_single_batch"]
            - arms["plain"]["kmer_stage_ms_single_batch"],
            "step_delta_ms": arms["labelled"]["step_ms_median"] - arms["plain"]["step_ms_median"]}
        del subs
        torch.cuda.empty_cache()
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

"""Cost of the fold-back screen (tgsf_set_foldback / --foldback) on a B200.

Workloads, generated on the GPU and kept resident (tgsf_submit_device) like bench.py: config[1] (synthetic ONT,
200 k reads, ~4.7 Gbases, -p 0, so the `kmer` stage holds the screen alone) and a config[4]-sized HiFi batch (200 k
reads of config[4], ~3 Gbases, -k 11 -p 5000, so the `kmer` stage also holds K4).  Per workload and arm (screen off /
on): the step device time (median of the timed steps after warm-up, four sub-batches two in flight, max(end) -
min(start) on the device clock like bench.py), the `kmer` stage time of a pass with one batch in flight, and for the
arm with the screen the screened windows per second of the stage difference, and the pieces cut.

    python profiles/foldback_bench.py [--steps 7] [--out results.json]   # JSON on stdout without --out
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from tgsfilter_b200 import _capi, synth  # noqa: E402
from tgsfilter_b200.engine import FilterEngine  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], stdout=subprocess.PIPE,
                         text=True, check=True).stdout.strip().splitlines()[0]
    return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))


def run_arm(params, subs, steps, warmup, enable):
    with FilterEngine(params) as eng:
        eng.set_foldback(enable)

        def submit(j):
            b, q, o, offs, nb = subs[j]
            eng.submit_device(b.data_ptr(), q.data_ptr(), o.data_ptr(), len(offs) - 1, int(nb))

        kmer_ms, windows, n_emit = 0.0, 0, 0
        for j in range(len(subs)):
            submit(j)
            _, pieces = eng.collect()
            kmer_ms += eng.last_stage_ms()["kmer"]
            n_emit += len(pieces)
        stats = eng.foldback_stats()
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
    return {"step_ms_median": statistics.median(steps_ms), "step_ms": steps_ms,
            "kmer_stage_ms_single_batch": kmer_ms, "pieces": n_emit,
            "fold_stats_single_pass": list(stats) if enable else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=200_000)
    ap.add_argument("--steps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    import torch
    dev = torch.device("cuda:0")
    info = gpu_info()
    res = {"gpu": info, "workloads": {}}
    for name, cfg in (("config[1] ONT", 2), ("config[4] HiFi", 5)):
        params = synth.config_params(cfg)
        params.n_slots = 2
        params.max_read_len = 4 << 20
        subs = [bench.gen_workload_gpu(cfg, args.reads // 4, bench.batch_seed(cfg, 0, j), dev) for j in range(4)]
        torch.cuda.synchronize()
        bases = int(sum(int(s[4]) for s in subs))
        arms = {arm: run_arm(params, subs, args.steps, args.warmup, arm == "foldback") for arm in ("off", "foldback")}
        # windows the screen looks at: every 15-base window of the pieces K5 emitted (= the pieces of the off arm)
        win = 0
        with FilterEngine(params) as eng:
            for j in range(4):
                b, q, o, offs, nb = subs[j]
                eng.submit_device(b.data_ptr(), q.data_ptr(), o.data_ptr(), len(offs) - 1, int(nb))
                _, pieces = eng.collect()
                L = pieces["len"][pieces["status"] != _capi.PIECE_QC_ONLY].astype(np.int64)
                win += int(np.maximum(L - 14, 0).sum())
        dk = arms["foldback"]["kmer_stage_ms_single_batch"] - arms["off"]["kmer_stage_ms_single_batch"]
        w = {"reads": args.reads, "bases": bases, "arms": arms, "screened_windows": win,
             "screen_ms_single_batch": dk, "windows_per_s": win / (dk * 1e-3) if dk > 0 else None,
             "step_overhead_ms": arms["foldback"]["step_ms_median"] - arms["off"]["step_ms_median"]}
        res["workloads"][name] = w
        print(name, json.dumps({k: v for k, v in w.items() if k != "arms"}), flush=True)
        del subs
        torch.cuda.empty_cache()
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

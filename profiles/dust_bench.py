"""Cost of the low-complexity screen (tgsf_set_dust / --dust) on a B200.

Pipeline: config[1] (synthetic ONT, 200 k reads, ~4.7 Gbases, -p 0), generated on the GPU and kept resident
(tgsf_submit_device) like bench.py.  Per arm (screen off / on at the defaults, level 7 and 0.5): the step device time
(median of the timed steps after warm-up, four sub-batches two in flight, max(end) - min(start) on the device clock
like bench.py), the `kmer` stage time of a pass with one batch in flight (the screen alone in that stage, -p 0), the
screened windows per second of the stage difference, and the pieces dropped.

Stand-alone: tgsf_dust_detect on 15 kb and 1 Mb random pieces with 5 % planted homopolymer and dinucleotide runs
(~300 Mbases each): host wall time of the call (median of five; it creates a context, copies the pieces in and the
counts out, and waits for its stream), as bases per second.

    python profiles/dust_bench.py [--steps 7] [--out results.json]   # JSON on stdout without --out
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


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], stdout=subprocess.PIPE,
                         text=True, check=True).stdout.strip().splitlines()[0]
    return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))


def run_arm(params, subs, steps, warmup, dust):
    with FilterEngine(params) as eng:
        if dust:
            eng.set_dust(7, 0.5)

        def submit(j):
            b, q, o, offs, nb = subs[j]
            eng.submit_device(b.data_ptr(), q.data_ptr(), o.data_ptr(), len(offs) - 1, int(nb))

        kmer_ms, dropped, windows = 0.0, 0, 0
        for j in range(len(subs)):
            submit(j)
            _, pieces = eng.collect()
            kmer_ms += eng.last_stage_ms()["kmer"]
            dropped += int((pieces["status"] == _capi.PIECE_LOWCOMPLEX).sum())
            screened = pieces["status"] != _capi.PIECE_QC_ONLY
            windows += int(np.maximum(pieces["len"][screened].astype(np.int64) - 63, 0).sum())
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
            "kmer_stage_ms_single_batch": kmer_ms, "pieces_dropped": dropped, "windows": windows}


def detect_pieces(rng, piece_len, total):
    n = max(1, total // piece_len)
    bases = synth._ACGT[rng.integers(0, 4, n * piece_len, dtype=np.uint8)]
    for p in range(0, n * piece_len, 2000):  # 5 %: a 100-base homopolymer or dinucleotide run every 2 kb
        bases[p:p + 100] = np.frombuffer((b"A" * 100) if (p // 2000) % 2 else (b"CA" * 50), dtype=np.uint8)
    offs = np.arange(n + 1, dtype=np.uint64) * np.uint64(piece_len)
    return np.ascontiguousarray(bases), offs


def time_detect(bases, offs, reps=5):
    lib = _capi.load()
    n = len(offs) - 1
    out = np.zeros(n, dtype=np.uint32)
    _capi.check(lib.tgsf_dust_detect(0, bases.ctypes.data, offs.ctypes.data, n, 7, out.ctypes.data), "warm-up")
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        _capi.check(lib.tgsf_dust_detect(0, bases.ctypes.data, offs.ctypes.data, n, 7, out.ctypes.data),
                    "tgsf_dust_detect")
        ts.append(time.perf_counter() - t0)
    s = statistics.median(ts)
    return {"pieces": n, "bases": int(offs[-1]), "call_s_median": s, "call_s": ts,
            "bases_per_s": int(offs[-1]) / s, "masked_bases": int(out.sum())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=200_000)
    ap.add_argument("--steps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--detect-bases", type=int, default=300_000_000)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    import torch
    dev = torch.device("cuda:0")
    res = {"gpu": gpu_info()}
    cfg = 2  # config[1]
    params = synth.config_params(cfg)
    params.n_slots = 2
    params.max_read_len = 4 << 20
    subs = [bench.gen_workload_gpu(cfg, args.reads // 4, bench.batch_seed(cfg, 0, j), dev) for j in range(4)]
    torch.cuda.synchronize()
    bases = int(sum(int(s[4]) for s in subs))
    arms = {arm: run_arm(params, subs, args.steps, args.warmup, arm == "dust") for arm in ("off", "dust")}
    dk = arms["dust"]["kmer_stage_ms_single_batch"] - arms["off"]["kmer_stage_ms_single_batch"]
    win = arms["off"]["windows"]
    res["config[1]"] = {"reads": args.reads, "bases": bases, "arms": arms, "screen_ms_single_batch": dk,
                        "windows_per_s": win / (dk * 1e-3) if dk > 0 else None,
                        "step_overhead_ms": arms["dust"]["step_ms_median"] - arms["off"]["step_ms_median"]}
    print("config[1]", json.dumps({k: v for k, v in res["config[1]"].items() if k != "arms"}), flush=True)
    del subs
    torch.cuda.empty_cache()
    rng = np.random.default_rng(5)
    res["detect"] = {}
    for name, L in (("15 kb", 15_000), ("1 Mb", 1_000_000)):
        b, o = detect_pieces(rng, L, args.detect_bases)
        res["detect"][name] = time_detect(b, o)
        print("tgsf_dust_detect", name, json.dumps({k: v for k, v in res["detect"][name].items() if k != "call_s"}),
              flush=True)
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

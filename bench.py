#!/usr/bin/env python
"""bench.py — filtered Gbases/s of the per-read filter/trim hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--config C] [--strong] [--reads R] [--dump-outputs DIR]

One "step" = one pass of the whole hot path (K1 raw scan -> K3 adapter search -> K5 regions ->
[K4] -> K1 clean scan) over the workload's batches.  Workload (`--config`, or TGSF_BENCH_CONFIG;
BASELINE config index + 1): default 2 = configs[1], 200 000 synthetic ONT reads, N50 ~30 kb, planted
5' adapter, `-x ont` with adapter auto-identify + end trim.
  weak scaling (default): every rank processes its own dataset of the config's full size; no data-path
      collective, the QC counters are combined with one NCCL allreduce after the timed region.
  strong scaling (`--strong`, or TGSF_BENCH_STRONG=1): ONE dataset of the config's full size, cut into
      16 batches that are dealt round-robin to the ranks (tgsfilter_b200.shard); the counter allreduce is
      INSIDE the reported time of every step.
Datasets of more than 400 000 reads are fed as several batches through the context's two slots.

`value`  : input bases / device time, inputs resident in HBM.  Device time of a step = last kernel end
           - first kernel start of its batches on the device clock (tgsf_last_span; batches in the two
           slots run on two streams and overlap) [+ the allreduce in strong mode], max over ranks.
`e2e`    : same metric through the C-ABI with pinned HOST buffers holding what a parser produces (byte bases, Phred
           bytes, offsets): H2D + unpack + kernels + D2H of the results inside the timed region (wall clock between
           barriers, max over ranks).  Two feeds are timed and the faster is reported (the other: `e2e_other_feed`):
           plain bytes (tgsf_submit, 2 B/base over PCIe) and the adaptive feed, where host threads pack the bases to
           2 bits INSIDE the timed region ahead of the submit loop and a sub-batch goes out packed when its packed copy
           is ready, as bytes otherwise.
`roofline`: dominant kernel; the others under `roofline_kernels`.
`cpu_baseline` / `--impl reference`: the UNMODIFIED reference CLI (oracle/_ref/tgsfilter) on this box's
           host cores over the SAME workload (rank 0's dataset, written as FASTQ to tmpfs).  The
           reference arm runs the full dataset every step unless that would exceed its time budget
           (TGSF_REF_BUDGET_S, default 600 s for all warm-up + timed steps); then every step is the
           largest prefix of the dataset that fits, and `cpu_baseline.sample` says so.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

CONFIG_READS = {1: 20_000, 2: 200_000, 3: 50_000, 4: 1_000_000, 5: 2_000_000}
CONFIG_CLI = {1: ["-x", "hifi"], 2: ["-x", "ont"], 3: ["-x", "ont", "-M", "35", "-T", "50"],
              4: ["-x", "clr", "-q", "7", "-Q", "15", "-e", "150", "-b", "1"],
              5: ["-x", "hifi", "-k", "11", "-p", "5000"]}
CONFIG_TYPE = {1: "hifi", 2: "ont", 3: "ont", 4: "clr", 5: "hifi"}
REF_CLI = os.path.join(ROOT, "oracle", "_ref", "tgsfilter")
SUB_READS = 400_000      # weak mode: datasets above this many reads are fed as several batches
STRONG_BATCHES = 16      # strong mode: the dataset is always dealt as this many batches
SEED0 = 20261017


def batch_seed(cfg: int, rank: int, j: int) -> int:
    return SEED0 + cfg + 1000 * rank + 100000 * j


def plan_batches(cfg: int, n_total: int, world: int, rank: int, strong: bool, split: int = 0):
    """[(global batch index, reads, seed)] this rank generates and processes."""
    if strong:
        nb = min(STRONG_BATCHES, n_total)
        sizes = [n_total // nb + (1 if j < n_total % nb else 0) for j in range(nb)]
        return [(j, sizes[j], batch_seed(cfg, 0, j)) for j in range(nb) if j % world == rank]
    nb = max(1, math.ceil(n_total / SUB_READS), split)
    sizes = [n_total // nb + (1 if j < n_total % nb else 0) for j in range(nb)]
    return [(j, sizes[j], batch_seed(cfg, rank, j)) for j in range(nb)]


def workload_name(cfg: int, n_reads: int, strong: bool) -> str:
    names = {1: "config[0] synthetic HiFi FASTQ ~15 kb, -x hifi",
             2: "config[1] synthetic ONT FASTQ N50 ~30 kb, planted 5' adapter, -x ont (auto-identify + end trim)",
             3: "config[2] synthetic ONT ultra-long N50 ~100 kb, planted middle adapters, -M 35 -T 50",
             4: "config[3] synthetic PacBio CLR, -q 7 -Q 15 -e 150 -b 1",
             5: "config[4] synthetic HiFi, -k 11 -p 5000"}
    return f"{names[cfg]}; {n_reads} reads " + ("in total, dealt to the GPUs" if strong else "per GPU")


def static_config(cfg: int, n_reads: int, strong: bool) -> dict:
    """The `config` object: a pure function of the command line, identical in both arms."""
    return {"workload": workload_name(cfg, n_reads, strong), "cli": " ".join(CONFIG_CLI[cfg]),
            "reads": n_reads, "reads_are": "total over all GPUs" if strong else "per GPU",
            "batches": "16, dealt round-robin" if strong else "ceil(reads / 400000), at least --split; two in flight",
            "seed": SEED0 + cfg,
            "l2": "inputs (2 B/base, >= 0.5 GB per launch) are larger than the 126 MB L2"}


# ------------------------------------------------------------------------------------------------
# synthetic workload, generated on the GPU (same distributions as tgsfilter_b200.synth)
# ------------------------------------------------------------------------------------------------
def gen_workload_gpu(config: int, n_reads: int, seed: int, device):
    import torch
    from tgsfilter_b200 import synth
    from tgsfilter_b200.params import ADAPTER_LIB

    rng = np.random.default_rng(seed)
    lens = synth._lengths(config, n_reads, rng)
    offsets = np.zeros(n_reads + 1, dtype=np.int64)
    np.cumsum(lens, out=offsets[1:])
    total = int(offsets[-1])
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    bases = torch.empty(total + 64, dtype=torch.uint8, device=device)
    quals = torch.empty(total + 64, dtype=torch.uint8, device=device)
    bases[total:] = 65
    quals[total:] = 33
    mu, sigma = synth._QUAL[config]
    mean_q = rng.normal(mu, sigma, n_reads).astype(np.float32)
    if config in (1, 5):
        low = rng.random(n_reads) < 0.05
        mean_q[low] = rng.normal(15, 4, int(low.sum())).astype(np.float32)
    d_mean = torch.from_numpy(mean_q).to(device)
    d_lens = torch.from_numpy(lens).to(device)
    group = max(1, n_reads // 32)
    for lo in range(0, n_reads, group):
        hi = min(n_reads, lo + group)
        s, e = int(offsets[lo]), int(offsets[hi])
        code = torch.randint(0, 4, (e - s,), dtype=torch.uint8, device=device, generator=g)
        # A=65 C=67 G=71 T=84
        b = 65 + 2 * code + 2 * (code >= 2).to(torch.uint8) + 11 * (code == 3).to(torch.uint8)
        bases[s:e] = b
        q = torch.repeat_interleave(d_mean[lo:hi], d_lens[lo:hi])
        q = q + 5.0 * torch.randn(e - s, dtype=torch.float32, device=device, generator=g)
        quals[s:e] = (q.round_().clamp_(1, 60) + 33).to(torch.uint8)
        del code, b, q
    d_off = torch.from_numpy(offsets).to(device)

    def plant(reads_idx, pos, variants, vlen, which):
        """bases[offsets[r] + pos + j] = variants[which][j] for j < vlen[which]"""
        if len(reads_idx) == 0:
            return
        r = torch.from_numpy(reads_idx).to(device)
        p = torch.from_numpy(pos).to(device)
        w = torch.from_numpy(which).to(device)
        V = torch.from_numpy(variants).to(device)
        VL = torch.from_numpy(vlen).to(device)
        J = torch.arange(V.shape[1], device=device)[None, :]
        mask = J < VL[w][:, None]
        dest = (d_off[r] + p)[:, None] + J
        bases[dest[mask]] = V[w][mask]

    def variant_pool(ad, err, count):
        vs = [synth.mutate(ad, err, rng) for _ in range(count)]
        ml = max(len(v) for v in vs)
        arr = np.full((count, ml), 65, dtype=np.uint8)
        for i, v in enumerate(vs):
            arr[i, :len(v)] = np.frombuffer(v, dtype=np.uint8)
        return arr, np.array([len(v) for v in vs], dtype=np.int64)

    if config in (2, 3):
        ad = ADAPTER_LIB[8]
        V, VL = variant_pool(ad, 0.10, 1024)
        sel = np.nonzero((rng.random(n_reads) < 0.80) & (lens > 200))[0]
        plant(sel, rng.integers(0, 31, len(sel)), V, VL, rng.integers(0, 1024, len(sel)))
        frac_mid, err_mid = (0.01, 0.10) if config == 2 else (0.10, 0.05)
        V2, VL2 = variant_pool(ad, err_mid, 1024)
        sel = np.nonzero((rng.random(n_reads) < frac_mid) & (lens > 1000))[0]
        pos = (400 + rng.random(len(sel)) * (lens[sel] - 900)).astype(np.int64)
        plant(sel, pos, V2, VL2, rng.integers(0, 1024, len(sel)))
    elif config in (1, 5):
        ad = ADAPTER_LIB[0]
        V, VL = variant_pool(ad, 0.03, 512)
        u = rng.random(n_reads)
        sel = np.nonzero(u < 0.015)[0]
        plant(sel, np.zeros(len(sel), np.int64), V, VL, rng.integers(0, 512, len(sel)))
        sel = np.nonzero((u >= 0.015) & (u < 0.030))[0]
        plant(sel, lens[sel] - 60, V, VL, rng.integers(0, 512, len(sel)))
        sel = np.nonzero((u >= 0.030) & (u < 0.033))[0]
        pos = (300 + rng.random(len(sel)) * (lens[sel] - 700)).astype(np.int64)
        plant(sel, pos, V, VL, rng.integers(0, 512, len(sel)))
    if config == 5:
        # 30 % of reads carry a 6-12 kb tandem repeat (unit 50-500 bp, 1 % error; substitutions only here,
        # tgsfilter_b200.synth also plants indels), so that repeatLen straddles the -p 5000 bound
        sel = np.nonzero(rng.random(n_reads) < 0.30)[0]
        unit_len = rng.integers(50, 501, len(sel))
        span = np.minimum(rng.integers(6000, 12001, len(sel)), lens[sel] - 200)
        ok = span > unit_len
        sel, unit_len, span = sel[ok], unit_len[ok], span[ok]
        pos = (100 + rng.random(len(sel)) * np.maximum(1, lens[sel] - span - 150)).astype(np.int64)
        pool = torch.randint(0, 4, (1 << 22,), dtype=torch.uint8, device=device, generator=g)
        pool = 65 + 2 * pool + 2 * (pool >= 2).to(torch.uint8) + 11 * (pool == 3).to(torch.uint8)
        unit_off = rng.integers(0, (1 << 22) - 512, len(sel))
        step = 20000
        for lo in range(0, len(sel), step):
            hi = min(len(sel), lo + step)
            sp = torch.from_numpy(span[lo:hi]).to(device)
            first = torch.cumsum(sp, 0) - sp
            rid = torch.repeat_interleave(torch.arange(hi - lo, device=device), sp)
            j = torch.arange(int(sp.sum().item()), device=device) - first[rid]
            ul = torch.from_numpy(unit_len[lo:hi]).to(device)[rid]
            uo = torch.from_numpy(unit_off[lo:hi]).to(device)[rid]
            val = pool[uo + j % ul]
            err = torch.rand(val.shape, device=device, generator=g) < 0.01
            val = torch.where(err, pool[(uo + j * 7 + 13) % (1 << 22)], val)
            dest = (d_off[torch.from_numpy(sel[lo:hi]).to(device)] + torch.from_numpy(pos[lo:hi]).to(device))[rid] + j
            bases[dest] = val
            del sp, first, rid, j, ul, uo, val, err, dest
    if config == 4:
        k = 12
        r = np.arange(n_reads)
        J = torch.arange(k, device=device)[None, :]
        at = torch.rand((n_reads, k), device=device, generator=g) < 0.70
        pick_at = torch.randint(0, 2, (n_reads, k), device=device, generator=g) * 19 + 65   # A / T
        pick_cg = torch.randint(0, 2, (n_reads, k), device=device, generator=g) * 4 + 67    # C / G
        val = torch.where(at, pick_at, pick_cg).to(torch.uint8)
        dest = d_off[:-1][:, None] + J
        mask = J < d_lens[:, None]
        bases[dest[mask]] = val[mask]
        del r
    torch.cuda.synchronize(device)
    return bases, quals, d_off, offsets, total


class ClockSampler:
    """nvidia-smi sampler running during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def __enter__(self):
        if shutil.which("nvidia-smi") is None:
            return self
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits", "-lms", "100"],
                                     stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        self.t = threading.Thread(target=self._read, daemon=True)
        self.t.start()
        time.sleep(0.3)
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for nme, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except (ValueError, IndexError):
                continue
        busy = sorted(sm)[len(sm) // 2:] if sm else []  # upper half ~ samples under load
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


class ClockSampler:
    """nvidia-smi sampler running during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def __enter__(self):
        if shutil.which("nvidia-smi") is None:
            return self
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits", "-lms", "100"],
                                     stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        self.t = threading.Thread(target=self._read, daemon=True)
        self.t.start()
        time.sleep(0.3)
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for nme, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except (ValueError, IndexError):
                continue
        busy = sorted(sm)[len(sm) // 2:] if sm else []  # upper half ~ samples under load
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# reference on the host CPU
# ------------------------------------------------------------------------------------------------
def ref_threads() -> int:
    n = os.cpu_count() or 2
    return max(1, min(32, n - 1))  # the reference's own clamp, T.cpp:488-499


def write_reference_fastq(cfg: int, plan, path: str, max_reads: int = 0):
    """The reads of `plan` (rank 0's batches) as one FASTQ file; same generator and seeds as the GPU arm when a
    CUDA device is there (it is on the bench box), the numpy generator of tgsfilter_b200.synth otherwise.
    Returns (reads, bases, generator name)."""
    from tgsfilter_b200 import synth
    use_gpu = False
    try:
        import torch
        use_gpu = torch.cuda.is_available()
    except Exception:
        pass
    reads = bases = 0
    with open(path, "wb", buffering=1 << 24) as f:
        for j, n, seed in plan:
            if max_reads and reads >= max_reads:
                break
            take = n if not max_reads else min(n, max_reads - reads)
            if use_gpu:
                import torch
                dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
                d_b, d_q, _, offsets, total = gen_workload_gpu(cfg, n, seed, dev)
                hb, hq = d_b[:total].cpu().numpy(), d_q[:total].cpu().numpy()
                del d_b, d_q
                torch.cuda.empty_cache()
            else:
                b = synth.make_config(cfg, n, with_names=False)
                hb, hq, offsets = b.bases, b.quals, b.offsets.astype(np.int64)
            synth.write_fastq_to(f, hb, hq, offsets[:take + 1], b"b%d_" % j)
            reads += take
            bases += int(offsets[take])
            del hb, hq
    return reads, bases, "bench.gen_workload_gpu" if use_gpu else "tgsfilter_b200.synth (numpy; no CUDA device here)"


def run_reference_once(cfg: int, fq_path: str, threads: int) -> float:
    out = os.path.join(os.path.dirname(fq_path), "ref_out.fq")
    t0 = time.perf_counter()
    pr = subprocess.run([REF_CLI, "-i", fq_path, "-o", out, "-t", str(threads)] + CONFIG_CLI[cfg],
                        stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, cwd=os.path.dirname(fq_path))
    dt = time.perf_counter() - t0
    if pr.returncode != 0:
        raise RuntimeError("reference CLI failed: " + pr.stderr.decode()[-400:])
    try:
        os.unlink(out)
    except OSError:
        pass
    return dt


def shm_dir():
    return "/dev/shm" if os.path.isdir("/dev/shm") else None


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cfg, strong = args.config, args.strong
    n_total = args.reads or CONFIG_READS[cfg]
    if not os.path.exists(REF_CLI):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/tgsfilter not built"}))
        return 0
    threads = ref_threads()
    budget = float(os.environ.get("TGSF_REF_BUDGET_S", "600"))
    plan = plan_batches(cfg, n_total, 1, 0, strong, args.split)
    tmpdir = tempfile.mkdtemp(prefix="tgsf_ref_", dir=shm_dir())
    t_begin = time.perf_counter()
    try:
        fq_path = os.path.join(tmpdir, "sample.fq")
        reads, bases, gen = write_reference_fastq(cfg, plan, fq_path, args.sample_reads)
        # one calibration run (it is also the first warm-up step): does (warmup + steps) x full fit the budget?
        t_full = run_reference_once(cfg, fq_path, threads)
        runs_left = max(args.warmup - 1, 0) + args.steps
        left = budget - (time.perf_counter() - t_begin)
        if runs_left * t_full > left and reads > 6000:
            frac = max(left / (runs_left * t_full), 0.02)
            reads_s = max(6000, int(reads * frac) // 1000 * 1000)
            reads, bases, gen = write_reference_fastq(cfg, plan, fq_path, reads_s)
            run_reference_once(cfg, fq_path, threads)
        for _ in range(max(args.warmup - 1, 0)):
            run_reference_once(cfg, fq_path, threads)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            run_reference_once(cfg, fq_path, threads)
        dt = time.perf_counter() - t0
    finally:
        shutil.rmtree(tmpdir, ignore_errors=True)
    value = bases * args.steps / dt / 1e9
    whole = reads == sum(n for _, n, _ in plan)
    sample = (f"{'the whole dataset' if whole else 'the first ' + str(reads) + ' reads of the dataset'} of rank 0 "
              f"({reads} reads, {bases} bases, generator {gen}), FASTQ on tmpfs -> FASTQ on tmpfs, unmodified "
              f"reference CLI -t {threads}, {dt / args.steps:.1f} s per step")
    line = {
        "impl": "reference", "metric": "filtered Gbases/s", "value": value, "unit": "Gbases/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong" if strong else "weak",
        "vs_baseline": None, "dtype": "u8/u64", "data": "synthetic",
        "config": static_config(cfg, n_total, strong),
        "cpu_baseline": {"value": value, "unit": "Gbases/s", "cores": threads, "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": "Gbases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
# outputs of the timed path (--dump-outputs)
# ------------------------------------------------------------------------------------------------
DUMP_LIMIT_BYTES = 64 << 20
DUMP_SEED = 20261018
READ_COLUMNS = ("sum_q", "status", "n_mid", "n_5p", "n_3p", "piece_begin", "n_pieces")
PIECE_COLUMNS = ("sum_q", "read", "start", "len", "repeat_len", "status")


def dump_outputs(out_dir: str, batch_ids, results, counters: np.ndarray, limit: int = DUMP_LIMIT_BYTES):
    """What a caller of the timed path receives for one step, as float64 .npy files (every value is an integer below
    2^53, so exactly):
      batch<j>_reads.npy   one row per read of batch j: row index, then READ_COLUMNS (tgsf_read_result)
      batch<j>_pieces.npy  one row per piece of batch j: row index, then PIECE_COLUMNS (tgsf_piece)
      counters.npy         the QC counter block the step added (tgsf_counters: DropInfo, histograms, tables)
    When the whole would exceed `limit` bytes, every per-row array keeps the same fraction of its rows, picked by a
    generator with a fixed seed; the row index column says which rows they are."""
    os.makedirs(out_dir, exist_ok=True)
    tables = {}
    for j, (reads, pieces) in zip(batch_ids, results):
        tables[f"batch{j}_reads"] = (reads, READ_COLUMNS)
        tables[f"batch{j}_pieces"] = (pieces, PIECE_COLUMNS)
    row_bytes = sum(len(a) * (len(cols) + 1) * 8 for a, cols in tables.values())
    frac = min(1.0, (limit - counters.size * 8) / max(row_bytes, 1))
    for name, (a, cols) in tables.items():
        rows = np.arange(len(a))
        if frac < 1.0:
            rng = np.random.default_rng([DUMP_SEED, len(a)])
            rows = np.sort(rng.choice(len(a), int(len(a) * frac), replace=False))
        out = np.empty((len(rows), len(cols) + 1), dtype=np.float64)
        out[:, 0] = rows
        for c, f in enumerate(cols, 1):
            out[:, c] = a[f][rows]
        np.save(os.path.join(out_dir, name + ".npy"), out)
    np.save(os.path.join(out_dir, "counters.npy"), counters.astype(np.float64))


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=int(os.environ.get("TGSF_BENCH_CONFIG", "2")),
                    help="BASELINE config index + 1 (2 = configs[1]); env TGSF_BENCH_CONFIG")
    ap.add_argument("--strong", action="store_true", default=os.environ.get("TGSF_BENCH_STRONG", "") not in ("", "0"),
                    help="strong scaling: one dataset dealt to the ranks, counter allreduce inside the step; env TGSF_BENCH_STRONG=1")
    ap.add_argument("--reads", type=int, default=0, help="reads in the dataset (0 = the config's full size)")
    ap.add_argument("--split", type=int, default=int(os.environ.get("TGSF_BENCH_SPLIT", "-1")),
                    help="weak mode: feed the dataset as at least this many batches (two are in flight at a time, so the "
                         "HBM-bound scans of one overlap the ALU-bound adapter scan of the other); default 2 for configs 2 and 3")
    ap.add_argument("--sample-reads", type=int, default=0, help="CPU reference: cap the reads per step (0 = whole dataset / time budget)")
    ap.add_argument("--slots", type=int, default=int(os.environ.get("TGSF_BENCH_SLOTS", "2")), help="batches in flight per context (1..4)")
    ap.add_argument("--e2e-chunks", type=int, default=16)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-fed measurement (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (per-read results, pieces, QC counters) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        raise SystemExit("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)
    if args.config not in CONFIG_READS:
        raise SystemExit(f"--config must be one of {sorted(CONFIG_READS)}")
    if args.split < 0:
        args.split = 2 if args.config in (2, 3) else 0
    if args.impl == "reference":
        return run_reference_arm(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    from tgsfilter_b200 import _capi, prepass
    from tgsfilter_b200.engine import FilterEngine
    from tgsfilter_b200.params import FilterParams
    from tgsfilter_b200.synth import ReadBatch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: tgsfilter_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)

    cfg, strong = args.config, args.strong
    n_total = args.reads or CONFIG_READS[cfg]
    read_type = CONFIG_TYPE[cfg]
    plan = plan_batches(cfg, n_total, world, rank, strong, args.split)

    # ---- resident batches + pinned host copies
    class B:
        pass
    batches = []
    for j, n, seed in plan:
        b = B()
        b.j, b.n_reads = j, n
        b.d_bases, b.d_quals, b.d_off, b.offsets, b.n_bases = gen_workload_gpu(cfg, n, seed, device)
        batches.append(b)
    local_bases = sum(b.n_bases for b in batches)
    local_reads = sum(b.n_reads for b in batches)
    want_e2e = not args.no_e2e
    for b in batches:
        if want_e2e or b is batches[0]:
            b.h_bases = torch.empty(b.n_bases, dtype=torch.uint8, pin_memory=True)
            b.h_quals = torch.empty(b.n_bases, dtype=torch.uint8, pin_memory=True)
            b.h_bases.copy_(b.d_bases[:b.n_bases])
            b.h_quals.copy_(b.d_quals[:b.n_bases])
    torch.cuda.synchronize()

    # ---- parameters exactly as the CLI would resolve them for this config (pre-pass on the first batch of the
    # dataset; in strong mode rank 0 owns that batch and broadcasts the decision)
    cli = CONFIG_CLI[cfg]
    p = FilterParams().apply_read_type(read_type)
    if "-q" in cli:
        p.min_q = float(cli[cli.index("-q") + 1])
    if "-Q" in cli:
        p.max_q = float(cli[cli.index("-Q") + 1])
    if "-p" in cli:
        p.min_repeat = int(cli[cli.index("-p") + 1])
    t0 = time.perf_counter()
    params = None
    if not strong or rank == 0:
        # the CLI samples the first 100 000 usable reads of the FILE: take the leading batches of the dataset
        # until they hold that many reads (batches that live on other ranks are regenerated here just for this)
        lead, have = [], 0
        full_plan = plan_batches(cfg, n_total, 1, 0, strong, args.split) if strong else plan
        by_j = {b.j: b for b in batches}
        for j, n, seed in full_plan:
            if have >= 100_000:
                break
            if j in by_j and hasattr(by_j[j], "h_bases"):
                b = by_j[j]
                lead.append((b.h_bases.numpy(), b.h_quals.numpy(), b.offsets))
            else:
                d_b, d_q, _, offs, tot = gen_workload_gpu(cfg, n, seed, device)
                lead.append((d_b[:tot].cpu().numpy(), d_q[:tot].cpu().numpy(), offs))
                del d_b, d_q
            have += n
        if len(lead) == 1:
            hb, hq, ho = lead[0]
        else:
            hb = np.concatenate([x[0] for x in lead])
            hq = np.concatenate([x[1] for x in lead])
            parts, base = [np.zeros(1, np.int64)], 0
            for x in lead:
                parts.append(x[2][1:] + base)
                base += int(x[2][-1])
            ho = np.concatenate(parts)
        host_batch = ReadBatch(hb, hq, ho.astype(np.uint64))
        params, _pre = prepass.run_prepass(host_batch, p, read_type, device=local_rank)
        del lead, hb, hq, host_batch
        torch.cuda.empty_cache()
    if strong and world > 1:
        box = [params]
        dist.broadcast_object_list(box, src=0)
        params = box[0]
    prepass_ms = (time.perf_counter() - t0) * 1e3
    params.n_slots = max(1, min(4, args.slots))
    n_slots = params.n_slots
    max_len = max(int(np.diff(b.offsets).max()) for b in batches)
    if max_len > 4_000_000:
        params.max_read_len = max_len
    eng = FilterEngine(params, device=local_rank)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # zero-copy view of the device counter block (allreduce operand)
    blk = scratch = None
    if world > 1:
        ptr, nwords = eng.counters_device_ptr()

        class _Blk:
            __cuda_array_interface__ = {"shape": (nwords,), "typestr": "<i8", "data": (ptr, False), "version": 3}
        blk = torch.as_tensor(_Blk(), device=device)
        scratch = torch.zeros(nwords, dtype=torch.int64, device=device)
        dist.all_reduce(scratch, op=dist.ReduceOp.SUM)  # NCCL sets its channels up lazily
        torch.cuda.synchronize()
    ar_ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))

    def step_resident(stage_acc, keep=None):
        """All local batches through the two slots; returns the step's device time in ms.  With a list as `keep`,
        the (per-read results, pieces) of every batch are appended to it in batch order."""
        spans = []
        inflight = 0

        def retire():
            res = eng.collect(want_results=keep is not None)
            if keep is not None:
                keep.append(res)
            spans.append(eng.last_span())
            st = eng.last_stage_ms()
            for k in stage_acc:
                stage_acc[k] += st[k]
        for b in batches:
            if inflight == n_slots:
                retire()
                inflight -= 1
            eng.submit_device(b.d_bases.data_ptr(), b.d_quals.data_ptr(), b.d_off.data_ptr(), b.n_reads, b.n_bases)
            inflight += 1
        while inflight:
            retire()
            inflight -= 1
        ms = max(e for _, e in spans) - min(s for s, _ in spans) if spans else 0.0
        if strong and world > 1:  # the QC counters of the dataset: one allreduce, inside the step
            ar_ev[0].record()
            scratch.copy_(blk)
            dist.all_reduce(scratch, op=dist.ReduceOp.SUM)
            ar_ev[1].record()
            ar_ev[1].synchronize()
            ms += ar_ev[0].elapsed_time(ar_ev[1])
        return ms

    # ---- sub-batches of the end-to-end path (host buffers; two slots -> copy / compute overlap)
    sub = []          # (batch, first base, reads, pinned offsets, bases, packed offset)
    pk_total = 0
    if want_e2e:
        per = max(1, args.e2e_chunks // len(batches))
        for b in batches:
            bounds = np.linspace(0, b.n_reads, per + 1).astype(np.int64)
            for a, c in zip(bounds[:-1], bounds[1:]):
                if c > a:
                    o = (b.offsets[a:c + 1] - b.offsets[a]).astype(np.uint64)
                    o_t = torch.from_numpy(o.view(np.int64)).pin_memory()
                    nb = int(b.offsets[c] - b.offsets[a])
                    sub.append((b, int(b.offsets[a]), int(c - a), o_t, nb, pk_total))
                    pk_total += ((nb + 3) // 4 + 63) // 64 * 64
        # pinned staging for the 2-bit packed bases of every sub-batch; the packing itself (tgsf_pack_bases, the
        # AVX2 packer src/TGSFilter.cpp uses) runs INSIDE the timed region on a pool of host threads
        h_packed = torch.empty(pk_total + 64, dtype=torch.uint8, pin_memory=True)
        torch.cuda.synchronize()
    d2h_bytes = 0

    import ctypes
    from concurrent.futures import ThreadPoolExecutor
    lib = _capi.load()
    host_cores = os.cpu_count() or 2
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    pack_threads = max(1, min(12, (host_cores - local_world) // max(local_world, 1)))
    if os.environ.get("TGSF_BENCH_PACK_THREADS"):
        pack_threads = max(1, int(os.environ["TGSF_BENCH_PACK_THREADS"]))
    pack_seconds = [0.0]
    pool = ThreadPoolExecutor(pack_threads)

    def pack_sub(b, s0, nb, po):
        """bases[s0 : s0 + nb] -> 2-bit codes at h_packed[po ...], in pack_threads ranges that are multiples of 32 bases
        (the synthetic bases are pure upper-case ACGT: a non-empty exception list is an error here)."""
        src, dst = b.h_bases.data_ptr() + s0, h_packed.data_ptr() + po
        per = ((nb + pack_threads - 1) // pack_threads + 31) // 32 * 32

        def one(lo):
            ne = ctypes.c_uint64(0)
            n = min(per, nb - lo)
            rc = lib.tgsf_pack_bases(src + lo, n, dst + lo // 4, None, None, 0, ctypes.byref(ne))
            return rc, ne.value
        tq = time.perf_counter()
        for rc, ne in pool.map(one, range(0, nb, per)):
            if rc != 0 or ne:
                raise RuntimeError(f"tgsf_pack_bases: status {rc}, {ne} exceptions")
        pack_seconds[0] += time.perf_counter() - tq

    adaptive_stats = {"packed": 0, "bytes": 0}

    def run_e2e_adaptive(steps):
        """The host-fed stream of `steps` passes as ONE sequence of sub-batches.  A packer thread (driving the pool above)
        runs ahead of the submit loop and packs sub-batch after sub-batch; the submit loop takes the 2-bit version when
        it is ready (1.25 B/base over PCIe) and sends the plain bytes (2 B/base, no host work) when the packer has not
        got there: with cores to spare everything goes packed, with few cores per GPU the two feeds mix by themselves."""
        nonlocal d2h_bytes
        n, total = len(sub), steps * len(sub)
        state = {}                      # global index -> 1 packing, 2 packed, 3 sent as bytes
        lock = threading.Condition()
        pos = [0]                       # sub-batches the submit loop has decided so far
        ahead_max = max(n - 3, 1)       # the staging region of sub-batch i is reused every n items: stay behind its last use

        def packer():
            g = 0
            while True:
                with lock:
                    g = max(g, pos[0] + 2)  # two sub-batches of lead so that the result is ready when it is wanted
                    while g < total and g - pos[0] > ahead_max:
                        lock.wait()
                        g = max(g, pos[0] + 2)
                    if g >= total:
                        return
                    state[g] = 1
                b, s0, nr, o_t, nb, po = sub[g % n]
                pack_sub(b, s0, nb, po)
                with lock:
                    state[g] = 2
                    lock.notify_all()
                g += 1
        th = threading.Thread(target=packer)
        th.start()
        d2h = 0
        inflight = 0
        for g in range(total):
            b, s0, nr, o_t, nb, po = sub[g % n]
            with lock:
                while state.get(g) == 1:
                    lock.wait()
                st = state.get(g, 0)
                if st == 0:
                    state[g] = 3
                pos[0] = g + 1
                lock.notify_all()
            if inflight == n_slots:
                r, pcs = eng.collect()
                d2h += r.nbytes + pcs.nbytes
                inflight -= 1
            if st == 2:
                eng.submit_packed_raw(h_packed.data_ptr() + po, b.h_quals.data_ptr() + s0, o_t.data_ptr(), nr)
                adaptive_stats["packed"] += nb
            else:
                eng.submit_raw(b.h_bases.data_ptr() + s0, b.h_quals.data_ptr() + s0, o_t.data_ptr(), nr)
                adaptive_stats["bytes"] += nb
            inflight += 1
        while inflight:
            r, pcs = eng.collect()
            d2h += r.nbytes + pcs.nbytes
            inflight -= 1
        th.join()
        d2h_bytes = d2h // max(steps, 1)

    def step_e2e_packed():  # warm-up form: one pass, everything packed
        inflight = 0
        for b, s0, nr, o_t, nb, po in sub:
            pack_sub(b, s0, nb, po)
            if inflight == n_slots:
                eng.collect()
                inflight -= 1
            eng.submit_packed_raw(h_packed.data_ptr() + po, b.h_quals.data_ptr() + s0, o_t.data_ptr(), nr)
            inflight += 1
        while inflight:
            eng.collect()
            inflight -= 1

    def step_e2e_bytes():
        inflight = 0
        for b, s0, nr, o_t, nb, po in sub:
            if inflight == n_slots:
                eng.collect()
                inflight -= 1
            eng.submit_raw(b.h_bases.data_ptr() + s0, b.h_quals.data_ptr() + s0, o_t.data_ptr(), nr)
            inflight += 1
        while inflight:
            eng.collect()
            inflight -= 1

    def timed_wall(fn, steps):
        barrier()
        e0 = time.perf_counter()
        for _ in range(steps):
            fn()
        barrier()
        t = torch.tensor([time.perf_counter() - e0], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- warm-up
    dummy = {k: 0.0 for k in _capi.STAGE_NAMES}
    for _ in range(args.warmup):
        step_resident(dummy)
    if want_e2e:
        step_e2e_bytes()
        step_e2e_packed()
    eng.reset_counters()

    # ---- timed: resident
    launches0 = eng.launch_count()
    stage_sum = {k: 0.0 for k in _capi.STAGE_NAMES}
    dump = args.dump_outputs is not None and rank == 0
    last_results, cnt_before_last = [], None
    barrier()
    with ClockSampler(local_rank) as clk:
        wall0 = time.perf_counter()
        dev_ms = 0.0
        for i in range(args.steps):
            last = dump and i == args.steps - 1
            if last:  # the counters accumulate over the steps: the last step's are the difference
                cnt_before_last = eng.counters().flat.copy()
            dev_ms += step_resident(stage_sum, last_results if last else None)
        barrier()
        wall_ms = (time.perf_counter() - wall0) * 1e3
    launches = eng.launch_count() - launches0
    clocks = clk.summary()
    cnt = eng.counters()
    if dump:
        dump_outputs(args.dump_outputs, [b.j for b in batches], last_results, cnt.flat - cnt_before_last)
        del last_results
    # per-kernel times for the rooflines: one more pass with ONE batch in flight (stages of batches that overlap in
    # the two slots stretch each other, so their event times are not kernel times)
    # ... and with the end-window kernels on the batch's main stream (TGSF_FORK_ENDS=0: a second context), because the
    # timed path runs them NEXT TO the middle scan, whose stage time would otherwise include them
    stage_serial = {k: 0.0 for k in _capi.STAGE_NAMES}
    serial_ms = 0.0
    os.environ["TGSF_FORK_ENDS"] = "0"
    try:
        eng_prof = FilterEngine(params, device=local_rank)
    finally:
        del os.environ["TGSF_FORK_ENDS"]
    for it in range(2):  # first pass: warm-up (allocations)
        for k in stage_serial:
            stage_serial[k] = 0.0
        serial_ms = 0.0
        for b in batches:
            eng_prof.submit_device(b.d_bases.data_ptr(), b.d_quals.data_ptr(), b.d_off.data_ptr(), b.n_reads, b.n_bases)
            eng_prof.collect(want_results=False)
            st = eng_prof.last_stage_ms()
            serial_ms += eng_prof.last_timing()[0]
            for k in stage_serial:
                stage_serial[k] += st[k]
    eng_prof.close()
    t_dev = torch.tensor([dev_ms], dtype=torch.float64, device=device)
    t_bases = torch.tensor([float(local_bases)], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t_dev, op=dist.ReduceOp.MAX)
        dist.all_reduce(t_bases, op=dist.ReduceOp.SUM)
    dev_ms_max = float(t_dev.item())
    total_bases = float(t_bases.item())

    # ---- timed: end to end (host buffers)
    e2e_value = e2e_packed_value = None
    pack_gbs = None
    if want_e2e:
        e2e_s = timed_wall(step_e2e_bytes, args.steps)
        pack_seconds[0] = 0.0
        adaptive_stats["packed"] = adaptive_stats["bytes"] = 0
        e2e_packed_s = timed_wall(lambda: run_e2e_adaptive(args.steps), 1)
        pack_s_per_step = pack_seconds[0] / args.steps
        packed_frac = adaptive_stats["packed"] / max(1, adaptive_stats["packed"] + adaptive_stats["bytes"])
        e2e_value = total_bases * args.steps / e2e_s / 1e9
        e2e_packed_value = total_bases * args.steps / e2e_packed_s / 1e9
        # host packer speed (one thread), for context
        b0 = batches[0]
        nb_probe = min(b0.n_bases, 256 << 20)
        probe_out = np.empty(nb_probe // 4 + 16, dtype=np.uint8)
        ne = ctypes.c_uint64(0)
        tp0 = time.perf_counter()
        lib.tgsf_pack_bases(b0.h_bases.data_ptr(), nb_probe, probe_out.ctypes.data, None, None, 0, ctypes.byref(ne))
        pack_gbs = nb_probe / (time.perf_counter() - tp0) / 1e9

    # ---- final counter allreduce over NVLink (weak mode: outside the timed region; reported)
    allreduce_ms = None
    if world > 1:
        torch.cuda.synchronize()
        a0 = time.perf_counter()
        dist.all_reduce(blk, op=dist.ReduceOp.SUM)
        torch.cuda.synchronize()
        allreduce_ms = (time.perf_counter() - a0) * 1e3

    value = total_bases * args.steps / (dev_ms_max / 1e3) / 1e9

    # ---- rooflines (this rank's batches)
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
    lens = np.concatenate([np.diff(b.offsets) for b in batches])
    drop = cnt.drop_info
    E = params.end_len
    word_cols_all = 0
    for a in params.adapters:
        q = len(a)
        nw = (q + 63) // 64
        mid = lens - 2 * E
        word_cols_all += nw * int(mid[mid >= q].sum())
    stage_sum = {k: v * args.steps for k, v in stage_serial.items()}  # (the code below divides by steps)
    active_frac = 1.0 - (int(drop[1]) / args.steps) / max(1, local_bases)
    word_cols = word_cols_all * active_frac
    mid_ms = stage_sum["mid_scan"] / args.steps
    sm_clock = clocks.get("sm_mhz") or float(peaks.get("sm_max_mhz", 1965.0))
    int_peak = 148 * 128 * sm_clock * 1e6 / 1e12  # T int32-op/s at the clock seen under load
    achieved_int = word_cols * 34 / (mid_ms / 1e3) / 1e12 if mid_ms > 0 else 0.0
    raw_ms = stage_sum["raw_scan"] / args.steps
    clean_ms = stage_sum["clean"] / args.steps
    k1_gbs = 2 * local_bases / (raw_ms / 1e3) / 1e9 if raw_ms > 0 else 0.0
    step_ms = dev_ms / args.steps if dev_ms else 0.0
    stage_total = sum(stage_sum.values()) / args.steps
    kept_bases = local_bases - int(drop[1]) // args.steps  # bases entering the clean pass (upper bound)
    clean_gbs = 2 * kept_bases / (clean_ms / 1e3) / 1e9 if clean_ms > 0 else 0.0
    kmer_ms = stage_sum["kmer"] / args.steps
    share = (lambda ms: ms / stage_total if stage_total else None)
    rl_mid = {"kernel": "k_mid_scan (K3 Myers HW scan, middle windows)", "bound": "int_alu",
              "achieved": achieved_int, "peak": int_peak, "unit": "Tint32op/s",
              "frac": achieved_int / int_peak if int_peak else None, "traffic": None,
              "work": "34 int32-op equivalents per 64-bit word-column (SURVEY.md §8d), "
                      f"{word_cols:.4g} word-columns per launch set",
              "peak_def": f"148 SMs x 128 lanes x {sm_clock:.0f} MHz (median SM clock under load)",
              "note": "ALU-pipe bound (ncu: pipe_alu ~92 % busy); logic ops cannot use the FMA pipe, so "
                      "the 128-lane peak is not reachable: see DESIGN.md §4",
              "ms": mid_ms, "share_of_step": share(mid_ms)}
    rl_raw = {"kernel": "k_scan_tiles_dyn raw pass (K1)", "bound": "hbm", "achieved": k1_gbs, "peak": hbm_peak,
              "unit": "GB/s", "frac": k1_gbs / hbm_peak, "traffic": None, "peak_source": hbm_src,
              "work": "2 B per input base", "ms": raw_ms, "share_of_step": share(raw_ms)}
    rl_clean = {"kernel": "k_scan_tiles_dyn clean pass (K1)", "bound": "hbm", "achieved": clean_gbs,
                "peak": hbm_peak, "unit": "GB/s", "frac": clean_gbs / hbm_peak, "traffic": None,
                "peak_source": hbm_src, "work": "2 B per kept base (upper bound: bases of reads passing -q/-Q)",
                "ms": clean_ms, "share_of_step": share(clean_ms)}
    # K4: no memory roofline applies (1 B/base of HBM traffic is < 5 % of peak); the kernel is bound by instruction
    # issue.  Peak = inserts/s if every issue slot of the GPU issued one of the kernel's own instructions each cycle:
    # 4 slots x 148 SMs x clock / (warp-instructions per insert, from the ncu capture in profiles/).
    kmer_inserts = kept_bases / (kmer_ms / 1e3) / 1e9 if kmer_ms > 0 else 0.0
    k4_prof = {}
    try:
        with open(os.path.join(ROOT, "profiles", "r2_kmer_issue.json")) as f:
            k4_prof = json.load(f)
    except Exception:
        pass
    wi = k4_prof.get("warp_instructions_per_insert")
    kmer_peak = 4 * 148 * sm_clock * 1e6 / wi / 1e9 if wi else None
    rl_kmer = {"kernel": "k_kmer_tag16 (K4, k <= 12: owner-byte dense round + position-tag list rounds in shared memory, "
                         "2 CTAs/SM, producer warps; k = 13..16: the same with u16 entries; pieces > 65 kb: k_kmer_smem / hash; k > 16: hash)",
               "bound": "issue", "achieved": kmer_inserts, "peak": kmer_peak, "unit": "Ginserts/s",
               "frac": kmer_inserts / kmer_peak if kmer_peak else None, "traffic": None,
               "work": "1 set insert per kept base",
               "peak_def": (f"4 issue slots x 148 SMs x {sm_clock:.0f} MHz / {wi} warp-instructions per insert "
                            f"(ncu, {k4_prof.get('source')})") if wi else "no ncu capture committed",
               "hbm_view": {"achieved_gbs": kmer_inserts, "frac_of_hbm": kmer_inserts / hbm_peak,
                            "work": "1 B per kept base (SURVEY.md §8d)"},
               "ms": kmer_ms, "share_of_step": share(kmer_ms)}
    # measured DRAM traffic per launch (one ncu --set full capture of this same command, committed under profiles/;
    # the launches of the step's FIRST batch); only valid for the workload it was captured on
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            tr = json.load(f)
        b0 = batches[0]
        if tr.get("config") == cfg and tr.get("reads_per_launch") == b0.n_reads and tr.get("seed") == plan[0][2]:
            lens0 = np.diff(b0.offsets)
            mid0 = lens0 - 2 * E
            qmin = min(len(a) for a in params.adapters)
            rl_mid["traffic"] = tr["k_mid_scan"]["dram_bytes"]
            # 1 B per middle-window column of the reads that pass -q/-Q; one pass serves both adapters
            rl_mid["algorithmic_bytes"] = int(int(mid0[mid0 >= qmin].sum()) * active_frac)
            rl_raw["traffic"] = tr["k_scan_tiles_raw"]["dram_bytes"]
            rl_raw["algorithmic_bytes"] = 2 * b0.n_bases
            rl_clean["traffic"] = tr["k_scan_tiles_clean"]["dram_bytes"]
            for r in (rl_mid, rl_raw, rl_clean):
                r["traffic_note"] = "per launch of the step's first batch (%d reads), ncu --set full, %s" % (b0.n_reads, tr.get("source"))
    except Exception:
        pass
    by_stage = {"mid_scan": rl_mid, "raw_scan": rl_raw, "clean": rl_clean, "kmer": rl_kmer}
    dominant = max(by_stage, key=lambda k: by_stage[k]["ms"])
    roofline = by_stage[dominant]
    roofline_kernels = {k: v for k, v in by_stage.items() if k != dominant and v["ms"] > 0}
    roofline_kernels["stage_ms_per_step"] = {k: v / args.steps for k, v in stage_sum.items()}
    roofline_kernels["stage_ms_note"] = ("from one extra pass with a single batch in flight and every kernel on the batch's "
                                         f"main stream (sum over the batches: {serial_ms:.3f} ms); the timed steps keep two "
                                         "batches in flight and run the end-window search next to the middle scan")

    line = {
        "metric": "filtered Gbases/s", "value": value, "unit": "Gbases/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms_max / args.steps,
        "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "u8/u64",
        "data": "synthetic",
        "config": static_config(cfg, n_total, strong),
        "workload_detail": {"reads_this_rank": local_reads, "bases_this_rank": local_bases, "bases_all_ranks": int(total_bases),
                            "batches_this_rank": len(batches), "adapters": [a.decode() for a in params.adapters],
                            "head_trim": params.head_trim, "tail_trim": params.tail_trim,
                            "timing": "device clock: first kernel start to last kernel end of the step's batches "
                                      "(+ counter allreduce in strong mode), max over ranks"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "roofline_kernels": roofline_kernels,
        "wall_ms_per_step_resident": wall_ms / args.steps,
        "prepass_ms": prepass_ms,
        "allreduce_ms": allreduce_ms,
        "drop_info_per_step": [int(x) // args.steps for x in drop],
    }
    if want_e2e:
        nsub = len(sub)
        e2e_b = {"value": e2e_value, "unit": "Gbases/s",
                 "h2d_bytes_per_step": int(2 * local_bases + 8 * (local_reads + nsub)) * world,
                 "d2h_bytes_per_step": int(d2h_bytes) * world, "chunks": nsub, "slots": 2,
                 "input_format": "byte bases + Phred bytes + offsets in pinned host memory (tgsf_submit): nothing to prepare "
                                 "on the host, 2 B/base over PCIe"}
        h2d_adaptive = (adaptive_stats["packed"] * 1.25 + adaptive_stats["bytes"] * 2.0) / args.steps + 8 * (local_reads + nsub)
        e2e_p = {"value": e2e_packed_value, "unit": "Gbases/s",
                 "h2d_bytes_per_step": int(h2d_adaptive) * world,
                 "d2h_bytes_per_step": int(d2h_bytes) * world, "chunks": nsub, "slots": n_slots,
                 "input_format": "byte bases + Phred bytes + offsets in pinned host memory; a packer thread driving "
                                 f"{pack_threads} host threads per rank packs the bases to 2 bits INSIDE the timed region "
                                 "(tgsf_pack_bases, the packer src/TGSFilter.cpp uses), running ahead of the submit loop; a "
                                 "sub-batch goes out packed (tgsf_submit_packed, 1.25 B/base over PCIe) when its packed copy is "
                                 "ready and as plain bytes (tgsf_submit, 2 B/base) when the packer has not got there",
                 "packed_fraction_of_bases_this_rank": packed_frac,
                 "pack_threads_per_rank": pack_threads, "host_cores": host_cores,
                 "host_pack_ms_per_step": pack_s_per_step * 1e3, "wall_ms_per_step": e2e_packed_s / args.steps * 1e3,
                 "host_pack_gbases_per_s_per_thread": pack_gbs}
        # the host picks the feed that is faster on the box it runs on: packing pays while there are host cores to spare
        best, other = (e2e_p, e2e_b) if e2e_packed_value >= e2e_value else (e2e_b, e2e_p)
        line["e2e"] = best
        line["e2e_other_feed"] = other

    if rank == 0 and world == 1 and not args.no_cpu_baseline and os.path.exists(REF_CLI):
        # the reference on the same dataset, once (bounded: at most ~5 Gbases, ~2 Gbases with -p)
        tmpdir = tempfile.mkdtemp(prefix="tgsf_ref_", dir=shm_dir())
        try:
            cap_bases = 2.0e9 if "-p" in cli else 5.0e9
            mean_len = local_bases / max(local_reads, 1)
            cap_reads = 0 if local_bases <= cap_bases else int(cap_bases / mean_len)
            fq_path = os.path.join(tmpdir, "sample.fq")
            del batches[1:]
            r_reads, r_bases, gen = write_reference_fastq(cfg, plan, fq_path, args.sample_reads or cap_reads)
            threads = ref_threads()
            secs = run_reference_once(cfg, fq_path, threads)
            whole = r_reads == local_reads
            line["cpu_baseline"] = {"value": r_bases / secs / 1e9, "unit": "Gbases/s", "cores": threads, "kind": "reference",
                                    "sample": f"{'the whole dataset' if whole else 'the first ' + str(r_reads) + ' reads'} "
                                              f"({r_reads} reads, {r_bases} bases) through the unmodified reference CLI, "
                                              f"-t {threads}, FASTQ on tmpfs, one run of {secs:.1f} s"}
        except Exception as exc:  # keep the GPU line even if the CPU leg fails
            line["cpu_baseline"] = {"value": None, "unit": "Gbases/s", "cores": 0, "kind": "reference",
                                    "sample": f"failed: {exc}"}
        finally:
            shutil.rmtree(tmpdir, ignore_errors=True)
    eng.close()
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())

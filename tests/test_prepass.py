"""The pre-pass (tgsf_prepass: k_base_content and k_lib_search) against the CPU oracle at the shapes the CLI gives it,
and the CLI's pre-pass decisions (-A) against an expectation built from the oracle without the GPU.

The CLI samples up to max(-n, -N) reads (100 000 by default) and cuts checkLen = max(-E, -e, 100) bases from each end
(T.cpp:897-904, 949-982), so both kernels see any row count and any row length.  Every comparison is exact.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import oracle_lib
from tgsfilter_b200 import _capi, prepass, synth
from tgsfilter_b200.params import ADAPTER_LIB, FilterParams, rev_comp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "src", "tgsfilter")
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
PRE_ROWS_PER_CTA = 8  # k_base_content: one row per warp, 8 warps per CTA, at most 4 CTAs per SM in one pass
RES_THREADS = 128     # k_lib_search: one row per thread, at most 4 CTAs of 128 threads per SM in one pass


def _sm_count() -> int:
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _min_k(q: int, min_sim: float) -> int:
    """k of the library search: minSim clamped to 0.9, then int((1 - minSim) * qLen) + 1 in float32 (T.cpp:1151-1161)."""
    s = np.float32(min_sim)
    if float(s) < 0.9:
        s = np.float32(0.9)
    return int((np.float32(1) - s) * np.float32(q)) + 1


def _oracle_search(ends: np.ndarray, lib, min_sim: float) -> np.ndarray:
    """oracle_lib.adapter_search over chunks of rows on every core (ctypes releases the GIL), maps summed."""
    oracle_lib.load()
    workers = os.cpu_count() or 1
    step = max(1, -(-ends.shape[0] // (4 * workers)))
    chunks = [ends[i:i + step] for i in range(0, ends.shape[0], step)]
    if len(chunks) <= 1:
        return oracle_lib.adapter_search(ends, lib, min_sim)
    with ThreadPoolExecutor(workers) as ex:
        return sum(ex.map(lambda c: oracle_lib.adapter_search(c, lib, min_sim), chunks))


# ---- argument checks (no GPU) ------------------------------------------------------------------
def _call_prepass(*, ends=True, row_len=8, lib=(b"ACGTACGT",), lib_len=None, n_lib=None, counts=(True, True),
                  maps=(True, True)):
    lib_so = _capi.load()
    rows = np.zeros((2, max(row_len, 1)), dtype=np.uint8)
    cnt = np.zeros((max(row_len, 1), 4), dtype=np.int32)
    m = np.zeros(2048, dtype=np.int64)
    seqs = lens = None
    if lib is not None:
        seqs = (C.c_char_p * max(len(lib), 1))(*lib)
        lens = (C.c_int32 * max(len(lib), 1))(*([len(a) for a in lib] if lib_len is None else lib_len))
        seqs, lens = C.cast(seqs, C.POINTER(C.c_char_p)), C.cast(lens, C.POINTER(C.c_int32))
    rc = lib_so.tgsf_prepass(0, rows.ctypes.data if ends else None, rows.ctypes.data if ends else None, 2, row_len,
                             seqs, lens, len(lib or ()) if n_lib is None else n_lib, 0.9,
                             cnt.ctypes.data if counts[0] else None, cnt.ctypes.data if counts[1] else None,
                             m.ctypes.data if maps[0] else None, m.ctypes.data if maps[1] else None)
    return rc, lib_so.tgsf_last_error().decode()


@pytest.mark.parametrize("case", [
    dict(row_len=0), dict(ends=False), dict(counts=(False, True)), dict(counts=(True, False)),
    dict(n_lib=0), dict(n_lib=1025), dict(maps=(False, True)), dict(maps=(True, False)),
    dict(lib=(b"",)), dict(lib=(b"A" * 2049,)), dict(lib=(b"ACGT", b"A" * 2049)), dict(lib=(b"ACGT",), lib_len=[-1]),
], ids=["row_len_0", "no_ends", "no_counts5", "no_counts3", "n_lib_0", "n_lib_1025", "no_map5", "no_map3",
        "empty_adapter", "adapter_2049", "second_adapter_2049", "negative_length"])
def test_prepass_rejects_bad_arguments_before_touching_the_gpu(case):
    """Without a GPU every call below would fail with TGSF_ERR_CUDA if it reached the device first."""
    rc, err = _call_prepass(**case)
    assert rc == _capi.TGSF_ERR_INVALID, (rc, err)
    assert err.startswith("prepass"), err


def _skewed_counts(n: int, check_len: int, rng) -> np.ndarray:
    """[check_len][4] table of n sampled ends whose first 30 columns are A-rich, fading towards column 30."""
    p_a = np.full(check_len, 0.25)
    p_a[:30] = 0.25 + 0.6 * (30 - np.arange(30)) / 30
    a = rng.binomial(n, p_a)
    out = np.zeros((check_len, 4), dtype=np.int32)
    out[:, 0] = a
    for i in range(check_len):
        out[i, 1:] = rng.multinomial(n - a[i], [1 / 3] * 3)
    return out


@pytest.mark.parametrize("n,end_bias", [(100_000, 1.0), (30_000, 0.3), (1500, 1.0), (300, 0.3), (7, 1.0)])
def test_base_content_trim_python_matches_the_oracle(n, end_bias):
    """The CLI tests below build their expectation with prepass.base_content_trim; it must decide like the oracle's
    restatement of CheckBaseContent, float32 maxDiff included."""
    rng = np.random.default_rng(n)
    trims = []
    for check_len in (100, 150, 3500):
        t = _skewed_counts(n, check_len, rng)
        trims.append(prepass.base_content_trim(t, n, end_bias))
        assert trims[-1] == oracle_lib.base_content_trim(t, n, end_bias)
    assert any(trims)


# ---- k_base_content ----------------------------------------------------------------------------
COUNT_ROW_LENS = [1, 31, 32, 33, 100, 150, 3072, 3073, 4000, 8192, 8193, 12000]


@pytest.mark.gpu
@pytest.mark.parametrize("n_kind", ["0", "1", "7", "400", "grid"])
@pytest.mark.parametrize("row_len", COUNT_ROW_LENS)
def test_base_content_counts_vs_oracle(row_len, n_kind):
    """Counts-only call (the CLI's -a path) on uniformly random bytes 0..255: lower case, N, IUPAC, 0x00 and >= 0x80
    must not count.  'grid' is more rows than k_base_content covers in one grid-stride pass."""
    sms = _sm_count()
    n = 4 * sms * PRE_ROWS_PER_CTA + 5 if n_kind == "grid" else int(n_kind)
    rng = np.random.default_rng(row_len * 10 + len(n_kind))
    e5 = rng.integers(0, 256, (n, row_len), dtype=np.uint8)
    e3 = rng.integers(0, 256, (n, row_len), dtype=np.uint8)
    c5, c3, m5, m3 = prepass.device_prepass(e5, e3, None, 0.9)
    o5, o3 = oracle_lib.base_content_counts(e5), oracle_lib.base_content_counts(e3)
    if n * row_len >= 256:  # the fixture can tell a zero table and swapped outputs from the right answer
        assert o5.any() and not np.array_equal(o5, o3)
    assert np.array_equal(c5, o5)
    assert np.array_equal(c3, o3)
    assert m5 is None and m3 is None


# ---- k_lib_search -----------------------------------------------------------------------------
def _edit(seq: np.ndarray, e: int, rng) -> np.ndarray:
    """seq with e edits (substitution by another base, deletion, insertion) at distinct positions."""
    out = list(seq)
    for p in sorted(rng.choice(len(seq), size=min(e, len(seq)), replace=False).tolist(), reverse=True):
        op = int(rng.integers(3))
        if op == 0:
            out[p] = int(ACGT[(int(np.nonzero(ACGT == out[p])[0][0]) + int(rng.integers(1, 4))) % 4])
        elif op == 1:
            del out[p]
        else:
            out.insert(p, int(ACGT[rng.integers(4)]))
    return np.array(out, dtype=np.uint8)


def _put(row: np.ndarray, seq: np.ndarray, start: int) -> None:
    """row[start:start + len(seq)] = seq, clipped to the row (start may be negative)."""
    lo, hi = max(start, 0), min(start + len(seq), len(row))
    if lo < hi:
        row[lo:hi] = seq[lo - start:hi - start]


def _planted_rows(n: int, row_len: int, lib, min_sims, seed: int, frac: float = 0.5):
    """n random ACGT rows; about frac of them carry a library adapter (or its reverse complement) at column 0, ending at
    the last column, running off the row end by minK - 1, minK or minK + 1 bases, or edited minK - 1, minK or minK + 1
    times, with minK that of one of min_sims.  Adapters longer than the row are cut to it.  Returns (rows, plants):
    plants = [(row, adapter index)] of the forward adapters that were cut or edited."""
    rng = np.random.default_rng(seed)
    rows = ACGT[rng.integers(0, 4, (n, row_len), dtype=np.uint8)]
    lib_arr = [np.frombuffer(a, dtype=np.uint8) for a in lib]
    rc_arr = [np.frombuffer(rev_comp(a), dtype=np.uint8) for a in lib]
    planted = np.nonzero(rng.random(n) < frac)[0]
    a_idx = rng.integers(0, len(lib), n)
    rc = rng.random(n) < 0.5
    kind = rng.integers(0, 4, n)
    ms = rng.integers(0, len(min_sims), n)
    delta = rng.integers(-1, 2, n)
    where = rng.random(n)
    plants = []
    for r in planted.tolist():
        a = int(a_idx[r])
        seq = rc_arr[a] if rc[r] else lib_arr[a]
        e = max(0, _min_k(len(seq), min_sims[ms[r]]) + int(delta[r]))
        k = int(kind[r])
        if k == 0:
            _put(rows[r], seq, 0)
        elif k == 1:
            _put(rows[r], seq, row_len - len(seq))
        elif k == 2:
            _put(rows[r], seq, row_len - len(seq) + max(e, 1))
        else:
            seq = _edit(seq, e, rng)
            _put(rows[r], seq, int(where[r] * max(row_len - len(seq) + 1, 1)))
        if k >= 2 and not rc[r]:
            plants.append((r, a))
    return np.ascontiguousarray(rows), plants


def _assert_plants_straddle_min_k(rows, plants, lib, min_sim, limit=400):
    """Some planted rows align with d == minK (a hit) and some with d == minK + 1 (a miss)."""
    ds = set()
    for r, a in plants[:limit]:
        d = oracle_lib.align_hw(lib[a], rows[r].tobytes(), -1)[0]["edit_distance"]
        ds.add(d - _min_k(len(lib[a]), min_sim))
        if {0, 1} <= ds:
            return
    raise AssertionError(f"no plant on both sides of minK at min_sim {min_sim}: d - minK in {sorted(ds)}")


LIB_MIN_SIMS = [0.5, 0.9, 0.93, 0.99, 1.0]
_rows_cache: dict = {}
_oracle_cache: dict = {}


def _lib_case(shape: str, row_len: int):
    key = (shape, row_len)
    if key not in _rows_cache:
        n = max(100_000, 4 * _sm_count() * RES_THREADS + 1) if shape == "grid" else int(shape)
        e5, p5 = _planted_rows(n, row_len, ADAPTER_LIB, LIB_MIN_SIMS, seed=row_len * 2 + 1)
        e3, p3 = _planted_rows(n, row_len, ADAPTER_LIB, LIB_MIN_SIMS, seed=row_len * 2 + 2)
        _rows_cache.clear()  # one shape at a time: the 100 000-row cases are large
        _rows_cache[key] = (e5, p5, e3, p3)
    return _rows_cache[key]


def _oracle_maps(key, ends, lib, min_sim):
    """The oracle's maps depend on min_sim only through the per-adapter k: cases with the same k share them."""
    k = (key, tuple(_min_k(len(a), min_sim) for a in lib))
    if k not in _oracle_cache:
        _oracle_cache[k] = _oracle_search(ends, lib, min_sim)
    return _oracle_cache[k]


@pytest.mark.gpu
@pytest.mark.parametrize("min_sim", LIB_MIN_SIMS)
@pytest.mark.parametrize("shape,row_len", [("grid", 100), ("grid", 150), ("2000", 1000), ("2000", 4000)])
def test_library_search_vs_oracle(shape, row_len, min_sim):
    """The 22-adapter library search.  'grid' is more sampled ends than k_lib_search covers in one grid-stride pass
    (4 CTAs x 128 threads per SM): the CLI's default 100 000-read sample on a B200.  min_sim 0.5 runs as 0.9."""
    e5, p5, e3, p3 = _lib_case(shape, row_len)
    n = e5.shape[0]
    if shape == "grid":
        assert n > 4 * _sm_count() * RES_THREADS
    c5, c3, m5, m3 = prepass.device_prepass(e5, e3, ADAPTER_LIB, min_sim)
    o5 = _oracle_maps((shape, row_len, 5), e5, ADAPTER_LIB, min_sim)
    o3 = _oracle_maps((shape, row_len, 3), e3, ADAPTER_LIB, min_sim)
    assert o5.any() and o3.any() and not np.array_equal(o5, o3)
    _assert_plants_straddle_min_k(e5, p5, ADAPTER_LIB, min_sim)
    _assert_plants_straddle_min_k(e3, p3, ADAPTER_LIB, min_sim)
    assert np.array_equal(m5, o5), np.nonzero(m5 != o5)
    assert np.array_equal(m3, o3), np.nonzero(m3 != o3)
    assert np.array_equal(c5, oracle_lib.base_content_counts(e5))
    assert np.array_equal(c3, oracle_lib.base_content_counts(e3))


def _random_lib(lengths, seed):
    rng = np.random.default_rng(seed)
    return [ACGT[rng.integers(0, 4, q, dtype=np.uint8)].tobytes() for q in lengths]


# Myers word counts: 1 (1-64 bp), 2 (65-128), 3 (129-192), 4 (193-256), 8 (257-512), 16 (513-1024), 32 (1025-2048)
ANY_LIB_CASES = {
    "short": (120, 3000, [1, 22, 63, 64, 65, 128, 129], (0.9, 0.95)),  # 128 and 129 are longer than the row
    "long": (1900, 200, [200, 256, 257, 512, 1024, 2048], (0.9,)),      # 2048 is longer than the row
    "lib1024": (150, 256, list(np.random.default_rng(7).integers(1, 130, 1024)), (0.9, 0.97)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(ANY_LIB_CASES))
def test_any_library_vs_oracle(case):
    """tgsf_prepass with a library of the caller's: every Myers word count, adapters longer than the row, and the
    largest library the ABI takes (1024 adapters)."""
    row_len, n, lengths, min_sims = ANY_LIB_CASES[case]
    lib = _random_lib([int(q) for q in lengths], seed=len(lengths) + row_len)
    e5, p5 = _planted_rows(n, row_len, lib, min_sims, seed=11 + row_len, frac=0.8)
    e3, p3 = _planted_rows(n, row_len, lib, min_sims, seed=12 + row_len, frac=0.8)
    for min_sim in min_sims:
        c5, c3, m5, m3 = prepass.device_prepass(e5, e3, lib, min_sim)
        o5, o3 = _oracle_search(e5, lib, min_sim), _oracle_search(e3, lib, min_sim)
        assert o5.any() and o3.any() and not np.array_equal(o5, o3)
        _assert_plants_straddle_min_k(e5, p5, lib, min_sim)
        assert np.array_equal(m5, o5), (min_sim, np.nonzero(m5 != o5))
        assert np.array_equal(m3, o3), (min_sim, np.nonzero(m3 != o3))
        if min_sim == 0.9 and case == "short":  # every adapter hits somewhere, the two longer than the row included
            assert (o5 > 0).all()
        if min_sim == 0.9 and case == "long":
            assert o5[-1] > 0 and len(lib[-1]) > row_len
    assert np.array_equal(c5, oracle_lib.base_content_counts(e5))


# ---- the CLI's pre-pass ------------------------------------------------------------------------
SKEW = 30  # bases at each read end with a composition that fades towards the middle


def _cli_reads(n: int, lo: int, hi: int, seed: int, ad5=None, ad3=None, frac=0.4):
    """n reads of lo..hi bases (FASTQ qualities Phred+33 5..40).  The first SKEW bases are A-rich and the last SKEW
    G-rich, most at the very ends; ad5 / ad3 (library adapters) are planted with 5 % errors within 15 bases of the
    5' end / as their reverse complement at the 3' end of a fraction frac of the reads."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(lo, hi + 1, n)
    offsets = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(lens, out=offsets[1:])
    bases = ACGT[rng.integers(0, 4, int(offsets[-1]), dtype=np.uint8)]
    p = 0.25 + 0.6 * (SKEW - np.arange(SKEW)) / SKEW
    other = np.frombuffer(b"CGT", dtype=np.uint8)
    start = offsets[:-1].astype(np.int64)[:, None] + np.arange(SKEW)
    bases[start] = np.where(rng.random((n, SKEW)) < p, ord("A"), other[rng.integers(0, 3, (n, SKEW))])
    end = offsets[1:].astype(np.int64)[:, None] - 1 - np.arange(SKEW)
    other = np.frombuffer(b"ACT", dtype=np.uint8)
    bases[end] = np.where(rng.random((n, SKEW)) < p, ord("G"), other[rng.integers(0, 3, (n, SKEW))])
    for ad, at_end in ((ad5, False), (ad3, True)):
        if ad is None:
            continue
        for r in np.nonzero(rng.random(n) < frac)[0].tolist():
            s, e = int(offsets[r]), int(offsets[r + 1])
            m = np.frombuffer(synth.mutate(rev_comp(ad) if at_end else ad, 0.05, rng), dtype=np.uint8)
            pos = e - len(m) - int(rng.integers(0, 15)) if at_end else s + int(rng.integers(0, 15))
            bases[pos:pos + len(m)] = m
    quals = (rng.integers(5, 41, int(offsets[-1])) + 33).astype(np.uint8)
    return synth.ReadBatch(bases, quals, offsets)


def _prepass_lines(stderr: str):
    keep = ("INFO: trim 5'", "INFO: trim 3'", "INFO: 5' adapter", "INFO: 3' adapter", "INFO: mean depth",
            "INFO: set ")
    return [ln for ln in stderr.splitlines() if ln.startswith(keep)]


def _expected(batch, *, read_type, min_len=1000, bc_len=150, end_len=150, bc_num=100000, ad_num=100000,
              end_bias=1.0, mid_sim=None, adapter_file=None, only_ad=True):
    """What the CLI prints for the pre-pass, from prepass.sample_ends, the oracle's counts and search and
    prepass.resolve.  Returns (lines, result, sampled ends)."""
    params = FilterParams(min_len=max(min_len, 100), bc_len=bc_len, end_len=end_len,
                          mid_sim=0.0 if mid_sim is None else mid_sim).apply_read_type(read_type)
    e5, e3, _, _, _ = prepass.sample_ends(batch, params, ad_num, bc_num)
    c5, c3 = oracle_lib.base_content_counts(e5), oracle_lib.base_content_counts(e3)
    m5 = m3 = None
    if adapter_file is None:
        m5 = _oracle_search(e5, ADAPTER_LIB, params.mid_sim)
        m3 = _oracle_search(e3, ADAPTER_LIB, params.mid_sim)
    res = prepass.resolve(c5, c3, m5, m3, n=e5.shape[0], end_bias=end_bias, mid_sim=params.mid_sim, bc_len=bc_len,
                          read_type=read_type, adapter_file=adapter_file)
    lines = res.log[:2]
    if adapter_file is None:
        lines += res.log[2:4] + [f"INFO: mean depth of 5' adapter: {res.dep5p:g}",
                                 f"INFO: mean depth of 3' adapter: {res.dep3p:g}"]
        if not only_ad:  # -A ends the run before the default adapter is set
            lines += res.log[4:]
    return lines, res, e5


def _run_cli(tmp_path, batch, args, fasta=False):
    if not os.path.exists(EXE):
        subprocess.run(["make", "-C", os.path.join(ROOT, "src")], check=True, stdout=subprocess.DEVNULL)
    fi = tmp_path / ("in.fa" if fasta else "in.fq")
    if fasta:
        fi.write_bytes(batch.to_fasta())
    else:
        synth.write_fastq(str(fi), batch.bases, batch.quals, batch.offsets)
    pr = subprocess.run([EXE, "-i", str(fi)] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=900,
                        cwd=tmp_path)
    err = pr.stderr.decode("utf-8", "replace")
    assert pr.returncode == 0, err[-2000:]
    return err


CLI_CASES = {
    # id: (reads, their length range, CLI arguments, _expected arguments, planted adapters, sampled ends' shape);
    # a few reads are shorter than max(-l, 2 * checkLen) and must not be sampled
    "default_sizes": (103_000, (295, 900), ["-x", "ont", "-A", "-l", "300"],
                      dict(read_type="ont", min_len=300), (ADAPTER_LIB[4], ADAPTER_LIB[8]), (100_000, 150)),
    "bc_len_3500": (1600, (6980, 7600), ["-x", "ont", "-A", "-e", "3500", "-n", "1500", "-N", "1500"],
                    dict(read_type="ont", bc_len=3500, bc_num=1500, ad_num=1500), (ADAPTER_LIB[0], ADAPTER_LIB[0]),
                    (1500, 3500)),
    "end_len_9000": (340, (17980, 18600), ["-x", "hifi", "-A", "-E", "9000", "-n", "300", "-N", "300"],
                     dict(read_type="hifi", end_len=9000, bc_num=300, ad_num=300), (ADAPTER_LIB[0], None),
                     (300, 9000)),
    "bias_0.3_sim_0.95": (30_000, (300, 900), ["-x", "ont", "-A", "-l", "300", "-b", "0.3", "-S", "0.95"],
                          dict(read_type="ont", min_len=300, end_bias=0.3, mid_sim=0.95),
                          (ADAPTER_LIB[12], ADAPTER_LIB[20]), (30_000, 150)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CLI_CASES))
def test_cli_prepass_vs_oracle(case, tmp_path):
    """`tgsfilter -A`: the trims, the adapters picked and their mean depth, at the default sample size, past 3072 and
    past 8192 columns and with a non-default -b / -S."""
    n, (lo, hi), args, exp_args, (ad5, ad3), shape = CLI_CASES[case]
    batch = _cli_reads(n, lo, hi, seed=n, ad5=ad5, ad3=ad3)
    lines, res, e5 = _expected(batch, **exp_args)
    assert e5.shape == shape
    assert res.trim5p > 0 and res.trim3p > 0 and (res.adapter5p or res.adapter3p), lines
    assert _prepass_lines(_run_cli(tmp_path, batch, args)) == lines


@pytest.mark.gpu
def test_cli_prepass_counts_only_with_adapter_file(tmp_path):
    """-E 3500 -a: the base content alone is counted (no library search) and the main pass runs with the file's
    adapters and both trims."""
    batch = _cli_reads(300, 7000, 7400, seed=3500, ad5=ADAPTER_LIB[8])
    (tmp_path / "adapters.fa").write_bytes(b">rapid\n" + ADAPTER_LIB[8] + b"\n")
    lines, res, e5 = _expected(batch, read_type="ont", end_len=3500, adapter_file=[ADAPTER_LIB[8]])
    assert e5.shape == (300, 3500) and res.trim5p > 0 and res.trim3p > 0, lines
    err = _run_cli(tmp_path, batch, ["-x", "ont", "-E", "3500", "-a", "adapters.fa", "-o", "out.fq"])
    assert _prepass_lines(err) == lines
    given = {ln.split(":", 2)[2] for ln in err.splitlines() if ln.startswith("INFO: input adapter")}
    assert given == set(a.decode() for a in res.adapters) == {ADAPTER_LIB[8].decode(), ADAPTER_LIB[9].decode()}
    assert (tmp_path / "out.fq").stat().st_size > 0


@pytest.mark.gpu
def test_cli_prepass_fasta_sets_the_default_adapter(tmp_path):
    """FASTA input (no qualities) through the whole run: no adapter in the sample, so the read type's default adapter
    is set after the pre-pass."""
    batch = _cli_reads(3000, 300, 900, seed=31)
    lines, res, _ = _expected(batch, read_type="hifi", min_len=300, only_ad=False)
    assert res.trim5p > 0 and res.trim3p > 0 and not res.adapter5p and not res.adapter3p, lines
    assert lines[-1] == "INFO: set PacBio blunt adapter to trim: " + ADAPTER_LIB[0].decode()
    err = _run_cli(tmp_path, batch, ["-x", "hifi", "-l", "300", "-o", "out.fa"], fasta=True)
    assert _prepass_lines(err) == lines

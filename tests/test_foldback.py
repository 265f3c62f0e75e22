"""Fold-back screen (tgsf_set_foldback / --foldback): the oracle against a plain Python restatement, every rule at its
boundary, the ABI's and the CLI's argument checks, and on the GPU field-by-field parity with tgsfo_run_foldback
(tests/foldback_oracle.c)."""
from __future__ import annotations

import gzip
import os
import subprocess

import numpy as np
import pytest

import foldback_oracle
import oracle_lib
from tgsfilter_b200 import _capi, records, synth
from tgsfilter_b200.params import ADAPTER_LIB, FilterParams, rev_comp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "src", "tgsfilter")
_CODE = {ord(c): i for i, c in enumerate("ACGT")} | {ord(c): i for i, c in enumerate("acgt")}
_M32 = 0xFFFFFFFF


# ---- plain restatement -----------------------------------------------------------------------------
def _fmix32(h: int) -> int:
    h ^= h >> 16
    h = (h * 0x85EBCA6B) & _M32
    h ^= h >> 13
    h = (h * 0xC2B2AE35) & _M32
    return h ^ (h >> 16)


def _codes(w: bytes):
    f = r = 0
    for j, b in enumerate(w):
        c = _CODE.get(b)
        if c is None:
            return None
        f = (f << 2) | c
        r |= (3 - c) << (2 * j)
    return f, r


def _detect(s: bytes):
    """(fold, anchors, centre, min_gap) of one piece, straight from the rules."""
    L = len(s)
    occ = {}
    for i in range(L - 14):
        fr = _codes(s[i:i + 15])
        if fr is None:
            continue
        f, r = fr
        key = min(f, r)
        if _fmix32(key) & 7:
            continue
        occ.setdefault(key, []).append((0 if f < r else 1, i))
    bins = {}
    for v in occ.values():
        if len(v) == 2 and {o for o, _ in v} == {0, 1}:
            p0 = next(p for o, p in v if o == 0)
            p1 = next(p for o, p in v if o == 1)
            d = p0 + p1 + 15
            bins.setdefault(d >> 7, []).append((d, abs(p1 - p0) - 15))
    if not bins:
        return (-1, 0, -1, -1)
    best = max(bins, key=lambda b: (len(bins.get(b, [])) + len(bins.get(b + 1, [])), -b))
    peak = bins.get(best, []) + bins.get(best + 1, [])
    V = len(peak)
    c = sum(d for d, _ in peak) // (2 * V)
    g = min(g for _, g in peak)
    cut = V >= 8 and g <= 500 and 400 * V >= min(c, L - c) and 0 < c < L
    return (c if cut else -1, V, c, g)


# ---- reads -----------------------------------------------------------------------------------------
def _rand(rng, n) -> bytes:
    return synth._ACGT[rng.integers(0, 4, n, dtype=np.uint8)].tobytes()


def _fold_read(rng, arm: int, frac: float = 0.8, err: float = 0.001) -> bytes:
    """X·rc(X'): an arm, then the reverse complement of its last frac·arm bases, both with errors."""
    x = _rand(rng, arm)
    back = x[arm - int(arm * frac):]
    return synth.mutate(x, err, rng) + synth.mutate(rev_comp(back), err, rng)


_SAMPLED = None


def _sampled_kmers():
    """Distinct 15-mers w with f < r whose canonical key is sampled: each placed once as w and once as rc(w) is an
    anchor."""
    global _SAMPLED
    if _SAMPLED is None:
        rng = np.random.default_rng(77)
        out, seen = [], set()
        while len(out) < 400:
            w = _rand(rng, 15)
            f, r = _codes(w)
            if f < r and not _fmix32(f) & 7 and f not in seen:
                seen.add(f)
                out.append(w)
        _SAMPLED = out
    return _SAMPLED


def _placed(L: int, pairs) -> bytes:
    """A piece of L bases, N everywhere except one sampled 15-mer at p0 and its reverse complement at p1 per pair:
    exactly those anchors (no two 15-mers touch, so no other window is valid)."""
    s = bytearray(b"N" * L)
    starts = sorted(p for pair in pairs for p in pair)
    assert all(b - a >= 16 for a, b in zip(starts, starts[1:])) and starts[0] >= 0 and starts[-1] + 15 <= L
    for w, (p0, p1) in zip(_sampled_kmers(), pairs):
        s[p0:p0 + 15] = w
        s[p1:p1 + 15] = rev_comp(w)
    return bytes(s)


def _designed(L: int, anchors) -> bytes:
    """_placed with each anchor given as (d, g)."""
    pairs = [((d - g - 30) // 2, (d - g - 30) // 2 + g + 15) for d, g in anchors]
    assert all(p0 + p1 + 15 == d for (p0, p1), (d, _) in zip(pairs, anchors))
    return _placed(L, pairs)


def _cluster(d: int, V: int, g0: int = 26):
    return [(d, g0 + 40 * j) for j in range(V)]


# ---- CPU: the oracle's detector ---------------------------------------------------------------------
def _detector_cases():
    rng = np.random.default_rng(11)
    seqs = [b"", b"ACGT", _rand(rng, 14), _rand(rng, 15), _rand(rng, 16)]
    seqs += [_rand(rng, int(n)) for n in (500, 3000, 12000)]
    for arm in (300, 1500, 4000, 9000):
        seqs.append(_fold_read(rng, arm))
    seqs.append(_fold_read(rng, 3000, err=0.05))
    seqs.append(_fold_read(rng, 3000, err=0.10))
    r = bytearray(_fold_read(rng, 5000))  # N and lowercase bytes
    for j in rng.integers(0, len(r), 40):
        r[j] = b"NnacgtRY"[int(rng.integers(0, 8))]
    seqs.append(bytes(r))
    seqs.append(_fold_read(rng, 4000).lower())
    unit = _rand(rng, 300)  # tandem repeat: repeated keys are no anchors
    seqs.append((unit * 30) + rev_comp(unit * 10))
    seqs.append(b"A" * 2000 + b"T" * 2000)
    x = _rand(rng, 3000)  # inverted repeats with a 200-base and a 2 kb spacer
    seqs.append(x + _rand(rng, 200) + rev_comp(x))
    seqs.append(x + _rand(rng, 2000) + rev_comp(x))
    return seqs


def test_oracle_detector_matches_restatement():
    seqs = _detector_cases()
    got = foldback_oracle.detect(seqs)
    for s, g in zip(seqs, got):
        assert tuple(int(v) for v in g) == _detect(s), len(s)
    folds = [i for i in range(5, 15) if got["fold"][i] >= 0]
    assert len(folds) >= 7
    assert got["fold"][-1] == -1 and got["fold"][-2] >= 0  # the 2 kb spacer fails the gap rule, 200 b does not


@pytest.mark.parametrize("arm", [1000, 5000, 10000])
def test_oracle_cuts_planted_folds_near_the_junction(arm):
    rng = np.random.default_rng(arm)
    for err, tol in ((0.001, 3), (0.05, 25)):
        x = _rand(rng, arm)
        a = synth.mutate(x, err, rng)
        s = a + synth.mutate(rev_comp(x[arm - int(0.8 * arm):]), err, rng)
        r = foldback_oracle.detect([s])[0]
        assert r["fold"] >= 0 and abs(int(r["fold"]) - len(a)) <= tol, (err, r, len(a))


BOUNDARY = [
    # name, piece, expected (fold, anchors, centre, min_gap)
    ("V=8", (2000, _cluster(2000, 8)), (1000, 8, 1000, 26)),
    ("V=7", (2000, _cluster(2000, 7)), (-1, 7, 1000, 26)),
    ("g=500", (2000, _cluster(2000, 8, 500)), (1000, 8, 1000, 500)),
    ("g=501", (2000, _cluster(2001, 8, 501)), (-1, 8, 1000, 501)),
    ("400V=shorter", (10000, _cluster(6400, 8)), (3200, 8, 3200, 26)),
    ("400V=shorter+1", (10000, _cluster(6402, 8)), (-1, 8, 3201, 26)),
    ("400V=shorter (3' arm)", (10000, _cluster(2 * 6800, 8)), (6800, 8, 6800, 26)),
    ("400V=shorter+1 (3' arm)", (10000, _cluster(2 * 6799, 8)), (-1, 8, 6799, 26)),
]


@pytest.mark.parametrize("name,piece,expect", BOUNDARY, ids=[b[0] for b in BOUNDARY])
def test_oracle_rule_boundaries(name, piece, expect):
    s = _designed(*piece)
    assert _detect(s) == expect
    assert tuple(int(v) for v in foldback_oracle.detect([s])[0]) == expect


def _tie_pieces():
    # two clusters of 8 in bins 15 and 46: b = 14 and b = 15 tie with b = 45 and 46, the smallest b wins
    a = _designed(8000, _cluster(1980, 8) + _cluster(5900, 8))
    # the same with 9 anchors at 5900: that cluster wins
    b = _designed(8000, _cluster(1980, 8) + _cluster(5900, 9))
    # 4 anchors at d = 1940, 2100 and 2260 (bins 15, 16, 17): b = 15 (bins 15 + 16) ties with b = 16 (bins 16 + 17)
    c = _placed(8000, [(200 + 20 * i, d - 215 - 20 * i) for i, d in enumerate([1940] * 4 + [2100] * 4 + [2260] * 4)])
    return [a, b, c]


def test_oracle_bin_ties_take_the_smallest_bin():
    a, b, c = _tie_pieces()
    assert _detect(a) == tuple(int(v) for v in foldback_oracle.detect([a])[0]) == (990, 8, 990, 26)
    assert _detect(b) == tuple(int(v) for v in foldback_oracle.detect([b])[0]) == (2950, 9, 2950, 26)
    rc = foldback_oracle.detect([c])[0]
    assert _detect(c) == tuple(int(v) for v in rc)
    assert int(rc["anchors"]) == 8 and int(rc["centre"]) == (4 * 1940 + 4 * 2100) // 16


def _plain_params(**kw) -> FilterParams:
    p = FilterParams(min_q=-1.0, head_trim=0, tail_trim=0, min_len=1, filter=False, **kw)
    return p.apply_read_type("ont")


def test_oracle_arm_tie_and_min_len():
    """c = L - c keeps the 5' arm; a kept arm of exactly -l stays, one base shorter is dropped without a counter."""
    tie = _designed(4000, _cluster(4000, 8))  # c = 2000 = L - c
    three = _designed(5000, _cluster(2 * 3000, 8))  # c = 3000: the 3' arm [3000, 5000) is shorter, keep [0, 3000)
    five = _designed(5000, _cluster(2 * 1500, 8))  # c = 1500: keep [1500, 5000)
    seqs = [tie, three, five]
    batch = synth.pack_reads(seqs, [b"I" * len(s) for s in seqs])
    for min_len, dropped in ((2000, []), (2001, [0]), (3500, [0, 1]), (3501, [0, 1, 2])):
        params = _plain_params()
        params.min_len = min_len
        _, pieces, cnt, stats = foldback_oracle.run(params, batch)
        _, _, cnt0 = oracle_lib.run(params, batch)
        assert list(pieces["start"]) == [0, 0, 1500] and list(pieces["len"]) == [2000, 3000, 3500]
        status = [_capi.PIECE_FOLDBACK if i in dropped else _capi.PIECE_EMIT for i in range(3)]
        assert list(pieces["status"]) == status
        assert all(pieces["sum_q"][i] == 0 and pieces["repeat_len"][i] == -1 for i in dropped)
        arms = [2000, 3000, 3500]
        assert list(stats) == [3, 2000 + 2000 + 1500, len(dropped), sum(arms[i] for i in dropped)]
        # the dropped arms never reach the clean step; DropInfo[0..12] is that of the uncut run
        L = oracle_lib.layout(params)
        assert np.array_equal(cnt[L.drop_info:L.drop_info + 13], cnt0[L.drop_info:L.drop_info + 13])


def test_oracle_replays_the_tail_on_the_arm():
    """With -p and -q, a cut piece's counters are those of its arm: the oracle's counter block equals tgsfo_run on a
    batch whose folded reads were replaced by their kept arms."""
    rng = np.random.default_rng(5)
    seqs, quals = [], []
    for i in range(40):
        s = _fold_read(rng, int(rng.integers(2000, 6000))) if i % 3 == 0 else _rand(rng, int(rng.integers(1000, 8000)))
        seqs.append(s)
        quals.append(bytes(rng.integers(45, 75, len(s), dtype=np.uint8)))
    batch = synth.pack_reads(seqs, quals)
    params = _plain_params(kmer=11, min_repeat=3)
    params.min_q = 15.0
    params.filter = True
    params.min_len = 500
    params.adapters = []
    _, pieces, cnt, stats = foldback_oracle.run(params, batch)
    cut = [i for i in range(len(seqs)) if pieces["len"][i] < len(seqs[i])]
    assert len(cut) >= 10 and stats[0] == len(cut)
    arms = [seqs[i][int(pieces["start"][i]):int(pieces["start"][i] + pieces["len"][i])] for i in range(len(seqs))]
    aq = [quals[i][int(pieces["start"][i]):int(pieces["start"][i] + pieces["len"][i])] for i in range(len(seqs))]
    _, p_arm, c_arm = oracle_lib.run(params, synth.pack_reads(arms, aq))
    L = oracle_lib.layout(params)
    clean = np.zeros(L.n_u64, dtype=bool)  # the raw side still counts the uncut reads
    for off, n in [(L.clean_hist, 256), (L.drop_info + 13, 4)] + \
            [(getattr(L, t), L.bc_len * 5) for t in ("clean5p_cnt", "clean5p_qual", "clean3p_cnt", "clean3p_qual")] + \
            [(getattr(L, t), L.max_bins * 5) for t in ("clean_bin_cnt", "clean_bin_qual")]:
        clean[off:off + n] = True
    assert np.array_equal(cnt[clean], c_arm[clean])
    for f in ("sum_q", "len", "repeat_len", "status"):
        assert np.array_equal(pieces[f], p_arm[f]), f


# ---- CPU: argument checks -----------------------------------------------------------------------------
def test_abi_rejects_bad_arguments_without_a_device():
    lib = _capi.load()
    out = np.zeros(2, dtype=_capi.FOLD_RESULT_DTYPE)
    seq = np.frombuffer(b"ACGT" * 10, dtype=np.uint8)
    good = np.array([0, 20, 40], dtype=np.uint64)
    assert lib.tgsf_fold_detect(0, seq.ctypes.data, good.ctypes.data, 0, None) == _capi.TGSF_OK
    for s, o, n, r in ((seq.ctypes.data, None, 2, out.ctypes.data), (seq.ctypes.data, good.ctypes.data, 2, None),
                       (None, good.ctypes.data, 2, out.ctypes.data),
                       (seq.ctypes.data, np.array([1, 20, 40], dtype=np.uint64).ctypes.data, 2, out.ctypes.data),
                       (seq.ctypes.data, np.array([0, 30, 20], dtype=np.uint64).ctypes.data, 2, out.ctypes.data),
                       (seq.ctypes.data, np.array([0, 1 << 31], dtype=np.uint64).ctypes.data, 1, out.ctypes.data)):
        assert lib.tgsf_fold_detect(0, s, o, n, r) == _capi.TGSF_ERR_INVALID
    stats = np.zeros(4, dtype=np.uint64)
    assert lib.tgsf_set_foldback(None, 1) == _capi.TGSF_ERR_INVALID
    assert lib.tgsf_foldback_stats(None, stats.ctypes.data) == _capi.TGSF_ERR_INVALID


@pytest.mark.parametrize("extra", [["--qc"], ["-A"], ["-F"]])
def test_cli_rejects_foldback_with(tmp_path, extra):
    if not os.path.exists(EXE):
        pytest.skip("src/tgsfilter not built")
    fq = tmp_path / "r.fq"
    fq.write_bytes(b"@r\n" + b"ACGT" * 300 + b"\n+\n" + b"I" * 1200 + b"\n")
    cmd = [EXE, "-i", str(fq), "-x", "ont", "-o", str(tmp_path / "o.fq"), "--foldback"] + extra
    pr = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=60)
    assert pr.returncode != 0
    assert "--foldback" in pr.stderr.decode()
    assert not (tmp_path / "o.fq").exists()


# ---- GPU ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_fold_detect_matches_oracle():
    """Pieces from 16 b to 1 Mb, through both the shared-memory path (<= 40 960 b) and the global one."""
    from tgsfilter_b200.engine import fold_detect
    rng = np.random.default_rng(21)
    seqs = _detector_cases() + [_designed(*p) for _, p, _ in BOUNDARY] + _tie_pieces()
    for arm in (20, 800, 8000, 16000, 20000, 20500, 21000, 40000, 150000, 500000):
        seqs.append(_fold_read(rng, arm, err=0.01))
    for n in (16, 40960, 40961, 65536, 200000, 1_000_000):
        seqs.append(_rand(rng, n))
    seqs.append(_rand(rng, 300000) + _fold_read(rng, 350000, err=0.02))
    seqs.append((_rand(rng, 500) * 200)[:100000])  # repeats only
    got = fold_detect(seqs)
    want = foldback_oracle.detect(seqs)
    for f in ("fold", "anchors", "centre", "min_gap"):
        assert np.array_equal(got[f], want[f]), (f, np.nonzero(got[f] != want[f])[0][:5])
    assert (got["fold"] >= 0).sum() >= 20


def _with_folds(batch, frac, seed, fasta=False):
    """Replace a share of the reads by X·rc(X') reads of the same length (qualities kept)."""
    rng = np.random.default_rng(seed)
    b = batch.bases.copy()
    planted = []
    for r in range(batch.n_reads):
        s, e = int(batch.offsets[r]), int(batch.offsets[r + 1])
        if e - s < 400 or rng.random() >= frac:
            continue
        fr = _fold_read(rng, int((e - s) / 1.7), frac=float(rng.uniform(0.4, 0.9)), err=float(rng.uniform(0.001, 0.05)))
        fr = (fr + _rand(rng, e - s))[:e - s]
        b[s:e] = np.frombuffer(fr, dtype=np.uint8)
        planted.append(r)
    b[5::9973] = ord("n")
    return synth.ReadBatch(b, None if fasta else batch.quals, batch.offsets, batch.names), planted


def _run_gpu(params, batch, path="submit", contam=None, enable=True):
    from tgsfilter_b200.engine import FilterEngine
    with FilterEngine(params) as eng:
        if contam is not None:
            eng.set_contaminants(contam[0], k=contam[1], min_frac=contam[2])
        if enable:
            eng.set_foldback(True)
        if path == "submit":
            eng.submit(batch)
        elif path == "packed":
            eng.submit_packed(batch)
        else:
            import torch
            d_b = torch.from_numpy(batch.bases).cuda()
            d_q = None if batch.quals is None else torch.from_numpy(batch.quals).cuda()
            d_o = torch.from_numpy(batch.offsets.astype(np.int64)).cuda()
            torch.cuda.synchronize()
            eng.submit_device(d_b.data_ptr(), None if d_q is None else d_q.data_ptr(), d_o.data_ptr(),
                              batch.n_reads, batch.n_bases, keep=(d_b, d_q, d_o))
        reads, pieces = eng.collect()
        return reads, pieces, eng.counters().flat, eng.foldback_stats(), eng.launch_count()


def _assert_parity(got, want):
    reads, pieces, cnt, stats = got[:4]
    o_reads, o_pieces, o_cnt, o_stats = want
    assert np.array_equal(reads, o_reads)
    assert len(pieces) == len(o_pieces)
    for f in o_pieces.dtype.names:
        assert np.array_equal(pieces[f], o_pieces[f]), (f, np.nonzero(pieces[f] != o_pieces[f])[0][:5])
    assert np.array_equal(cnt, o_cnt)
    assert tuple(int(x) for x in o_stats) == stats


GPU_CASES = [
    # cfg, n, path, fasta, extra params, contaminant set
    (1, 300, "submit", False, {}, False),   # hifi
    (2, 400, "packed", False, {}, False),   # ont
    (4, 400, "device", False, {}, False),   # clr
    (3, 60, "submit", False, {"max_read_len": 1 << 20}, False),  # long ONT reads: the global path
    (2, 300, "submit", True, {}, False),    # FASTA
    (2, 300, "packed", False, {"discard": True}, False),  # -D
    (5, 200, "submit", False, {"min_repeat": 20}, False),  # -k 11 -p 20
    (1, 200, "device", False, {"kmer": 17, "min_repeat": 40}, False),
    (2, 300, "submit", False, {}, True),    # --contam with the fold screen
    (4, 300, "packed", False, {"kmer": 12, "min_repeat": 3}, True),
]


@pytest.mark.gpu
@pytest.mark.parametrize("cfg,n,path,fasta,extra,with_contam", GPU_CASES)
def test_gpu_foldback_parity(cfg, n, path, fasta, extra, with_contam):
    batch, planted = _with_folds(synth.make_config(cfg, n, max_len=None if cfg == 3 else 200_000), 0.25, cfg, fasta)
    params = synth.config_params(cfg)
    for key, v in extra.items():
        setattr(params, key, v)
    contam = None
    if with_contam:
        genome = synth.make_contaminant(48_502)
        batch, _, _ = synth.mix_contaminants(batch, genome, 0.08, 0.04, chimeras=0.05, seed=cfg)
        contam = ([genome], 17, 0.05)
    got = _run_gpu(params, batch, path, contam)
    want = foldback_oracle.run(params, batch, contam)
    _assert_parity(got, want)
    assert want[3][0] >= len(planted) // 3 > 0


@pytest.mark.gpu
def test_gpu_foldback_through_the_pool_overflow_retry():
    from test_gpu_parity import _pool_overflow_case
    params, pool = _pool_overflow_case()
    rng = np.random.default_rng(9)
    extra = [_fold_read(rng, int(rng.integers(1500, 6000))) for _ in range(40)]
    seqs = [pool.read(i)[0].tobytes() for i in range(pool.n_reads)] + extra
    batch = synth.pack_reads(seqs, [bytes([50] * len(s)) for s in seqs])
    got = _run_gpu(params, batch)
    want = foldback_oracle.run(params, batch)
    _assert_parity(got, want)
    assert want[3][0] >= 30


@pytest.mark.gpu
def test_gpu_foldback_off_changes_nothing():
    """Never enabled, enabled then disabled: reads, pieces, counters and launches equal; stats stay zero."""
    from tgsfilter_b200.engine import FilterEngine
    batch, _ = _with_folds(synth.make_config(2, 300), 0.3, 2)
    params = synth.config_params(2)
    r0, p0, c0, s0, l0 = _run_gpu(params, batch, enable=False)
    with FilterEngine(params) as eng:
        eng.set_foldback(True)
        eng.set_foldback(False)
        r1, p1 = eng.run(batch)
        c1, s1, l1 = eng.counters().flat, eng.foldback_stats(), eng.launch_count()
    assert np.array_equal(r0, r1) and np.array_equal(p0, p1) and np.array_equal(c0, c1)
    assert s0 == s1 == (0, 0, 0, 0) and l0 == l1
    o_reads, o_pieces, o_cnt = oracle_lib.run(params, batch)
    assert np.array_equal(p0, o_pieces) and np.array_equal(c0, o_cnt)


@pytest.mark.gpu
def test_gpu_foldback_state_and_stats():
    """TGSF_ERR_STATE while a batch is outstanding; stats add up over batches and reset with the counters."""
    from tgsfilter_b200.engine import FilterEngine
    batch, _ = _with_folds(synth.make_config(1, 150), 0.3, 1)
    params = synth.config_params(1)
    want = foldback_oracle.run(params, batch)[3]
    with FilterEngine(params) as eng:
        assert eng._lib.tgsf_set_foldback(eng._ctx, 2) == _capi.TGSF_ERR_INVALID
        eng.set_foldback(True)
        eng.submit(batch)
        for call in (lambda: eng.set_foldback(False), eng.foldback_stats):
            with pytest.raises(_capi.TgsfError) as e:
                call()
            assert e.value.code == _capi.TGSF_ERR_STATE
        eng.collect()
        eng.run(batch)
        assert eng.foldback_stats() == tuple(2 * int(x) for x in want) and want[0] > 0
        eng.reset_counters()
        assert eng.foldback_stats() == (0, 0, 0, 0)


@pytest.mark.gpu
def test_gpu_foldback_deflate_blocks():
    from tgsfilter_b200.engine import FilterEngine
    from test_contam import _gz_members
    batch, _ = _with_folds(synth.make_config(2, 200), 0.3, 12)
    params = synth.config_params(2)
    params.min_len = 3000  # some arms are dropped
    params.gz_blocks = True
    with FilterEngine(params) as eng:
        eng.set_foldback(True)
        eng.submit(batch)
        blob, spans = eng.collect_gz()
        _, pieces = eng.collect()
    _, o_pieces, _, o_stats = foldback_oracle.run(params, batch)
    assert np.array_equal(pieces, o_pieces)
    dropped = pieces["status"] == _capi.PIECE_FOLDBACK
    assert o_stats[0] > 0 and dropped.sum() > 0 and (spans["bytes"][dropped] == 0).all()
    members, texts = _gz_members(batch, o_pieces, blob, spans, fastq=True)
    assert gzip.decompress(b"".join(members)) == b"".join(texts)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [1, 2, 3, 4, 5])
def test_gpu_unplanted_configs_cut_what_the_oracle_predicts(cfg):
    """No folds are planted: the screen cuts exactly the pieces the oracle cuts (printed for the record)."""
    n = {1: 300, 2: 600, 3: 80, 4: 600, 5: 200}[cfg]
    batch = synth.make_config(cfg, n)
    params = synth.config_params(cfg)
    params.max_read_len = 1 << 20
    got = _run_gpu(params, batch)
    want = foldback_oracle.run(params, batch)
    _assert_parity(got, want)
    print(f"config[{cfg}]: {batch.n_reads} reads, {batch.n_bases} bases, {int(want[3][0])} pieces cut")


# ---- CLI on the GPU ----------------------------------------------------------------------------------
def _fastq_records(data: bytes):
    lines = data.split(b"\n")
    return sorted(b"\n".join(lines[i:i + 4]) for i in range(0, len(lines) - 3, 4))


def _info(stderr: bytes, needle: str):
    return [ln for ln in stderr.decode().splitlines() if needle in ln]


@pytest.fixture(scope="module")
def cli_inputs(tmp_path_factory):
    d = tmp_path_factory.mktemp("foldback_cli")
    batch, _ = _with_folds(synth.make_config(2, 2000), 0.2, 31)
    fq = d / "reads.fq"
    fq.write_bytes(batch.to_fastq())
    ad = d / "ad.fa"
    ad.write_bytes(b">ad\n" + ADAPTER_LIB[8] + b"\n")
    return d, batch, fq, ad


def _cli(d, fq, args, env=None, out_name="o.fq"):
    out = d / out_name
    pr = subprocess.run([EXE, "-i", str(fq), "-o", str(out), "-x", "ont", "-5", "0", "-3", "0", "-q", "10"] + args,
                        stdout=subprocess.PIPE, stderr=subprocess.PIPE, env={**os.environ, **(env or {})}, timeout=600)
    assert pr.returncode == 0, pr.stderr.decode()[-2000:]
    return (out.read_bytes() if out.exists() else b""), pr.stderr


@pytest.mark.gpu
def test_cli_foldback_matches_oracle(cli_inputs):
    d, batch, fq, ad = cli_inputs
    out, err = _cli(d, fq, ["-a", str(ad), "--foldback", "-l", "2000"])
    params = FilterParams(min_q=10.0, head_trim=0, tail_trim=0, min_len=2000,
                          adapters=[ADAPTER_LIB[8], rev_comp(ADAPTER_LIB[8])]).apply_read_type("ont")
    _, o_pieces, _, st = foldback_oracle.run(params, batch)
    expect = sorted(t.rstrip(b"\n") for t, _, _ in records.format_records(batch, o_pieces, fastq=True))
    assert _fastq_records(out) == expect
    assert st[0] > 100 and st[2] > 0
    assert _info(err, "fold-back") == [
        f"INFO: {st[0]} reads were cut at a fold-back junction, removing {st[1]} bases.",
        f"INFO: {st[2]} reads were discarded with {st[3]} bases as too short after a fold-back cut."]
    out2, err2 = _cli(d, fq, ["-a", str(ad), "--foldback", "-l", "2000", "--gpus", "2"],
                      env={"TGSF_SHARE_DEVICES": "1", "TGSF_BATCH_MB": "4"}, out_name="o2.fq")
    assert _fastq_records(out2) == expect
    assert [ln for ln in _info(err2, "INFO:") if "written to" not in ln] == \
        [ln for ln in _info(err, "INFO:") if "written to" not in ln]
    out3, _ = _cli(d, fq, ["-a", str(ad), "--foldback", "-l", "2000"], out_name="o3.fq.gz")
    assert _fastq_records(gzip.decompress(out3)) == expect
    _, err0 = _cli(d, fq, ["-a", str(ad), "-l", "2000"], out_name="o0.fq")
    assert not _info(err0, "fold-back")


@pytest.mark.gpu
def test_cli_foldback_then_downsample(cli_inputs):
    d, _, fq, ad = cli_inputs
    out, err = _cli(d, fq, ["-a", str(ad), "--foldback", "-g", "1m", "-d", "5"], out_name="ds.fq")
    assert len(_info(err, "fold-back junction")) == 1
    assert out.count(b"\n+\n") > 0

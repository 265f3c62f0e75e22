"""Low-complexity screen (tgsf_set_dust / --dust): the oracle against a plain Python restatement, every rule at its
boundary, the ABI's and the CLI's argument checks, and on the GPU tgsf_dust_detect and field-by-field parity with
tgsfo_run_dust (tests/dust_oracle.c)."""
from __future__ import annotations

import gzip
import os
import subprocess

import numpy as np
import pytest

import dust_oracle
import oracle_lib
from tgsfilter_b200 import _capi, records, synth
from tgsfilter_b200.params import ADAPTER_LIB, FilterParams, rev_comp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "src", "tgsfilter")
_CODE = np.full(256, -1, dtype=np.int64)
for _i, _c in enumerate(b"ACGT"):
    _CODE[_c] = _CODE[_c + 32] = _i


# ---- plain restatement -----------------------------------------------------------------------------
def _scores(s: bytes) -> np.ndarray:
    """S of every window s[j, j+64) (-1 when a byte of it is not ACGT/acgt)."""
    c = _CODE[np.frombuffer(s, dtype=np.uint8)] if s else np.zeros(0, dtype=np.int64)
    out = np.full(max(len(s) - 63, 0), -1, dtype=np.int64)
    for j in range(len(out)):
        w = c[j:j + 64]
        if (w < 0).any():
            continue
        t = 16 * w[:62] + 4 * w[1:63] + w[2:64]
        n = np.bincount(t, minlength=64)
        out[j] = int((n * (n - 1) // 2).sum())
    return out


def _masked(s: bytes, level: int, scores=None) -> int:
    """M: the bases covered by the masked windows, straight from the union."""
    sc = _scores(s) if scores is None else scores
    covered = set()
    for j in np.nonzero(sc > 61 * level)[0]:
        covered.update(range(int(j), int(j) + 64))
    return len(covered)


# ---- pieces ----------------------------------------------------------------------------------------
def _rand(rng, n) -> bytes:
    return synth._ACGT[rng.integers(0, 4, n, dtype=np.uint8)].tobytes()


def _repeat(rng, unit_len: int, n: int, err: float) -> bytes:
    """n bases of a random unit repeated, each base substituted by another with probability err."""
    s = np.frombuffer((_rand(rng, unit_len) * (n // unit_len + 1))[:n], dtype=np.uint8).copy()
    hit = np.nonzero(rng.random(n) < err)[0]
    s[hit] = synth._ACGT[(_CODE[s[hit]] + rng.integers(1, 4, len(hit))) % 4]
    return s.tobytes()


def _detector_cases():
    rng = np.random.default_rng(31)
    seqs = [b"", b"ACGT", b"A" * 63, b"A" * 64, b"A" * 65, b"a" * 64, _rand(rng, 63), _rand(rng, 64), _rand(rng, 65),
            b"A" * 63 + b"N", b"N" + b"A" * 64, b"CA" * 32, (b"CA" * 33)[:65]]
    seqs += [_rand(rng, int(n)) for n in rng.integers(66, 1500, 6)]
    for unit in range(1, 9):  # planted repeats of units 1-8 with 0, 5 and 10 % errors inside random flanks
        for err in (0.0, 0.05, 0.10):
            n = int(rng.integers(80, 600))
            seqs.append(_rand(rng, int(rng.integers(0, 300))) + _repeat(rng, unit, n, err) +
                        _rand(rng, int(rng.integers(0, 300))))
    for unit in (1, 2, 3):  # N bytes inside and at the edges of repeats
        r = bytearray(_repeat(rng, unit, 400, 0.0))
        r[200] = ord("N")
        seqs.append(_rand(rng, 100) + b"N" + bytes(r) + b"N" + _rand(rng, 100))
        r[30:33] = b"NNN"
        seqs.append(bytes(r) + b"n" + _rand(rng, 50))
    seqs.append(_repeat(rng, 2, 500, 0.02).lower())  # lower case
    mixed = bytearray(_repeat(rng, 3, 600, 0.03))
    for j in rng.integers(0, len(mixed), 200):
        mixed[j] = mixed[j] | 0x20
    seqs.append(bytes(mixed))
    seqs.append(_repeat(rng, 6, 600, 0.0))  # vertebrate telomere-like: kept at level 7
    return seqs


# ---- CPU: the oracle's detector ---------------------------------------------------------------------
def test_oracle_scores_match_restatement():
    rng = np.random.default_rng(3)
    for s in _detector_cases()[::4] + [_repeat(rng, u, 300, 0.05) for u in (1, 2, 4)]:
        assert np.array_equal(dust_oracle.scores(s), _scores(s)), len(s)


def test_oracle_detector_matches_restatement():
    seqs = _detector_cases()
    scores = [_scores(s) for s in seqs]
    for level in (1, 3, 5, 7, 12, 20, 29, 30):
        got = dust_oracle.masked(seqs, level)
        want = [_masked(s, level, sc) for s, sc in zip(seqs, scores)]
        assert list(got) == want, level
    at7 = dust_oracle.masked(seqs, 7)
    assert at7[2] == 0 and at7[3] == 64 and at7[4] == 65 and at7[5] == 64 and at7[9] == 0 and at7[10] == 64
    assert at7[-1] == 0  # the 6-base unit stays unmasked at the default level


def test_oracle_level_7_masks_short_units():
    """Units 1-3 at 5 % substitutions and perfect 4-base units are masked over most of their length at level 7;
    6- and 7-base units and random sequence are not masked at all."""
    rng = np.random.default_rng(8)
    for unit, err in ((1, 0.05), (2, 0.05), (3, 0.05), (4, 0.0)):
        s = _repeat(rng, unit, 600, err)
        assert dust_oracle.masked([s], 7)[0] >= 0.9 * 600, (unit, err)
    for unit in (6, 7):
        assert dust_oracle.masked([_repeat(rng, unit, 600, 0.0)], 7)[0] == 0, unit
    assert dust_oracle.masked([_rand(rng, 30000)], 1)[0] < 30000 // 2
    assert dust_oracle.masked([_rand(rng, 30000)], 2)[0] == 0


_HILL = {}


def _window_with_score(target: int) -> bytes:
    """A 64-base window whose S is exactly target (found by a seeded hill climb on single-base changes)."""
    if target in _HILL:
        return _HILL[target]
    rng = np.random.default_rng(target)
    for start in range(20):
        w = bytearray((_rand(rng, int(rng.integers(1, 6))) * 64)[:64] if start else _rand(rng, 64))
        for j in rng.integers(0, 64, 12 if start else 0):
            w[j] = b"ACGT"[int(rng.integers(0, 4))]
        cur = abs(int(_scores(bytes(w))[0]) - target)
        for _ in range(6000):
            if cur == 0:
                _HILL[target] = bytes(w)
                return bytes(w)
            j = int(rng.integers(0, 64))
            old = w[j]
            w[j] = b"ACGT"[int(rng.integers(0, 4))]
            d = abs(int(_scores(bytes(w))[0]) - target)
            if d <= cur:
                cur = d
            else:
                w[j] = old
    raise AssertionError(f"no window with S = {target}")


SCORE_LEVELS = (1, 7, 15)  # S = 61 level and 61 level + 1 are both reachable there (not at every level)


def _score_boundary_pieces():
    out = []
    for level in SCORE_LEVELS:
        for s, m in ((_window_with_score(61 * level), 0), (_window_with_score(61 * level + 1), 64)):
            out.append((level, s, m))
            out.append((level, b"N" + s + b"n", m))
    return out


def test_oracle_score_boundary():
    """S = 61 level is not masked, S = 61 level + 1 is."""
    for level, s, m in _score_boundary_pieces():
        sc = _scores(s)
        assert sorted(set(sc[sc >= 0].tolist())) in ([61 * level], [61 * level + 1])
        assert _masked(s, level) == m and dust_oracle.masked([s], level)[0] == m, (level, len(s))


def _two_windows(gap: int) -> bytes:
    """A piece whose only masked windows at level 29 are j = 0 and j = gap = L - 64: A^62, a spacer, T^62.  Window 0
    (A^62 + 2 spacer bases) and window gap (2 spacer bases + T^62) hold 60 equal triplets (S = 1770 > 1769); every
    window between them at most 59 (S <= 1711 + a few)."""
    spacer = (b"GC" * 8)[:gap - 60]
    return b"A" * 62 + spacer + b"T" * 62


GAP_CASES = [  # name, piece, masked starts, M at level 29
    ("overlap by 63", b"A" * 65, [0, 1], 65),
    ("63 apart", _two_windows(63), [0, 63], 127),
    ("64 apart (abut)", _two_windows(64), [0, 64], 128),
    ("65 apart", _two_windows(65), [0, 65], 128),
]


@pytest.mark.parametrize("name,s,starts,m", GAP_CASES, ids=[g[0] for g in GAP_CASES])
def test_oracle_union_of_masked_windows(name, s, starts, m):
    sc = _scores(s)
    assert list(np.nonzero(sc > 61 * 29)[0]) == starts and starts[-1] == len(s) - 64
    assert _masked(s, 29, sc) == m and dust_oracle.masked([s], 29)[0] == m


def _plain_params(**kw) -> FilterParams:
    p = FilterParams(min_q=-1.0, head_trim=0, tail_trim=0, min_len=1, filter=False, **kw)
    return p.apply_read_type("ont")


def _threshold_batch():
    """Pieces of 1 000 bases: A^(64+r), C, then random bases, M = 66 + r at level 29 (windows r + 1 and r + 2 still hold
    61 and 60 equal triplets).  With min_frac 0.076 (ppm 76 000) the piece with M = 76 is dropped (M 10^6 = ppm L)
    and the one with M = 75 kept; L = 63 and 64 border the length rule."""
    rng = np.random.default_rng(4)
    seqs = [b"A" * (64 + r) + b"C" + _rand(rng, 1000 - 65 - r) for r in (10, 9)]
    seqs += [b"A" * 63, b"A" * 64, b"C" * 64 + b"N" * 30]
    return seqs, synth.pack_reads(seqs, [bytes(rng.integers(40, 70, len(s), dtype=np.uint8)) for s in seqs])


def test_oracle_piece_threshold():
    seqs, batch = _threshold_batch()
    assert list(dust_oracle.masked(seqs, 29)) == [76, 75, 0, 64, 64]
    params = _plain_params()
    _, pieces, cnt, _ = dust_oracle.run(params, batch, level=29, min_frac=0.076)
    assert list(pieces["status"]) == [_capi.PIECE_LOWCOMPLEX, _capi.PIECE_EMIT, _capi.PIECE_EMIT,
                                      _capi.PIECE_LOWCOMPLEX, _capi.PIECE_LOWCOMPLEX]
    assert pieces["sum_q"][0] == 0 and pieces["sum_q"][1] > 0
    # a dropped piece's clean step is taken back out: the clean side equals a run over the kept reads only, the raw
    # side a run over all of them
    _, _, c_all = oracle_lib.run(params, batch)
    keep = synth.pack_reads([seqs[1], seqs[2]], [bytes(batch.quals[int(batch.offsets[i]):int(batch.offsets[i + 1])])
                                                 for i in (1, 2)])
    _, _, c_keep = oracle_lib.run(params, keep)
    L = oracle_lib.layout(params)
    clean = np.zeros(L.n_u64, dtype=bool)
    for off, n in [(L.clean_hist, 256)] + \
            [(getattr(L, t), L.bc_len * 5) for t in ("clean5p_cnt", "clean5p_qual", "clean3p_cnt", "clean3p_qual")] + \
            [(getattr(L, t), L.max_bins * 5) for t in ("clean_bin_cnt", "clean_bin_qual")]:
        clean[off:off + n] = True
    assert np.array_equal(cnt[clean], c_keep[clean])
    raw = np.zeros(L.n_u64, dtype=bool)
    for off, n in [(L.raw_hist, 256)] + [(getattr(L, t), L.max_bins * 5) for t in ("raw_bin_cnt", "raw_bin_qual")]:
        raw[off:off + n] = True
    assert np.array_equal(cnt[raw], c_all[raw])
    _, p2, _, _ = dust_oracle.run(params, batch, level=29, min_frac=0.0761)
    assert p2["status"][0] == _capi.PIECE_EMIT


def test_oracle_keeps_repeat_and_contam_fields_of_dropped_pieces():
    rng = np.random.default_rng(6)
    genome = _rand(rng, 5000)
    seqs = [_repeat(rng, 2, 3000, 0.01), genome[:2500] + _repeat(rng, 1, 2500, 0.0), _repeat(rng, 300, 3000, 0.0)]
    batch = synth.pack_reads(seqs, [b"I" * len(s) for s in seqs])
    params = _plain_params(kmer=11, min_repeat=1)
    _, pieces, _, _ = dust_oracle.run(params, batch, contam=([genome], 17, 0.9))
    _, p0, _, _ = dust_oracle.run(params, batch, contam=([genome], 17, 0.9), level=30, min_frac=1.0)
    assert list(pieces["status"]) == [_capi.PIECE_LOWCOMPLEX, _capi.PIECE_LOWCOMPLEX, _capi.PIECE_EMIT]
    for f in ("repeat_len", "contam_hits"):
        assert np.array_equal(pieces[f], p0[f]), f
    assert pieces["contam_hits"][1] > 0 and pieces["repeat_len"][0] >= 1


# ---- CPU: argument checks -----------------------------------------------------------------------------
def test_abi_rejects_bad_arguments_without_a_device():
    lib = _capi.load()
    out = np.zeros(2, dtype=np.uint32)
    seq = np.frombuffer(b"ACGT" * 40, dtype=np.uint8)
    good = np.array([0, 80, 160], dtype=np.uint64)
    assert lib.tgsf_dust_detect(0, seq.ctypes.data, good.ctypes.data, 0, 7, None) == _capi.TGSF_OK
    bad = ((None, good.ctypes.data, 2, 7, out.ctypes.data), (seq.ctypes.data, None, 2, 7, out.ctypes.data),
           (seq.ctypes.data, good.ctypes.data, 2, 7, None),
           (seq.ctypes.data, np.array([1, 80, 160], dtype=np.uint64).ctypes.data, 2, 7, out.ctypes.data),
           (seq.ctypes.data, np.array([0, 100, 80], dtype=np.uint64).ctypes.data, 2, 7, out.ctypes.data),
           (seq.ctypes.data, np.array([0, 1 << 31], dtype=np.uint64).ctypes.data, 1, 7, out.ctypes.data),
           (seq.ctypes.data, good.ctypes.data, 2, 31, out.ctypes.data),
           (seq.ctypes.data, good.ctypes.data, 2, -1, out.ctypes.data),
           (seq.ctypes.data, good.ctypes.data, 2, 0, out.ctypes.data))
    for args in bad:
        assert lib.tgsf_dust_detect(0, *args) == _capi.TGSF_ERR_INVALID, args
    assert lib.tgsf_set_dust(None, 7, 0.5) == _capi.TGSF_ERR_INVALID


def _cli_reject(tmp_path, args):
    if not os.path.exists(EXE):
        pytest.skip("src/tgsfilter not built")
    fq = tmp_path / "r.fq"
    fq.write_bytes(b"@r\n" + b"ACGT" * 300 + b"\n+\n" + b"I" * 1200 + b"\n")
    cmd = [EXE, "-i", str(fq), "-x", "ont", "-o", str(tmp_path / "o.fq")] + args
    pr = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=60)
    assert pr.returncode != 0
    assert not (tmp_path / "o.fq").exists()
    return pr.stderr.decode()


@pytest.mark.parametrize("extra", [["--qc"], ["-A"], ["-F"]])
def test_cli_rejects_dust_with(tmp_path, extra):
    assert "--dust" in _cli_reject(tmp_path, ["--dust"] + extra)


@pytest.mark.parametrize("args", [["--dust-level", "0"], ["--dust-level", "31"], ["--dust-frac", "0"],
                                  ["--dust-frac", "1.5"]])
def test_cli_rejects_dust_values(tmp_path, args):
    assert args[0] in _cli_reject(tmp_path, ["--dust"] + args)


# ---- GPU ---------------------------------------------------------------------------------------------
def _straddling(rng, L: int, borders, unit_lens=(1, 2, 3)) -> bytes:
    """Random L bases with a short repeat (64-400 bases, some with N runs and lower case) across each border."""
    s = bytearray(_rand(rng, L))
    for i, b in enumerate(borders):
        n = int(rng.integers(64, 400))
        r = bytearray(_repeat(rng, unit_lens[i % len(unit_lens)], n, 0.02))
        if i % 3 == 1:
            r[n // 2:n // 2 + 5] = b"NNNNN"
        if i % 4 == 2:
            r = bytearray(bytes(r).lower())
        lo = max(0, min(L - n, b - int(rng.integers(0, n))))
        s[lo:lo + n] = r
    return bytes(s)


def _gpu_detect_cases():
    rng = np.random.default_rng(41)
    seqs = _detector_cases() + [s for _, s, _ in _score_boundary_pieces()] + [g[1] for g in GAP_CASES]
    seqs += _threshold_batch()[0]
    seqs += [b"A", _rand(rng, 1), _rand(rng, 62)]
    # a single chunk: lane borders at multiples of ceil((L - 63) / 32) windows
    for L in (2000, 5000, 16447):
        span = (L - 63 + 31) // 32
        seqs.append(_straddling(rng, L, [span * k + 31 for k in range(1, 32, 3)]))
    # several chunks: repeats across the chunk borders (16 384 windows) and their halos
    for L in (16448, 40000, 100_000):
        seqs.append(_straddling(rng, L, [16384 * k + d for k in range(1, L // 16384 + 1) for d in (-40, 0, 30, 63)]))
    big = bytearray(_straddling(rng, 1_000_000, list(range(10_000, 1_000_000, 9_000))))
    big[500_000:500_200] = b"N" * 200
    seqs.append(bytes(big))
    seqs.append(_repeat(rng, 2, 200_000, 0.03))
    return seqs


@pytest.mark.gpu
def test_gpu_dust_detect_matches_oracle():
    from tgsfilter_b200.engine import dust_detect
    seqs = _gpu_detect_cases()
    for level in (7, 1, 29):
        got = dust_detect(seqs, level)
        want = dust_oracle.masked(seqs, level)
        assert np.array_equal(got, want), (level, np.nonzero(got != want)[0][:5])
    assert (dust_detect(seqs, 7) > 0).sum() >= 40


def _with_junk(batch, frac, seed, fasta=False):
    """Replace a share of the reads by low-complexity sequence of the same length: whole reads, or a stretch of 20-90 %
    of the read (on both sides of the 0.5 default), units 1-4 with up to 5 % errors (qualities kept)."""
    rng = np.random.default_rng(seed)
    b = batch.bases.copy()
    planted = []
    for r in range(batch.n_reads):
        s, e = int(batch.offsets[r]), int(batch.offsets[r + 1])
        if e - s < 200 or rng.random() >= frac:
            continue
        n = e - s if rng.random() < 0.4 else int((e - s) * rng.uniform(0.2, 0.9))
        junk = _repeat(rng, int(rng.integers(1, 5)), n, float(rng.uniform(0.0, 0.05)))
        lo = s + int(rng.integers(0, e - s - n + 1))
        b[lo:lo + n] = np.frombuffer(junk, dtype=np.uint8)
        planted.append(r)
    b[5::9973] = ord("n")
    return synth.ReadBatch(b, None if fasta else batch.quals, batch.offsets, batch.names), planted


def _run_gpu(params, batch, path="submit", contam=None, foldback=False, dust=(7, 0.5)):
    from tgsfilter_b200.engine import FilterEngine
    with FilterEngine(params) as eng:
        if contam is not None:
            eng.set_contaminants(contam[0], k=contam[1], min_frac=contam[2])
        if foldback:
            eng.set_foldback(True)
        if dust is not None:
            eng.set_dust(*dust)
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
        stats = eng.foldback_stats() if foldback else None
        return reads, pieces, eng.counters().flat, stats, eng.launch_count()


def _assert_parity(got, want):
    reads, pieces, cnt, stats = got[:4]
    o_reads, o_pieces, o_cnt, o_stats = want
    assert np.array_equal(reads, o_reads)
    assert len(pieces) == len(o_pieces)
    for f in o_pieces.dtype.names:
        assert np.array_equal(pieces[f], o_pieces[f]), (f, np.nonzero(pieces[f] != o_pieces[f])[0][:5])
    assert np.array_equal(cnt, o_cnt)
    if o_stats is not None:
        assert tuple(int(x) for x in o_stats) == stats


GPU_CASES = [
    # cfg, n, path, fasta, extra params, contaminant set, fold-back screen, (level, min_frac)
    (1, 300, "submit", False, {}, False, False, (7, 0.5)),    # hifi
    (2, 400, "packed", False, {}, False, False, (7, 0.5)),    # ont
    (4, 400, "device", False, {}, False, False, (7, 0.5)),    # clr
    (3, 60, "submit", False, {"max_read_len": 1 << 20}, False, False, (7, 0.5)),  # long ONT reads: many chunks
    (2, 300, "submit", True, {}, False, False, (7, 0.5)),     # FASTA
    (2, 300, "packed", False, {"discard": True}, False, False, (7, 0.5)),  # -D
    (5, 200, "submit", False, {"min_repeat": 20}, False, False, (7, 0.5)),  # -k 11 -p 20
    (1, 200, "device", False, {"kmer": 17, "min_repeat": 40}, False, False, (4, 0.2)),
    (2, 300, "submit", False, {}, True, False, (7, 0.5)),     # --contam
    (2, 300, "packed", False, {}, False, True, (7, 0.5)),     # --foldback
    (4, 300, "submit", False, {"kmer": 12, "min_repeat": 3}, True, True, (9, 0.5)),  # both
]


@pytest.mark.gpu
@pytest.mark.parametrize("cfg,n,path,fasta,extra,with_contam,foldback,dust", GPU_CASES)
def test_gpu_dust_parity(cfg, n, path, fasta, extra, with_contam, foldback, dust):
    batch = synth.make_config(cfg, n, max_len=None if cfg == 3 else 200_000)
    if foldback:
        from test_foldback import _with_folds
        batch, _ = _with_folds(batch, 0.2, cfg + 50, fasta)
    batch, planted = _with_junk(batch, 0.2, cfg, fasta)
    params = synth.config_params(cfg)
    for key, v in extra.items():
        setattr(params, key, v)
    contam = None
    if with_contam:
        genome = synth.make_contaminant(48_502)
        batch, _, _ = synth.mix_contaminants(batch, genome, 0.08, 0.04, chimeras=0.05, seed=cfg)
        contam = ([genome], 17, 0.05)
    got = _run_gpu(params, batch, path, contam, foldback, dust)
    want = dust_oracle.run(params, batch, dust[0], dust[1], contam, foldback)
    _assert_parity(got, want)
    assert (want[1]["status"] == _capi.PIECE_LOWCOMPLEX).sum() >= len(planted) // 4 > 0


@pytest.mark.gpu
def test_gpu_dust_thresholds_in_the_pipeline():
    _, batch = _threshold_batch()
    params = _plain_params()
    got = _run_gpu(params, batch, dust=(29, 0.076))
    want = dust_oracle.run(params, batch, 29, 0.076)
    _assert_parity(got, want)
    assert list(want[1]["status"]) == [_capi.PIECE_LOWCOMPLEX, _capi.PIECE_EMIT, _capi.PIECE_EMIT,
                                       _capi.PIECE_LOWCOMPLEX, _capi.PIECE_LOWCOMPLEX]


@pytest.mark.gpu
def test_gpu_dust_through_the_pool_overflow_retry():
    from test_gpu_parity import _pool_overflow_case
    params, pool = _pool_overflow_case()
    rng = np.random.default_rng(9)
    extra = [_repeat(rng, int(rng.integers(1, 4)), int(rng.integers(1500, 6000)), 0.02) for _ in range(20)]
    extra += [_rand(rng, int(rng.integers(1500, 6000))) for _ in range(20)]
    seqs = [pool.read(i)[0].tobytes() for i in range(pool.n_reads)] + extra
    batch = synth.pack_reads(seqs, [bytes([50] * len(s)) for s in seqs])
    got = _run_gpu(params, batch)
    want = dust_oracle.run(params, batch)
    _assert_parity(got, want)
    assert (want[1]["status"] == _capi.PIECE_LOWCOMPLEX).sum() >= 20


@pytest.mark.gpu
def test_gpu_dust_two_batches_in_flight():
    from tgsfilter_b200.engine import FilterEngine
    b1, _ = _with_junk(synth.make_config(2, 300), 0.2, 61)
    b2, _ = _with_junk(synth.make_config(4, 300), 0.2, 62)
    params = synth.config_params(2)
    w1 = dust_oracle.run(params, b1)
    w2 = dust_oracle.run(params, b2)
    with FilterEngine(params) as eng:
        eng.set_dust(7, 0.5)
        eng.submit(b1)
        eng.submit(b2)
        r1, p1 = eng.collect()
        r2, p2 = eng.collect()
        cnt = eng.counters().flat
    _assert_parity((r1, p1, w1[2], None), w1)
    _assert_parity((r2, p2, w2[2], None), w2)
    assert np.array_equal(cnt, w1[2] + w2[2])
    assert (p1["status"] == _capi.PIECE_LOWCOMPLEX).any() and (p2["status"] == _capi.PIECE_LOWCOMPLEX).any()


@pytest.mark.gpu
def test_gpu_dust_off_changes_nothing():
    """Never set, set then turned off with level 0: reads, pieces, counters and launches equal the oracle's plain run."""
    from tgsfilter_b200.engine import FilterEngine
    batch, _ = _with_junk(synth.make_config(2, 300), 0.3, 2)
    params = synth.config_params(2)
    r0, p0, c0, _, l0 = _run_gpu(params, batch, dust=None)
    with FilterEngine(params) as eng:
        eng.set_dust(7, 0.5)
        eng.set_dust(0, 0.5)
        r1, p1 = eng.run(batch)
        c1, l1 = eng.counters().flat, eng.launch_count()
    assert np.array_equal(r0, r1) and np.array_equal(p0, p1) and np.array_equal(c0, c1) and l0 == l1
    o_reads, o_pieces, o_cnt = oracle_lib.run(params, batch)
    assert np.array_equal(p0, o_pieces) and np.array_equal(c0, o_cnt)
    r2, p2, c2, _, l2 = _run_gpu(params, batch)
    assert l2 > l0 and (p2["status"] == _capi.PIECE_LOWCOMPLEX).any()


@pytest.mark.gpu
def test_gpu_dust_state_and_arguments():
    from tgsfilter_b200.engine import FilterEngine
    batch = synth.make_config(1, 50)
    with FilterEngine(synth.config_params(1)) as eng:
        for level, frac in ((31, 0.5), (-1, 0.5), (7, 0.0), (7, 1.5), (7, float("nan"))):
            assert eng._lib.tgsf_set_dust(eng._ctx, level, frac) == _capi.TGSF_ERR_INVALID
        assert eng._lib.tgsf_set_dust(eng._ctx, 0, 0.0) == _capi.TGSF_OK
        eng.submit(batch)
        with pytest.raises(_capi.TgsfError) as e:
            eng.set_dust(7, 0.5)
        assert e.value.code == _capi.TGSF_ERR_STATE
        eng.collect()


@pytest.mark.gpu
def test_gpu_dust_only_qc_is_a_no_op():
    from tgsfilter_b200.engine import FilterEngine
    batch, _ = _with_junk(synth.make_config(2, 200), 0.3, 7)
    params = FilterParams(filter=False, only_qc=True, adapters=[])
    r0, p0, c0, _, l0 = _run_gpu(params, batch, dust=None)
    with FilterEngine(params) as eng:
        eng.set_dust(7, 0.5)
        r1, p1 = eng.run(batch)
        c1, l1 = eng.counters().flat, eng.launch_count()
    assert np.array_equal(r0, r1) and np.array_equal(p0, p1) and np.array_equal(c0, c1) and l0 == l1
    assert (p1["status"] == _capi.PIECE_QC_ONLY).all()


@pytest.mark.gpu
def test_gpu_dust_deflate_blocks():
    from tgsfilter_b200.engine import FilterEngine
    from test_contam import _gz_members
    batch, _ = _with_junk(synth.make_config(2, 200), 0.3, 12)
    params = synth.config_params(2)
    params.gz_blocks = True
    with FilterEngine(params) as eng:
        eng.set_dust(7, 0.5)
        eng.submit(batch)
        blob, spans = eng.collect_gz()
        _, pieces = eng.collect()
    _, o_pieces, _, _ = dust_oracle.run(params, batch)
    assert np.array_equal(pieces, o_pieces)
    dropped = pieces["status"] == _capi.PIECE_LOWCOMPLEX
    assert dropped.sum() > 0 and (spans["bytes"][dropped] == 0).all()
    members, texts = _gz_members(batch, o_pieces, blob, spans, fastq=True)
    assert gzip.decompress(b"".join(members)) == b"".join(texts)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [1, 2, 3, 4, 5])
def test_gpu_unplanted_configs_drop_nothing(cfg):
    """Config-shaped reads without planted junk, config 5's 50-500 bp tandem repeats included: no piece is dropped at
    the defaults, and the results equal the oracle's."""
    n = {1: 300, 2: 600, 3: 80, 4: 600, 5: 200}[cfg]
    batch = synth.make_config(cfg, n)
    params = synth.config_params(cfg)
    params.max_read_len = 1 << 20
    got = _run_gpu(params, batch)
    want = dust_oracle.run(params, batch)
    _assert_parity(got, want)
    assert not (got[1]["status"] == _capi.PIECE_LOWCOMPLEX).any()


# ---- CLI on the GPU ----------------------------------------------------------------------------------
def _fastq_records(data: bytes):
    lines = data.split(b"\n")
    return sorted(b"\n".join(lines[i:i + 4]) for i in range(0, len(lines) - 3, 4))


def _info(stderr: bytes, needle: str):
    return [ln for ln in stderr.decode().splitlines() if needle in ln]


@pytest.fixture(scope="module")
def cli_inputs(tmp_path_factory):
    """ONT reads with planted junk reads, and junk pieces: reads split by a middle adapter with one side junk."""
    d = tmp_path_factory.mktemp("dust_cli")
    batch, _ = _with_junk(synth.make_config(2, 2000), 0.1, 31)
    rng = np.random.default_rng(32)
    b = batch.bases.copy()
    for r in rng.choice(batch.n_reads, 150, replace=False):
        s, e = int(batch.offsets[r]), int(batch.offsets[r + 1])
        if e - s < 3000:
            continue
        mid = s + (e - s) // 2
        ad = synth.mutate(ADAPTER_LIB[8], 0.02, rng)
        b[mid:mid + len(ad)] = np.frombuffer(ad, dtype=np.uint8)
        junk = _repeat(rng, int(rng.integers(1, 4)), mid - s - 200, 0.02)
        lo = s + 100 if rng.random() < 0.5 else mid + len(ad) + 100
        hi = min(lo + len(junk), e)
        b[lo:hi] = np.frombuffer(junk[:hi - lo], dtype=np.uint8)
    batch = synth.ReadBatch(b, batch.quals, batch.offsets, batch.names)
    fq = d / "reads.fq"
    fq.write_bytes(batch.to_fastq())
    ad = d / "ad.fa"
    ad.write_bytes(b">ad\n" + ADAPTER_LIB[8] + b"\n")
    return d, batch, fq, ad


def _cli(d, fq, args, env=None, out_name="o.fq"):
    out = d / out_name
    pr = subprocess.run([EXE, "-i", str(fq), "-o", str(out), "-x", "ont", "-5", "0", "-3", "0", "-q", "10",
                         "-l", "1000"] + args,
                        stdout=subprocess.PIPE, stderr=subprocess.PIPE, env={**os.environ, **(env or {})}, timeout=600)
    assert pr.returncode == 0, pr.stderr.decode()[-2000:]
    return (out.read_bytes() if out.exists() else b""), pr.stderr


def _cli_expect(batch, level, frac):
    params = FilterParams(min_q=10.0, head_trim=0, tail_trim=0, min_len=1000,
                          adapters=[ADAPTER_LIB[8], rev_comp(ADAPTER_LIB[8])]).apply_read_type("ont")
    _, o_pieces, _, _ = dust_oracle.run(params, batch, level, frac)
    expect = sorted(t.rstrip(b"\n") for t, _, _ in records.format_records(batch, o_pieces, fastq=True))
    dropped = o_pieces["status"] == _capi.PIECE_LOWCOMPLEX
    return expect, int(dropped.sum()), int(o_pieces["len"][dropped].sum()), o_pieces


@pytest.mark.gpu
def test_cli_dust_matches_oracle(cli_inputs):
    d, batch, fq, ad = cli_inputs
    out, err = _cli(d, fq, ["-a", str(ad), "--dust"])
    expect, n, nb, o_pieces = _cli_expect(batch, 7, 0.5)
    assert _fastq_records(out) == expect
    split = np.bincount(o_pieces["read"][o_pieces["status"] == _capi.PIECE_LOWCOMPLEX], minlength=batch.n_reads)
    assert n > 150 and ((split > 0) & (np.bincount(o_pieces["read"], minlength=batch.n_reads) > 1)).sum() > 20
    assert _info(err, "low complexity") == [f"INFO: {n} reads were discarded with {nb} bases as low complexity."]
    lines = _info(err, "INFO:")
    assert lines.index(_info(err, "low complexity")[0]) == lines.index(_info(err, "short length")[0]) + 2
    out2, err2 = _cli(d, fq, ["-a", str(ad), "--dust", "--gpus", "2"],
                      env={"TGSF_SHARE_DEVICES": "1", "TGSF_BATCH_MB": "4"}, out_name="o2.fq")
    assert _fastq_records(out2) == expect
    assert [ln for ln in _info(err2, "INFO:") if "written to" not in ln] == \
        [ln for ln in _info(err, "INFO:") if "written to" not in ln]
    out3, _ = _cli(d, fq, ["-a", str(ad), "--dust"], out_name="o3.fq.gz")
    assert _fastq_records(gzip.decompress(out3)) == expect
    _, err0 = _cli(d, fq, ["-a", str(ad)], out_name="o0.fq")
    assert not _info(err0, "low complexity")


@pytest.mark.gpu
def test_cli_dust_level_and_frac(cli_inputs):
    d, batch, fq, ad = cli_inputs
    out, err = _cli(d, fq, ["-a", str(ad), "--dust", "--dust-level", "4", "--dust-frac", "0.3"], out_name="l4.fq")
    expect, n, nb, _ = _cli_expect(batch, 4, 0.3)
    assert _fastq_records(out) == expect
    assert _info(err, "low complexity") == [f"INFO: {n} reads were discarded with {nb} bases as low complexity."]

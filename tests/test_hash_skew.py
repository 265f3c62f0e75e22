"""The repeat check's hash kernel (k_kmer) and the fold-back screen's hash tables on pieces built to crowd one hash
pass, against the oracle.

Natural sequence spreads its keys over the passes within about 1 %, so the code that runs when a pass fills its table
never runs on it.  The generators here restate the kernels' hashes and partition rules and build pieces base by base,
taking a base whose new key lands in the pass they aim at whenever one does.  The CPU tests check that each piece does
what it was built for (they also parse the constants they rely on from the kernel headers, so that a changed constant
fails here instead of quietly making the pieces harmless); the GPU tests compare the kernels bit-exact with the oracle
on them."""
from __future__ import annotations

import functools
import os
import random
import re

import numpy as np
import pytest

import foldback_oracle
import oracle_lib
from tgsfilter_b200 import _capi, records, synth
from tgsfilter_b200.params import ADAPTER_LIB, FilterParams, rev_comp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "tgsfilter_b200", "csrc")
EXE = os.path.join(ROOT, "src", "tgsfilter")
_M32 = 0xFFFFFFFF
_M64 = (1 << 64) - 1


def _source(name: str) -> str:
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _defines(*names: str) -> dict:
    """The integer #defines of the kernel headers, evaluated (u suffixes dropped, earlier defines substituted)."""
    out = {}
    for name in names:
        for m in re.finditer(r"^#define\s+(\w+)\s+([^/\n]+)", _source(name), re.M):
            expr = re.sub(r"\b(0x[0-9a-fA-F]+|\d+)u\b", r"\1", m.group(2).strip())
            expr = re.sub(r"\b[A-Z][A-Z0-9_]+\b", lambda t: str(out.get(t.group(0), t.group(0))), expr)
            try:
                out[m.group(1)] = int(eval(expr, {"__builtins__": {}}))
            except Exception:
                pass
    return out


D = _defines("kmer16.cuh", "kmer.cuh", "foldback.cuh")


# ---- k_kmer (kmer.cuh): hash, partition, table ------------------------------------------------------------------
def mix32(x: int) -> int:
    x ^= x >> 33
    x = (x * 0xFF51AFD7ED558CCD) & _M64
    x ^= x >> 33
    x = (x * 0xC4CEB9FE1A85EC53) & _M64
    x ^= x >> 33
    return x & _M32


def kmer_slots(k: int) -> int:
    """Table slots of k_kmer at k: u32 keys for k <= 15, u64 above (launch_kmer)."""
    return D["KMER_SMEM_BYTES"] // (4 if k <= 15 else 8)


def kmer_limit(k: int) -> int:
    """Distinct keys one pass may hold; one more splits the pass."""
    return kmer_slots(k) // 4 * 3


def kmer_passes(total: int, k: int) -> int:
    half = kmer_slots(k) // 2
    return (total + half - 1) // half


def kmer_pass(h: int, passes: int) -> int:
    return ((h >> 8) * passes) >> 24


_BASE = {ord("C"): 1, ord("G"): 2, ord("T"): 3}  # every other byte is A's code (T.cpp:1709-1724)


def kmer_keys(seq: bytes, k: int) -> set:
    mask = (1 << (2 * k)) - 1
    km, keys = 0, set()
    for i, b in enumerate(seq):
        km = ((km << 2) | _BASE.get(b, 0)) & mask
        if i >= k - 1:
            keys.add(km)
    return keys


def kmer_pass_fill(seq: bytes, k: int, passes: int = 0) -> list:
    """Distinct keys per pass of k_kmer (at the piece's own pass count unless given)."""
    passes = passes or kmer_passes(len(seq) - k + 1, k)
    fill = [0] * passes
    for key in kmer_keys(seq, k):
        fill[kmer_pass(mix32(key), passes)] += 1
    return fill


def repeat_len(seq: bytes, k: int) -> int:
    total = len(seq) - k + 1
    return total - 1 if total <= 0 else total - len(kmer_keys(seq, k))


@functools.lru_cache(maxsize=None)
def skewed_kmer_piece(k: int, L: int, target_fill: int, seed: int) -> bytes:
    """L bases whose pass 0 of k_kmer gets target_fill distinct keys (or as many as the greedy walk finds, if fewer):
    while it has fewer, take a base whose new k-mer is a new pass-0 key if any is; after that, a base whose k-mer is
    not and after which the walk can go on for three more bases without one."""
    rng = random.Random(seed)
    passes = kmer_passes(L - k + 1, k)
    mask = (1 << (2 * k)) - 1
    codes = [rng.randrange(4) for _ in range(k - 1)]
    km = 0
    for c in codes:
        km = (km << 2) | c
    seen = set()

    def new0(x):
        return x not in seen and kmer_pass(mix32(x), passes) == 0

    def free(x, depth):
        return not new0(x) and (depth == 0 or any(free(((x << 2) | c) & mask, depth - 1) for c in range(4)))

    for _ in range(L - k + 1):
        opts = [0, 1, 2, 3]
        rng.shuffle(opts)
        cand = [((km << 2) | c) & mask for c in opts]
        if len(seen) < target_fill:
            pick = next((j for j, x in enumerate(cand) if new0(x)), 0)
        else:
            pick = next((j for j, x in enumerate(cand) if free(x, 3)), None)
            assert pick is not None, "the walk is stuck: try another seed"
        km = cand[pick]
        codes.append(opts[pick])
        if kmer_pass(mix32(km), passes) == 0:
            seen.add(km)
    return bytes(b"ACGT"[c] for c in codes)


def _tandem(rng: np.random.Generator, L: int, unit: int) -> bytes:
    u = synth._ACGT[rng.integers(0, 4, unit, dtype=np.uint8)].tobytes()
    return (u * (L // unit + 1))[:L]


def _rand(rng: np.random.Generator, L: int) -> bytes:
    return synth._ACGT[rng.integers(0, 4, L, dtype=np.uint8)].tobytes()


# k = 13 .. 16: pieces of more than KMER16_MAX_KMERS k-mers, which k_kmer_tag16 hands to k_kmer; k > 16: k_kmer takes
# every piece
KMER_K = [13, 15, 16, 17, 21, 31]


def _kmer_len(k: int) -> int:
    return 82_000 if k <= 16 else 28_000


def kmer_cases(k: int):
    """(name, piece) of one batch at k: two pieces over the table's slots, two one key above the pass limit, two at
    the limit, and ordinary random and tandem-repeat pieces of the same length."""
    L = _kmer_len(k)
    lim, slots = kmer_limit(k), kmer_slots(k)
    out = []
    for j in range(2):
        out.append((f"over_slots_{j}", skewed_kmer_piece(k, L, slots + 500, 10 * k + j)))
        out.append((f"limit_plus_1_{j}", skewed_kmer_piece(k, L, lim + 1, 20 * k + j)))
        out.append((f"at_limit_{j}", skewed_kmer_piece(k, L, lim, 30 * k + j)))
    rng = np.random.default_rng(k)
    out += [("random_0", _rand(rng, L)), ("random_1", _rand(rng, L - 777))]
    out += [("tandem_0", _tandem(rng, L, 5000)), ("tandem_1", _rand(rng, L // 2) + _tandem(rng, L - L // 2, 300))]
    return out


# ---- fold-back screen (foldback.cuh): sampling, key, tables -----------------------------------------------------
def fold_fmix32(h: int) -> int:
    h ^= h >> 16
    h = (h * 0x85EBCA6B) & _M32
    h ^= h >> 13
    h = (h * 0xC2B2AE35) & _M32
    return h ^ (h >> 16)


def fold_smem_limit() -> int:
    return D["FOLD_SMEM_SLOTS"] // 4 * 3


def fold_global_limit() -> int:
    return D["FOLD_GLOBAL_SLOTS"] // 4 * 3


def fold_global_passes(L: int) -> int:
    w = L - (D["FOLD_K"] - 1)
    return (w + D["FOLD_GLOBAL_WINDOWS_PER_PASS"] - 1) // D["FOLD_GLOBAL_WINDOWS_PER_PASS"]


def fold_sampled_keys(seq: bytes) -> set:
    """Distinct canonical 15-mer keys of the sampled windows (ACGT only; the generators below make no other byte)."""
    K = D["FOLD_K"]
    mask = (1 << (2 * K)) - 1
    f = r = 0
    keys = set()
    for i, b in enumerate(seq):
        c = "ACGT".index(chr(b))
        f = ((f << 2) | c) & mask
        r = (r >> 2) | ((3 - c) << (2 * (K - 1)))
        if i >= K - 1:
            key = min(f, r)
            if not fold_fmix32(key) & D["FOLD_SAMPLE_MASK"]:
                keys.add(key)
    return keys


def fold_pass_fill(seq: bytes, passes: int) -> list:
    fill = [0] * passes
    for key in fold_sampled_keys(seq):
        fill[(fold_fmix32(key) * passes) >> 32] += 1
    return fill


@functools.lru_cache(maxsize=None)
def skewed_fold_piece(L: int, seed: int) -> bytes:
    """L bases, taking a base whose canonical 15-mer is sampled whenever one is."""
    rng = random.Random(seed)
    K = D["FOLD_K"]
    mask = (1 << (2 * K)) - 1
    codes = [rng.randrange(4) for _ in range(K - 1)]
    f = r = 0
    for c in codes:
        f = ((f << 2) | c) & mask
        r = (r >> 2) | ((3 - c) << (2 * (K - 1)))
    for _ in range(L - K + 1):
        opts = [0, 1, 2, 3]
        rng.shuffle(opts)
        pick = opts[0]
        for c in opts:
            nf, nr = ((f << 2) | c) & mask, (r >> 2) | ((3 - c) << (2 * (K - 1)))
            if not fold_fmix32(min(nf, nr)) & D["FOLD_SAMPLE_MASK"]:
                pick = c
                break
        f, r = ((f << 2) | pick) & mask, (r >> 2) | ((3 - pick) << (2 * (K - 1)))
        codes.append(pick)
    return bytes(b"ACGT"[c] for c in codes)


@functools.lru_cache(maxsize=None)
def skewed_fold_read(arm: int, err: float, seed: int, frac: float = 0.8) -> bytes:
    """X·rc(X'): a skewed arm X, then the reverse complement of its last frac·arm bases, both with errors."""
    rng = np.random.default_rng(seed)
    x = skewed_fold_piece(arm, seed)
    return synth.mutate(x, err, rng) + synth.mutate(rev_comp(x[arm - int(arm * frac):]), err, rng)


FOLD_ARMS = (3000, 8000, 16_000, 22_000, 60_000)


def fold_pieces():
    """The fold_detect cases: skewed pieces through the shared-memory limit, past its length, through the global
    path's pass doubling, skewed folds, and ordinary pieces beside them."""
    rng = np.random.default_rng(3)
    seqs = [skewed_fold_piece(20_000, 1), skewed_fold_piece(40_960, 2), skewed_fold_piece(40_961, 3),
            skewed_fold_piece(190_000, 4)]
    seqs += [skewed_fold_read(arm, 0.01, 10 + i) for i, arm in enumerate(FOLD_ARMS)]
    seqs += [_rand(rng, 20_000), _rand(rng, 40_960)]
    return seqs


# ---- CPU: the constants the generators rely on -------------------------------------------------------------------
def test_kernel_constants_match_the_restatement():
    assert D["KMER_SMEM_BYTES"] == 128 * 1024 and D["KMER_MAX_PASSES"] == 1 << 24
    assert D["KMER16_MAX_KMERS"] == 65_000
    assert (kmer_slots(13), kmer_slots(15), kmer_slots(16), kmer_slots(31)) == (32_768, 32_768, 16_384, 16_384)
    assert (D["FOLD_K"], D["FOLD_SAMPLE_MASK"], D["FOLD_SMEM_SLOTS"], D["FOLD_SMEM_MAX_LEN"]) == (15, 7, 8192, 40_960)
    assert (D["FOLD_GLOBAL_SLOTS"], D["FOLD_GLOBAL_WINDOWS_PER_PASS"], D["FOLD_MAX_PASSES"]) == (65_536, 196_608, 1 << 14)
    kmer = _source("kmer.cuh")
    assert "min(SLOTS / 4u * 3u, fill_cap)" in kmer
    assert "(u32)(((u64)(h >> 8) * passes) >> 24) != pass" in kmer
    assert "((u32)total + SLOTS / 2 - 1) / (SLOTS / 2)" in kmer
    assert "return (u32)x;" in kmer and "0xff51afd7ed558ccdull" in kmer and "0xc4ceb9fe1a85ec53ull" in kmer
    fold = _source("foldback.cuh")
    assert "const u32 limit = T.slots / 4u * 3u;" in fold
    assert "(u32)(((u64)h * passes) >> 32) != pass" in fold
    assert "h *= 0x85ebca6bu;" in fold and "h *= 0xc2b2ae35u;" in fold
    launch = _source("tgsf_cuda.cu")
    assert "else if (P.kmer <= 15)\n        k_kmer<u32>" in launch


def test_split_pass_is_two_passes_of_the_finer_partition():
    """Partition p of P passes is exactly partitions 2p and 2p + 1 of 2P, so a split pass loses nothing done."""
    rng = random.Random(5)
    for _ in range(20_000):
        x, P = rng.randrange(1 << 24), rng.randrange(1, 1 << 23)
        assert kmer_pass(x << 8, 2 * P) // 2 == kmer_pass(x << 8, P)
    for x in (0, 1, (1 << 24) - 1):
        for P in (1, 3, 6, 1 << 23):
            assert kmer_pass(x << 8, 2 * P) // 2 == kmer_pass(x << 8, P)


# ---- CPU: the pieces do what they were built to do ---------------------------------------------------------------
@pytest.mark.parametrize("k", KMER_K)
def test_skewed_kmer_pieces_crowd_one_pass(k):
    L = _kmer_len(k)
    lim, slots = kmer_limit(k), kmer_slots(k)
    for name, s in kmer_cases(k):
        assert len(s) >= L - 777
        total = len(s) - k + 1
        if k <= 16:
            assert total > D["KMER16_MAX_KMERS"]
        fill = kmer_pass_fill(s, k)
        if name.startswith("over_slots"):
            assert fill[0] > slots, fill
            assert max(kmer_pass_fill(s, k, 2 * len(fill))) <= lim  # one split is enough
        elif name.startswith("limit_plus_1"):
            assert fill[0] == lim + 1 and max(fill[1:]) < lim, fill
        elif name.startswith("at_limit"):
            assert fill[0] == lim and max(fill[1:]) < lim, fill
        else:
            assert max(fill) < lim * 3 // 4, fill


def test_skewed_fold_pieces_overflow_both_tables():
    s = skewed_fold_piece(40_960, 2)
    assert len(s) == D["FOLD_SMEM_MAX_LEN"]  # the longest piece the shared-memory path takes
    assert len(fold_sampled_keys(s)) > fold_smem_limit()
    assert len(fold_sampled_keys(skewed_fold_piece(20_000, 1))) > fold_smem_limit()
    big = skewed_fold_piece(190_000, 4)
    P = fold_global_passes(len(big))
    assert P == 1
    assert max(fold_pass_fill(big, P)) > fold_global_limit()
    assert max(fold_pass_fill(big, 2 * P)) <= fold_global_limit()
    for i in (2, 3):  # skewed folds short enough for the shared-memory path overflow its table too
        r = skewed_fold_read(FOLD_ARMS[i], 0.01, 10 + i)
        assert len(r) <= D["FOLD_SMEM_MAX_LEN"] and len(fold_sampled_keys(r)) > fold_smem_limit()


@functools.lru_cache(maxsize=None)
def colliding_kmers(k: int = 17, seed: int = 7):
    """Two k-mers whose mix32 >> 8 agree: they share a pass at every pass count (birthday search)."""
    rng = random.Random(seed)
    seen = {}
    tries = 0
    while True:
        tries += 1
        x = rng.randrange(1 << (2 * k))
        h = mix32(x) >> 8
        if h in seen and seen[h] != x:
            return seen[h], x, tries
        seen[h] = x


def _kmer_text(x: int, k: int) -> bytes:
    return bytes(b"ACGT"[(x >> (2 * (k - 1 - i))) & 3] for i in range(k))


def test_colliding_kmers_share_every_pass():
    a, b, tries = colliding_kmers()
    assert a != b and tries < 20_000
    piece = _kmer_text(a, 17) + _kmer_text(b, 17)
    assert {a, b} <= kmer_keys(piece, 17)
    for P in (1, 2, 3, 1000, D["KMER_MAX_PASSES"]):
        assert kmer_pass(mix32(a), P) == kmer_pass(mix32(b), P)


# ---- GPU: k_kmer ---------------------------------------------------------------------------------------------------
def _kmer_params(k: int, p: int, max_read_len: int = 1 << 20) -> FilterParams:
    return FilterParams(min_len=50, min_q=0.0, kmer=k, min_repeat=p, qtype=33, adapters=[],
                        max_read_len=max_read_len)


def _both_ways(seqs, k: int) -> int:
    """A -p bound some of the pieces fall below and some do not."""
    reps = sorted({repeat_len(s, k) for s in seqs})
    assert len(reps) >= 2
    return reps[len(reps) // 2]


def _kmer_batch(k: int):
    seqs = [s for _, s in kmer_cases(k)]
    return synth.pack_reads(seqs, [b"I" * len(s) for s in seqs]), seqs


@pytest.mark.gpu
@pytest.mark.parametrize("sm", [None, "1"], ids=["grid", "one_sm"])
@pytest.mark.parametrize("k", KMER_K)
def test_gpu_kmer_on_skewed_pieces_matches_oracle(k, sm, monkeypatch):
    """Pieces that overflow a pass, pass its limit by one key and sit at it, beside ordinary pieces; on one SM a
    single CTA takes them all in a row."""
    from test_gpu_parity import _compare
    if sm:
        monkeypatch.setenv("TGSF_SM_COUNT", sm)
    batch, seqs = _kmer_batch(k)
    p = _both_ways(seqs, k)
    _, pieces, _ = _compare(_kmer_params(k, p), batch)
    assert len(pieces) == len(seqs) and list(pieces["len"]) == [len(s) for s in seqs]
    assert list(pieces["repeat_len"]) == [repeat_len(s, k) for s in seqs]
    st = pieces["status"]
    assert (st == _capi.PIECE_SHORT_REPEAT).any() and (st == _capi.PIECE_EMIT).any()


@pytest.mark.gpu
def test_gpu_kmer_fill_cap_config5_k21(monkeypatch):
    """TGSF_KMER_FILL_CAP=64: nearly every pass of every piece is split, the counts stay exact."""
    from test_gpu_parity import _compare
    monkeypatch.setenv("TGSF_KMER_FILL_CAP", "64")
    batch = synth.make_config(5, 200)
    params = synth.config_params(5)
    params.kmer = 21
    _, pieces, _ = _compare(params, batch)
    st = pieces["status"]
    assert (st == _capi.PIECE_SHORT_REPEAT).any() and (st == _capi.PIECE_EMIT).any()


@pytest.mark.gpu
def test_gpu_kmer_fill_cap_long_pieces_k13(monkeypatch):
    from test_gpu_parity import _compare, _repeat_batch
    monkeypatch.setenv("TGSF_KMER_FILL_CAP", "64")
    batch = _repeat_batch(113, long_read=[450000, 19000, 33000, 64990, 65100])
    _, pieces, _ = _compare(_kmer_params(13, 200, 500000), batch)
    assert (pieces["status"] != 0).any() and (pieces["status"] == 0).any()


@pytest.mark.gpu
def test_gpu_kmer_pass_cap_fails_the_batch(monkeypatch):
    """Two k-mers that share a pass at every pass count, one key allowed per pass: the split reaches KMER_MAX_PASSES
    and tgsf_collect reports the batch as failed.  The context takes the next batch as usual."""
    from tgsfilter_b200.engine import FilterEngine
    monkeypatch.setenv("TGSF_KMER_FILL_CAP", "1")
    a, b, _ = colliding_kmers()
    piece = _kmer_text(a, 17) + _kmer_text(b, 17)
    bad = synth.pack_reads([piece], [b"I" * len(piece)])
    rng = np.random.default_rng(1)
    good_seqs = [_rand(rng, 300), _tandem(rng, 500, 40)]
    good = synth.pack_reads(good_seqs, [b"I" * len(s) for s in good_seqs])
    params = _kmer_params(17, 5, 0)
    params.min_len = 1  # the piece is 34 bases
    with FilterEngine(params) as eng:
        with pytest.raises(_capi.TgsfError) as e:
            eng.run(bad)
        assert e.value.code == _capi.TGSF_ERR_CAPACITY and "hash pass" in str(e.value)
        reads, pieces = eng.run(good)
    o_reads, o_pieces, _ = oracle_lib.run(params, good)
    assert np.array_equal(reads, o_reads) and np.array_equal(pieces, o_pieces)


# ---- GPU: fold-back ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_fold_detect_on_skewed_pieces_matches_oracle():
    from tgsfilter_b200.engine import fold_detect
    seqs = fold_pieces()
    got = fold_detect(seqs)
    want = foldback_oracle.detect(seqs)
    for f in ("fold", "anchors", "centre", "min_gap"):
        assert np.array_equal(got[f], want[f]), (f, np.nonzero(got[f] != want[f])[0][:5])
    assert (want["fold"][4:9] >= 0).sum() >= 4


def _pipeline_batch():
    """Skewed k = 21 pieces, skewed folds and the skewed fold-back pieces in one batch."""
    kseqs = [s for name, s in kmer_cases(21) if not name.startswith(("random", "tandem"))]
    fseqs = fold_pieces()
    rng = np.random.default_rng(8)
    seqs = kseqs + fseqs + [_tandem(rng, 9000, 700), _rand(rng, 15_000)]
    return synth.pack_reads(seqs, [b"I" * len(s) for s in seqs]), seqs, len(kseqs)


def _fold_params(p: int) -> FilterParams:
    return FilterParams(min_q=10.0, head_trim=0, tail_trim=0, min_len=2000, kmer=21, min_repeat=p,
                        adapters=[ADAPTER_LIB[8], rev_comp(ADAPTER_LIB[8])], max_read_len=1 << 20).apply_read_type("ont")


@pytest.mark.gpu
@pytest.mark.parametrize("sm", [None, "1"], ids=["grid", "one_sm"])
def test_gpu_foldback_and_kmer_split_in_one_batch(sm, monkeypatch):
    from test_foldback import _assert_parity, _run_gpu
    if sm:
        monkeypatch.setenv("TGSF_SM_COUNT", sm)
    batch, seqs, n_kmer = _pipeline_batch()
    params = _fold_params(_both_ways(seqs[:n_kmer] + seqs[-2:], 21))
    want = foldback_oracle.run(params, batch)
    _assert_parity(_run_gpu(params, batch), want)
    pieces = want[1]
    whole = [int(pieces["len"][np.nonzero(pieces["read"] == i)[0][0]]) for i in range(n_kmer)]
    assert whole == [len(s) for s in seqs[:n_kmer]]  # k_kmer saw the crowded pieces whole
    assert want[3][0] >= 4  # and the fold screen cut skewed folds
    st = pieces["status"]
    assert (st == _capi.PIECE_SHORT_REPEAT).any() and (st == _capi.PIECE_EMIT).any()


@pytest.mark.gpu
def test_cli_skewed_reads_match_oracle(tmp_path):
    from test_foldback import _cli, _fastq_records, _info
    if not os.path.exists(EXE):
        pytest.skip("src/tgsfilter not built")
    batch, seqs, _ = _pipeline_batch()
    plain = synth.make_config(5, 300)  # a third of its reads carry tandem repeats: -k 21 -p 1 keeps those
    seqs = seqs + [plain.read(i)[0].tobytes() for i in range(plain.n_reads)]
    quals = [b"I" * len(s) for s in seqs[:batch.n_reads]] + \
        [plain.read(i)[1].tobytes() for i in range(plain.n_reads)]
    names = [b"r%d" % i for i in range(len(seqs))]
    batch = synth.pack_reads(seqs, quals, names)
    fq = tmp_path / "reads.fq"
    fq.write_bytes(batch.to_fastq())
    ad = tmp_path / "ad.fa"
    ad.write_bytes(b">ad\n" + ADAPTER_LIB[8] + b"\n")
    out, err = _cli(tmp_path, fq, ["-a", str(ad), "--foldback", "-l", "2000", "-k", "21", "-p", "1"])
    params = _fold_params(1)
    _, o_pieces, _, st = foldback_oracle.run(params, batch)
    expect = sorted(t.rstrip(b"\n") for t, _, _ in records.format_records(batch, o_pieces, fastq=True))
    assert _fastq_records(out) == expect and len(expect) > 50
    assert st[0] >= 4
    assert _info(err, "fold-back") == [
        f"INFO: {st[0]} reads were cut at a fold-back junction, removing {st[1]} bases.",
        f"INFO: {st[2]} reads were discarded with {st[3]} bases as too short after a fold-back cut."]

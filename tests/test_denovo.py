"""De novo adapter assembly (--adapter-denovo): k_end_kmers / tgsf_end_kmer_counts against a numpy count, the host
assembly (prepass.assemble_adapter) on planted row sets, and the CLI on synthetic ONT reads with an adapter that is
not in the library.

Row sets for the assembly rules use 'N' outside the planted sequences, so every count is exact and each rule can be
put on its boundary.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tgsfilter_b200 import _capi, prepass, synth
from tgsfilter_b200.params import ADAPTER_LIB, FilterParams, rev_comp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "src", "tgsfilter")
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
K = prepass.DENOVO_K
_CODE = np.full(256, -1, dtype=np.int64)
_CODE[np.frombuffer(b"ACGT", dtype=np.uint8)] = np.arange(4)


def np_counts(rows: np.ndarray, k: int, split: int):
    """(outer, inner) [4^k] u32 counts of the valid windows row[j, j+k) with j < split / j >= split."""
    outer = np.zeros(1 << (2 * k), dtype=np.uint32)
    inner = np.zeros_like(outer)
    n, c = rows.shape
    w = c - k + 1
    if n == 0 or w <= 0:
        return outer, inner
    step = max(1, (1 << 22) // c)
    for lo in range(0, n, step):
        v = _CODE[rows[lo:lo + step]]
        code = np.zeros((v.shape[0], w), dtype=np.int64)
        valid = np.ones((v.shape[0], w), dtype=bool)
        for i in range(k):
            code = (code << 2) | np.maximum(v[:, i:i + w], 0)
            valid &= v[:, i:i + w] >= 0
        for table, sl in ((outer, slice(0, min(split, w))), (inner, slice(min(split, w), w))):
            x = code[:, sl][valid[:, sl]]
            u, cnt = np.unique(x, return_counts=True)
            table[u] += cnt.astype(np.uint32)
    return outer, inner


def assemble(rows: np.ndarray) -> bytes:
    n, c = rows.shape
    O, I = np_counts(rows, K, prepass.denovo_split(c))
    return prepass.assemble_adapter(O, I, n, K, c)


def blank(n: int, c: int = 150) -> np.ndarray:
    return np.full((n, c), ord("N"), dtype=np.uint8)


def put(rows: np.ndarray, r, col: int, seq: bytes) -> None:
    rows[r, col:col + len(seq)] = np.frombuffer(seq, dtype=np.uint8)


def rand_seq(n: int, seed: int) -> bytes:
    return ACGT[np.random.default_rng(seed).integers(0, 4, n)].tobytes()


def edit_distance(a: bytes, b: bytes) -> int:
    prev = list(range(len(b) + 1))
    for i in range(1, len(a) + 1):
        cur = [i] + [0] * len(b)
        for j in range(1, len(b) + 1):
            cur[j] = min(prev[j] + 1, cur[j - 1] + 1, prev[j - 1] + (a[i - 1] != b[j - 1]))
        prev = cur
    return prev[-1]


def infix_distance(q: bytes, t: bytes) -> int:
    """Edit distance of q against its best substring of t (free ends in t)."""
    prev = [0] * (len(t) + 1)
    for i in range(1, len(q) + 1):
        cur = [i] + [0] * len(t)
        for j in range(1, len(t) + 1):
            cur[j] = min(prev[j] + 1, cur[j - 1] + 1, prev[j - 1] + (q[i - 1] != t[j - 1]))
        prev = cur
    return min(prev)


# ---- the assembly rules (CPU) --------------------------------------------------------------------------------
ADAPTER = b"GATTCCAGTACGGTCATAGCTGTTACGA"  # 28 bases, >= 3 distinct bases and no long run in every 12-mer


def test_assembles_a_planted_adapter_with_random_flanks():
    """Random lead-in and random read body: the extension stops at both ends by the 1/2 cut."""
    rng = np.random.default_rng(1)
    rows = ACGT[rng.integers(0, 4, (3000, 150), dtype=np.uint8)]
    ad = rand_seq(45, 2)
    for r in np.nonzero(rng.random(3000) < 0.5)[0]:
        put(rows, r, int(rng.integers(0, 20)), ad)
    assert assemble(rows) == ad


def test_half_cut_boundary():
    """The branch after the adapter is followed while 2 x its count >= the seed's count, not below."""
    tail, other = b"CATGGACTTAGCAGTCCGAT", b"TGCACTGATCAGGCTAACTG"
    for n_tail, expect in ((200, ADAPTER + tail), (199, ADAPTER)):
        rows = blank(1000)
        put(rows, slice(0, 400), 0, ADAPTER)
        put(rows, slice(0, n_tail), len(ADAPTER), tail)
        put(rows, slice(n_tail, n_tail + 150), len(ADAPTER), other)  # fewer rows than the tail: never the best branch
        assert assemble(rows) == expect, n_tail


def test_extension_tie_takes_the_first_base():
    """Two branches with the same count: A before C before G before T, on the right and on the left."""
    b1, b2 = b"CATGGACTTAGCAGTCCGAT", b"GTCAACTGATCAGGCTAACT"
    rows = blank(1000)
    put(rows, slice(0, 400), 40, ADAPTER)
    put(rows, slice(0, 200), 40 + len(ADAPTER), b2)
    put(rows, slice(200, 400), 40 + len(ADAPTER), b1)
    put(rows, slice(0, 200), 40 - len(b1), b1[::-1])  # left branches end in T / C next to the adapter
    put(rows, slice(200, 400), 40 - len(b2), b2[::-1])
    left = b1[::-1] if b1[0] < b2[0] else b2[::-1]
    assert assemble(rows) == left + ADAPTER + b1


def test_seed_tie_takes_the_smallest_code():
    """Two adapters in as many rows: the seed is the smallest code of all their k-mers, and only its adapter is
    assembled."""
    other = b"TCAGGCATTGACCGTAGTCAAGTGCT"
    rows = blank(1000)
    put(rows, slice(0, 300), 0, ADAPTER)
    put(rows, slice(300, 600), 0, other)
    codes = {}
    for s in (ADAPTER, other):
        for j in range(len(s) - K + 1):
            codes[int(sum(int(_CODE[b]) << (2 * (K - 1 - i)) for i, b in enumerate(s[j:j + K])))] = s
    assert assemble(rows) == codes[min(codes)]


def test_cycle_in_a_tandem_adapter_stops_the_extension():
    """A tandem of a 15-base unit: the path stops when a k-mer comes round again, one unit plus k - 1 bases long."""
    unit = b"ACGTTGCAGCATGAC"
    rows = blank(1000)
    put(rows, slice(0, 500), 0, unit * 5)
    cand = assemble(rows)
    assert len(cand) == len(unit) + K - 1
    assert cand in unit * 5


def test_length_cap():
    """A 140-base adapter: the candidate stops at 100 bases, the whole extension included."""
    ad = rand_seq(140, 3)
    rows = blank(500, 150)
    put(rows, slice(0, 300), 0, ad)
    cand = assemble(rows)
    assert len(cand) == prepass.DENOVO_MAX_LEN and cand in ad


@pytest.mark.parametrize("length", [19, 20])
def test_shorter_than_20_is_rejected(length):
    ad = ADAPTER[:length]
    rows = blank(500)
    put(rows, slice(0, 200), 0, ad)
    assert assemble(rows) == (ad if length >= prepass.DENOVO_MIN_LEN else b"")


@pytest.mark.parametrize("n,rows_with,ok", [(1000, 20, True), (1000, 19, False), (3000, 30, True), (3000, 29, False)])
def test_support_rule(n, rows_with, ok):
    """O >= max(20, ceil(n / 100))."""
    rows = blank(n)
    put(rows, slice(0, rows_with), 0, ADAPTER)
    assert assemble(rows) == (ADAPTER if ok else b"")


@pytest.mark.parametrize("inner,ok", [(9, True), (10, False)])
def test_enrichment_rule(inner, ok):
    """O >= 4 (I + 1): 40 outer copies allow 9 inner copies of every k-mer, not 10."""
    rows = blank(1000)
    put(rows, slice(0, 40), 0, ADAPTER)
    put(rows, slice(40, 40 + inner), 100, ADAPTER)  # windows from column 100 on: the inner half of a 150-base row
    assert assemble(rows) == (ADAPTER if ok else b"")


@pytest.mark.parametrize("seq,ok", [
    ((b"AACCAACCACAC" * 4)[:40], False),               # two distinct bases in every 12-mer
    ((b"AAAAACG" * 6)[:40], False),                    # a run of 5 in every 12-mer
    (b"AAAACGTTTTGCAAAAGTCCCCATGGGGACTTTTCAGGGG", True),  # runs of 4 are allowed
])
def test_seed_complexity_rules(seq, ok):
    """Low-complexity sequence in many rows cannot seed; a valid adapter in fewer rows is then assembled."""
    rows = blank(2000)
    put(rows, slice(0, 800), 0, seq)
    put(rows, slice(800, 900), 0, ADAPTER)
    assert assemble(rows) == (seq if ok else ADAPTER)


def test_no_rows_and_short_rows():
    O = np.zeros(1 << (2 * K), dtype=np.uint32)
    assert prepass.assemble_adapter(O, O, 0, K, 150) == b""
    assert prepass.assemble_adapter(O, O, 100, K, K - 1) == b""
    with pytest.raises(ValueError):
        prepass.assemble_adapter(O[:-1], O[:-1], 100, K, 150)


# ---- the ABI's argument checks (CPU: a call that reached the device would fail with TGSF_ERR_CUDA) -------------
def _call(rows, n, row_len, k, outer=True, inner=True):
    so = _capi.load()
    t = np.ones(1 << (2 * min(max(k, 1), 13)), dtype=np.uint32)
    rc = so.tgsf_end_kmer_counts(0, None if rows is None else rows.ctypes.data, n, row_len, k, 0,
                                 t.ctypes.data if outer else None, t.ctypes.data if inner else None)
    return rc, so.tgsf_last_error().decode(), t


ROWS8 = np.zeros(64, dtype=np.uint8)


@pytest.mark.parametrize("args", [
    dict(rows=ROWS8, n=2, row_len=8, k=0), dict(rows=ROWS8, n=2, row_len=8, k=14), dict(rows=ROWS8, n=2, row_len=8, k=-3),
    dict(rows=None, n=2, row_len=8, k=4), dict(rows=ROWS8, n=2, row_len=8, k=4, outer=False),
    dict(rows=ROWS8, n=2, row_len=8, k=4, inner=False),
    dict(rows=ROWS8, n=1 << 31, row_len=3, k=2), dict(rows=ROWS8, n=(1 << 32) - 1, row_len=14, k=13),
], ids=["k0", "k14", "k_negative", "no_rows", "no_outer", "no_inner", "2^32_windows", "2^33-2_windows"])
def test_end_kmer_counts_rejects_bad_arguments_before_touching_the_gpu(args):
    rc, err, _ = _call(**args)
    assert rc == _capi.TGSF_ERR_INVALID, (rc, err)
    assert err.startswith("end_kmer_counts"), err


@pytest.mark.parametrize("n,row_len,k", [(0, 150, 12), (0, 5, 1), (5, 11, 12), (3, 0, 1)])
def test_end_kmer_counts_without_windows_zeroes_the_tables_on_the_host(n, row_len, k):
    rows = np.zeros(max(n * row_len, 1), dtype=np.uint8)
    rc, err, t = _call(rows, n, row_len, k)
    assert rc == _capi.TGSF_OK, err
    assert not t.any()


# ---- the CLI's argument checks (CPU) ------------------------------------------------------------------------
@pytest.mark.parametrize("args", [["-a", "{fa}"], ["--qc"], ["-F", "-r", "10"]], ids=["a", "qc", "F"])
def test_cli_rejects_adapter_denovo_with(tmp_path, args):
    """These fail in argument parsing, before any device call (so also without a GPU)."""
    if not os.path.exists(EXE):
        pytest.skip("src/tgsfilter not built")
    fa = tmp_path / "a.fa"
    fa.write_bytes(b">a\n" + ADAPTER + b"\n")
    fq = tmp_path / "r.fq"
    fq.write_bytes(b"@r\n" + b"ACGT" * 300 + b"\n+\n" + b"I" * 1200 + b"\n")
    cmd = [EXE, "-i", str(fq), "-x", "ont", "-o", str(tmp_path / "o.fq"), "--adapter-denovo"] + \
        [a.format(fa=fa) for a in args]
    pr = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=60)
    assert pr.returncode != 0
    err = pr.stderr.decode()
    assert "Error:" in err and "--adapter-denovo" in err, err
    assert not (tmp_path / "o.fq").exists()


# ---- k_end_kmers on the GPU ---------------------------------------------------------------------------------
def _sm_count() -> int:
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


_NOISY = np.frombuffer(b"ACGTacgtN\0", dtype=np.uint8)
_NOISY_P = np.array([0.23] * 4 + [0.01] * 4 + [0.02, 0.02])
_rows_cache: dict = {}


def _noisy_rows(n: int, row_len: int) -> np.ndarray:
    key = (n, row_len)
    if key not in _rows_cache:
        _rows_cache.clear()
        rng = np.random.default_rng(n * 7919 + row_len)
        _rows_cache[key] = _NOISY[rng.choice(len(_NOISY), size=(n, row_len), p=_NOISY_P / _NOISY_P.sum())]
    return _rows_cache[key]


@pytest.mark.gpu
@pytest.mark.parametrize("n_kind", ["0", "1", "7", "grid"])
@pytest.mark.parametrize("row_len", [1, 11, 12, 13, 150, 3073])
@pytest.mark.parametrize("k", [1, 5, 11, 12, 13])
def test_end_kmer_counts_vs_numpy(k, row_len, n_kind):
    """Rows of ACGT sprinkled with acgt, N and NUL.  'grid' is more rows than one grid-stride pass of k_end_kmers covers
    (8 warps x 8 CTAs per SM).  The split is the assembly's for row_len >= k, else 3."""
    n = 64 * _sm_count() + 5 if n_kind == "grid" else int(n_kind)
    rows = _noisy_rows(n, row_len)
    split = prepass.denovo_split(row_len, k) if row_len >= k else 3
    O, I = prepass.device_end_kmers(rows, k, split)
    eO, eI = np_counts(rows, k, split)
    assert np.array_equal(O, eO)
    assert np.array_equal(I, eI)
    if n >= 7 and row_len >= 150:
        assert O.any() and I.any()


@pytest.mark.gpu
@pytest.mark.parametrize("split", [0, 1, 69, 138, 139, 1000])
def test_end_kmer_counts_cli_sample(split):
    """The CLI's default sample: 100 000 rows of 150 bases at k = 12, split anywhere from 0 to past the last window."""
    rows = _noisy_rows(100_000, 150)
    O, I = prepass.device_end_kmers(rows, 12, split)
    eO, eI = np_counts(rows, 12, split)
    assert np.array_equal(O, eO) and np.array_equal(I, eI)


# ---- the CLI on the GPU -------------------------------------------------------------------------------------
def _novel_adapter() -> bytes:
    """A seeded random 45-mer more than 30 % edits away from every library adapter and its reverse complement."""
    for seed in range(100):
        ad = rand_seq(45, 4500 + seed)
        if all(infix_distance(ad, t) > 0.3 * 45 and infix_distance(t, ad) > 0.3 * len(t)
               for a in ADAPTER_LIB for t in (a, rev_comp(a))):
            return ad
    raise AssertionError("no novel adapter")


NOVEL = _novel_adapter()


def _ont_reads(n, seed, lo=1000, hi=3000, ad5=None, ad3=None, f5=0.8, f3=0.6):
    """n ONT-like reads of lo..hi bases, Phred+33 qualities 5..40; ad5 with 10 % errors after a 0-30-base lead-in at
    the 5' end of a fraction f5 of the reads, the reverse complement of ad3 likewise at the 3' end of f3."""
    rng = np.random.default_rng(seed)
    seqs = []
    for _ in range(n):
        s = ACGT[rng.integers(0, 4, int(rng.integers(lo, hi + 1)))].tobytes()
        if ad5 is not None and rng.random() < f5:
            s = rand_seq(int(rng.integers(0, 31)), int(rng.integers(1 << 30))) + synth.mutate(ad5, 0.10, rng) + s
        if ad3 is not None and rng.random() < f3:
            s = s + synth.mutate(rev_comp(ad3), 0.10, rng) + rand_seq(int(rng.integers(0, 31)), int(rng.integers(1 << 30)))
        seqs.append(s)
    quals = [(rng.integers(5, 41, len(s)) + 33).astype(np.uint8).tobytes() for s in seqs]
    return synth.pack_reads(seqs, quals)


def _write(path, batch):
    synth.write_fastq(str(path), batch.bases, batch.quals, batch.offsets)


def _run(cwd, fq, args, env=None):
    if not os.path.exists(EXE):
        subprocess.run(["make", "-C", os.path.join(ROOT, "src")], check=True, stdout=subprocess.DEVNULL)
    os.makedirs(cwd, exist_ok=True)
    pr = subprocess.run([EXE, "-i", str(fq)] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=900,
                        cwd=cwd, env={**os.environ, **(env or {})})
    err = pr.stderr.decode("utf-8", "replace")
    assert pr.returncode == 0, err[-2000:]
    return err


PREPASS = ("INFO: trim 5'", "INFO: trim 3'", "INFO: de novo", "INFO: mean depth", "INFO: 5' adapter",
           "INFO: 3' adapter", "INFO: set ")


def _prepass_lines(err: str):
    return [ln for ln in err.splitlines() if ln.startswith(PREPASS)]


def _denovo_lines(err: str):
    return [ln for ln in err.splitlines() if ln.startswith(("INFO: de novo", "INFO: mean depth of de novo"))]


def _line_value(err: str, prefix: str) -> str:
    (ln,) = [ln for ln in err.splitlines() if ln.startswith(prefix)]
    return ln[len(prefix):]


@pytest.fixture(scope="module")
def novel(tmp_path_factory):
    d = tmp_path_factory.mktemp("denovo")
    batch = _ont_reads(6000, 45, ad5=NOVEL, ad3=NOVEL)
    fq = d / "reads.fq"
    _write(fq, batch)
    return d, batch, fq


@pytest.mark.gpu
def test_cli_assembles_a_novel_adapter(novel):
    d, batch, fq = novel
    err = _run(d / "a", fq, ["-x", "ont", "-A", "--adapter-denovo"])
    c5 = _line_value(err, "INFO: de novo 5' adapter: ").encode()
    c3 = _line_value(err, "INFO: de novo 3' adapter: ").encode()
    # the 3' rows are the reverse complement of the read tails: they carry the adapter in its own orientation
    assert edit_distance(c5, NOVEL) <= 4, (c5, NOVEL)
    assert edit_distance(c3, NOVEL) <= 4, (c3, NOVEL)
    params = FilterParams().apply_read_type("ont")
    _, res = prepass.run_prepass(batch, params, "ont", denovo=True)
    i = next(j for j, ln in enumerate(res.log) if ln.startswith("INFO: 3' adapter")) + 1
    expect = res.log[:i] + [f"INFO: mean depth of 5' adapter: {res.dep5p:g}",
                            f"INFO: mean depth of 3' adapter: {res.dep3p:g}"]
    assert _prepass_lines(err) == expect
    assert res.adapter5p == c5 and res.adapter3p == c3
    assert res.dep5p >= 6000 / 100 and res.dep3p >= 6000 / 100
    # without the flag the library finds nothing and the run falls back to the rapid adapter
    err0 = _run(d / "b", fq, ["-x", "ont", "-o", "out.fq"])
    assert not _denovo_lines(err0)
    assert "INFO: set NanoPore rapid adapter to trim: " + ADAPTER_LIB[8].decode() in err0.splitlines()


def _filter_info(err: str):
    """The counter lines of the main pass (input, drop and trim counts, output)."""
    return [ln for ln in err.splitlines() if ln.startswith("INFO: ") and
            (" reads " in ln or " bases were trimmed" in ln) and "written to" not in ln]


@pytest.mark.gpu
def test_cli_denovo_run_equals_the_run_with_its_candidates(novel):
    """The full run with --adapter-denovo filters exactly like -a with the printed candidates."""
    d, batch, fq = novel
    err = _run(d / "dn", fq, ["-x", "ont", "-o", "out.fq", "--adapter-denovo"], env={"TGSF_DUMP_COUNTERS": "cnt.bin"})
    c5 = _line_value(err, "INFO: de novo 5' adapter: ")
    c3 = _line_value(err, "INFO: de novo 3' adapter: ")
    assert c5 and c3
    (d / "fa").mkdir()
    (d / "fa" / "cand.fa").write_bytes(f">c5\n{c5}\n>c3\n{c3}\n".encode())
    err_a = _run(d / "fa", fq, ["-x", "ont", "-o", "out.fq", "-a", "cand.fa"], env={"TGSF_DUMP_COUNTERS": "cnt.bin"})
    assert (d / "dn" / "out.fq").read_bytes() == (d / "fa" / "out.fq").read_bytes()
    assert (d / "dn" / "cnt.bin").read_bytes() == (d / "fa" / "cnt.bin").read_bytes()
    assert _filter_info(err) == _filter_info(err_a)
    counts = {ln.split(" ", 2)[2]: int(ln.split(" ")[1]) for ln in _filter_info(err) if "have adapter" in ln}
    num5p = sum(v for key, v in counts.items() if "5'" in key)
    planted = int(round(0.8 * batch.n_reads))
    print(f"num5p {num5p} of about {planted} planted 5' adapters")
    assert num5p >= 0.6 * planted, counts


def _repeat_reads(n, seed):
    """Reads of 1-3 kb; 30 % carry a 300-bp interspersed repeat with 2 % errors at a uniformly random position."""
    rng = np.random.default_rng(seed)
    rep = rand_seq(300, seed + 1)
    seqs = []
    for _ in range(n):
        s = ACGT[rng.integers(0, 4, int(rng.integers(1000, 3001)))].tobytes()
        if rng.random() < 0.30:
            m = synth.mutate(rep, 0.02, rng)
            p = int(rng.integers(0, len(s) - len(m) + 1))
            s = s[:p] + m + s[p + len(m):]
        seqs.append(s)
    quals = [(rng.integers(5, 41, len(s)) + 33).astype(np.uint8).tobytes() for s in seqs]
    return synth.pack_reads(seqs, quals), rep


def _poly_reads(n, seed):
    """Reads of 1-3 kb; 70 % start with 10-40 T and end with 10-40 A."""
    rng = np.random.default_rng(seed)
    seqs = []
    for _ in range(n):
        s = ACGT[rng.integers(0, 4, int(rng.integers(1000, 3001)))].tobytes()
        if rng.random() < 0.7:
            s = b"T" * int(rng.integers(10, 41)) + s + b"A" * int(rng.integers(10, 41))
        seqs.append(s)
    quals = [(rng.integers(5, 41, len(s)) + 33).astype(np.uint8).tobytes() for s in seqs]
    return synth.pack_reads(seqs, quals)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["random", "repeat", "poly", "config2"])
def test_cli_no_false_adapters(case, tmp_path):
    """No candidate is accepted, and records, report and every other line equal the run without the flag."""
    rep = None
    if case == "random":
        batch = _ont_reads(4000, 7)
    elif case == "repeat":
        batch, rep = _repeat_reads(20000, 11)
    elif case == "poly":
        batch = _poly_reads(4000, 13)
    else:
        batch = synth.make_config(2, 3000)
    fq = tmp_path / "reads.fq"
    _write(fq, batch)
    if rep is not None:  # the repeat's top k-mer clears the support: only the enrichment rule rejects it
        params = FilterParams().apply_read_type("ont")
        e5, _, _, _, _ = prepass.sample_ends(batch, params)
        n = e5.shape[0]
        O, I = np_counts(e5, K, prepass.denovo_split(e5.shape[1]))
        codes = [int(sum(int(_CODE[b]) << (2 * (K - 1 - i)) for i, b in enumerate(rep[j:j + K])))
                 for j in range(len(rep) - K + 1)]
        top = max(codes, key=lambda x: O[x])
        assert O[top] >= max(20, -(-n // 100)), (O[top], n)
        assert O[top] < 4 * (int(I[top]) + 1)
    env = {"TGSF_DUMP_COUNTERS": "cnt.bin"}
    err = _run(tmp_path / "dn", fq, ["-x", "ont", "-o", "out.fq", "--adapter-denovo"], env=env)
    err0 = _run(tmp_path / "plain", fq, ["-x", "ont", "-o", "out.fq"], env=env)
    dn = _denovo_lines(err)
    ends = ["3'"] if case == "config2" else ["5'", "3'"]
    assert dn == sum(([f"INFO: de novo {e} adapter: ", f"INFO: mean depth of de novo {e} adapter: 0"] for e in ends),
                     [])
    if case == "config2":
        assert "INFO: 5' adapter: " + ADAPTER_LIB[8].decode() in err0.splitlines()
    assert [ln for ln in err.splitlines() if ln not in dn] == err0.splitlines()
    for f in ("out.fq", "cnt.bin"):
        assert (tmp_path / "dn" / f).read_bytes() == (tmp_path / "plain" / f).read_bytes(), f
    assert _report(tmp_path / "dn" / "out.html") == _report(tmp_path / "plain" / "out.html")


def _report(path):
    """The HTML report without its last paragraph, which states the wall-clock time it was written at."""
    lines = path.read_bytes().splitlines()
    assert lines[-3].startswith(b"<p>Generated by tgsfilter"), lines[-3:]
    return lines[:-3] + lines[-2:]

"""The integer rules of the per-read path that decide where a read is cut and which pieces are kept, each tested
with plants on both sides of its threshold.

Adapter copies are built from explicit edit scripts (S substitutions, I inserted and D deleted bases) so that the
distance d, the aligned target length tl and the match count M = alen - d of every plant are known.  A plain int64
semi-global DP (``_hw``), which shares no code with the Myers kernels or the oracle, checks each fixture before it
goes to the GPU; the traceback length alen comes from ``oracle_lib.align_hw`` (pinned to edlib elsewhere).  From
(q, tl, d, thr) the file predicts which branch of ``mlen_decision`` every plant takes and whether it passes, and
the CPU tests assert that every boundary below has plants on both sides:

- end windows (``k_ends``): d against k_end, M against thr_end, all three ``mlen_decision`` outcomes, similarity
  thresholds hit exactly and moved by float rounding, checkLen 4 / 5 / 6, copies at the window's edges and
  several locations at one distance;
- middle window (``k_mid_scan`` / ``k_mid_count`` / ``k_mid_emit``): the window length against qLen, d against
  k_mid, M against thr_mid, degenerate match lengths, chunk minima above the u8 tag's 254 and the extra_len clip;
- pieces: fp64 mean quality at min_q / max_q and at the histogram's bin edges, piece lengths at min_len / max_len.

On the GPU every case is compared bit for bit with the oracle (``_compare``) and its intended outcome is asserted
directly; with the reference build the same fixtures go through the reference against the oracle."""
import dataclasses
import fractions
import functools

import numpy as np
import pytest

import oracle_lib
import ref_lib
from test_gpu_parity import _compare
from test_launch_regimes import _concat, _filler
from tgsfilter_b200 import _capi, records, synth
from tgsfilter_b200.params import FilterParams

ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
OFF = 1 << 20  # a match length no adapter reaches: switches the end or middle search off

needs_ref = pytest.mark.skipif(not ref_lib.available(), reason="oracle/_ref not built")


# ---------------------------------------------------------------------------------------------------------------
# plain reference and threshold arithmetic
# ---------------------------------------------------------------------------------------------------------------

def _last_row(q: bytes, t: bytes, free_start: bool) -> np.ndarray:
    """Last row of the unit-cost edit matrix of q (rows) against t (columns), int64.  free_start: row 0 is zero
    (the alignment may start at any column), else row 0 is j (global)."""
    qa, ta = np.frombuffer(q, np.uint8), np.frombuffer(t, np.uint8)
    j = np.arange(len(ta) + 1, dtype=np.int64)
    row = np.zeros_like(j) if free_start else j.copy()
    for i in range(1, len(qa) + 1):
        c = np.empty_like(j)
        c[0] = i
        c[1:] = np.minimum(row[:-1] + (ta != qa[i - 1]), row[1:] + 1)
        row = np.minimum.accumulate(c - j) + j  # row[j] = min(c[j], row[j - 1] + 1)
    return row


def _hw(q: bytes, t: bytes):
    """Best semi-global distance of q in t, every end column at that distance and the smallest start of the first
    of them (the start whose global distance to q is d)."""
    row = _last_row(q, t, True)
    d = int(row.min())
    ends = (np.nonzero(row == d)[0] - 1).tolist()  # column -1: the empty alignment, only when d == qLen
    e = ends[0]
    if e < 0:
        return d, ends, None
    back = _last_row(q[::-1], t[:e + 1][::-1], False)  # back[j] = NW(q, t[e - j + 1 .. e])
    start = e + 1 - int(np.nonzero(back == d)[0].max())
    return d, ends, start


def _min_mlen(q: int, sim: float) -> int:
    """Smallest m with (float)m / qLen >= sim, qLen + 1 if none (the float test of T.cpp:1250 / 1287)."""
    s = np.float32(sim)
    return next((m for m in range(q + 1) if np.float32(m) / np.float32(q) >= s), q + 1)


def _thresholds(q: int, match_len: int, sim: float):
    """(k, thr) as fill_thresholds sets them."""
    thr = max(_min_mlen(q, sim), match_len)
    k = min(q - match_len + 1, q - 1)
    return (0 if thr > q else k), thr


def _end_extra(q: int, sim: float) -> int:
    return int(np.float32(q) / np.float32(sim))


def mlen_decision(q, tl, d, thr):
    c = d - (tl - q)
    if q - ((c + 1) >> 1) < thr:
        return 0
    if q - c >= thr:
        return 1
    return -1


def _classify(ad: bytes, window: bytes, match_len: int, sim: float):
    """What one (adapter, window) search must give: the DP's distance and end columns, the branch and the
    outcome of the integer rules, checked against the reference's float expressions on the oracle's alignment."""
    q = len(ad)
    k, thr = _thresholds(q, match_len, sim)
    d, ends, start = _hw(ad, window)
    res, locs = oracle_lib.align_hw(ad, window, -1)
    assert res["edit_distance"] == d and [e for _, e in locs] == ends, (ad, window)
    if start is not None:
        # every location's smallest start is at least the first one's: two optimal paths that cross can swap
        # their tails, so a later location never starts further left
        assert locs[0][0] == start and min(s for s, _ in locs) == start
    alen = res["align_len"]
    tl = ends[0] - (start if start is not None else 0) + 1
    branch = mlen_decision(q, tl, d, thr) if d <= k else None
    passes = d <= k and (branch == 1 or (branch == -1 and alen - d >= thr))
    mlen = alen - d
    ref_max_k = q - match_len + 1
    ref_passes = ((ref_max_k < 0 or d <= ref_max_k) and mlen >= match_len
                  and np.float32(mlen) / np.float32(q) >= np.float32(sim))
    assert passes == ref_passes, (q, d, alen, k, thr, sim)
    return dict(q=q, d=d, k=k, thr=thr, M=mlen, tl=tl, branch=branch, passes=passes, ends=ends, start=start,
                traceback=None if branch != -1 else alen - d >= thr)


def _rand(rng, n, alphabet=ACGT):
    return alphabet[rng.integers(0, len(alphabet), n)].tobytes()


def plant(ad: bytes, S: int, I: int, D: int, rng) -> bytes:
    """Copy of ad with S substitutions, I inserted and D deleted bases at spread-out interior positions (never
    within 3 bases of either end, never two edits next to each other): d = S + I + D, tl = q - D + I,
    M = q - S - D when the script is optimal, which the DP checks."""
    q = len(ad)
    n = S + I + D
    slots = np.linspace(3, q - 4, n + 2)[1:-1].round().astype(int) if n else np.zeros(0, int)
    assert n <= 1 or np.diff(slots).min() >= 2, (q, S, I, D)
    ops = np.array(["S"] * S + ["I"] * I + ["D"] * D)
    rng.shuffle(ops)
    out = bytearray()
    edits = dict(zip(slots.tolist(), ops.tolist()))
    for i, b in enumerate(ad):
        op = edits.get(i)
        if op == "D":
            continue
        if op == "S":
            out.append(int(next(x for x in ACGT[rng.permutation(4)] if x != b)))
            continue
        out.append(b)
        if op == "I":
            nxt = ad[i + 1] if i + 1 < q else -1
            out.append(int(next(x for x in ACGT[rng.permutation(4)] if x != b and x != nxt)))
    return bytes(out)


def _scripts(k):
    """Edit scripts around d = k and M = thr = q - k + 1 (the match length of these cases is q - k + 1)."""
    s = [(0, 0, 0), (k - 2, 0, 0), (k - 1, 0, 0), (k, 0, 0), (k + 1, 0, 0), (0, k, 0), (0, k + 1, 0),
         (0, 0, k - 1), (0, 0, k), (1, 0, k - 2), (2, 0, k - 2), (1, 0, k - 1), (1, 2, k - 3), (0, 3, 3)]
    return [x for x in s if min(x) >= 0 and sum(x) <= k + 1]


class Case:
    """A batch, its parameters and the per-read outcome every device must reach."""

    def __init__(self, params, seqs, quals=None):
        self.params = params
        self.seqs = seqs
        self.quals = quals if quals is not None else [b"5" * len(s) for s in seqs]
        self.expect = {}   # read field -> expected int array
        self.plants = []   # classification dicts (one per planted search)

    @functools.cached_property
    def batch(self):
        return synth.pack_reads(self.seqs, self.quals)

    def expect_field(self, name, values):
        self.expect[name] = np.asarray(values, dtype=np.int64)


def _end_windows(case, match_len, sim):
    """Classify every (adapter, read end) search of an end case and set the expected n_5p / n_3p."""
    P = case.params
    n5, n3 = [], []
    for s in case.seqs:
        t5 = t3 = 0
        for ad in P.adapters:
            check = min(P.end_len + _end_extra(len(ad), sim), len(s))
            if check < 5:
                continue
            c5 = _classify(ad, s[:check], match_len, sim)
            c3 = _classify(ad, s[len(s) - check:], match_len, sim)
            c5["side"], c3["side"], c5["check"], c3["check"] = 5, 3, check, check
            case.plants += [c5, c3]
            t5 += len(c5["ends"]) if c5["passes"] else 0
            t3 += len(c3["ends"]) if c3["passes"] else 0
        n5.append(t5)
        n3.append(t3)
    case.expect_field("n_5p", n5)
    case.expect_field("n_3p", n3)


def _base_params(**kw):
    p = FilterParams(min_len=1, min_q=0.0, max_q=255.0, head_trim=0, tail_trim=0, extra_len=0, end_len=0,
                     end_match_len=OFF, mid_match_len=OFF, end_sim=0.5, mid_sim=0.5)
    for k, v in kw.items():
        setattr(p, k, v)
    return p


# ---------------------------------------------------------------------------------------------------------------
# end-window cases
# ---------------------------------------------------------------------------------------------------------------

END_LENGTHS = (22, 64, 65, 128, 150, 256, 257, 600)


@functools.lru_cache(maxsize=None)
def end_scripts_case(L):
    """Adapters of length L (NW = 1 .. 16 after round_nw), 2 or 3 of them, match length L - k + 1 (k_end = k).
    Every read carries one scripted copy at its 5' end and one at its 3' end."""
    rng = np.random.default_rng(1000 + L)
    k = 4 if L == 22 else 7
    n_ad = 3 if L in (64, 128, 256, 600) else 2
    ads = [_rand(rng, L) for _ in range(n_ad)]
    sim = 0.5
    P = _base_params(end_match_len=L - k + 1, end_sim=sim, end_len=10, adapters=ads)
    check = P.end_len + _end_extra(L, sim)
    seqs = []
    scripts = _scripts(k)
    for i, sc5 in enumerate(scripts):
        sc3 = scripts[(i + 5) % len(scripts)]
        a5, a3 = ads[i % n_ad], ads[(i + 1) % n_ad]
        c5, c3 = plant(a5, *sc5, rng), plant(a3, *sc3, rng)
        head = _rand(rng, 6) + c5
        tail = c3 + _rand(rng, 6)
        mid = _rand(rng, 2 * check - len(head) - len(tail) + 40)
        seqs.append(head + mid + tail)
    case = Case(P, seqs)
    _end_windows(case, P.end_match_len, sim)
    return case


SIM_CASES = ((64, 0.75), (128, 0.875), (100, 0.97), (200, 0.97), (150, 0.8), (22, 1.0))


@functools.lru_cache(maxsize=None)
def end_similarity_case():
    """The similarity decides the threshold (end_match_len 4): copies with M = thr - 1, thr, thr + 1 made of
    substitutions only or of substitutions and deleted bases, for (qLen, end_sim) pairs at which
    (float)thr / qLen == end_sim exactly and pairs at which float rounding moves the threshold by one match."""
    rng = np.random.default_rng(77)
    cases = []
    for L, sim in SIM_CASES:
        ad = _rand(rng, L)
        P = _base_params(end_match_len=4, end_sim=sim, end_len=8, adapters=[ad])
        _, thr = _thresholds(L, 4, sim)
        check = P.end_len + _end_extra(L, sim)
        seqs = []
        for dm in (-1, 0, 1):
            e = L - (thr + dm)  # edits that cost a match
            for sc in ((e, 0, 0), (e - e // 3, 0, e // 3), (e, 1, 0)):
                if min(sc) < 0:
                    continue
                cp = plant(ad, *sc, rng)
                head = _rand(rng, 4) + cp
                seqs.append(head + _rand(rng, 2 * check - len(head) + 30) + cp)
        case = Case(P, seqs)
        _end_windows(case, 4, sim)
        case.sim = (L, sim, thr)
        cases.append(case)
    return cases


@functools.lru_cache(maxsize=None)
def end_small_match_len_cases():
    """end_match_len 0 and 1 (k_end capped at qLen - 1) and end_sim 0.01, whose end_extra (2 200) is longer than
    every read, so checkLen is the read length: windows over G/T only (d = qLen, no alignment has a match) and
    with one or two adapter bases (d = qLen - 1, qLen - 2)."""
    rng = np.random.default_rng(5)
    ad = _rand(rng, 22, np.frombuffer(b"AC", np.uint8))
    out = []
    for em in (0, 1):
        P = _base_params(end_match_len=em, end_sim=0.01, end_len=20, adapters=[ad])
        gt = np.frombuffer(b"GT", np.uint8)
        seqs = [_rand(rng, 300, gt), _rand(rng, 150, gt) + b"A" + _rand(rng, 149, gt),
                _rand(rng, 140, gt) + b"AC" + _rand(rng, 160, gt), _rand(rng, 290, gt) + b"C" + _rand(rng, 3, gt)]
        case = Case(P, seqs)
        _end_windows(case, em, 0.01)
        out.append(case)
    return out


@functools.lru_cache(maxsize=None)
def end_edge_case():
    """Window edges with only exact copies passing (end_match_len = qLen, end_sim 1.0): reads of 4, 5 and 6 bases
    (checkLen 4 is skipped, 5 and 6 are scanned) with a 4-base adapter, and for a 22-base adapter 5' copies ending
    at the window's last column and one past it, 3' copies starting at its first column and one before it, two
    exact copies in one 5' window (te from the last end column) and in one 3' window (ts from the leftmost)."""
    rng = np.random.default_rng(9)
    short = b"ACGT"
    ad = b"GATTACAGGCTTCAGTCCATGA"
    P = _base_params(end_match_len=4, end_sim=1.0, end_len=30, adapters=[short, ad])
    # the 22-base adapter's threshold: end_match_len 4 < 22, so only the similarity (1.0) keeps it exact
    check = P.end_len + _end_extra(len(ad), 1.0)  # 52
    gt = np.frombuffer(b"GT", np.uint8)  # no A/C run, so the 4-base adapter only matches where planted
    seqs = [b"ACGT", b"ACGTG", b"TACGTG", b"ACGTT"]

    def read(c5_at=None, c3_at=None, extra5=(), extra3=()):
        L = 300
        s = bytearray(_rand(rng, L, gt))
        for at in ((c5_at,) if c5_at is not None else ()) + tuple(extra5):
            s[at:at + 22] = ad
        for at in ((c3_at,) if c3_at is not None else ()) + tuple(extra3):
            s[L - at - 22:L - at] = ad  # at = distance from the read end to the copy's end
        return bytes(s)

    seqs += [read(c5_at=check - 22), read(c5_at=check - 21),                  # 5' copy ends at check - 1 / check
             read(c3_at=check - 22), read(c3_at=check - 21),                  # 3' copy starts at tLen - check / - 1
             read(c5_at=2, extra5=(25,)), read(c3_at=1, extra3=(24,))]        # two locations at d = 0
    case = Case(P, seqs)
    _end_windows(case, 4, 1.0)
    return case


def _end_cases():
    return ([end_scripts_case(L) for L in END_LENGTHS] + list(end_similarity_case())
            + list(end_small_match_len_cases()) + [end_edge_case()])


# ---------------------------------------------------------------------------------------------------------------
# middle-window cases
# ---------------------------------------------------------------------------------------------------------------

def _mid_windows(case, match_len, sim):
    P = case.params
    n = []
    for s in case.seqs:
        tot = 0
        win = s[P.end_len:len(s) - P.end_len]
        for ad in P.adapters:
            if len(win) < len(ad) or _thresholds(len(ad), match_len, sim)[0] <= 0:
                continue
            c = _classify(ad, win, match_len, sim)
            c["tsm"] = len(win)
            case.plants.append(c)
            tot += len(c["ends"]) if c["passes"] else 0
        n.append(tot)
    case.expect_field("n_mid", n)


MID_LENGTHS = (22, 64, 150, 300)


@functools.lru_cache(maxsize=None)
def mid_scripts_case(L):
    rng = np.random.default_rng(2000 + L)
    k = 4 if L == 22 else 7
    ads = [_rand(rng, L), _rand(rng, L)]
    P = _base_params(mid_match_len=L - k + 1, mid_sim=0.5, end_len=40, extra_len=5, adapters=ads)
    seqs = []
    for i, sc in enumerate(_scripts(k)):
        cp = plant(ads[i % 2], *sc, rng)
        seqs.append(_rand(rng, P.end_len + 30) + cp + _rand(rng, P.end_len + 200 + 37 * i))
    # window lengths qLen - 1, qLen, qLen + 1 around an exact copy (it starts the window)
    for w in (L - 1, L, L + 1):
        seqs.append(_rand(rng, P.end_len) + (ads[0] + _rand(rng, 2))[:w] + _rand(rng, P.end_len))
    case = Case(P, seqs)
    _mid_windows(case, P.mid_match_len, 0.5)
    return case


@functools.lru_cache(maxsize=None)
def mid_degenerate_case():
    """mid_match_len 22 with adapters of 21 bases (mid_match_len > qLen: k_mid <= 0, never hits) and 22 bases
    (mid_match_len == qLen: exact copies only), plus extra_len 60, which clips ts at 0 and te at tLen."""
    rng = np.random.default_rng(31)
    a21, a22 = _rand(rng, 21), _rand(rng, 22)
    P = _base_params(mid_match_len=22, mid_sim=0.5, end_len=25, extra_len=60, adapters=[a21, a22])
    seqs = []
    for cp in (a21, a22, plant(a22, 1, 0, 0, rng)):
        seqs.append(_rand(rng, 25) + cp + _rand(rng, 200) + cp + _rand(rng, 25))
    case = Case(P, seqs)
    _mid_windows(case, 22, 0.5)
    return case


def _sat_copy(ad, S, rng):
    """Copy of an A/C adapter with S positions turned into G/T: no alignment can match a G/T base, so d = S."""
    cp = bytearray(ad)
    for i in rng.choice(np.arange(1, len(ad) - 1), S, replace=False):
        cp[int(i)] = int(rng.choice(np.frombuffer(b"GT", np.uint8)))
    return bytes(cp)


@functools.lru_cache(maxsize=None)
def mid_tag_case():
    """A 350-base A/C adapter with k_mid = 331 in G/T reads: copies at exact distances 253 .. 256, each ending in
    its own 1 024-column chunk.  Chunk minima 254, 255 and 256 all carry the tag 254; only the chunk whose exact
    minimum is the read's best may be counted and emitted."""
    rng = np.random.default_rng(41)
    ad = _rand(rng, 350, np.frombuffer(b"AC", np.uint8))
    P = _base_params(mid_match_len=20, mid_sim=0.05, end_len=64, extra_len=3, adapters=[ad])
    gt = np.frombuffer(b"GT", np.uint8)
    seqs, pos = [], 0
    for dists in ((253, 254, 255, 256), (254, 255, 256), (255, 256), (256, 255, 255), (256, 256)):
        # the read starts on a chunk boundary after a short spacer read
        spacer = (-pos) % 1024 or 1024
        seqs.append(_rand(rng, spacer, gt))
        pos += spacer
        s = bytearray(_rand(rng, 1024 * (len(dists) + 1), gt))
        for i, d in enumerate(dists):
            end = 1024 * (i + 1) + 600
            s[end - 349:end + 1] = _sat_copy(ad, d, rng)
        seqs.append(bytes(s))
        pos += len(s)
    quals = [b"#" * len(s) if i % 2 == 0 else b"5" * len(s) for i, s in enumerate(seqs)]
    P.min_q = 5.0
    case = Case(P, seqs, quals)
    case.designed = list(range(1, len(seqs), 2))
    _mid_windows(case, 20, 0.05)
    return case


def _mid_cases():
    return [mid_scripts_case(L) for L in MID_LENGTHS] + [mid_degenerate_case(), mid_tag_case()]


# ---------------------------------------------------------------------------------------------------------------
# piece cases
# ---------------------------------------------------------------------------------------------------------------

def _qual(values, qtype):
    return bytes(int(v) + qtype for v in values)


@functools.lru_cache(maxsize=None)
def quality_cases():
    """Reads whose fp64 mean quality is exactly min_q or max_q (10.0, 18.5), a hair either side, 7.1 against
    min_q = 7.1f (kept: 7.1 > (double)7.1f) and 7.099 (dropped), and exact integer means (histogram bin edges)."""
    out = []
    rng = np.random.default_rng(3)
    for qtype in (33, 64):
        for min_q, max_q in ((10.0, 18.5), (18.5, 30.0), (7.1, 10.0)):
            P = _base_params(min_q=min_q, max_q=max_q, qtype=qtype)
            quals = [[10] * 50, [10] * 49 + [9], [10] * 49 + [11], [18, 19] * 25, [18, 19] * 24 + [18, 18],
                     [18, 19] * 24 + [19, 19], [7] * 9 + [8], [7] * 901 + [8] * 99, [7] * 900 + [8] * 100,
                     [12] * 40, [11] * 39 + [12], [30] * 8, [31] * 7 + [30]]
            seqs = [_rand(rng, len(v)) for v in quals]
            case = Case(P, seqs, [_qual(v, qtype) for v in quals])
            means = [sum(v) / len(v) for v in quals]
            case.means = means
            case.expect_field("status", [_capi.READ_LOWQ if (m < np.float64(np.float32(min_q))
                                                             or m > np.float64(np.float32(max_q)))
                                         else _capi.READ_EVALUATED for m in means])
            out.append(case)
    return out


@functools.lru_cache(maxsize=None)
def piece_length_case():
    """min_len 100, max_len 200, head and tail trims of 10: pieces of 99, 100, 200 and 201 bases from whole reads and
    from both sides of a middle split, and reads of 9, 10, 19, 20 and 21 bases (trims equal to the read and above)."""
    rng = np.random.default_rng(4)
    ad = b"GATTACAGGCTTCAGTCCATGA"
    P = _base_params(min_len=100, max_len=200, head_trim=10, tail_trim=10, mid_match_len=22, end_len=0,
                     adapters=[ad])
    seqs = [_rand(rng, n + 20) for n in (99, 100, 200, 201)]
    for a, b in ((99, 100), (200, 201), (100, 200)):
        seqs.append(_rand(rng, 10 + a) + ad + _rand(rng, b + 10))
    seqs += [_rand(rng, n) for n in (9, 10, 19, 20, 21)]
    case = Case(P, seqs)
    case.expect_field("n_pieces", [0, 1, 1, 0, 1, 1, 2, 0, 0, 0, 0, 0])
    case.pieces = [100, 200, 100, 200, 100, 200]
    return case


@functools.lru_cache(maxsize=None)
def short_trim_case():
    """min_len 1 with head and tail trims of 10: reads of 9 and 10 bases (each trim covers the read), 19 and 20
    (the trims meet or overlap), 21 and 22 (a 1- and a 2-base piece between them)."""
    rng = np.random.default_rng(6)
    P = _base_params(min_len=1, head_trim=10, tail_trim=10)
    case = Case(P, [_rand(rng, n) for n in (9, 10, 19, 20, 21, 22)])
    case.expect_field("n_pieces", [0, 0, 0, 0, 1, 1])
    case.pieces = [1, 2]
    return case


def _piece_cases():
    return list(quality_cases()) + [piece_length_case(), short_trim_case()]


ALL_CASES = {**{f"end{L}": (lambda L=L: end_scripts_case(L)) for L in END_LENGTHS},
             "end_sim": lambda: end_similarity_case(),
             "end_small_match": lambda: end_small_match_len_cases(),
             "end_edges": lambda: [end_edge_case()],
             **{f"mid{L}": (lambda L=L: mid_scripts_case(L)) for L in MID_LENGTHS},
             "mid_degenerate": lambda: [mid_degenerate_case()],
             "mid_tag": lambda: [mid_tag_case()],
             "quality": lambda: quality_cases(),
             "pieces": lambda: [piece_length_case()],
             "short_trims": lambda: [short_trim_case()]}


def _cases(name):
    c = ALL_CASES[name]()
    return list(c) if isinstance(c, (list, tuple)) else [c]


# ---------------------------------------------------------------------------------------------------------------
# CPU: the fixtures reach their branches
# ---------------------------------------------------------------------------------------------------------------

def test_reference_dp_matches_the_oracle_on_edit_scripts():
    rng = np.random.default_rng(0)
    for L in (16, 22, 70):
        ad = _rand(rng, L)
        for sc in ((0, 0, 0), (1, 0, 0), (0, 1, 0), (0, 0, 1), (1, 1, 1)):
            w = _rand(rng, 7) + plant(ad, *sc, rng) + _rand(rng, 5)
            d, ends, start = _hw(ad, w)
            res, locs = oracle_lib.align_hw(ad, w, -1)
            assert (d, ends, start) == (res["edit_distance"], [e for _, e in locs], locs[0][0])


def _plants_at_k(plants):
    return [p for p in plants if p["k"] > 0]


def _check_branch_coverage(plants):
    live = _plants_at_k(plants)
    ds = {p["d"] - p["k"] for p in live}
    assert {-1, 0, 1} <= ds, ds
    ms = {p["M"] - p["thr"] for p in live if p["d"] <= p["k"]}
    assert {-1, 0, 1} <= ms, ms
    branches = {p["branch"] for p in live if p["branch"] is not None}
    assert branches == {-1, 0, 1}, branches
    assert {p["traceback"] for p in live if p["branch"] == -1} == {True, False}
    assert any(p["passes"] for p in live) and any(p["d"] <= p["k"] and not p["passes"] for p in live)


def test_end_fixtures_cover_every_branch():
    plants = [p for c in _end_cases() for p in c.plants]
    _check_branch_coverage(plants)
    # per adapter length: d = k - 1 / k / k + 1 and both outcomes of d = k
    for L in END_LENGTHS:
        pl = [p for p in end_scripts_case(L).plants if p["q"] == L]
        assert {p["d"] - p["k"] for p in pl} >= {-1, 0, 1}, L
        assert {p["passes"] for p in pl if p["d"] == p["k"]} == {True, False}, L
    # both sides of the window are searched and both pass somewhere
    assert {p["side"] for p in plants if p["passes"]} == {3, 5}


def test_similarity_fixtures_hit_exact_and_rounded_thresholds():
    kinds, per_kind = set(), {}
    for case in end_similarity_case():
        L, sim, thr = case.sim
        s = np.float32(sim)
        exact = np.float32(thr) / np.float32(L) == s
        rounded = thr != int(np.ceil(fractions.Fraction(float(s)) * L))
        kind = "exact" if exact and not rounded else "rounded" if rounded else "other"
        kinds.add(kind)
        per_kind.setdefault(kind, set()).update(p["M"] - thr for p in case.plants if p["d"] <= p["k"])
        assert {p["passes"] for p in case.plants} == {True, False}
    assert {"exact", "rounded"} <= kinds
    assert {-1, 0, 1} <= per_kind["exact"] and {-1, 0, 1} <= per_kind["rounded"], per_kind
    # end_sim 1.0 is present; a double-precision ceil would move the rounded ones
    assert any(c.sim[1] == 1.0 for c in end_similarity_case())
    assert any(int(np.ceil(np.float64(np.float32(c.sim[1])) * c.sim[0])) != c.sim[2] for c in end_similarity_case())


def test_small_end_match_lengths_cap_k_and_exclude_d_equal_qlen():
    for case in end_small_match_len_cases():
        assert all(p["k"] == 21 for p in case.plants)
        assert all(p["check"] == len(s) for p, s in zip(case.plants[::2], case.seqs))
        ds = {p["d"] for p in case.plants}
        assert {22, 21, 20} <= ds
        assert not any(p["passes"] for p in case.plants if p["d"] == 22)
        assert any(p["passes"] for p in case.plants if p["d"] == 21)
    assert _end_extra(22, 0.01) > 300


def test_window_edge_fixtures():
    case = end_edge_case()
    assert [min(case.params.end_len + _end_extra(4, 1.0), len(s)) for s in case.seqs[:4]] == [4, 5, 6, 5]
    n5, n3 = case.expect["n_5p"], case.expect["n_3p"]
    assert n5[:4].tolist() == [0, 1, 1, 1] and n3[:4].tolist() == [0, 1, 1, 1]
    # copies at the window's last column / first column pass, one column further they do not
    assert n5[4:6].tolist() == [1, 0] and n3[6:8].tolist() == [1, 0]
    # two locations at one distance in one window
    assert n5[8] == 2 and n3[9] == 2


def test_mid_fixtures_cover_every_branch_and_window_length():
    plants = [p for c in _mid_cases() if c is not mid_tag_case() for p in c.plants]
    _check_branch_coverage(plants)
    for L in MID_LENGTHS:
        case = mid_scripts_case(L)
        assert case.expect["n_mid"][-3:].tolist()[0] == 0 and min(case.expect["n_mid"][-2:]) >= 1, L
    deg = mid_degenerate_case()
    assert _thresholds(21, 22, 0.5)[0] <= 0 and _thresholds(22, 22, 0.5) == (1, 22)
    assert deg.expect["n_mid"].tolist() == [0, 2, 0]


def test_tag_fixture_has_distinct_minima_behind_one_tag():
    case = mid_tag_case()
    k, thr = _thresholds(350, 20, 0.05)
    assert k > 256 and thr == 20
    best = [p["d"] for p in case.plants if p["d"] <= p["k"]]
    assert best == [253, 254, 255, 255, 256]
    assert all(p["passes"] for p in case.plants if p["d"] <= p["k"])
    n_mid = case.expect["n_mid"][case.designed]
    assert (n_mid >= 1).all()


def test_quality_fixtures_sit_on_the_thresholds():
    for case in quality_cases():
        P = case.params
        lo, hi = np.float64(np.float32(P.min_q)), np.float64(np.float32(P.max_q))
        m = np.array(case.means)
        assert (m == lo).any() or P.min_q == 7.1
        assert ((m < lo) & (m > lo - 0.05)).any() or P.min_q == 7.1
        assert (m == np.floor(m)).sum() >= 3  # integer means: bin edges of the histograms
    seven = [c for c in quality_cases() if c.params.min_q == 7.1][0]
    assert 7.1 in seven.means and 7.099 in seven.means and 7.1 > np.float64(np.float32(7.1)) > 7.099


# ---------------------------------------------------------------------------------------------------------------
# GPU: every case against the oracle, and its intended outcome
# ---------------------------------------------------------------------------------------------------------------

def _run_case(case, **kw):
    reads, pieces, _ = _compare(case.params, case.batch, **kw)
    for f, v in case.expect.items():
        idx = getattr(case, "designed", None)
        got = reads[f].astype(np.int64)
        np.testing.assert_array_equal(got if idx is None or f != "n_mid" else got[idx],
                                      v if idx is None or f != "n_mid" else v[idx], err_msg=f)
    return reads, pieces


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(ALL_CASES))
def test_cases_vs_oracle(name):
    for case in _cases(name):
        reads, pieces = _run_case(case)
        if hasattr(case, "pieces"):
            assert sorted(pieces["len"].tolist()) == sorted(case.pieces)


@pytest.mark.gpu
def test_mid_scripts_in_multi_chunk_runs(monkeypatch):
    """The 150-base middle cases after 12 Mbases of low-quality filler at TGSF_SM_COUNT=1: 1 024-column chunks in
    runs of 4.  One more read's middle window starts on a run boundary and spans five chunks; exact copies cross
    the three chunk boundaries inside the run and the run's closing boundary."""
    monkeypatch.setenv("TGSF_SM_COUNT", "1")
    case = mid_scripts_case(150)
    fill = _filler(12_000_000, seed=91)
    params = dataclasses.replace(case.params, min_q=5.0)
    run, chunk = 4096, 1024
    rng = np.random.default_rng(92)
    pos = sum(len(s) for s in fill[0]) + sum(len(s) for s in case.seqs)
    mb = (pos + params.end_len + 200 + run - 1) // run * run  # the designed read's middle window starts here
    spacer = mb - params.end_len - pos
    read = bytearray(_rand(rng, 2 * params.end_len + 5 * chunk))
    ad = params.adapters[0]
    for b in (1, 2, 3, 4):  # copy ends 40 columns after chunk boundary b (b = 4: the run's end)
        end = params.end_len + b * chunk + 40
        read[end - len(ad) + 1:end + 1] = ad
    runs = Case(params, [_rand(rng, spacer), bytes(read)], [b"#" * spacer, b"5" * len(read)])
    _mid_windows(runs, params.mid_match_len, 0.5)
    assert runs.expect["n_mid"].tolist() == [0, 4]
    batch = _concat(fill, (case.seqs, case.quals), (runs.seqs, runs.quals))

    def shape(eng):
        assert eng.launch_shape() == (1, 10)
        assert eng.mid_run_shift() == 2

    reads, _, _ = _compare(params, batch, on_engine=shape)
    n_fill, n_case = len(fill[0]), len(case.seqs)
    np.testing.assert_array_equal(reads["n_mid"][n_fill:n_fill + n_case].astype(np.int64), case.expect["n_mid"])
    assert int(reads["n_mid"][-1]) == 4


# ---------------------------------------------------------------------------------------------------------------
# CPU with the reference build: the oracle's reading of the reference on the same fixtures
# ---------------------------------------------------------------------------------------------------------------

@needs_ref
@pytest.mark.ref
@pytest.mark.parametrize("name", list(ALL_CASES))
def test_cases_oracle_vs_reference(name):
    for case in _cases(name):
        params, batch = case.params, case.batch
        ref = ref_lib.perread(params, batch, 1)
        reads, pieces, cnt = oracle_lib.run(params, batch)
        L = oracle_lib.layout(params)
        np.testing.assert_array_equal(ref["drop_info"], cnt[L.drop_info:L.drop_info + 17])
        np.testing.assert_array_equal(ref["raw_hist"], cnt[L.raw_hist:L.raw_hist + 256])
        np.testing.assert_array_equal(ref["clean_hist"], cnt[L.clean_hist:L.clean_hist + 256])
        for t in ref_lib.TABLES:
            rows_total = L.bc_len if ("5p" in t or "3p" in t) else L.max_bins
            off = getattr(L, t)
            mine = cnt[off:off + rows_total * 5].reshape(rows_total, 5)
            np.testing.assert_array_equal(mine[:ref[t].shape[0]], ref[t], err_msg=t)
        assert records.format_records(batch, pieces) == ref["records"]

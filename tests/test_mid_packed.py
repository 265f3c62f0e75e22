"""The packed middle scan (k_mid_scan_packed) against the CPU oracle.

A pair of adapters of at most 50 bp is scanned as one 96-bit vector in which each adapter keeps its last 48 rows.
That suffix score is a lower bound on the whole adapter's score, so the scan only flags chunks and an exact 64-bit
re-check decides them.  These tests plant copies that fool the filter (the suffix scores <= k, the whole adapter
k + 1), copies at exactly k and k + 1 around chunk and run boundaries, reads that carry only one adapter of the pair,
and adapter sets at the edges of the routing rule.  Copies are built from insertions, which keep the match count at
q, so a copy at distance <= k passes the reference's match thresholds and shows up as a middle region.
Comparisons are bit-exact."""
import numpy as np
import pytest

from test_gpu_parity import _compare, _long_adapter_batch, params_rev
from test_launch_regimes import ACGT, _filler
from test_mid_runs import CHUNK, RUN, TARGET_BASES, _Layout, _expect_runs
from tgsfilter_b200 import synth
from tgsfilter_b200.params import ADAPTER_LIB, FilterParams, rev_comp

pytestmark = pytest.mark.gpu

RAPID = ADAPTER_LIB[8]
K = 16  # config_params(3): k = q - 35 + 1 for the 50-bp rapid adapter


def _hw(query: bytes, text: bytes) -> int:
    """Edit distance of query against its best substring of text (free start and end in the text)."""
    prev = list(range(len(query) + 1))
    best = prev[-1]
    for t in text:
        cur = [0]
        for i, ch in enumerate(query):
            cur.append(min(prev[i] + (ch != t), prev[i + 1] + 1, cur[i] + 1))
        prev = cur
        best = min(best, cur[-1])
    return best


def _copy(ad, rng, n_ins, lead_subs=0, lo=None):
    """ad with its first lead_subs bases substituted and n_ins random insertions at positions >= lo."""
    cp = bytearray(ad)
    for i in range(lead_subs):
        cp[i] = int(ACGT[(int(np.nonzero(ACGT == cp[i])[0][0]) + 2) % 4])
    lo = max(lead_subs, 1) if lo is None else lo
    for pos in sorted(rng.choice(np.arange(lo, len(ad) - 1), n_ins, replace=False))[::-1]:
        cp[int(pos):int(pos)] = bytes([int(ACGT[rng.integers(0, 4)])])
    return bytes(cp)


def _exact(ad, rng, d, lead_subs=0, suffix_max=None):
    """A copy whose distance to ad (in 40 bases of random context on both sides) is exactly d; with suffix_max, the
    distance of ad's last 48 bases must also be at most suffix_max."""
    for _ in range(500):
        cp = _copy(ad, rng, d - lead_subs, lead_subs)
        ctx = ACGT[rng.integers(0, 4, 40)].tobytes() + cp + ACGT[rng.integers(0, 4, 40)].tobytes()
        if _hw(ad, ctx) != d:
            continue
        if suffix_max is not None and _hw(ad[-48:], ctx) > suffix_max:
            continue
        return cp
    raise AssertionError("no copy found")


def _n_mid(r, lay):
    return r["n_mid"][[i for i, _ in lay.designed]]


def test_helpers_agree_on_distances():
    rng = np.random.default_rng(1)
    near = _exact(RAPID, rng, K + 1, lead_subs=2, suffix_max=K)
    assert _hw(RAPID, near) == K + 1 and _hw(RAPID[-48:], near) <= K
    assert _hw(RAPID, RAPID) == 0 and _hw(RAPID, _copy(RAPID, rng, 3)) <= 3


@pytest.mark.parametrize("ad", [RAPID, rev_comp(RAPID)], ids=["rapid", "rapid_rc"])
def test_near_misses_fool_the_filter_only(ad, monkeypatch):
    """Copies whose 48-row suffix scores <= k while the whole adapter scores k + 1: the filter flags their chunks and
    the exact re-check must report nothing."""
    monkeypatch.setenv("TGSF_SM_COUNT", "1")
    params = synth.config_params(3)
    lay = _Layout(TARGET_BASES - 40 * RUN, params.end_len, seed=91)
    for i in range(24):
        mb = lay.next_run()
        plants = [(mb + 300 + j * CHUNK + 17 * i, _exact(ad, lay.rng, K + 1, lead_subs=2, suffix_max=K))
                  for j in range(RUN // CHUNK)]
        lay.read(mb, RUN, plants)
    batch = lay.batch()
    r, _, _ = _compare(params, batch, on_engine=_expect_runs(batch.n_bases))
    assert (_n_mid(r, lay) == 0).all()


def test_threshold_copies_around_chunk_and_run_boundaries(monkeypatch):
    """Copies at exactly k (found) and k + 1 (not found) of both adapters whose end column lies just before, on and
    after chunk boundaries inside a run and at the run's ends."""
    monkeypatch.setenv("TGSF_SM_COUNT", "1")
    params = synth.config_params(3)
    ads = [RAPID, rev_comp(RAPID)]
    deltas = [-66, -65, -17, -1, 0, 1, 15, 16, 64, 65]
    n_chunks = 2 * (RUN // CHUNK) + 1
    lay = _Layout(TARGET_BASES - 12 * (n_chunks * CHUNK + 6000), params.end_len, seed=92)
    found = []
    for i in range(len(deltas)):
        mb = lay.next_run()
        d = K if i % 2 == 0 else K + 1
        plants = [(mb + j * CHUNK + deltas[(i + j) % len(deltas)], _exact(ads[(i + j) % 2], lay.rng, d))
                  for j in range(1, n_chunks)]
        lay.read(mb, n_chunks * CHUNK, plants)
        found.append(d == K)
    batch = lay.batch()
    r, _, _ = _compare(params, batch, on_engine=_expect_runs(batch.n_bases))
    n = _n_mid(r, lay)
    assert (n[np.array(found)] >= 1).all() and (n[~np.array(found)] == 0).all()


@pytest.mark.parametrize("which", [0, 1])
def test_one_adapter_of_the_pair_only(which, monkeypatch):
    """Reads that carry copies of one adapter of the pair only (exact and at k), many per chunk: the other field
    shares every column with it and must stay empty."""
    monkeypatch.setenv("TGSF_SM_COUNT", "1")
    params = synth.config_params(3)
    ad = [RAPID, rev_comp(RAPID)][which]
    lay = _Layout(TARGET_BASES - 30 * RUN, params.end_len, seed=93 + which)
    for i in range(16):
        mb = lay.next_run()
        plants = [(mb + 200 + 150 * j, ad if j % 2 == 0 else _exact(ad, lay.rng, K)) for j in range(20)]
        lay.read(mb, RUN, plants)
    batch = lay.batch()
    r, _, _ = _compare(params, batch, on_engine=_expect_runs(batch.n_bases))
    assert (_n_mid(r, lay) >= 1).all()


def _random_adapter(rng, n):
    return ACGT[rng.integers(0, 4, n)].tobytes()


@pytest.mark.parametrize("lens", [(45, 45), (48, 50), (50, 50), (50, 51), (50, 50, 50)],
                         ids=["45_45", "48_50", "50_50", "50_51", "three_50"])
def test_routing_edges(lens, monkeypatch):
    """Pairs that fit whole (45/45), lose 0 and 2 rows (48/50), both lose 2 (50/50), a pair that is not packed
    (50/51) and three adapters where the third runs on its own."""
    monkeypatch.setenv("TGSF_SM_COUNT", "1")
    rng = np.random.default_rng(sum(lens))
    ads = [_random_adapter(rng, n) for n in lens]
    reads = _long_adapter_batch(ads + [params_rev(a) for a in ads], n=120, seed=len(lens))
    core = ([reads.read(i)[0].tobytes() for i in range(reads.n_reads)],
            [reads.read(i)[1].tobytes() for i in range(reads.n_reads)])
    fill = _filler(TARGET_BASES - reads.n_bases, seed=95)
    half = len(fill[0]) // 2
    seqs = fill[0][:half] + core[0] + fill[0][half:]
    quals = fill[1][:half] + core[1] + fill[1][half:]
    batch = synth.pack_reads(seqs, quals)
    params = FilterParams(min_len=500, min_q=7.0, qtype=33, adapters=ads).apply_read_type("ont")
    r, _, _ = _compare(params, batch, on_engine=_expect_runs(batch.n_bases))
    assert (r["n_mid"] > 0).sum() >= 5


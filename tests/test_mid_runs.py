"""The middle scan's runs of chunks against the CPU oracle.

k_mid_scan hands out runs of up to 2^run_shift consecutive chunks of a read's middle window: a thread restarts
the q+k-1 column halo before a run's first chunk only and carries the exact Myers state across the chunk
boundaries inside the run, closing each chunk's minimum there.  A run covers 4 096 columns.  A benchmark batch
(config[1], ~2.35 Gbases on 148 SMs) runs with 1 024-column chunks and runs of 4 chunks; TGSF_SM_COUNT=1 reaches
that same shape with a ~12 Mbase batch, and runs of 2 chunks of 2 048 columns with a ~18 Mbase batch, padded with
low-quality filler reads that the QC drops.  Comparisons are bit-exact."""
import numpy as np
import pytest

from test_gpu_parity import _compare, _long_adapter_batch, params_rev
from test_launch_regimes import ACGT, _concat, _filler
from tgsfilter_b200 import synth
from tgsfilter_b200.params import ADAPTER_LIB, FilterParams

pytestmark = pytest.mark.gpu

TARGET_BASES = 12_000_000
TARGET_BASES_SHIFT_11 = 18_000_000


def _shape(n_bases, sm=1):
    """(chunk_shift, run_shift) that slot_reserve picks for a batch of n_bases on `sm` SMs."""
    cs = 10
    while cs < 12 and (n_bases >> (cs + 1)) >= sm * 8192:
        cs += 1
    return cs, 12 - cs


CS, RS = _shape(TARGET_BASES)
CHUNK, RUN = 1 << CS, 1 << (CS + RS)


def _expect_runs(n_bases):
    cs, rs = _shape(n_bases)
    assert rs >= 1, "the batch must run with runs of several chunks"

    def check(eng):
        assert eng.launch_shape() == (1, cs)
        assert eng.mid_run_shift() == rs
    return check


class _Layout:
    """Builds a batch whose reads sit at chosen absolute offsets of the bases stream: low-quality spacer reads
    (dropped by the QC like the filler) move each designed read so that its middle window starts where asked."""

    def __init__(self, lead_bases, end_len, seed, run=RUN):
        self.run = run
        self.rng = np.random.default_rng(seed)
        self.end_len = end_len
        self.seqs, self.quals = _filler(lead_bases, seed=seed)
        self.pos = sum(len(s) for s in self.seqs)
        self.designed = []

    def _spacer(self, n):
        self.seqs.append(ACGT[self.rng.integers(0, 4, n)].tobytes())
        self.quals.append(b"#" * n)
        self.pos += n

    def read(self, mb, window, plants):
        """A read whose middle window is [mb, mb + window) (absolute); plants: [(absolute end column, copy)]."""
        rs = mb - self.end_len
        assert rs > self.pos, (rs, self.pos)
        self._spacer(rs - self.pos)
        L = window + 2 * self.end_len
        s = bytearray(ACGT[self.rng.integers(0, 4, L)].tobytes())
        for end, cp in plants:
            start = end - (len(cp) - 1) - rs
            assert self.end_len <= start and start + len(cp) <= L - self.end_len
            s[start:start + len(cp)] = cp
        self.seqs.append(bytes(s))
        self.quals.append(b"5" * L)
        self.designed.append((len(self.seqs) - 1, len(plants)))
        self.pos += L

    def next_run(self, margin=2000):
        """First run boundary at least `margin` bases ahead of the stream's end."""
        return (self.pos + margin + self.run - 1) // self.run * self.run

    def batch(self):
        return synth.pack_reads(self.seqs, self.quals)


def _mutated(ad, rng, n_sub=2):
    cp = bytearray(ad)
    for k in rng.choice(np.arange(3, len(ad) - 3), n_sub, replace=False):
        cp[int(k)] = int(ACGT[(int(np.nonzero(ACGT == cp[int(k)])[0][0]) + 1) % 4])
    return bytes(cp)


def _check_found(r, layout):
    idx = [i for i, _ in layout.designed]
    assert (r["n_mid"][idx] >= 1).all(), r["n_mid"][idx]


def test_runs_reach_the_bench_shape():
    assert (CS, RS) == _shape(2_350_000_000, sm=148) == (10, 2)
    assert _shape(TARGET_BASES_SHIFT_11) == (11, 1)


@pytest.mark.parametrize("target", [TARGET_BASES, TARGET_BASES_SHIFT_11])
def test_copies_around_chunk_boundaries_inside_runs(target, monkeypatch):
    """Copies of a 50-bp adapter (k = 16, q + k - 1 = 65) whose end column lies 0, 1, 15, 16, 64 or 65 columns
    before or after a chunk boundary: boundaries inside a run, at a run's start and at a run's end.  Every read's
    window is R * 2 + 1 chunks long and starts on a run boundary."""
    monkeypatch.setenv("TGSF_SM_COUNT", "1")
    params = synth.config_params(3)
    ad = ADAPTER_LIB[8]
    deltas = [-66, -65, -17, -16, -2, -1, 0, 1, 15, 16, 64, 65]
    cs, rs = _shape(target)
    chunk = 1 << cs
    n_chunks = 2 * (1 << rs) + 1
    lay = _Layout(target - 12 * (n_chunks * chunk + 6000), params.end_len, seed=71, run=chunk << rs)
    for k in range(len(deltas)):
        mb = lay.next_run()
        plants = []
        for i in range(1, n_chunks):
            d = deltas[(k + i) % len(deltas)]
            plants.append((mb + i * chunk + d, _mutated(ad, lay.rng)))
        lay.read(mb, n_chunks * chunk, plants)
    batch = lay.batch()
    r, _, _ = _compare(params, batch, on_engine=_expect_runs(batch.n_bases))
    _check_found(r, lay)


def test_window_shapes_and_equal_minima(monkeypatch):
    """Middle windows of one partial chunk, exactly R chunks (aligned to a run and not), R * m + 1 chunks, and two
    equal minima (exact copies, and copies with the same substitution count) in different chunks of one run."""
    monkeypatch.setenv("TGSF_SM_COUNT", "1")
    params = synth.config_params(3)
    ad = ADAPTER_LIB[8]
    lay = _Layout(TARGET_BASES - 80 * RUN, params.end_len, seed=72)
    R = RUN // CHUNK
    # one partial chunk
    mb = lay.next_run() + 200
    lay.read(mb, 600, [(mb + 300, _mutated(ad, lay.rng))])
    # exactly R chunks, aligned to a run
    mb = lay.next_run()
    lay.read(mb, RUN, [(mb + 100, ad), (mb + RUN - 1, _mutated(ad, lay.rng))])
    # R chunks, not aligned: a partial first and last chunk
    mb = lay.next_run() + 300
    lay.read(mb, RUN - 600, [(mb + CHUNK, _mutated(ad, lay.rng)), (mb + RUN - 700, ad)])
    # R * m + 1 chunks for m = 1, 2, 3
    for m in (1, 2, 3):
        mb = lay.next_run()
        lay.read(mb, (R * m + 1) * CHUNK, [(mb + (R * m) * CHUNK + 70, _mutated(ad, lay.rng)),
                                           (mb + R * CHUNK - 3, _mutated(ad, lay.rng))])
    # equal minima in two chunks of one run: exact copies, then copies with two substitutions each
    for cp_a, cp_b in ((ad, ad), (_mutated(ad, lay.rng), _mutated(ad, lay.rng))):
        mb = lay.next_run()
        lay.read(mb, RUN, [(mb + 500, cp_a), (mb + 2 * CHUNK + 700, cp_b)])
    batch = lay.batch()
    r, _, _ = _compare(params, batch, on_engine=_expect_runs(batch.n_bases))
    _check_found(r, lay)
    assert (r["n_mid"][[i for i, _ in lay.designed[-2:]]] >= 2).all()


def test_long_adapters_in_runs(monkeypatch):
    """300- and 1 500-bp adapters (one and six Myers words, the latter from global memory) at the run shape."""
    monkeypatch.setenv("TGSF_SM_COUNT", "1")
    rng = np.random.default_rng(73)
    ads = [ACGT[rng.integers(0, 4, n)].tobytes() for n in (300, 1500)]
    adapters = []
    for a in ads:
        adapters += [a, params_rev(a)]
    reads = _long_adapter_batch(ads, n=40, seed=74)
    core = ([reads.read(i)[0].tobytes() for i in range(reads.n_reads)],
            [reads.read(i)[1].tobytes() for i in range(reads.n_reads)])
    fill = _filler(TARGET_BASES - reads.n_bases, seed=75)
    half = len(fill[0]) // 2
    batch = _concat((fill[0][:half], fill[1][:half]), core, (fill[0][half:], fill[1][half:]))
    params = FilterParams(min_len=500, min_q=7.0, qtype=33, adapters=adapters).apply_read_type("ont")
    r, _, _ = _compare(params, batch, on_engine=_expect_runs(batch.n_bases))
    assert (r["n_mid"] > 0).sum() >= 5


@pytest.mark.parametrize("config", [1, 2, 3, 4, 5])
def test_configs_in_runs(config, monkeypatch):
    monkeypatch.setenv("TGSF_SM_COUNT", "1")
    core = synth.make_config(config, 150)
    seqs = [core.read(i)[0].tobytes() for i in range(core.n_reads)]
    quals = [core.read(i)[1].tobytes() for i in range(core.n_reads)]
    fill = _filler(max(TARGET_BASES - core.n_bases, 1), seed=80 + config)
    batch = _concat(fill, (seqs, quals))
    _compare(synth.config_params(config), batch, on_engine=_expect_runs(batch.n_bases))

"""The kernels in the launch regimes of large runs, against the CPU oracle.

The parity suite feeds batches of at most a few hundred Mbases to the full grid.  A benchmark step is one batch
of ~4.7 Gbases: the middle scan then cuts the reads into chunks of 2048 columns instead of 1024, absolute
offsets pass 2^32, every scan warp works through hundreds of tiles and every CTA accumulates its shared-memory
bins over many reads.  TGSF_SM_COUNT=n sizes every grid (and the chunk-size rule) for n SMs, so small batches
reach those shapes; every test asserts through ``FilterEngine.launch_shape`` the SM count and chunk shift it
set out to reach.  Comparisons are bit-exact, like the rest of the suite."""
import functools
import gzip

import numpy as np
import pytest

import contam_oracle
import oracle_lib
from test_contam import _case_batch, _run_gpu, _set
from test_gpu_parity import (_compare, _fuzz_case, _gz_members, _info, _long_adapter_batch, _pool_overflow_case,
                             _repeat_batch, _run_host_cli, params_rev)
from tgsfilter_b200 import _capi, synth
from tgsfilter_b200.engine import Counters, FilterEngine
from tgsfilter_b200.params import ADAPTER_LIB, FilterParams

pytestmark = pytest.mark.gpu

# slot_reserve: shift s + 1 once n_bases >> (s + 1) >= sm_count * 8192, so at one SM
SHIFT_11_BASES = 1 << 24  # 16 777 216
SHIFT_12_BASES = 1 << 25  # 33 554 432
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


def _expect_shape(sm, shift=None):
    def check(eng):
        got_sm, got_shift = eng.launch_shape()
        assert got_sm == sm, f"grids sized for {got_sm} SMs, wanted {sm}"
        if shift is not None:
            assert got_shift == shift, f"chunk shift {got_shift}, wanted {shift}"
    return check


def _shift_target(shift):
    """A batch size (bases) that gives `shift` at one SM, just above its threshold."""
    return {10: 12_000_000, 11: SHIFT_11_BASES + 700_000, 12: SHIFT_12_BASES + 700_000}[shift]


def _filler(n_bases, seed):
    """Random reads of ~50 kb at Q2: below every min_q used here, so the oracle and the GPU drop them after the
    raw QC scan.  They only move the batch size (and with it the chunk shift) and the absolute offsets."""
    rng = np.random.default_rng(seed)
    seqs, left = [], n_bases
    while left > 0:
        L = int(min(left, rng.integers(30_000, 70_000)))
        seqs.append(ACGT[rng.integers(0, 4, L)].tobytes())
        left -= L
    return seqs, [b"#" * len(s) for s in seqs]


def _concat(*parts):
    seqs, quals = [], []
    for s, q in parts:
        seqs += s
        quals += q
    return synth.pack_reads(seqs, quals)


@functools.lru_cache(maxsize=None)
def _config3_reads():
    return synth.make_config(3, 700)


def _config3_batch(n_bases):
    full = _config3_reads()
    k = int(np.searchsorted(full.offsets.astype(np.int64), n_bases)) + 1
    assert k <= full.n_reads
    return full.slice(0, k)


# ---- chunk shifts 10 / 11 / 12 against the oracle -------------------------------------------------------
@pytest.mark.parametrize("shift", [10, 11, 12])
def test_config3_at_each_chunk_shift(shift, monkeypatch):
    """Config 3 (middle adapters, -M 35 -T 50) with the chunk lengths of large batches (one SM)."""
    monkeypatch.setenv("TGSF_SM_COUNT", "1")
    batch = _config3_batch(_shift_target(shift))
    r, _, _ = _compare(synth.config_params(3), batch, on_engine=_expect_shape(1, shift))
    assert (r["n_mid"] > 0).sum() >= 5


@pytest.mark.parametrize("shift", [10, 11, 12])
def test_long_adapters_at_each_chunk_shift(shift, monkeypatch):
    """300 / 600 / 1 500-bp adapters: the restart halo of the 1 500-bp one is longer than a 1 024-column chunk."""
    monkeypatch.setenv("TGSF_SM_COUNT", "1")
    rng = np.random.default_rng(9)
    ads = [ACGT[rng.integers(0, 4, n)].tobytes() for n in (300, 600, 1500)]
    adapters = []
    for a in ads:
        adapters += [a, params_rev(a)]
    reads = _long_adapter_batch(ads, n=30, seed=20 + shift)
    core = ([reads.read(i)[0].tobytes() for i in range(reads.n_reads)],
            [reads.read(i)[1].tobytes() for i in range(reads.n_reads)])
    fill = _filler(_shift_target(shift) - reads.n_bases, seed=shift)
    half = len(fill[0]) // 2
    batch = _concat((fill[0][:half], fill[1][:half]), core, (fill[0][half:], fill[1][half:]))
    params = FilterParams(min_len=500, min_q=7.0, qtype=33, adapters=adapters).apply_read_type("ont")
    r, _, _ = _compare(params, batch, on_engine=_expect_shape(1, shift))
    assert (r["n_mid"] > 0).sum() >= 5 and (r["n_5p"] > 0).any() and (r["n_3p"] > 0).any()


def _boundary_batch(shift):
    """Reads with substitution-mutated copies of ADAPTER_LIB[8] whose last base (the alignment's end column)
    falls at chosen distances from absolute multiples of 1 024, 2 048 and 4 096 bytes of the stream: one column
    before, at and after a chunk start, and across the restart halo (q + k_mid - 1 = 65 columns, rounded to 80)."""
    ad = ADAPTER_LIB[8]
    q, halo = len(ad), 80
    rng = np.random.default_rng(300 + shift)
    deltas = [-1, 0, 1, -2, 2, -halo - 1, -halo, -halo + 1, halo - 1, halo, halo + 1, -q, -q + 1, q - 1, q,
              -15, -16, -17, 15, 16, 17] + [int(x) for x in rng.integers(-halo, halo + 1, 13)]
    plan = [(m, d) for m in (1024, 2048, 4096) for d in deltas]
    lead = _filler(_shift_target(shift) - 51 * 12_032, seed=40 + shift)
    base = sum(len(s) for s in lead[0])
    seqs, plants = [], []
    pos = base
    for i in range(0, len(plan), 2):
        L = 12_000 + int(rng.integers(0, 64))
        s = bytearray(ACGT[rng.integers(0, 4, L)].tobytes())
        lo = pos + 150 + q + halo + 200  # middle window starts at end_len = 150
        for j, (m, d) in enumerate(plan[i:i + 2]):
            b = (lo + j * 6000 + m - 1) // m * m  # an absolute multiple of m inside the read
            end = b + d
            start = end - (q - 1) - pos
            assert 150 < start and start + q < L - 150
            cp = bytearray(ad)
            for k in rng.choice(np.arange(3, q - 3), 2, replace=False):  # interior substitutions
                cp[int(k)] = int(ACGT[(int(np.nonzero(ACGT == cp[int(k)])[0][0]) + 1) % 4])
            s[start:start + q] = cp
            plants.append(end)
        seqs.append(bytes(s))
        pos += L
    batch = _concat(lead, (seqs, [b"5" * len(x) for x in seqs]))
    return batch, len(lead[0]), plants


@pytest.mark.parametrize("shift", [10, 11, 12])
def test_adapters_at_chunk_boundaries(shift, monkeypatch):
    monkeypatch.setenv("TGSF_SM_COUNT", "1")
    batch, first, plants = _boundary_batch(shift)
    params = synth.config_params(3)
    r, p, _ = _compare(params, batch, on_engine=_expect_shape(1, shift))
    # both copies of every planted read were found
    assert (r["n_mid"][first:] >= 2).all(), r["n_mid"][first:]
    cb = np.array(plants, dtype=np.int64) & ((1 << shift) - 1)
    assert (cb == 0).any() and (cb == 1).any() and (cb == (1 << shift) - 1).any()


# ---- grid shapes ------------------------------------------------------------------------------------------
GRIDS = [("1", {}), ("5", {}), ("1", {"TGSF_RES_CTAS": "1", "TGSF_MID_CTAS": "1", "TGSF_FORK_ENDS": "0"}),
         ("5", {"TGSF_RES_CTAS": "1", "TGSF_MID_CTAS": "1", "TGSF_FORK_ENDS": "0"})]
KNOBS = ("TGSF_SM_COUNT", "TGSF_RES_CTAS", "TGSF_MID_CTAS", "TGSF_FORK_ENDS")


def _each_grid(monkeypatch):
    """Yields the SM count of each grid shape with the environment set for it."""
    for sm, extra in GRIDS:
        for k in KNOBS:
            monkeypatch.delenv(k, raising=False)
        monkeypatch.setenv("TGSF_SM_COUNT", sm)
        for k, v in extra.items():
            monkeypatch.setenv(k, v)
        yield int(sm)
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)


def _config_case(cfg, n):
    params = synth.config_params(cfg)
    if cfg == 5:
        params.min_repeat = 40
    return params, synth.make_config(cfg, n, max_len=250000)


def _kmer_case(k):
    params = FilterParams(min_len=50, min_q=0.0, kmer=k, min_repeat=200, qtype=33, adapters=[], max_read_len=500000)
    return params, _repeat_batch(100 + k, long_read=[450000, 19000, 33000, 64990, 65100])


ORACLE_CASES = ([f"config{c}" for c in range(1, 6)] + [f"fuzz{s}" for s in range(8)]
                + [f"kmer{k}" for k in (5, 11, 12, 13, 16, 21)] + ["pool_overflow"])


def _oracle_case(name):
    if name.startswith("config"):
        cfg = int(name[6:])
        return _config_case(cfg, {1: 400, 2: 300, 3: 60, 4: 600, 5: 300}[cfg])
    if name.startswith("fuzz"):
        return _fuzz_case(int(name[4:]))
    if name.startswith("kmer"):
        return _kmer_case(int(name[4:]))
    return _pool_overflow_case()


@pytest.mark.parametrize("name", ORACLE_CASES)
def test_grid_shapes_vs_oracle(name, monkeypatch):
    """The same input on 1 and 5 SMs, with the default resolve / middle-scan grids and with one CTA per SM and the
    end windows on the main stream: results must not depend on how the work is spread."""
    params, batch = _oracle_case(name)
    oracle = oracle_lib.run(params, batch)
    for sm in _each_grid(monkeypatch):
        _compare(params, batch, oracle=oracle, on_engine=_expect_shape(sm))


@pytest.mark.parametrize("set_name,cfg,n,k,path", [("small", 1, 200, 17, "submit"), ("large", 3, 60, 11, "device")])
def test_grid_shapes_contaminant_screen(set_name, cfg, n, k, path, monkeypatch):
    genome, cset = _set(set_name)
    batch, _ = _case_batch(cfg, n, genome)
    params = synth.config_params(cfg)
    o_reads, o_pieces, o_cnt = contam_oracle.run(params, batch, (cset, k, 0.05))
    for sm in _each_grid(monkeypatch):
        with FilterEngine(params) as eng:
            assert eng.launch_shape()[0] == sm
        _, reads, pieces, cnt = _run_gpu(params, batch, cset, k, 0.05, path)
        assert np.array_equal(reads, o_reads) and np.array_equal(pieces, o_pieces) and np.array_equal(cnt, o_cnt)
        assert (pieces["status"] == _capi.PIECE_CONTAM).any()


def test_grid_shapes_deflate_and_packed_submit(monkeypatch):
    """GPU deflate blocks must inflate to the records, and the 2-bit packed submit must equal the oracle."""
    params, batch = _config_case(3, 40)
    params.gz_blocks = True
    p2, b2 = synth.config_params(2), synth.make_config(2, 150, max_len=30000)
    o_reads, o_pieces, _ = oracle_lib.run(params, batch)
    o2 = oracle_lib.run(p2, b2)
    for sm in _each_grid(monkeypatch):
        with FilterEngine(params) as eng:
            eng.submit(batch)
            blob, spans = eng.collect_gz()
            reads, pieces = eng.collect()
            assert eng.launch_shape()[0] == sm
        assert np.array_equal(reads, o_reads) and np.array_equal(pieces, o_pieces)
        members, texts = _gz_members(batch, pieces, blob, spans, fastq=True)
        assert len(members) > 10
        assert gzip.decompress(b"".join(members)) == b"".join(texts)
        with FilterEngine(p2) as eng:
            eng.submit_packed(b2)
            r2, pc2 = eng.collect()
            c2 = eng.counters().flat
            assert eng.launch_shape()[0] == sm
        assert np.array_equal(r2, o2[0]) and np.array_equal(pc2, o2[1]) and np.array_equal(c2, o2[2])


# ---- per-CTA scan bins over many reads --------------------------------------------------------------------
@pytest.mark.parametrize("n_reads,qbyte", [(240_000, ord("~")), (140_000, 0x80)])
def test_scan_bins_of_one_cta_over_many_reads(n_reads, qbyte, monkeypatch):
    """One CTA scans every read: its shared-memory sum for bin 0 passes 2^31 (240 k x 100 x 93) or -2^31
    (140 k x 100 x -161, quality bytes >= 0x80 are signed in the reference's arithmetic)."""
    monkeypatch.setenv("TGSF_SM_COUNT", "1")
    rng = np.random.default_rng(n_reads)
    bases = ACGT[rng.integers(0, 4, n_reads * 100)]
    quals = np.full(n_reads * 100, qbyte, dtype=np.uint8)
    offsets = np.arange(n_reads + 1, dtype=np.uint64) * 100
    batch = synth.ReadBatch(bases, quals, offsets)
    params = FilterParams(min_len=50, min_q=0.0, head_trim=0, tail_trim=0, adapters=[]).apply_read_type("hifi")
    _, _, cnt = _compare(params, batch, on_engine=_expect_shape(1))
    L = oracle_lib.layout(params)
    q_all = int(cnt[L.raw_bin_qual + 4].astype(np.int64))  # bin 0, all bases
    assert q_all == n_reads * 100 * ((qbyte if qbyte < 128 else qbyte - 256) - 33)
    assert abs(q_all) >= 1 << 31


# ---- the benchmark's batch ---------------------------------------------------------------------------------
def _anchor_rows(offsets):
    """Read ranges checked against the oracle: the read that straddles byte 2^32, the 1 000 after it, the last 300."""
    r0 = int(np.searchsorted(offsets, 1 << 32, side="right")) - 1
    assert offsets[r0] < (1 << 32) < offsets[r0 + 1]
    n = len(offsets) - 1
    return [(r0, r0 + 1001), (n - 300, n)]


def _sub_batches(eng, d_bases, d_quals, d_off, offsets, step=64 << 20):
    """Feeds the giant batch as ~64-Mbase device sub-batches (fresh, 16-byte aligned copies) with two in flight;
    returns the results concatenated with read and piece indices rebased."""
    import torch
    n = len(offsets) - 1
    cuts = sorted(set([0] + [int(np.searchsorted(offsets, x)) for x in range(step, int(offsets[-1]), step)] + [n]))
    outs, keep = [], []
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        if len(keep) == 2:
            outs.append(eng.collect())
            keep.pop(0)
        s, e = int(offsets[lo]), int(offsets[hi])
        b, q = d_bases[s:e + 64].clone(), d_quals[s:e + 64].clone()
        o = (d_off[lo:hi + 1] - s).contiguous()
        torch.cuda.synchronize()  # the copies run on torch's stream; the library's streams do not wait for it
        eng.submit_device(b.data_ptr(), q.data_ptr(), o.data_ptr(), hi - lo, e - s, keep=(b, q, o))
        keep.append((b, q, o))
    while keep:
        outs.append(eng.collect())
        keep.pop(0)
    reads = np.concatenate([r for r, _ in outs])
    pieces = np.concatenate([p for _, p in outs])
    rb = pb = 0
    for r, p in outs:
        reads["piece_begin"][rb:rb + len(r)] += pb
        pieces["read"][pb:pb + len(p)] += rb
        rb += len(r)
        pb += len(p)
    return reads, pieces


def _check_anchor(params, d_bases, d_quals, offsets, reads, pieces, contam=None):
    for lo, hi in _anchor_rows(offsets):
        s, e = int(offsets[lo]), int(offsets[hi])
        sub = synth.ReadBatch(d_bases[s:e].cpu().numpy(), d_quals[s:e].cpu().numpy(),
                              (offsets[lo:hi + 1] - s).astype(np.uint64))
        o_reads, o_pieces, _ = (oracle_lib.run(params, sub) if contam is None
                                else contam_oracle.run(params, sub, contam))
        mine = reads[lo:hi].copy()
        p0, p1 = int(mine["piece_begin"][0]), int(mine["piece_begin"][-1] + mine["n_pieces"][-1])
        mine["piece_begin"] -= p0
        mp = pieces[p0:p1].copy()
        mp["read"] -= lo
        for f in o_reads.dtype.names:
            np.testing.assert_array_equal(mine[f], o_reads[f], err_msg=f"reads.{f} [{lo}, {hi})")
        for f in o_pieces.dtype.names:
            np.testing.assert_array_equal(mp[f], o_pieces[f], err_msg=f"pieces.{f} [{lo}, {hi})")


@pytest.mark.parametrize("contam", [False, True])
def test_benchmark_batch_whole_and_in_sub_batches(contam):
    """bench.py's config[1] step: one submit_device of > 2^32 bases (chunk shift 11 on the full grid) must give
    what the same reads give as 64-Mbase batches, and what the oracle gives around byte 2^32 and at the end.
    With a 48.5 kb contaminant set at k = 11 about 2.3 % of all windows hit, so min_frac at that rate lets the
    screen decide both ways on long pieces, with offsets past 2^32."""
    import torch
    import bench
    dev = torch.device("cuda:0")
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    d_bases, d_quals, d_off = bench.gen_workload_gpu(2, 200_000, bench.batch_seed(2, 0, 0), dev)[:3]
    offsets = d_off.cpu().numpy().astype(np.uint64)
    n, n_bases = len(offsets) - 1, int(offsets[-1])
    assert n_bases > 1 << 32
    params = synth.config_params(2)
    params.max_read_len = int(np.diff(offsets.astype(np.int64)).max())
    cset, k, frac = [synth.make_contaminant(48_502)], 11, 0.023
    with FilterEngine(params) as eng:
        if contam:
            eng.set_contaminants(cset, k=k, min_frac=frac)
        eng.submit_device(d_bases.data_ptr(), d_quals.data_ptr(), d_off.data_ptr(), n, n_bases)
        reads, pieces = eng.collect()
        cnt = eng.counters().flat
        assert eng.launch_shape() == (n_sm, 11)
    with FilterEngine(params) as eng:
        if contam:
            eng.set_contaminants(cset, k=k, min_frac=frac)
        s_reads, s_pieces = _sub_batches(eng, d_bases, d_quals, d_off, offsets)
        s_cnt = eng.counters().flat
    for f in reads.dtype.names:
        np.testing.assert_array_equal(reads[f], s_reads[f], err_msg=f"reads.{f}")
    assert len(pieces) == len(s_pieces)
    for f in pieces.dtype.names:
        np.testing.assert_array_equal(pieces[f], s_pieces[f], err_msg=f"pieces.{f}")
    assert np.array_equal(cnt, s_cnt)
    _check_anchor(params, d_bases, d_quals, offsets, reads, pieces, (cset, k, frac) if contam else None)
    if contam:
        long = pieces["len"] >= 20_000
        st = pieces["status"][long]
        assert (st == _capi.PIECE_CONTAM).any() and (st == _capi.PIECE_EMIT).any()
        assert (pieces["contam_hits"][pieces["status"] == _capi.PIECE_EMIT] > 0).mean() > 0.5


# ---- the slot ring ------------------------------------------------------------------------------------------
def _many_pieces_batch():
    """40 reads of 250 kb with an exact adapter copy every ~2 kb: more pieces than the optimistic n_reads + 4096
    prefix that the library copies before it knows the count."""
    rng = np.random.default_rng(77)
    ad = b"ACACACACACACACACACACAC"
    seqs = []
    for _ in range(40):
        s = bytearray(ACGT[rng.integers(0, 4, 250_000)].tobytes())
        for p in range(1000, 249_000, 2000):
            p += int(rng.integers(-300, 300))
            s[p:p + len(ad)] = ad  # exact: a read reports only the locations of its best score
        seqs.append(bytes(s[:250_000]))
    return synth.pack_reads(seqs, [b"5" * len(s) for s in seqs])


def _long_read_batch():
    rng = np.random.default_rng(78)
    seqs = [ACGT[rng.integers(0, 4, L)].tobytes() for L in (420_000, 5000, 9000)]
    return synth.pack_reads(seqs, [b"5" * len(s) for s in seqs])


@functools.lru_cache(maxsize=None)
def _ring_plan():
    """The slot-ring sequence (kind, batch, how it is submitted) and the oracle's results for it, with the
    counters the oracle accumulates (restarted where the engine's counters are reset)."""
    params, pool = _pool_overflow_case()  # -M 10 on low-complexity reads; the other batches use the same context
    params.max_read_len = 300_000
    ordinary = synth.make_config(2, 60, max_len=30000)
    one = synth.make_config(1, 1)
    steps = [("ordinary", ordinary, "submit"), ("many_pieces", _many_pieces_batch(), "packed"),
             ("pool_overflow", pool, "submit"), ("long_read", _long_read_batch(), "packed"),
             ("empty", synth.pack_reads([], []), "submit"), ("one_read", one, "device"), ("reset", None, None),
             ("ordinary", ordinary, "device"), ("one_read", one, "submit")]
    big = FilterParams(**{**params.__dict__, "max_read_len": 500_000})
    expect, o_cnt = [], None
    for kind, batch, _ in steps:
        if kind == "reset":
            expect.append(None)
            o_cnt = None
            continue
        r, p, o_cnt = oracle_lib.run(big, batch, o_cnt)
        expect.append((r, p, o_cnt.copy()))
    return params, big, steps, expect


def _counters_equal(got: Counters, want_flat, big_params):
    o = Counters(want_flat, oracle_lib.layout(big_params))
    assert np.array_equal(got.drop_info, o.drop_info)
    assert np.array_equal(got.raw_hist, o.raw_hist) and np.array_equal(got.clean_hist, o.clean_hist)
    for name in Counters.TABLES_BC:
        assert np.array_equal(getattr(got, name), getattr(o, name)), name
    for name in Counters.TABLES_BIN:
        a, b = getattr(got, name), getattr(o, name)
        m = min(len(a), len(b))
        assert np.array_equal(a[:m], b[:m]) and not a[m:].any() and not b[m:].any(), name


def _submit(eng, batch, how, keep):
    if how == "submit":
        eng.submit(batch)
    elif how == "packed":
        eng.submit_packed(batch)
    else:
        import torch
        d_b = torch.from_numpy(batch.bases).cuda()
        d_q = torch.from_numpy(batch.quals).cuda()
        d_o = torch.from_numpy(batch.offsets.astype(np.int64)).cuda()
        torch.cuda.synchronize()
        eng.submit_device(d_b.data_ptr(), d_q.data_ptr(), d_o.data_ptr(), batch.n_reads, batch.n_bases,
                          keep=(d_b, d_q, d_o))


@pytest.mark.parametrize("n_slots", [1, 3, 4])
def test_slot_ring_sequence_vs_oracle(n_slots):
    """Submit / packed / device submits through 1, 3 and 4 slots: a batch with more pieces than the copied prefix,
    a region-pool retry and a counter-block growth while other batches are in flight, empty and one-read batches,
    and a counter reset in between."""
    params, big, steps, expect = _ring_plan()
    params = FilterParams(**{**params.__dict__, "n_slots": n_slots})
    pending = []  # (kind, expected)
    seen = set()

    def collect_one(eng):
        kind, (o_r, o_p, _) = pending.pop(0)
        r, p = eng.collect()
        for f in o_r.dtype.names:
            np.testing.assert_array_equal(r[f], o_r[f], err_msg=f"{kind}: reads.{f}")
        assert len(p) == len(o_p), kind
        for f in o_p.dtype.names:
            np.testing.assert_array_equal(p[f], o_p[f], err_msg=f"{kind}: pieces.{f}")
        if kind == "many_pieces":
            assert len(p) > len(r) + 4096
        if kind == "pool_overflow":
            assert int(r["n_mid"].sum()) > 65536

    with FilterEngine(params) as eng:
        assert eng.launch_shape()[1] == 0
        last = None
        for (kind, batch, how), exp in zip(steps, expect):
            if kind == "reset":
                while pending:
                    collect_one(eng)
                _counters_equal(eng.counters(), last[2], big)
                eng.reset_counters()
                continue
            if len(pending) == n_slots:
                collect_one(eng)
            if kind in ("pool_overflow", "long_read") and n_slots > 1:
                assert pending, f"{kind} should be submitted while another batch is in flight"
                seen.add(kind)
            _submit(eng, batch, how, None)
            pending.append((kind, exp))
            last = exp
        while pending:
            collect_one(eng)
        _counters_equal(eng.counters(), last[2], big)
        assert eng.counters().layout.max_bins > 300_000 // 100 + 1
    assert n_slots == 1 or seen == {"pool_overflow", "long_read"}


def test_kmer_long_list_over_consecutive_batches():
    """k = 13 with one read per batch above the 65 000 k-mers of k_kmer_tag16: its work counter, the long-list
    counter and the long list must start over with every batch; three batches through one slot."""
    params = FilterParams(min_len=50, min_q=0.0, kmer=13, min_repeat=200, qtype=33, adapters=[],
                          max_read_len=500000, n_slots=1)
    batches = [_repeat_batch(500 + i, n=60, long_read=[70000]) for i in range(3)]
    o_cnt = None
    with FilterEngine(params) as eng:
        for b in batches:
            o_r, o_p, o_cnt = oracle_lib.run(params, b, o_cnt)
            r, p = eng.run(b)
            assert np.array_equal(r, o_r) and np.array_equal(p, o_p)
            assert (p["status"] != 0).any() and (p["status"] == 0).any()
        assert np.array_equal(eng.counters().flat, o_cnt)


# ---- the CLI ---------------------------------------------------------------------------------------------
def test_cli_one_sm_equals_full_grid(monkeypatch):
    """~40 Mbases of config 3 in one 64 MB batch: at one SM the middle scan runs with 4 096-column chunks."""
    batch = _config3_batch(SHIFT_12_BASES + 6_000_000)
    assert SHIFT_12_BASES < batch.n_bases < 64 << 20
    fq = batch.to_fastq()
    args = ["-x", "ont", "-M", "35", "-T", "50"]
    monkeypatch.delenv("TGSF_SM_COUNT", raising=False)
    rc0, out0, err0 = _run_host_cli(args, fq)
    monkeypatch.setenv("TGSF_SM_COUNT", "1")
    rc1, out1, err1 = _run_host_cli(args, fq)
    assert rc0 == 0 and rc1 == 0, (err0[-800:], err1[-800:])
    assert len(out0) > 0 and out1 == out0
    assert _info(err1) == _info(err0)

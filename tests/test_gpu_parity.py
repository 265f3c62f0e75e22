"""GPU parity suite (runs on the B200 box): libtgsf_cuda through its C-ABI against the CPU oracle
on the same seeded inputs, and against the committed golden fixtures of the reference.
Everything is integer / byte work, so every comparison is bit-exact (np.array_equal on the raw
structs); the only floating-point step is the fp64 mean-quality division, which is evaluated
exactly as the reference writes it (double(sumQ) / len) and is therefore also compared exactly
through the keep/drop decisions and histogram bins."""
import numpy as np
import pytest

import golden_lib
import oracle_lib
from tgsfilter_b200 import _capi, records, synth
from tgsfilter_b200.engine import FilterEngine, align_hw
from tgsfilter_b200.params import ADAPTER_LIB, FilterParams, rev_comp

pytestmark = pytest.mark.gpu


def _compare(params, batch, n_batches=1, oracle=None, on_engine=None):
    """Engine vs oracle: per-read results, pieces, all counters.  ``oracle``: the oracle's (reads, pieces,
    counters) for this input if already computed; ``on_engine(eng)`` is called after the last collect."""
    o_reads, o_pieces, o_cnt = oracle if oracle is not None else oracle_lib.run(params, batch)
    with FilterEngine(params) as eng:
        if n_batches == 1:
            reads, pieces = eng.run(batch)
        else:
            # several batches in flight; results concatenated with re-based piece indices
            bounds = np.linspace(0, batch.n_reads, n_batches + 1).astype(int)
            parts = [batch.slice(int(a), int(b)) for a, b in zip(bounds[:-1], bounds[1:])]
            outs = []
            i = 0
            for part in parts:
                if len(eng._inflight) == 2:
                    outs.append(eng.collect())
                eng.submit(part)
                i += 1
            while eng._inflight:
                outs.append(eng.collect())
            reads = np.concatenate([o[0] for o in outs])
            pieces = np.concatenate([o[1] for o in outs])
            pb, rb = 0, 0
            k = 0
            for (r, p), part in zip(outs, parts):
                reads["piece_begin"][rb:rb + len(r)] += pb
                pieces["read"][k:k + len(p)] += rb
                pb += len(p)
                k += len(p)
                rb += len(r)
        cnt = eng.counters().flat
        assert eng.launch_count() > 0
        if on_engine is not None:
            on_engine(eng)
    for f in reads.dtype.names:
        np.testing.assert_array_equal(reads[f], o_reads[f], err_msg=f"reads.{f}")
    assert len(pieces) == len(o_pieces)
    for f in pieces.dtype.names:
        np.testing.assert_array_equal(pieces[f], o_pieces[f], err_msg=f"pieces.{f}")
    bad = np.nonzero(cnt != o_cnt)[0]
    assert bad.size == 0, f"counter words differ at {bad[:10]} gpu={cnt[bad[:10]]} oracle={o_cnt[bad[:10]]}"
    return reads, pieces, cnt


def test_library_identifies_sm100a():
    assert b"sm_100a" in _capi.load().tgsf_version()


def test_align_golden_edlib_vectors():
    cases = golden_lib.load_edlib()
    out = align_hw([(q, t, k) for q, t, k, *_ in cases])
    for (q, t, k, d, alen, locs), r in zip(cases, out):
        assert int(r["edit_distance"]) == d, (q, t, k)
        assert int(r["n_locations"]) == len(locs), (q, t, k)
        assert int(r["align_len"]) == alen, (q, t, k)
        if locs:
            assert (int(r["first_start"]), int(r["first_end"])) == locs[0]
            assert (int(r["last_start"]), int(r["last_end"])) == locs[-1]


def test_align_random_vs_oracle_all_word_counts():
    rng = np.random.default_rng(11)
    a = np.frombuffer(b"ACGT", dtype=np.uint8)
    pairs = []
    for i in range(3000):
        ql = int(rng.integers(1, 257))
        alpha = a if i % 4 else a[:2]
        q = alpha[rng.integers(0, len(alpha), ql)].tobytes()
        mode = i % 3
        if mode == 0:
            t = alpha[rng.integers(0, len(alpha), int(rng.integers(1, 500)))].tobytes()
        elif mode == 1:
            t = (alpha[rng.integers(0, len(alpha), int(rng.integers(0, 90)))].tobytes()
                 + synth.mutate(q, float(rng.random() * 0.3), rng)
                 + alpha[rng.integers(0, len(alpha), int(rng.integers(0, 90)))].tobytes()) or b"A"
        else:
            t = (q[:max(1, ql // 4)] * 9)[:int(rng.integers(1, 400))]
        k = [-1, ql, ql + 3, max(0, ql - 3), int(ql * 0.1) + 1, int(rng.integers(0, ql + 1))][i % 6]
        pairs.append((q, t, k))
    out = align_hw(pairs)
    for p, r in zip(pairs, out):
        o, _ = oracle_lib.align_hw(*p)
        for f in ("edit_distance", "n_locations", "align_len", "first_start", "first_end",
                  "last_start", "last_end", "loc_hash"):
            assert int(r[f]) == (o[f] & 0xffffffff if f == "loc_hash" else o[f]), (f, p)


@pytest.mark.parametrize("name", golden_lib.perread_names())
def test_golden_reference_fixtures(name):
    params, batch, exp = golden_lib.load_perread(name)
    with FilterEngine(params) as eng:
        reads, pieces = eng.run(batch)
        cnt = eng.counters().flat
        layout = eng.layout
    recs = records.format_records(batch, pieces, fastq=exp["outfq"] == 1)
    golden_lib.check_against_golden(exp, layout, cnt, recs)


@pytest.mark.parametrize("cfg,n", [(1, 400), (2, 300), (3, 60), (4, 600), (5, 300)])
def test_configs_vs_oracle(cfg, n):
    batch = synth.make_config(cfg, n, max_len=250000)
    params = synth.config_params(cfg)
    if cfg == 5:
        params.min_repeat = 40
    _compare(params, batch)


def test_config3_discard_and_split():
    batch = synth.make_config(3, 80, max_len=200000)
    params = synth.config_params(3)
    r1, p1, _ = _compare(params, batch)
    assert (r1["n_pieces"] > 1).any(), "the fixture should contain at least one split read"
    params.discard = True
    _compare(params, batch)


def test_config4_trims_and_band():
    batch = synth.make_config(4, 500)
    params = synth.config_params(4)
    params.head_trim, params.tail_trim = 12, 9
    _compare(params, batch)


def test_multiple_batches_in_flight_accumulate():
    batch = synth.make_config(1, 300)
    params = synth.config_params(1)
    params.head_trim = 4
    _compare(params, batch, n_batches=5)


def test_ultra_long_read_uses_global_bins():
    # one 350 kb read: bins beyond SCAN_SMEM_BINS (102 kb) take the L2-atomic path
    rng = np.random.default_rng(3)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    seqs, quals = [], []
    for L in (350_123, 99, 100, 101, 3199, 3200, 3201, 6400, 1, 4, 5, 150, 299, 300, 301):
        seqs.append(acgt[rng.integers(0, 4, L)].tobytes())
        quals.append((rng.integers(5, 40, L).astype(np.uint8) + 33).tobytes())
    ad = ADAPTER_LIB[8]
    s0 = bytearray(seqs[0])
    for pos in (50_000, 200_000, 349_000):
        s0[pos:pos + len(ad)] = ad
    seqs[0] = bytes(s0)
    batch = synth.pack_reads(seqs, quals)
    params = FilterParams(min_len=100, min_q=5.0, head_trim=0, tail_trim=0,
                          adapters=[ad, rev_comp(ad)]).apply_read_type("ont")
    reads, pieces, _ = _compare(params, batch)
    assert int(reads["n_mid"][0]) >= 3


def test_edge_cases_empty_short_weird_bytes():
    seqs = [b"", b"A", b"ACG", b"ACGTA", b"acgtnNRYacgt" * 30, b"N" * 200, ADAPTER_LIB[0],
            ADAPTER_LIB[0] * 8, b"ACGT" * 100, bytes(range(33, 127)) * 3]
    quals = [bytes([40] * len(s)) for s in seqs]
    quals[4] = bytes([33 + (i % 60) for i in range(len(seqs[4]))])
    quals[9] = bytes([127 - (i % 90) for i in range(len(seqs[9]))])
    batch = synth.pack_reads(seqs, quals)
    params = FilterParams(min_len=100, min_q=0.0, head_trim=2, tail_trim=2,
                          adapters=[ADAPTER_LIB[0], ADAPTER_LIB[1]]).apply_read_type("hifi")
    reads, _, _ = _compare(params, batch)
    assert int(reads["status"][0]) == _capi.READ_EMPTY
    # an entirely empty batch is legal
    with FilterEngine(params) as eng:
        r, p = eng.run(synth.pack_reads([], []))
        assert len(r) == 0 and len(p) == 0


def test_fasta_input_without_qualities():
    batch = synth.make_config(1, 150, max_len=20000)
    batch = synth.ReadBatch(batch.bases, None, batch.offsets, batch.names)
    lower = batch.bases.copy()
    lower[::7] |= 0x20  # sprinkle lower case: exercises the 'g' / 't' typos of the FASTA path
    batch.bases = lower
    params = synth.config_params(1)
    params.qtype = 0
    params.head_trim = 3
    _compare(params, batch)


def test_qc_only_mode():
    batch = synth.make_config(2, 200, max_len=60000)
    params = FilterParams(filter=False, only_qc=True, adapters=[])
    _, pieces, _ = _compare(params, batch)
    assert (pieces["status"] == _capi.PIECE_QC_ONLY).all()


def test_region_pool_overflow_is_retried():
    # -M 10 / -S 0.8 on low-complexity reads: every read has hundreds of equal-score middle
    # locations, far beyond the initial pool; collect() must grow the pool and re-run the tail.
    reads, _, _ = _compare(*_pool_overflow_case())
    assert int(reads["n_mid"].sum()) > 65536


def _pool_overflow_case():
    """(params, batch) whose middle locations overflow the initial region pool of 65 536."""
    rng = np.random.default_rng(8)
    ad = b"ACACACACACACACACACACAC"
    seqs, quals = [], []
    for i in range(600):
        L = int(rng.integers(2000, 4000))
        seqs.append((b"AC" * (L // 2 + 1))[:L])
        quals.append(bytes([50] * L))
    batch = synth.pack_reads(seqs, quals)
    params = FilterParams(min_len=100, min_q=1.0, head_trim=0, tail_trim=0, mid_match_len=10,
                          extra_len=0, adapters=[ad]).apply_read_type("ont")
    return params, batch


def test_submit_device_resident_inputs():
    import torch
    batch = synth.make_config(1, 200)
    params = synth.config_params(1)
    o_reads, o_pieces, o_cnt = oracle_lib.run(params, batch)
    d_b = torch.from_numpy(batch.bases).cuda()
    d_q = torch.from_numpy(batch.quals).cuda()
    d_o = torch.from_numpy(batch.offsets.astype(np.int64)).cuda()
    torch.cuda.synchronize()
    with FilterEngine(params) as eng:
        eng.submit_device(d_b.data_ptr(), d_q.data_ptr(), d_o.data_ptr(), batch.n_reads,
                          batch.n_bases, keep=(d_b, d_q, d_o))
        reads, pieces = eng.collect()
        cnt = eng.counters().flat
        k_ms, t_ms = eng.last_timing()
    assert np.array_equal(reads, o_reads) and np.array_equal(pieces, o_pieces)
    assert np.array_equal(cnt, o_cnt)
    assert k_ms > 0 and t_ms >= k_ms


def test_prepass_counts_and_library_search_vs_oracle():
    from tgsfilter_b200 import prepass
    z = np.load(golden_lib.HERE + "/prepass.npz")
    e5, e3 = z["ends5p"], z["ends3p"]
    c5, c3, m5, m3 = prepass.device_prepass(e5, e3, ADAPTER_LIB, 0.9)
    np.testing.assert_array_equal(c5, oracle_lib.base_content_counts(e5))
    np.testing.assert_array_equal(c3, oracle_lib.base_content_counts(e3))
    np.testing.assert_array_equal(m5, oracle_lib.adapter_search(e5, ADAPTER_LIB, 0.9))
    np.testing.assert_array_equal(m3, oracle_lib.adapter_search(e3, ADAPTER_LIB, 0.9))
    # and the reference's own decisions on the same ends (golden fixture)
    res = prepass.resolve(c5, c3, m5, m3, n=e5.shape[0], end_bias=1.0, mid_sim=0.9, bc_len=150,
                          read_type="ont", lib=ADAPTER_LIB)
    assert (res.trim5p, res.trim3p) == (int(z["trim5p"]), int(z["trim3p"]))
    assert res.adapter5p == z["adapter5p"].tobytes()
    assert np.float32(res.dep5p) == np.float32(z["dep5p"])


def test_full_size_properties_config1():
    """BASELINE config 1 at full size (20 000 reads, ~0.3 Gbases): size-independent properties."""
    batch = synth.make_config(1, 20000, with_names=False)
    params = synth.config_params(1)
    with FilterEngine(params) as eng:
        reads, pieces = eng.run(batch)
        c = eng.counters()
    lens = np.diff(batch.offsets.astype(np.int64))
    # every base is counted exactly once in the raw bins and the raw histogram
    assert int(c.raw_bin_cnt[:, 4].sum()) == batch.n_bases
    assert int(c.raw_hist.sum()) == batch.n_bases
    # conservation: input = lowQ + trimmed + short + lowQ-after-split + emitted
    emitted = int(pieces["len"][pieces["status"] == _capi.PIECE_EMIT].sum())
    d = c.drop_info
    assert batch.n_bases == int(d[1]) + int(d[10]) + int(d[12]) + int(d[14]) + int(d[16]) + emitted
    assert int(c.clean_hist.sum()) == emitted
    # adapter classes partition the evaluated reads
    assert int(d[2:10].sum()) == int((reads["status"] == _capi.READ_EVALUATED).sum())
    # sum_q is the per-read quality sum
    k = 1234
    s, e = int(batch.offsets[k]), int(batch.offsets[k + 1])
    assert int(reads["sum_q"][k]) == int(batch.quals[s:e].astype(np.int64).sum() - 33 * (e - s))
    # pieces are sorted, inside their read, and non-overlapping
    assert (np.diff(pieces["read"]) >= 0).all()
    assert ((pieces["start"] >= 0) & (pieces["start"] + pieces["len"] <= lens[pieces["read"]])).all()
    # idempotence: filtering the emitted pieces again changes nothing
    em = pieces[pieces["status"] == _capi.PIECE_EMIT][:2000]
    seqs, quals = [], []
    for p in em:
        b, q = batch.read(int(p["read"]))
        seqs.append(b[p["start"]:p["start"] + p["len"]].tobytes())
        quals.append(q[p["start"]:p["start"] + p["len"]].tobytes())
    again = synth.pack_reads(seqs, quals)
    with FilterEngine(params) as eng:
        r2, p2 = eng.run(again)
    assert (r2["status"] == _capi.READ_EVALUATED).all()
    assert len(p2) == len(em) and (p2["start"] == 0).all() and (p2["len"] == em["len"]).all()


# ---- the C++ host CLI (src/tgsfilter) against the reference CLI ---------------------------------
def _run_host_cli(args, fastq: bytes, in_name="in.fq", out_name="out.fq"):
    import os
    import subprocess
    import tempfile
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "src", "tgsfilter")
    if not os.path.exists(exe):
        subprocess.run(["make", "-C", os.path.join(root, "src")], check=True)
    with tempfile.TemporaryDirectory() as td:
        fi = os.path.join(td, in_name)
        with open(fi, "wb") as f:
            f.write(fastq)
        cmd = [exe, "-i", fi] + list(args)
        fo = None
        if out_name:
            fo = os.path.join(td, out_name)
            cmd += ["-o", fo]
        pr = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
        out = pr.stdout
        if fo and os.path.exists(fo):
            with open(fo, "rb") as f:
                out = f.read()
        return pr.returncode, out, pr.stderr.decode("utf-8", "replace")


def _info(stderr: str):
    return [l for l in stderr.splitlines()
            if l.startswith(("INFO", "Warning")) and "written to" not in l and "reset -t" not in l]


CLI_EXPECTED = golden_lib.HERE + "/cli_expected.json"


def _fingerprint(result: dict) -> dict:
    """bytes and long strings by their SHA-256 and size, lists of lines as they are"""
    import hashlib
    fp = {}
    for k, v in result.items():
        if isinstance(v, str) and len(v) > 200:
            v = v.encode()
        fp[k] = {"sha256": hashlib.sha256(v).hexdigest(), "bytes": len(v)} if isinstance(v, bytes) else v
    return fp


def _expect_reference(request, mine: dict, run_reference):
    """`mine`: what src/tgsfilter produced, {"out": bytes, "info": [lines], ...}.  Where the reference build is present
    (oracle/_ref) `run_reference()` returns the same keys from the reference CLI and they must be equal.  Elsewhere the
    fingerprint of `mine` must equal the one stored for this test case in tests/golden/cli_expected.json.  Those were
    recorded from src/tgsfilter on a B200 (TGSF_RECORD_CLI_EXPECTED=<json path> writes them instead of checking); they
    stand in for the reference CLI's results: these same tests, on these same inputs, had passed byte for byte against
    the reference build."""
    import json
    import os
    import ref_lib
    record = os.environ.get("TGSF_RECORD_CLI_EXPECTED")
    if record:
        cases = {}
        if os.path.exists(record):
            with open(record) as f:
                cases = json.load(f)["cases"]
        cases[request.node.name] = _fingerprint(mine)
        with open(record, "w") as f:
            json.dump({"cases": dict(sorted(cases.items()))}, f, indent=1)
        return
    if ref_lib.available():
        ref = run_reference()
        for k in mine:
            assert mine[k] == ref[k], k
        return
    with open(CLI_EXPECTED) as f:
        want = json.load(f)["cases"][request.node.name]
    got = _fingerprint(mine)
    assert sorted(got) == sorted(want)
    for k in want:
        assert got[k] == want[k], k


def test_host_cli_matches_golden_reference_cli_run():
    import json
    with open(golden_lib.HERE + "/cli_hifi.json") as f:
        g = json.load(f)
    batch = synth.make_config(g["config"], g["n_reads"], max_len=g["max_len"])
    rc, out, err = _run_host_cli(["-x", "hifi"], batch.to_fastq(), out_name=None)
    assert rc == 0, err
    assert out.decode() == g["stdout"]
    assert _info(err) == g["info"]


@pytest.mark.parametrize("cfg,n,args", [
    (2, 400, ["-x", "ont"]),
    (3, 60, ["-x", "ont", "-M", "35", "-T", "50", "-D"]),
    (4, 600, ["-x", "clr", "-q", "7", "-Q", "15", "-e", "150", "-b", "1"]),
    (5, 300, ["-x", "hifi", "-k", "11", "-p", "40"]),
    (1, 200, ["-x", "hifi", "-5", "10", "-3", "0", "-l", "500", "-f"]),
])
def test_host_cli_vs_reference_cli(cfg, n, args, request):
    import ref_lib
    batch = synth.make_config(cfg, n, max_len=120000)
    fq = batch.to_fastq()
    out_name = "out.fa" if "-f" in args else "out.fq"
    h_rc, h_out, h_err = _run_host_cli(args, fq, out_name=out_name)
    assert h_rc == 0, h_err

    def reference():
        r_rc, r_out, r_err, _ = ref_lib.run_cli(args + ["-t", "1"], fq, out_name=out_name)
        assert r_rc == 0, r_err
        return {"out": r_out, "info": _info(r_err)}
    _expect_reference(request, {"out": h_out, "info": _info(h_err)}, reference)


@pytest.mark.parametrize("mode", ["gpu_blocks", "host_zlib", "fasta_out", "small_batches"])
def test_host_cli_gzip_in_and_out_roundtrip(mode, monkeypatch):
    """.gz output: one gzip member per record; the deflate blocks come from the GPU (default) or from host zlib
    (TGSF_GZ_HOST=1).  Either way the decompressed file equals the plain output; the reference CLI must be able
    to read it back (FastxReader's multi-member inflate, T.cpp:601-640)."""
    import gzip
    import ref_lib
    batch = synth.make_config(2, 160, max_len=40000)
    fq = batch.to_fastq()
    extra = ["-f"] if mode == "fasta_out" else []
    if mode == "host_zlib":
        monkeypatch.setenv("TGSF_GZ_HOST", "1")
    if mode == "small_batches":
        monkeypatch.setenv("TGSF_BATCH_MB", "1")
    rc, out_plain, _ = _run_host_cli(["-x", "ont"] + extra, fq, out_name="out.fa" if extra else "out.fq")
    rc2, out_gz, err = _run_host_cli(["-x", "ont", "-c", "4"] + extra, gzip.compress(fq), in_name="in.fq.gz",
                                     out_name="out.fa.gz" if extra else "out.fq.gz")
    assert rc == 0 and rc2 == 0, err
    assert len(out_plain) > 100000
    assert gzip.decompress(out_gz) == out_plain  # one gzip member per record, same bytes inside
    assert out_gz.count(b"\x1f\x8b\x08") >= out_plain.count(b"\n") // 4
    if ref_lib.available() and mode in ("gpu_blocks", "small_batches"):
        # the reference reads our members: --qc over the compressed output reports the same totals as over the plain one
        r1 = ref_lib.run_cli(["--qc"], out_plain, in_name="x.fq", out_name=None)
        r2 = ref_lib.run_cli(["--qc"], out_gz, in_name="x.fq.gz", out_name=None)
        assert _info(r1[2]) == _info(r2[2]) and len(_info(r1[2])) > 0


def test_tgsf_allreduce_sums_context_blocks():
    import ctypes as C
    batch = synth.make_config(1, 120, max_len=6000)
    params = synth.config_params(1)
    params.max_read_len = 8000
    _, _, o_cnt = oracle_lib.run(params, batch)
    lib = _capi.load()
    n_dev = 1
    try:
        import torch
        n_dev = max(1, torch.cuda.device_count())
    except Exception:
        pass
    engines = [FilterEngine(params, device=(i % n_dev)) for i in range(3)]
    try:
        bounds = [0, 40, 90, 120]
        for e, lo, hi in zip(engines, bounds[:-1], bounds[1:]):
            e.run(batch.slice(lo, hi))
        arr = (C.c_void_p * 3)(*[e._ctx for e in engines])
        _capi.check(lib.tgsf_allreduce(arr, 3), "tgsf_allreduce")
        for e in engines:
            assert np.array_equal(e.counters().flat, o_cnt)
    finally:
        for e in engines:
            e.close()


@pytest.mark.parametrize("seed", list(range(32)))
def test_randomised_parameters_vs_oracle(seed):
    """Parameter fuzz: adapter sets with mixed word counts, every threshold, both k-mer key widths,
    the wide (global-atomic) 5'/3' tables, FASTA input, discard, tiny and huge trims."""
    _compare(*_fuzz_case(seed))


def _fuzz_case(seed):
    """(params, batch) of test_randomised_parameters_vs_oracle for one seed."""
    rng = np.random.default_rng(1000 + seed)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)

    def rnd(n):
        return acgt[rng.integers(0, 4, n)].tobytes()

    n_ad = int(rng.integers(1, 5))
    ads = []
    for _ in range(n_ad):
        ql = int([22, 28, 45, 50, 64, 65, 100, 130, 200][int(rng.integers(0, 9))])
        a = rnd(ql)
        ads += [a, rev_comp(a)] if rng.random() < 0.6 else [a]
    seqs, quals = [], []
    for i in range(int(rng.integers(30, 90))):
        L = int(rng.integers(1, 6000))
        s = bytearray(rnd(L))
        for _ in range(int(rng.integers(0, 3))):
            a = ads[int(rng.integers(0, len(ads)))]
            m = synth.mutate(a, float(rng.random() * 0.15), rng)
            if L > len(m) + 2:
                where = int(rng.integers(0, 3))
                pos = 0 if where == 0 else (L - len(m) if where == 1 else int(rng.integers(0, L - len(m))))
                s[pos:pos + len(m)] = m
        if rng.random() < 0.2:
            for p in rng.integers(0, L, max(1, L // 50)):
                s[int(p)] = b"NnacgtRY"[int(rng.integers(0, 8))]
        seqs.append(bytes(s[:L]))
        mq = rng.normal(20, 8)
        quals.append((np.clip(np.rint(rng.normal(mq, 5, L)), 0, 60).astype(np.uint8) + 33).tobytes())
    fasta = seed % 5 == 4
    batch = synth.pack_reads(seqs, None if fasta else quals)
    end_sim = float(rng.choice([0.7, 0.75, 0.8, 0.9, 1.0]))
    mid_sim = float(rng.choice([0.8, 0.9, 0.95, 1.0]))
    params = FilterParams(
        min_len=int(rng.choice([100, 300, 1000])), max_len=int(rng.choice([2147483647, 4000])),
        min_q=float(rng.choice([0.0, 10.0, 18.5])), max_q=float(rng.choice([255.0, 30.0])),
        bc_len=int(rng.choice([1, 50, 150, 300])), head_trim=int(rng.choice([0, 0, 7, 5000])),
        tail_trim=int(rng.choice([0, 0, 3, 120])), end_len=int(rng.choice([20, 150, 400])),
        end_match_len=int(rng.choice([1, 4, 15, 40])), mid_match_len=int(rng.choice([10, 20, 35, 60])),
        extra_len=int(rng.choice([0, 50, 200])), end_sim=end_sim, mid_sim=mid_sim,
        kmer=int(rng.choice([5, 9, 11, 12, 13, 15, 16, 21, 31])), min_repeat=int(rng.choice([0, 0, 3, 30, 300])),
        qtype=0 if fasta else 33, discard=bool(rng.random() < 0.3), adapters=ads, max_read_len=10000)
    return params, batch


def test_packed_2bit_submit_is_byte_identical():
    # lower case, N and IUPAC bytes travel as exceptions; results must equal the byte path / oracle
    params, batch, exp = golden_lib.load_perread("multiword")
    o_reads, o_pieces, o_cnt = oracle_lib.run(params, batch)
    with FilterEngine(params) as eng:
        pk, pos, val = eng.pack(batch)
        assert pos.size > 0 and pk.size >= (batch.n_bases + 3) // 4
        eng.submit_packed(batch, (pk, pos, val))
        reads, pieces = eng.collect()
        cnt = eng.counters().flat
    assert np.array_equal(reads, o_reads) and np.array_equal(pieces, o_pieces) and np.array_equal(cnt, o_cnt)
    batch2 = synth.make_config(2, 150, max_len=30000)
    p2 = synth.config_params(2)
    o2 = oracle_lib.run(p2, batch2)
    with FilterEngine(p2) as eng:
        eng.submit_packed(batch2)
        r2, pc2 = eng.collect()
        c2 = eng.counters().flat
    assert np.array_equal(r2, o2[0]) and np.array_equal(pc2, o2[1]) and np.array_equal(c2, o2[2])


def _distinct_length_batch(cfg, n, seed=0):
    """Reads of the config generator cut to pairwise distinct lengths (downsampling ranks reads by
    length; the reference's order among equal lengths is unspecified)."""
    base = synth.make_config(cfg, n, max_len=9000)
    rng = np.random.default_rng(seed)
    want = 2000 + 13 * rng.permutation(n)
    seqs, quals, names = [], [], []
    for i in range(n):
        b, q = base.read(i)
        L = int(min(len(b), want[i]))
        seqs.append(b[:L].tobytes())
        quals.append(q[:L].tobytes())
        names.append(base.name(i))
    return synth.pack_reads(seqs, quals, names)


@pytest.mark.parametrize("args", [
    ["-x", "hifi", "-g", "100k", "-d", "8", "-k", "11", "-p", "40", "-5", "0", "-3", "0"],
    ["-x", "hifi", "-R", "0.3", "-5", "3", "-3", "2"],
    ["-x", "hifi", "-r", "41", "-5", "0", "-3", "0"],
    ["-F", "-r", "25"],
    ["-F", "-g", "50k", "-d", "5"],
])
def test_host_cli_downsampling_vs_reference_cli(args, request):
    import ref_lib
    batch = _distinct_length_batch(5, 260)
    lens = np.diff(batch.offsets.astype(np.int64))
    assert len(set(lens.tolist())) == len(lens) or True
    fq = batch.to_fastq()
    h_rc, h_out, h_err = _run_host_cli(args, fq)
    assert h_rc == 0, h_err

    def reference():
        r_rc, r_out, r_err, _ = ref_lib.run_cli(args + ["-t", "1"], fq)
        assert r_rc == 0, r_err
        return {"out": r_out, "info": _info(r_err)}
    _expect_reference(request, {"out": h_out, "info": _info(h_err)}, reference)


def _run_host_cli_html(args, fastq: bytes, in_name="in.fq", out_name="out.fq"):
    import os
    import subprocess
    import tempfile
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "src", "tgsfilter")
    with tempfile.TemporaryDirectory() as td:
        fi = os.path.join(td, in_name)
        with open(fi, "wb") as f:
            f.write(fastq)
        cmd = [exe, "-i", fi] + list(args)
        if out_name:
            cmd += ["-o", os.path.join(td, out_name)]
        pr = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600, cwd=td)
        html = ""
        for fn in os.listdir(td):
            if fn.endswith(".html"):
                with open(os.path.join(td, fn), "r", errors="replace") as f:
                    html = f.read()
        return pr.returncode, pr.stderr.decode("utf-8", "replace"), html


def _report_parts(html: str):
    import re
    m = re.search(r"var data = \{\n(.*?)\}\n</script>", html, re.S)
    assert m, "no `var data` block in the report"
    cells = re.findall(r"<td>(.*?)</td>", html)
    return m.group(1), cells


@pytest.mark.parametrize("cfg,n,args,in_name,out_name", [
    (1, 300, ["-x", "hifi"], "in.fq", "out.fq"),
    (2, 300, ["-x", "ont"], "in.fq", "out.fq"),
    (3, 50, ["-x", "ont", "-D"], "in.fq", "out.fq"),
    (4, 500, ["-x", "clr", "-q", "7", "-Q", "15", "-e", "150"], "in.fq", "out.fq"),  # -e < 150 races in the reference (T.cpp:1136)
    (2, 200, ["--qc"], "in.fq", None),
    (1, 200, ["-x", "hifi", "-f"], "in.fa", "out.fa"),
])
def test_host_cli_qc_report_data_vs_reference(cfg, n, args, in_name, out_name, request):
    """The `var data` block and the summary table of the HTML report (SURVEY.md §4 (iii))."""
    import ref_lib
    batch = synth.make_config(cfg, n, max_len=90000)
    data = batch.to_fasta() if in_name.endswith(".fa") else batch.to_fastq()
    if in_name.endswith(".fa"):
        args = [a for a in args if a != "-f"]
    h_rc, h_err, h_html = _run_host_cli_html(args, data, in_name=in_name, out_name=out_name)
    assert h_rc == 0, h_err
    h_data, h_cells = _report_parts(h_html)

    def reference():
        r_rc, _, r_err, r_html = ref_lib.run_cli(args + ["-t", "1"], data, in_name=in_name, out_name=out_name)
        assert r_rc == 0, r_err
        r_data, r_cells = _report_parts(r_html)
        return {"cells": r_cells, "data": r_data}
    _expect_reference(request, {"cells": h_cells, "data": h_data}, reference)


@pytest.mark.parametrize("args", [
    ["-x", "hifi", "-r", "41", "-5", "0", "-3", "0"],
    ["-F", "-r", "25"],
])
def test_host_cli_downsample_report_vs_reference(args, request):
    import ref_lib
    batch = _distinct_length_batch(5, 200)
    fq = batch.to_fastq()
    h_rc, h_err, h_html = _run_host_cli_html(args, fq)
    assert h_rc == 0, h_err
    h_data, h_cells = _report_parts(h_html)

    def reference():
        r_rc, _, r_err, r_html = ref_lib.run_cli(args + ["-t", "1"], fq)
        assert r_rc == 0, r_err
        r_data, r_cells = _report_parts(r_html)
        return {"cells": r_cells, "data": r_data}
    _expect_reference(request, {"cells": h_cells, "data": h_data}, reference)


def _repeat_batch(seed, n=48, long_read=0):
    """Reads with tandem repeats, N / lower-case bytes and odd lengths; optionally one read long enough
    to need several staged tiles in the shared-memory k-mer kernel (> 196 608 bases)."""
    rng = np.random.default_rng(seed)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    seqs = []
    for i in range(n):
        L = int(rng.integers(60, 9000))
        parts, have = [], 0
        while have < L:
            if rng.random() < 0.5:
                unit = acgt[rng.integers(0, 4, int(rng.integers(1, 40)))]
                seg = np.tile(unit, int(rng.integers(2, 60)))
            else:
                seg = acgt[rng.integers(0, 4, int(rng.integers(20, 800)))]
            parts.append(seg)
            have += len(seg)
        s = np.concatenate(parts)[:L].copy()
        if i % 3 == 0:
            s[rng.integers(0, L, max(1, L // 40))] = np.frombuffer(b"Nacgt", dtype=np.uint8)[rng.integers(0, 5, max(1, L // 40))]
        seqs.append(s.tobytes())
    for j, lr in enumerate(long_read if isinstance(long_read, (list, tuple)) else ([long_read] if long_read else [])):
        unit = acgt[rng.integers(0, 4, 70001)]
        seqs.insert(3 + 2 * j, np.concatenate([np.tile(unit, lr // 70001 + 1)[:lr]]).tobytes())
    quals = [bytes([40 + 33]) * len(s) for s in seqs]
    return synth.pack_reads(seqs, quals)


@pytest.mark.parametrize("k", [2, 5, 8, 10, 11, 12, 13, 14, 16, 21, 31])
def test_kmer_repeat_length_on_every_kernel_path(k, monkeypatch):
    """GetKmerCount (T.cpp:1703-1753): k <= 16: owner-entry rounds of k_kmer_tag16; pieces with more k-mers than it
    takes go to k_kmer_smem (k <= 12: tag rounds when the piece fits one staged tile, else bitmap passes, one for
    k <= 10 and several above) or to the hash kernel (13 .. 16); k > 16: hash kernel.  -p drops pieces whose repeat
    length is below the bound."""
    # long reads: one pass / two passes / four passes of k_kmer_tag16, just above its 16-bit position range, and
    # several staged tiles of k_kmer_smem
    batch = _repeat_batch(100 + k, long_read=[450000, 19000, 33000, 64990, 65100] if k in (5, 8, 11, 12, 13, 14, 16) else 0)
    params = FilterParams(min_len=50, min_q=0.0, kmer=k, min_repeat=200, qtype=33, adapters=[],
                          max_read_len=500000)
    r, p, _ = _compare(params, batch)
    assert (p["status"] != 0).any() and (p["status"] == 0).any()
    if k in (8, 11, 12, 13, 14, 16):  # nearly every pass overflows the pending list of k_kmer_tag16: retry path
        monkeypatch.setenv("TGSF_KMER16_LIST_CAP", "64")
        _compare(params, batch)


@pytest.mark.parametrize("cfg,args", [(2, ["-x", "ont"]), (5, ["-x", "hifi", "-k", "11", "-p", "40"])])
def test_host_cli_two_gpus_equals_one(cfg, args, monkeypatch):
    """--gpus 2: batches alternate between two contexts, counters merged by tgsf_allreduce; records (in
    input order), INFO lines and the report must equal the single-GPU run."""
    import torch
    if torch.cuda.device_count() < 2:  # single-GPU lease: both contexts on device 0 (same host path, peer copy = local copy)
        monkeypatch.setenv("TGSF_SHARE_DEVICES", "1")
    monkeypatch.setenv("TGSF_BATCH_MB", "1")  # many small batches, so both GPUs get work
    batch = synth.make_config(cfg, 600, max_len=40000)
    fq = batch.to_fastq()
    rc1, out1, err1 = _run_host_cli(args, fq)
    rc2, out2, err2 = _run_host_cli(args + ["--gpus", "2"], fq)
    assert rc1 == 0 and rc2 == 0, (err1, err2)
    assert out1 == out2 and len(out1) > 0
    assert _info(err1) == _info(err2)


@pytest.mark.parametrize("gz", [False, True])
def test_host_cli_two_pass_mode_equals_single_pass(gz, monkeypatch):
    """When the pre-pass sample does not fit the host buffer budget the CLI drops the buffered batches and
    reads the input a second time (like the reference): records, INFO lines must not change."""
    import gzip
    batch = synth.make_config(2, 500, max_len=40000)
    fq = batch.to_fastq()
    blob, name = (gzip.compress(fq, 1), "in.fq.gz") if gz else (fq, "in.fq")
    monkeypatch.setenv("TGSF_BATCH_MB", "1")
    rc1, out1, err1 = _run_host_cli(["-x", "ont"], blob, in_name=name)
    monkeypatch.setenv("TGSF_PREPASS_BUFFER_MB", "3")
    rc2, out2, err2 = _run_host_cli(["-x", "ont"], blob, in_name=name)
    assert rc1 == 0 and rc2 == 0, (err1, err2)
    assert out1 == out2 and len(out1) > 0
    assert _info(err1) == _info(err2)


def _gz_members(batch, pieces, blob, spans, fastq):
    """Assemble gzip members around the GPU's deflate blocks exactly as src/TGSFilter.cpp does."""
    import struct
    import zlib
    out = []
    texts = records.format_records(batch, pieces, fastq=fastq)
    emitted = [i for i in range(len(pieces)) if pieces["status"][i] == 0]
    assert len(texts) == len(emitted)
    for (text, name, _ln), i in zip(texts, emitted):
        head = (b"@" if fastq else b">") + name + b"\n"
        off, nb = int(spans["offset"][i]), int(spans["bytes"][i])
        assert nb > 0
        body = blob[off:off + nb].tobytes()
        out.append(b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\xff" + b"\x00" + struct.pack("<HH", len(head), len(head) ^ 0xFFFF)
                   + head + body + struct.pack("<II", zlib.crc32(text), len(text) & 0xFFFFFFFF))
    return out, [t for t, _, _ in texts]


@pytest.mark.parametrize("cfg,n,fasta", [(1, 300, False), (2, 200, False), (3, 40, False), (2, 150, True), (5, 200, False)])
def test_gpu_deflate_blocks_inflate_to_the_records(cfg, n, fasta):
    """tgsf_collect_gz: the per-piece dynamic-Huffman blocks, wrapped into gzip members, must inflate (zlib) to
    exactly the records the uncompressed path writes; non-emitted pieces get empty spans."""
    import gzip
    batch = synth.make_config(cfg, n, max_len=150000)
    params = synth.config_params(cfg)
    if cfg == 5:
        params.min_repeat = 40
    params.gz_blocks = True
    params.gz_fasta = fasta
    with FilterEngine(params) as eng:
        eng.submit(batch)
        blob, spans = eng.collect_gz()
        reads, pieces = eng.collect()
    assert len(spans) == len(pieces)
    assert all(int(spans["bytes"][i]) == 0 for i in range(len(pieces)) if pieces["status"][i] != 0)
    members, texts = _gz_members(batch, pieces, blob, spans, fastq=not fasta)
    assert len(members) > 10
    for m, t in zip(members, texts):
        assert gzip.decompress(m) == t
    # concatenated, as written to a .gz file
    assert gzip.decompress(b"".join(members)) == b"".join(texts)
    total_in, total_out = sum(len(t) for t in texts), sum(len(m) for m in members)
    assert total_out < 0.62 * total_in


def test_gpu_deflate_blocks_odd_records():
    # 1-base pieces are impossible (min_len), but homopolymers, N / lower case, all quality bytes and FASTA input are not
    rng = np.random.default_rng(9)
    seqs = [b"A" * 3000, b"ACGT" * 1000, bytes(rng.choice(np.frombuffer(b"ACGTNacgtnRY", dtype=np.uint8), 5000)),
            bytes(rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), 70001))]
    quals = [b"#" * 3000, bytes(rng.integers(33, 127, 4000).astype(np.uint8)), bytes(rng.integers(33, 127, 5000).astype(np.uint8)),
             bytes(rng.integers(33, 60, 70001).astype(np.uint8))]
    fib = [1, 1]
    while len(fib) < 24:
        fib.append(fib[-1] + fib[-2])
    qf = rng.permutation(np.frombuffer(b"".join(bytes([40 + i]) * c for i, c in enumerate(fib)), dtype=np.uint8)).tobytes()
    seqs.append(bytes(rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), len(qf))))  # forces the 15-bit length limit
    quals.append(qf)
    import gzip
    for with_q in (True, False):
        batch = synth.pack_reads(seqs, quals if with_q else None)
        params = FilterParams(min_len=100, min_q=0.0, qtype=33 if with_q else 0, adapters=[], max_read_len=200000, gz_blocks=True)
        with FilterEngine(params) as eng:
            eng.submit(batch)
            blob, spans = eng.collect_gz()
            reads, pieces = eng.collect()
        members, texts = _gz_members(batch, pieces, blob, spans, fastq=with_q)
        assert len(members) == 5
        for m, t in zip(members, texts):
            assert gzip.decompress(m) == t


@pytest.mark.parametrize("args", [["-x", "hifi", "-g", "200k", "-d", "3"], ["-x", "hifi", "-F", "-r", "60"]])
def test_host_cli_downsampled_gzip_output_equals_plain(args):
    """Downsampling with a .gz output name: per-record members compressed by the -t threads in chunks; the
    decompressed file must equal the plain output."""
    import gzip
    batch = _distinct_length_batch(5, 260)
    fq = batch.to_fastq()
    rc1, plain, err1 = _run_host_cli(args, fq)
    rc2, gz, err2 = _run_host_cli(args, fq, out_name="out.fq.gz")
    assert rc1 == 0 and rc2 == 0, (err1, err2)
    assert len(plain) > 10000 and gzip.decompress(gz) == plain
    assert gz.count(b"\x1f\x8b\x08") >= plain.count(b"\n") // 4


def test_host_cli_multi_threaded_staging_equals_single(monkeypatch):
    """The batch staging (2-bit packing + quality copy into the pinned slot) is split over threads at 32-base
    boundaries; exception bytes (N, lower case) near the cuts must land at the right absolute positions."""
    rng = np.random.default_rng(21)
    batch = synth.make_config(2, 300, max_len=30000)
    fq = bytearray(batch.to_fastq())
    # sprinkle N / lower-case bases over the sequence lines
    lines = bytes(fq).split(b"\n")
    for i in range(1, len(lines), 4):
        ln = bytearray(lines[i])
        for p in rng.integers(0, len(ln), max(1, len(ln) // 40)):
            ln[int(p)] = b"Nacgtn"[int(rng.integers(0, 6))]
        lines[i] = bytes(ln)
    fq = b"\n".join(lines)
    monkeypatch.setenv("TGSF_STAGE_THREADS", "1")
    rc1, out1, err1 = _run_host_cli(["-x", "ont"], fq)
    monkeypatch.setenv("TGSF_STAGE_THREADS", "7")
    monkeypatch.setenv("TGSF_STAGE_MIN_SHIFT", "12")
    rc2, out2, err2 = _run_host_cli(["-x", "ont"], fq)
    assert rc1 == 0 and rc2 == 0, (err1, err2)
    assert out1 == out2 and len(out1) > 100000
    assert _info(err1) == _info(err2)


def test_host_cli_parallel_single_stream_gzip_input(monkeypatch):
    """A one-member .fastq.gz goes through src/pinflate.hpp (spans decoded in parallel against an unknown
    window, chain-validated): records and INFO lines must equal those of the plain input and of the
    sequential decoder (TGSF_SERIAL_INFLATE=1)."""
    import gzip
    batch = synth.make_config(2, 300, max_len=30000)
    fq = batch.to_fastq()
    gz = gzip.compress(fq, 6)
    assert len(gz) > 1_000_000
    rc0, out0, err0 = _run_host_cli(["-x", "ont"], fq)
    monkeypatch.setenv("TGSF_PINFLATE_MIN_BYTES", "100000")
    monkeypatch.setenv("TGSF_INFLATE_THREADS", "6")
    rc1, out1, err1 = _run_host_cli(["-x", "ont"], gz, in_name="in.fq.gz")
    monkeypatch.setenv("TGSF_SERIAL_INFLATE", "1")
    rc2, out2, err2 = _run_host_cli(["-x", "ont"], gz, in_name="in.fq.gz")
    assert rc0 == 0 and rc1 == 0 and rc2 == 0, (err0, err1, err2)
    assert out1 == out0 and out2 == out0 and len(out0) > 100000
    assert _info(err1) == _info(err0) and _info(err2) == _info(err0)


def test_host_cli_bam_and_sam_input(monkeypatch):
    """BAM / SAM input (read_bam, T.cpp:984-1040 pre-pass sampling and 1872-1916 main pass): the CLI parses the
    records itself (src/pipeline.hpp, BGZF blocks in parallel) and must write the records and INFO lines it writes
    for the equivalent FASTQ; the reference CLI (htslib) on the same BAM must agree where it is available."""
    import bam_lib
    import ref_lib
    fq = synth.make_config(2, 200, max_len=30000, with_names=False).to_fastq()
    bam, sam = bam_lib.from_fastq(fq)
    rc0, out0, err0 = _run_host_cli(["-x", "ont"], fq)
    rc1, out1, err1 = _run_host_cli(["-x", "ont"], bam, in_name="in.bam")
    rc2, out2, err2 = _run_host_cli(["-x", "ont"], sam, in_name="in.sam")
    monkeypatch.setenv("TGSF_BATCH_MB", "1")
    rc3, out3, err3 = _run_host_cli(["-x", "ont"], bam, in_name="in.bam")
    assert rc0 == 0 and rc1 == 0 and rc2 == 0 and rc3 == 0, (err0, err1, err2, err3)
    assert len(out0) > 100000 and out1 == out0 and out2 == out0 and out3 == out0
    assert _info(err1) == _info(err0) and _info(err2) == _info(err0) and _info(err3) == _info(err0)
    if ref_lib.available():
        r_rc, r_out, r_err, _ = ref_lib.run_cli(["-x", "ont", "-t", "1"], bam, in_name="in.bam")
        assert r_rc == 0 and r_out == out1 and _info(r_err) == _info(err1)


@pytest.mark.parametrize("kind", ["plain", "gz", "bam"])
def test_host_cli_adapter_identification_only(kind):
    """-A: adapter identification only (T.cpp:3071-3098).  The run ends right after the pre-pass; with streamed
    input (.gz, BAM) the ingest thread is still alive at that point and must not abort the process (exit 0, same
    INFO lines as the reference)."""
    import gzip
    import bam_lib
    import ref_lib
    fq = synth.make_config(2, 300, max_len=40000, with_names=False).to_fastq()
    data, name = fq, "in.fq"
    if kind == "gz":
        data, name = gzip.compress(fq, 1), "in.fq.gz"
    elif kind == "bam":
        data, name = bam_lib.from_fastq(fq)[0], "in.bam"
    rc, out, err = _run_host_cli(["-x", "ont", "-A"], data, in_name=name, out_name=None)
    assert rc == 0, (rc, err[-500:])
    assert any(l.startswith("INFO: 5' adapter:") for l in err.splitlines())
    if ref_lib.available():
        r_rc, _, r_err, _ = ref_lib.run_cli(["-x", "ont", "-A", "-t", "1"], data, in_name=name, out_name=None)
        assert r_rc == 0 and _info(err) == _info(r_err)


def _long_pairs(rng, n, q_lo, q_hi):
    a = np.frombuffer(b"ACGT", dtype=np.uint8)
    pairs = []
    for i in range(n):
        ql = int(rng.integers(q_lo, q_hi + 1))
        alpha = a if i % 4 else a[:2]
        q = alpha[rng.integers(0, len(alpha), ql)].tobytes()
        mode = i % 3
        if mode == 0:
            t = alpha[rng.integers(0, len(alpha), int(rng.integers(1, 2 * ql)))].tobytes()
        elif mode == 1:
            t = (alpha[rng.integers(0, len(alpha), int(rng.integers(0, 300)))].tobytes()
                 + synth.mutate(q, float(rng.random() * 0.25), rng)
                 + alpha[rng.integers(0, len(alpha), int(rng.integers(0, 300)))].tobytes()) or b"A"
        else:
            t = (q[:max(1, ql // 4)] * 9)[:int(rng.integers(1, 2 * ql))]
        k = [-1, ql, max(0, ql - 3), int(ql * 0.1) + 1, int(ql * 0.3), int(rng.integers(0, ql + 1))][i % 6]
        pairs.append((q, t, k))
    return pairs


def test_align_long_queries_vs_oracle_and_edlib():
    """Adapters longer than 256 bp (5..32 Myers words; the library runs them with 8, 16 or 32 words): tgsf_align_hw
    against the oracle's plain DP and, where the reference build is present, against the real edlibAlign
    (E.cpp:141-296 has no length limit) for queries up to 2 000 bp."""
    import ref_lib
    rng = np.random.default_rng(77)
    pairs = (_long_pairs(rng, 120, 257, 512) + _long_pairs(rng, 90, 513, 1024) + _long_pairs(rng, 60, 1025, 2000)
             + _long_pairs(rng, 12, 2040, 2048))
    out = align_hw(pairs)
    for p, r in zip(pairs, out):
        o, _ = oracle_lib.align_hw(*p)
        for f in ("edit_distance", "n_locations", "align_len", "first_start", "first_end",
                  "last_start", "last_end", "loc_hash"):
            assert int(r[f]) == (o[f] & 0xffffffff if f == "loc_hash" else o[f]), (f, len(p[0]), len(p[1]), p[2])
    if ref_lib.available():
        ref = ref_lib.edlib_batch(pairs)
        for p, r, (d, alen, locs) in zip(pairs, out, ref):
            assert int(r["edit_distance"]) == d and int(r["n_locations"]) == len(locs) and int(r["align_len"]) == alen, \
                (len(p[0]), len(p[1]), p[2])
            if locs:
                assert (int(r["first_start"]), int(r["first_end"])) == locs[0]
                assert (int(r["last_start"]), int(r["last_end"])) == locs[-1]


def test_align_hirschberg_sized_alignments_vs_oracle_and_edlib():
    """edlib leaves the traceback for Hirschberg's divide and conquer when the matrix of the located alignment would
    reach 1 MiB (E.cpp:1194-1215: adapters above ~1 250 bp with long, heavily mismatched hits); the split picks other
    optimal paths in ties, so the alignment LENGTH depends on it.  Library and oracle reproduce the split rule."""
    import ref_lib
    rng = np.random.default_rng(2024)
    a = np.frombuffer(b"ACGT", dtype=np.uint8)
    pairs = []
    for i in range(150):
        ql = int(rng.integers(1300, 2049))
        alpha = a if i % 3 else a[:2]
        q = alpha[rng.integers(0, len(alpha), ql)].tobytes()
        if i % 5 == 4:
            q = (q[:int(rng.integers(3, 40))] * 3000)[:ql]  # periodic query: masses of ties
        m = synth.mutate(q, float(rng.random() * 0.35), rng)
        t = (alpha[rng.integers(0, len(alpha), int(rng.integers(0, 200)))].tobytes() + m
             + alpha[rng.integers(0, len(alpha), int(rng.integers(0, 200)))].tobytes())
        pairs.append((q, t, [-1, ql, int(ql * 0.5)][i % 3]))
    out = align_hw(pairs)
    ref = ref_lib.edlib_batch(pairs) if ref_lib.available() else None
    big = 0
    for n, (p, r) in enumerate(zip(pairs, out)):
        o, _ = oracle_lib.align_hw(*p)
        for f in ("edit_distance", "n_locations", "align_len", "first_start", "first_end", "last_start", "last_end"):
            assert int(r[f]) == o[f], (f, len(p[0]), len(p[1]), p[2])
        tl = int(r["first_end"]) - int(r["first_start"]) + 1
        big += (20 * ((len(p[0]) + 63) // 64) + 8) * tl >= 1 << 20
        if ref is not None:
            d, alen, locs = ref[n]
            assert (o["edit_distance"], o["align_len"], o["n_locations"]) == (d, alen, len(locs)), (len(p[0]), len(p[1]), p[2])
    assert big >= 30  # the split really was exercised


def _long_adapter_batch(adapters, n=160, seed=5):
    """Reads with (mutated) copies of long adapters at the 5' end, the 3' end and in the middle."""
    rng = np.random.default_rng(seed)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    seqs = []
    for i in range(n):
        ad = adapters[i % len(adapters)]
        m = synth.mutate(ad, [0.0, 0.03, 0.08][i % 3], rng)
        lo = max(3000, 4 * len(m) + 1500)
        L = int(rng.integers(lo, lo + 5000))
        s = bytearray(acgt[rng.integers(0, 4, L)].tobytes())
        where = i % 5
        if where == 0:
            s[:len(m)] = m
        elif where == 1:
            s[L - len(m):] = m
        elif where == 2:
            p = int(rng.integers(len(m) + 500, L - 2 * len(m) - 500))
            s[p:p + len(m)] = m
        elif where == 3:
            s[10:10 + len(m)] = m
            p = int(rng.integers(len(m) + 800, L - 2 * len(m) - 500))
            s[p:p + len(m)] = params_rev(m)
        seqs.append(bytes(s[:L]))
    quals = [bytes([30 + 33]) * len(s) for s in seqs]
    return synth.pack_reads(seqs, quals, [b"r%d" % i for i in range(n)])


def params_rev(b: bytes) -> bytes:
    from tgsfilter_b200.params import rev_comp
    return rev_comp(bytes(b))


def test_long_adapters_per_read_vs_oracle():
    """-a adapters of 300, 600 and 1 500 bp (8, 16 and 32 words) through the whole per-read path."""
    rng = np.random.default_rng(9)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    ads = [acgt[rng.integers(0, 4, n)].tobytes() for n in (300, 600, 1500)]
    adapters = []
    for a in ads:
        adapters += [a, params_rev(a)]
    batch = _long_adapter_batch(ads, n=60)
    params = FilterParams(min_len=500, min_q=0.0, qtype=33, adapters=adapters).apply_read_type("ont")
    r, p, _ = _compare(params, batch)
    assert (r["n_5p"] > 0).any() and (r["n_3p"] > 0).any() and (r["n_mid"] > 0).any()


def test_many_adapters_per_read_vs_oracle():
    """More than 64 adapters in the set (the round-1 cap)."""
    rng = np.random.default_rng(10)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    ads = [acgt[rng.integers(0, 4, int(rng.integers(24, 70)))].tobytes() for _ in range(90)]
    batch = _long_adapter_batch(ads, n=120, seed=6)
    params = FilterParams(min_len=500, min_q=0.0, qtype=33, adapters=ads).apply_read_type("ont")
    _compare(params, batch)


def test_host_cli_long_adapter_file_vs_reference_cli(tmp_path, request):
    """-a with a 600-bp adapter (T.cpp:1218-1322 takes any adapter file; edlib has no length cap)."""
    import ref_lib
    rng = np.random.default_rng(12)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    ad = acgt[rng.integers(0, 4, 600)].tobytes()
    batch = _long_adapter_batch([ad], n=200, seed=8)
    fa = tmp_path / "adapters.fa"
    fa.write_bytes(b">long\n" + ad + b"\n")
    args = ["-x", "ont", "-a", str(fa)]
    fq = batch.to_fastq()
    h_rc, h_out, h_err = _run_host_cli(args, fq)
    assert h_rc == 0, h_err
    assert len(h_out) > 0

    def reference():
        r_rc, r_out, r_err, _ = ref_lib.run_cli(args + ["-t", "1"], fq)
        assert r_rc == 0, r_err
        return {"out": r_out, "info": _info(r_err)}
    _expect_reference(request, {"out": h_out, "info": _info(h_err)}, reference)


@pytest.mark.parametrize("args", [
    ["-x", "hifi", "-g", "100k", "-d", "8", "-k", "11", "-p", "40", "-5", "0", "-3", "0"],
    ["-x", "hifi", "-R", "0.3", "-5", "3", "-3", "2"],
    ["-x", "hifi", "-r", "41"],
    ["-F", "-R", "0.4"],
])
def test_host_cli_downsampling_in_memory_spill_and_selection_forms(args, monkeypatch, tmp_path):
    """Filter + downsample keeps the filtered records in host memory: no `<input>.tmp.<pid>` file appears next to
    the input while the run is going (the reference writes one, T.cpp:3129-3137).  Forcing the spill to the tmp file
    (buffer of 0 MB / of 1 MB, exceeded after the first batches) and the sort-based selection (the reference's form)
    must give the same records and INFO lines as the default (in memory, histogram cut-off)."""
    import os
    import subprocess
    import threading
    import time
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "src", "tgsfilter")
    batch = synth.make_config(5, 700, max_len=30000)  # ordinary lengths: many ties, also at the cut-off
    fq = tmp_path / "in.fq"
    fq.write_bytes(batch.to_fastq())
    monkeypatch.setenv("TGSF_BATCH_MB", "2")

    def run(env_extra, out_name):
        env = dict(os.environ)
        env.update(env_extra)
        seen = []
        stop = threading.Event()

        def watch():
            while not stop.is_set():
                seen.extend(f for f in os.listdir(tmp_path) if ".tmp." in f)
                time.sleep(0.002)
        th = threading.Thread(target=watch)
        th.start()
        pr = subprocess.run([exe, "-i", str(fq), "-o", str(tmp_path / out_name)] + args, stdout=subprocess.PIPE,
                            stderr=subprocess.PIPE, env=env, timeout=600)
        stop.set()
        th.join()
        assert pr.returncode == 0, pr.stderr.decode()[-800:]
        assert not [f for f in os.listdir(tmp_path) if ".tmp." in f]  # removed at the end in every mode
        return (tmp_path / out_name).read_bytes(), _info(pr.stderr.decode()), bool(seen)

    out0, info0, tmp0 = run({}, "a.fq")
    out1, info1, tmp1 = run({"TGSF_DOWNSAMPLE_BUFFER_MB": "0"}, "b.fq")
    out2, info2, _ = run({"TGSF_DOWNSAMPLE_BUFFER_MB": "1"}, "c.fq")
    out3, info3, _ = run({"TGSF_SELECT_SORT": "1"}, "d.fq")
    assert len(out0) > 0 and out1 == out0 and out2 == out0 and out3 == out0
    assert info1 == info0 and info2 == info0 and info3 == info0
    if "-F" not in args:
        assert not tmp0, "the default run wrote a tmp file"


def test_counter_block_grows_with_the_longest_read():
    """A context created for short reads (max_read_len 3 000) meets longer and longer reads batch after batch: the
    per-100 bp tables move to a larger layout before the batch is launched (the reference sizes them per read,
    T.cpp:1445), nothing accumulated so far is lost, and a read beyond the old limit is no longer an error."""
    from tgsfilter_b200.engine import Counters
    full = synth.make_config(2, 240, max_len=60000)
    lens = np.diff(full.offsets.astype(np.int64))
    order = np.argsort(lens, kind="stable")  # ascending: every batch brings longer reads than the one before
    seqs = [full.read(int(i))[0].tobytes() for i in order]
    quals = [full.read(int(i))[1].tobytes() for i in order]
    batches = [synth.pack_reads(seqs[a:a + 60], quals[a:a + 60]) for a in range(0, 240, 60)]
    params = synth.config_params(2)
    params.max_read_len = 3000
    with FilterEngine(params) as eng:
        for b in batches:
            eng.run(b)
        g = eng.counters()
    assert g.layout.max_bins > 3000 // 100 + 1
    big = synth.config_params(2)
    big.max_read_len = 100000
    o_cnt = None
    for b in batches:
        _, _, o_cnt = oracle_lib.run(big, b, o_cnt)
    o = Counters(o_cnt, oracle_lib.layout(big))
    assert np.array_equal(g.drop_info, o.drop_info)
    assert np.array_equal(g.raw_hist, o.raw_hist) and np.array_equal(g.clean_hist, o.clean_hist)
    for name in Counters.TABLES_BC:
        assert np.array_equal(getattr(g, name), getattr(o, name)), name
    for name in Counters.TABLES_BIN:
        a, b = getattr(g, name), getattr(o, name)
        m = min(len(a), len(b))
        assert np.array_equal(a[:m], b[:m]) and not a[m:].any() and not b[m:].any(), name


@pytest.mark.parametrize("args", [["-F", "-R", "0.35"], ["-F", "-g", "60k", "-d", "4"], ["-x", "hifi", "-R", "0.5", "-5", "0", "-3", "0"]])
def test_host_cli_downsampling_with_repeated_read_names(args, request):
    """Input with repeated read names: DownSampleTask keys the lengths by NAME (the last record of a name wins,
    T.cpp:2267) and keeps every record whose name was selected; with -F the fraction target counts EVERY record
    (get_fastx_SeqLen adds all of them to totalSize, T.cpp:2262), in filter mode only the ranked names (T.cpp:2318-2322)."""
    import ref_lib
    base = _distinct_length_batch(5, 180, seed=3)
    seqs, quals, names = [], [], []
    for i in range(base.n_reads):
        b, q = base.read(i)
        seqs.append(b.tobytes())
        quals.append(q.tobytes())
        names.append(base.name(i // 3 * 3) if i % 3 == 2 else base.name(i))  # every third record repeats an earlier name
    fq = synth.pack_reads(seqs, quals, names).to_fastq()
    h_rc, h_out, h_err = _run_host_cli(args, fq)
    assert h_rc == 0, h_err
    assert len(h_out) > 0

    def reference():
        r_rc, r_out, r_err, _ = ref_lib.run_cli(args + ["-t", "1"], fq)
        assert r_rc == 0, r_err
        return {"out": r_out, "info": _info(r_err)}
    _expect_reference(request, {"out": h_out, "info": _info(h_err)}, reference)


def test_host_cli_cram_input():
    """CRAM content (in a file named .bam, the only way it reaches the reference: GetFileType knows sam / bam only while
    hts_open sniffs the content, T.cpp:839-857, 984-1040).  The CLI decodes it through htslib when the build was
    pointed at one (src/Makefile HTS_DIR) and must write what it writes for the same reads as FASTQ, and what the
    reference CLI writes for the same file.  Fixture: tests/golden/reads_cram.bam (tests/golden/make_cram.py)."""
    import ref_lib
    with open(golden_lib.HERE + "/reads_cram.bam", "rb") as f:
        cram = f.read()
    assert cram[:4] == b"CRAM"
    fq = synth.make_config(2, 48, max_len=9000, with_names=False).to_fastq()
    rc1, out1, err1 = _run_host_cli(["-x", "ont"], cram, in_name="in.bam")
    if "needs a build with htslib" in err1:
        # a build without htslib must refuse CRAM with an error, not finish with an empty output
        assert rc1 != 0 and out1 == b"", (rc1, len(out1))
        pytest.skip("src/tgsfilter was built without htslib")
    rc0, out0, err0 = _run_host_cli(["-x", "ont"], fq)
    assert rc0 == 0 and rc1 == 0, (err0, err1)
    assert len(out0) > 10000 and out1 == out0
    assert _info(err1) == _info(err0)
    if ref_lib.available():
        r_rc, r_out, r_err, _ = ref_lib.run_cli(["-x", "ont", "-t", "1"], cram, in_name="in.bam")
        assert r_rc == 0 and r_out == out1 and _info(r_err) == _info(err1)

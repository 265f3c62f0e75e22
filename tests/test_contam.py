"""Contaminant screen (tgsf_set_contaminants / --contam): the oracle against a plain Python restatement, the
defaults on synthetic ONT data, the CLI's argument checks, and on the GPU field-by-field parity with
tgsfo_run_contam (tests/contam_oracle.c)."""
from __future__ import annotations

import gzip
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

import contam_oracle
import oracle_lib
from tgsfilter_b200 import _capi, records, synth
from tgsfilter_b200.params import ADAPTER_LIB, FilterParams, rev_comp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "src", "tgsfilter")
LAMBDA_LEN = 48_502
_CODE = {ord(c): i for i, c in enumerate("ACGT")} | {ord(c): i for i, c in enumerate("acgt")}


# ---- plain restatement -----------------------------------------------------------------------------
def _canon(seq: bytes, i: int, k: int):
    fwd = rev = 0
    for j in range(k):
        c = _CODE.get(seq[i + j])
        if c is None:
            return None
        fwd = (fwd << 2) | c
        rev |= (3 - c) << (2 * j)
    return min(fwd, rev)


def _keys(seqs, k):
    return {x for s in seqs for i in range(len(s) - k + 1) if (x := _canon(s, i, k)) is not None}


def _hits(seq: bytes, k: int, keys) -> int:
    return sum(1 for i in range(len(seq) - k + 1) if _canon(seq, i, k) in keys)


def _is_contam(hits: int, length: int, k: int, min_frac: float) -> bool:
    windows = length - k + 1
    ppm = int(np.round(np.float64(np.float32(min_frac)) * 1e6))
    return windows >= 1 and hits * 1_000_000 >= ppm * windows


def _noisy(rng, n, alphabet=b"ACGTacgtNRYn"):
    return bytes(rng.choice(np.frombuffer(alphabet, dtype=np.uint8), n))


def _plain_params(**kw) -> FilterParams:
    p = FilterParams(min_q=-1.0, head_trim=0, tail_trim=0, min_len=1, filter=False, **kw)
    return p.apply_read_type("ont")


@pytest.mark.parametrize("k", [11, 17, 21, 31])
def test_oracle_matches_restatement(k):
    """Hit counts, statuses and the distinct-key count of the oracle equal a plain Python restatement, on sets
    and pieces with lowercase, N and IUPAC bytes and pieces shorter than k."""
    rng = np.random.default_rng(1000 + k)
    genome = synth.make_contaminant(3000, seed=k)
    cset = [genome[:1200].lower(), _noisy(rng, 400), genome[1200:], b"ACG", b""]
    reads = []
    for i in range(40):
        kind = i % 4
        if kind == 0:  # from the set, both strands, some bytes disturbed
            s = int(rng.integers(0, 2000))
            r = bytearray(genome[s:s + int(rng.integers(k, 900))])
            if i % 8 == 0:
                r = bytearray(rev_comp(bytes(r)))
            for j in rng.integers(0, len(r), 3):
                r[j] = b"NnRa"[int(rng.integers(0, 4))]
            reads.append(bytes(r))
        elif kind == 1:
            reads.append(_noisy(rng, int(rng.integers(1, 600))))
        elif kind == 2:
            reads.append(_noisy(rng, int(rng.integers(1, k))))  # shorter than k
        else:
            reads.append(genome[:700] + _noisy(rng, 700))
    batch = synth.pack_reads(reads, [b"I" * len(r) for r in reads])
    keys = _keys(cset, k)
    assert contam_oracle.contam_kmers(cset, k) == len(keys)
    for frac in (0.05, 0.5, 1.0):
        _, pieces, cnt = contam_oracle.run(_plain_params(), batch, (cset, k, frac))
        _, pieces0, cnt0 = oracle_lib.run(_plain_params(), batch)
        assert len(pieces) == len(reads)
        for p, r in zip(pieces, reads):
            h = _hits(r, k, keys)
            assert int(p["contam_hits"]) == h
            assert (int(p["status"]) == _capi.PIECE_CONTAM) == _is_contam(h, len(r), k, frac)
        assert (pieces0["contam_hits"] == 0).all() and (pieces0["status"] == _capi.PIECE_EMIT).all()


def test_oracle_threshold_boundary():
    """hits * 10^6 >= ppm * windows, exactly at and one hit below the boundary."""
    k = 17
    genome = synth.make_contaminant(5000, seed=7)
    windows = 1000
    cases = []
    for frac in (0.05, 0.25, 0.5):
        need = -(-int(round(frac * 1e6)) * windows // 1_000_000)  # smallest hit count that is a contaminant
        for h in (need, need - 1):
            # h hits = a set segment of h + k - 1 bases, then bases that match nothing (poly-N)
            seq = genome[:h + k - 1] + b"N" * (windows - h) if h > 0 else b"N" * (windows + k - 1)
            cases.append((frac, h, seq))
    for frac, h, seq in cases:
        batch = synth.pack_reads([seq], [b"I" * len(seq)])
        _, pieces, _ = contam_oracle.run(_plain_params(), batch, ([genome], k, frac))
        assert int(pieces[0]["contam_hits"]) == h
        assert (int(pieces[0]["status"]) == _capi.PIECE_CONTAM) == _is_contam(h, len(seq), k, frac)


def test_oracle_contaminants_never_reach_the_clean_step():
    """Every read drawn from the set: all pieces the repeat check kept (emitted or low quality without the set)
    become contaminants, the clean-side counters and DropInfo[13/14] are zero, everything else is unchanged."""
    genome = synth.make_contaminant(LAMBDA_LEN)
    rng = np.random.default_rng(3)
    base = synth.make_config(2, 120)
    seqs = [synth.contaminant_read(genome, int(base.offsets[i + 1] - base.offsets[i]), 0.0, rng).tobytes()
            for i in range(base.n_reads)]
    batch = synth.ReadBatch(np.frombuffer(b"".join(seqs), dtype=np.uint8).copy(), base.quals, base.offsets, base.names)
    for fasta in (False, True):
        b = batch if not fasta else synth.ReadBatch(batch.bases, None, batch.offsets, batch.names)
        params = synth.config_params(2)
        reads0, pieces0, cnt0 = oracle_lib.run(params, b)
        reads, pieces, cnt = contam_oracle.run(params, b, ([genome], 17, 0.05))
        assert np.array_equal(reads, reads0)
        kept = np.isin(pieces0["status"], [_capi.PIECE_EMIT, _capi.PIECE_LOWQ])
        assert kept.sum() > 20 and (pieces["status"][kept] == _capi.PIECE_CONTAM).all()
        assert np.array_equal(pieces["status"][~kept], pieces0["status"][~kept])
        L = oracle_lib.layout(params)
        clean = [(L.clean_hist, 256)] + [(getattr(L, t), L.bc_len * 5) for t in
                                         ("clean5p_cnt", "clean5p_qual", "clean3p_cnt", "clean3p_qual")] + \
                [(getattr(L, t), L.max_bins * 5) for t in ("clean_bin_cnt", "clean_bin_qual")] + \
                [(L.drop_info + 13, 2)]
        mask = np.ones(L.n_u64, dtype=bool)
        for off, n in clean:
            assert (cnt[off:off + n] == 0).all()
            mask[off:off + n] = False
        assert np.array_equal(cnt[mask], cnt0[mask])


def test_oracle_rejects_bad_set():
    batch = synth.pack_reads([b"ACGT" * 10], [b"I" * 40])
    for args in (([b"ACGT" * 10], 10, 0.05), ([b"ACGT" * 10], 32, 0.05), ([b"ACGT" * 10], 17, 0.0),
                 ([b"ACGT" * 10], 17, 1.5), ([b"NNNN" * 10], 17, 0.05)):
        with pytest.raises(AssertionError):
            contam_oracle.run(_plain_params(), batch, args)


def _ont_batch(n, err, genome, seed):
    batch = synth.make_config(2, n)
    return synth.mix_contaminants(batch, genome, 0.05, err, chimeras=0.05, chimera_err=0.04, seed=seed)


@pytest.mark.parametrize("err", [0.04, 0.10])
def test_oracle_defaults_drop_planted_reads(err):
    """Default k = 17, min_frac = 0.05 on synthetic ONT reads: >= 99 % of the reads drawn from a 48.5 kb set
    (5 %, both strands) and of the chimeras (>= 30 % contaminant at 4 % error) are dropped, no other read is."""
    genome = synth.make_contaminant(LAMBDA_LEN)
    batch, planted, chim = _ont_batch(800, err, genome, seed=int(err * 1000))
    params = synth.config_params(2)
    reads, pieces, _ = contam_oracle.run(params, batch, ([genome], 17, 0.05))
    contam_reads = set(pieces["read"][pieces["status"] == _capi.PIECE_CONTAM].tolist())
    emit_reads = set(pieces["read"][pieces["status"] == _capi.PIECE_EMIT].tolist())
    screened = set(pieces["read"].tolist())  # reads that reached the piece loop
    target = [int(r) for r in np.concatenate([planted, chim]) if int(r) in screened]
    assert len(target) > 50
    dropped = [r for r in target if r in contam_reads and r not in emit_reads]
    assert len(dropped) >= 0.99 * len(target)
    others = screened - set(int(r) for r in np.concatenate([planted, chim]))
    assert not (others & contam_reads)


@pytest.mark.parametrize("args,msg", [
    (["--contam", "/nonexistent/contam.fa"], "--contam"),
    (["--contam", "{fa}", "--contam-k", "10"], "--contam-k"),
    (["--contam", "{fa}", "--contam-k", "32"], "--contam-k"),
    (["--contam", "{fa}", "--contam-frac", "0"], "--contam-frac"),
    (["--contam", "{fa}", "--contam-frac", "1.5"], "--contam-frac"),
    (["--contam", "{fa}", "--qc"], "--qc"),
])
def test_cli_rejects_bad_contam_options(tmp_path, args, msg):
    """These fail in argument parsing, before any device call (so also without a GPU)."""
    if not os.path.exists(EXE):
        pytest.skip("src/tgsfilter not built")
    fa = tmp_path / "c.fa"
    fa.write_bytes(b">c\nACGTACGTACGTACGTACGT\n")
    fq = tmp_path / "r.fq"
    fq.write_bytes(b"@r\n" + b"ACGT" * 300 + b"\n+\n" + b"I" * 1200 + b"\n")
    cmd = [EXE, "-i", str(fq), "-x", "ont", "-o", str(tmp_path / "o.fq")] + [a.format(fa=fa) for a in args]
    pr = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=60)
    assert pr.returncode != 0
    assert msg in pr.stderr.decode()
    assert not (tmp_path / "o.fq").exists()


# ---- GPU -------------------------------------------------------------------------------------------
def _sets():
    small = synth.make_contaminant(LAMBDA_LEN)
    large = synth.make_contaminant(5_000_000, seed=synth.SEED0 + 102)
    # soft-masked and N-interrupted records: the screen must treat them like the oracle does
    small_set = [small[:20000].lower(), small[20000:30000] + b"NNNNNRY" + small[30000:]]
    return {"small": (small, small_set), "large": (large, [large])}


_SETS = None


def _set(name):
    global _SETS
    if _SETS is None:
        _SETS = _sets()
    return _SETS[name]


def _case_batch(cfg, n, genome, fasta=False):
    batch = synth.make_config(cfg, n, max_len=200_000)
    batch, planted, chim = synth.mix_contaminants(batch, genome, 0.08, 0.04, chimeras=0.05, seed=cfg)
    b = batch.bases.copy()
    b[5::9973] = ord("n")  # lowercase / N bytes inside reads
    b[7::7919] = ord("a")
    batch = synth.ReadBatch(b, None if fasta else batch.quals, batch.offsets, batch.names)
    return batch, planted


def _run_gpu(params, batch, cset, k, frac, path):
    from tgsfilter_b200.engine import FilterEngine
    with FilterEngine(params) as eng:
        n_kmers = eng.set_contaminants(cset, k=k, min_frac=frac)
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
        cnt = eng.counters().flat
    return n_kmers, reads, pieces, cnt


GPU_CASES = [
    # cfg, n, k, set, path, fasta, extra params
    (1, 200, 17, "small", "submit", False, {}),
    (2, 300, 17, "small", "packed", False, {}),
    (3, 60, 11, "large", "device", False, {}),
    (4, 300, 31, "small", "submit", False, {}),
    (5, 150, 11, "small", "packed", False, {"min_repeat": 20}),  # config 5, -k 11 -p 20
    (2, 300, 17, "large", "submit", False, {"discard": True}),  # -D
    (1, 200, 17, "small", "device", True, {}),  # FASTA input
    (3, 60, 31, "large", "packed", False, {"kmer": 13, "min_repeat": 10}),
    (4, 200, 11, "small", "device", False, {"kmer": 12, "min_repeat": 3}),
]


@pytest.mark.gpu
@pytest.mark.parametrize("cfg,n,k,set_name,path,fasta,extra", GPU_CASES)
def test_gpu_contam_parity(cfg, n, k, set_name, path, fasta, extra):
    genome, cset = _set(set_name)
    batch, planted = _case_batch(cfg, n, genome, fasta)
    params = synth.config_params(cfg)
    for key, v in extra.items():
        setattr(params, key, v)
    n_kmers, reads, pieces, cnt = _run_gpu(params, batch, cset, k, 0.05, path)
    o_reads, o_pieces, o_cnt = contam_oracle.run(params, batch, (cset, k, 0.05))
    assert n_kmers == contam_oracle.contam_kmers(cset, k)
    assert np.array_equal(reads, o_reads)
    for f in o_pieces.dtype.names:
        assert np.array_equal(pieces[f], o_pieces[f]), f
    assert np.array_equal(cnt, o_cnt)
    assert (pieces["status"] == _capi.PIECE_CONTAM).sum() > 0
    assert (pieces["contam_hits"] > 0).sum() >= (pieces["status"] == _capi.PIECE_CONTAM).sum()


@pytest.mark.gpu
@pytest.mark.parametrize("set_name", ["small", "large"])
def test_gpu_contam_long_pieces(set_name):
    """Pieces of >= 500 kb: one drawn from the set, one ordinary, one half-and-half."""
    genome, cset = _set(set_name)
    rng = np.random.default_rng(5)
    a = synth.contaminant_read(genome, 600_000, 0.04, rng).tobytes()
    b = synth.make_contaminant(550_000, seed=55)
    c = synth.contaminant_read(genome, 260_000, 0.10, rng).tobytes() + synth.make_contaminant(260_000, seed=56)
    seqs = [a, b, c]
    batch = synth.pack_reads(seqs, [b"5" * len(s) for s in seqs], [b"a", b"b", b"c"])
    params = _plain_params(max_read_len=1 << 20)
    _, reads, pieces, cnt = _run_gpu(params, batch, cset, 17, 0.05, "submit")
    o_reads, o_pieces, o_cnt = contam_oracle.run(params, batch, (cset, 17, 0.05))
    assert np.array_equal(reads, o_reads) and np.array_equal(pieces, o_pieces) and np.array_equal(cnt, o_cnt)
    assert pieces["len"].max() >= 500_000
    assert list(pieces["status"]) == [_capi.PIECE_CONTAM, _capi.PIECE_EMIT, _capi.PIECE_CONTAM]


@pytest.mark.gpu
def test_gpu_unrelated_set_changes_nothing():
    """A set unrelated to the reads: emitted pieces, per-read results and the counter block equal a context
    without a set."""
    from tgsfilter_b200.engine import FilterEngine
    batch = synth.make_config(2, 300)
    params = synth.config_params(2)
    with FilterEngine(params) as eng:
        r0, p0 = eng.run(batch)
        c0 = eng.counters().flat
    _, r1, p1, c1 = _run_gpu(params, batch, [synth.make_contaminant(LAMBDA_LEN, seed=99)], 17, 0.05, "submit")
    assert np.array_equal(r0, r1) and np.array_equal(c0, c1)
    for f in p0.dtype.names:
        if f != "contam_hits":
            assert np.array_equal(p0[f], p1[f]), f
    assert (p0["contam_hits"] == 0).all()


@pytest.mark.gpu
def test_gpu_set_contaminants_errors():
    from tgsfilter_b200.engine import FilterEngine
    with FilterEngine(synth.config_params(1)) as eng:
        for seqs, k, frac in (([b"ACGT" * 20], 10, 0.05), ([b"ACGT" * 20], 32, 0.05), ([b"ACGT" * 20], 17, 0.0),
                              ([b"ACGT" * 20], 17, 1.01), ([b"N" * 100, b"ACG"], 17, 0.05)):
            with pytest.raises(_capi.TgsfError) as e:
                eng.set_contaminants(seqs, k=k, min_frac=frac)
            assert e.value.code == _capi.TGSF_ERR_INVALID
        assert eng.set_contaminants([b"ACGTTGCA" * 10], k=11) > 0
        eng.submit(synth.make_config(1, 20))
        with pytest.raises(_capi.TgsfError) as e:
            eng.set_contaminants([b"ACGTTGCA" * 10], k=11)
        assert e.value.code == _capi.TGSF_ERR_STATE
        eng.collect()
        # a second call replaces the set
        genome = synth.make_contaminant(LAMBDA_LEN)
        batch, _ = _case_batch(1, 100, genome)
        assert eng.set_contaminants([genome], k=17) == contam_oracle.contam_kmers([genome], 17)
        _, pieces = eng.run(batch)
    _, o_pieces, _ = contam_oracle.run(synth.config_params(1), batch, ([genome], 17, 0.05))
    assert np.array_equal(pieces, o_pieces)


def _gz_members(batch, pieces, blob, spans, fastq):
    out, texts = [], records.format_records(batch, pieces, fastq=fastq)
    emitted = [i for i in range(len(pieces)) if pieces["status"][i] == _capi.PIECE_EMIT]
    for (text, name, _), i in zip(texts, emitted):
        head = (b"@" if fastq else b">") + name + b"\n"
        off, nb = int(spans["offset"][i]), int(spans["bytes"][i])
        out.append(b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\xff" + b"\x00" + struct.pack("<HH", len(head), len(head) ^ 0xFFFF)
                   + head + blob[off:off + nb].tobytes() + struct.pack("<II", zlib.crc32(text), len(text) & 0xFFFFFFFF))
    return out, [t for t, _, _ in texts]


@pytest.mark.gpu
def test_gpu_contam_deflate_blocks():
    from tgsfilter_b200.engine import FilterEngine
    genome, cset = _set("small")
    batch, _ = _case_batch(2, 200, genome)
    params = synth.config_params(2)
    params.gz_blocks = True
    with FilterEngine(params) as eng:
        eng.set_contaminants(cset)
        eng.submit(batch)
        blob, spans = eng.collect_gz()
        _, pieces = eng.collect()
    _, o_pieces, _ = contam_oracle.run(params, batch, (cset, 17, 0.05))
    assert np.array_equal(pieces, o_pieces)
    contam = pieces["status"] == _capi.PIECE_CONTAM
    assert contam.sum() > 0 and (spans["bytes"][contam] == 0).all()
    members, texts = _gz_members(batch, o_pieces, blob, spans, fastq=True)
    assert gzip.decompress(b"".join(members)) == b"".join(texts)


# ---- CLI on the GPU ----------------------------------------------------------------------------------
def _fastq_records(data: bytes):
    lines = data.split(b"\n")
    return sorted(b"\n".join(lines[i:i + 4]) for i in range(0, len(lines) - 3, 4))


def _info(stderr: bytes, needle: str):
    return [ln for ln in stderr.decode().splitlines() if needle in ln]


@pytest.fixture(scope="module")
def cli_inputs(tmp_path_factory):
    d = tmp_path_factory.mktemp("contam_cli")
    genome = synth.make_contaminant(LAMBDA_LEN)
    batch, _, _ = synth.mix_contaminants(synth.make_config(2, 3000), genome, 0.05, 0.04, chimeras=0.03,
                                         chimera_err=0.04)
    fq = d / "reads.fq"
    fq.write_bytes(batch.to_fastq())
    fa = d / "contam.fa.gz"
    body = b"".join(genome[i:i + 60] + b"\n" for i in range(0, 30000, 60))
    body2 = b"".join(genome[i:i + 70].lower() + b"\n" for i in range(30000, len(genome), 70))
    fa.write_bytes(gzip.compress(b">part1 lambda-like\n" + body + b">part2\r\n" + body2))
    ad = d / "ad.fa"
    ad.write_bytes(b">ad\n" + ADAPTER_LIB[8] + b"\n")
    return d, batch, genome, [genome[:30000], genome[30000:]], fq, fa, ad


def _cli(d, fq, args, env=None, out_name="o.fq"):
    out = d / out_name
    pr = subprocess.run([EXE, "-i", str(fq), "-o", str(out), "-x", "ont", "-5", "0", "-3", "0", "-q", "10"] + args,
                        stdout=subprocess.PIPE, stderr=subprocess.PIPE, env={**os.environ, **(env or {})}, timeout=600)
    assert pr.returncode == 0, pr.stderr.decode()[-2000:]
    return (out.read_bytes() if out.exists() else b""), pr.stderr


@pytest.mark.gpu
def test_cli_contam_matches_oracle(cli_inputs):
    d, batch, genome, cset, fq, fa, ad = cli_inputs
    out, err = _cli(d, fq, ["-a", str(ad), "--contam", str(fa)])
    params = FilterParams(min_q=10.0, head_trim=0, tail_trim=0,
                          adapters=[ADAPTER_LIB[8], rev_comp(ADAPTER_LIB[8])]).apply_read_type("ont")
    _, o_pieces, _ = contam_oracle.run(params, batch, (cset, 17, 0.05))
    expect = sorted(t.rstrip(b"\n") for t, _, _ in records.format_records(batch, o_pieces, fastq=True))
    assert _fastq_records(out) == expect
    contam = o_pieces[o_pieces["status"] == _capi.PIECE_CONTAM]
    assert len(contam) > 100
    assert _info(err, "as contaminant") == [
        f"INFO: {len(contam)} reads were discarded with {int(contam['len'].sum())} bases as contaminant."]
    assert _info(err, "-mers loaded from") == [
        f"INFO: {contam_oracle.contam_kmers(cset, 17)} distinct 17-mers loaded from {fa}."]
    # two contexts on one device deal the batches between them: same records, same INFO lines
    out2, err2 = _cli(d, fq, ["-a", str(ad), "--contam", str(fa), "--gpus", "2"],
                      env={"TGSF_SHARE_DEVICES": "1", "TGSF_BATCH_MB": "4"}, out_name="o2.fq")
    assert _fastq_records(out2) == expect
    assert [ln for ln in _info(err2, "INFO:") if "written to" not in ln] == \
        [ln for ln in _info(err, "INFO:") if "written to" not in ln]
    # without --contam the new lines are absent
    _, err0 = _cli(d, fq, ["-a", str(ad)], out_name="o0.fq")
    assert not _info(err0, "contaminant") and not _info(err0, "-mers loaded")


@pytest.mark.gpu
def test_cli_contam_then_downsample(cli_inputs):
    d, _, _, _, fq, fa, ad = cli_inputs
    out, err = _cli(d, fq, ["-a", str(ad), "--contam", str(fa), "-g", "1m", "-d", "5"], out_name="ds.fq")
    assert len(_info(err, "as contaminant")) == 1
    assert out.count(b"\n+\n") > 0

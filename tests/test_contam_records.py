"""Per-record attribution of the contaminant screen (tgsf_set_contaminants_labelled, tgsf_contam_record_stats,
tgsf_contam_classify, --contam-report): the oracle (tests/contam_label_oracle.c) against a plain Python restatement,
the CLI's argument checks, and on the GPU field-by-field parity with the oracle."""
from __future__ import annotations

import os
import subprocess

import numpy as np
import pytest

import contam_label_oracle as clo
import contam_oracle
from tgsfilter_b200 import _capi, records, synth
from tgsfilter_b200.params import ADAPTER_LIB, FilterParams, rev_comp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "src", "tgsfilter")
LAMBDA_LEN = 48_502
_CODE = {ord(c): i for i, c in enumerate("ACGT")} | {ord(c): i for i, c in enumerate("acgt")}
SHARED = -2


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


def _labels(cset, k):
    lab = {}
    for r, s in enumerate(cset):
        for i in range(len(s) - k + 1):
            x = _canon(s, i, k)
            if x is not None:
                lab[x] = r if lab.get(x, r) == r else SHARED
    return lab


def _record_kmers(cset, lab):
    rk = np.zeros(len(cset) + 1, dtype=np.uint64)
    for v in lab.values():
        rk[len(cset) if v == SHARED else v] += 1
    return rk


def _attribute(seq: bytes, k: int, lab, n_rec: int):
    hits, votes = 0, {}
    for i in range(len(seq) - k + 1):
        v = lab.get(_canon(seq, i, k))
        if v is None:
            continue
        hits += 1
        if v != SHARED:
            votes[v] = votes.get(v, 0) + 1
    if votes:
        best = max(votes.values())
        return hits, min(r for r, c in votes.items() if c == best), best
    return hits, (n_rec if hits else -1), 0


def _noisy(rng, n, alphabet=b"ACGTacgtNRYn"):
    return bytes(rng.choice(np.frombuffer(alphabet, dtype=np.uint8), n))


def _tie(a: bytes, b: bytes, m: int, k: int) -> bytes:
    """m windows from a, m windows from b, separated by an N so no window spans both."""
    return a[:m + k - 1] + b"N" + b[:m + k - 1]


def _test_set(k, rng):
    g = synth.make_contaminant(6000, seed=3000 + k)
    return [g[:1500].lower(),            # 0: soft-masked
            _noisy(rng, 300),            # 1: lowercase, N and IUPAC bytes
            b"NRYNNNACGNNNN",            # 2: no valid k-mer
            g[1500:2500],                # 3
            g[1500:2500],                # 4: duplicate of 3: every key shared
            g[2500:3500],                # 5
            rev_comp(g[2500:3500]),      # 6: reverse complement of 5: every key shared
            g[3500:6000],                # 7
            b""]                         # 8: empty


def _test_pieces(cset, k, rng):
    g = b"".join(cset[i] for i in (0, 3, 5, 7))
    out = []
    for i in range(30):
        kind = i % 5
        if kind == 0:  # random segment of one record, either strand, some bytes disturbed
            rec = cset[int(rng.choice([0, 3, 5, 7]))]
            s = int(rng.integers(0, len(rec) - k))
            r = bytearray(rec[s:s + int(rng.integers(k, 700))])
            if i % 2:
                r = bytearray(rev_comp(bytes(r).upper()))
            for j in rng.integers(0, len(r), 2):
                r[j] = b"NnRa"[int(rng.integers(0, 4))]
            out.append(bytes(r))
        elif kind == 1:  # chimera of several records
            out.append(cset[0][:300] + cset[7][200:700] + _noisy(rng, 100) + cset[5][:200])
        elif kind == 2:
            out.append(_noisy(rng, int(rng.integers(1, 500))))
        elif kind == 3:
            out.append(_noisy(rng, int(rng.integers(0, k))))  # shorter than k
        else:
            out.append(g[int(rng.integers(0, 1000)):][:int(rng.integers(k, 2000))])
    m = 40
    out += [_tie(cset[7], cset[0].upper(), m, k), _tie(cset[0], cset[7], m, k),      # ties: smallest record
            _tie(cset[7][500:], cset[7][900:], m, k) + b"N" + cset[0][:m + k - 1],  # 2m for 7 beats m for 0
            cset[3][:200], cset[5][100:400], rev_comp(cset[6][:300]),              # shared keys only
            cset[3][:200] + b"N" + cset[7][:k]]                                     # shared + one window of 7
    return out


@pytest.mark.parametrize("k", [11, 17, 31])
def test_oracle_matches_restatement(k):
    rng = np.random.default_rng(400 + k)
    cset = _test_set(k, rng)
    lab = _labels(cset, k)
    n_kmers, rk = clo.labels(cset, k)
    assert n_kmers == len(lab) == contam_oracle.contam_kmers(cset, k)
    assert np.array_equal(rk, _record_kmers(cset, lab))
    assert rk[2] == rk[3] == rk[4] == rk[5] == rk[6] == rk[8] == 0 and rk[9] > 0 and int(rk.sum()) == n_kmers
    pieces = _test_pieces(cset, k, rng)
    got = clo.attribute(cset, k, pieces)
    for p, row in zip(pieces, got):
        assert tuple(int(x) for x in row) == _attribute(p, k, lab, len(cset))
    tail = [tuple(int(x) for x in r) for r in got[-7:]]
    assert tail[0][1:] == (0, 40) and tail[1][1:] == (0, 40) and tail[2][1:] == (7, 80)
    assert all(t[1:] == (9, 0) and t[0] > 0 for t in tail[3:6]) and tail[6][1:] == (7, 1)
    assert all(int(r[1]) == -1 and int(r[0]) == 0 for p, r in zip(pieces, got) if len(p) < k)
    cls = clo.classify(cset, k, 0.05, pieces)
    assert np.array_equal(cls["hits"], got[:, 0]) and cls["contam"].sum() > 0


@pytest.mark.parametrize("args,msg", [
    (["--contam-report", "{out}"], "--contam-report requires --contam"),
    (["--contam", "{fa}", "--contam-report", "{out}", "--qc"], "--qc"),
])
def test_cli_rejects_bad_report_options(tmp_path, args, msg):
    """These fail in argument parsing, before any device call (so also without a GPU)."""
    if not os.path.exists(EXE):
        pytest.skip("src/tgsfilter not built")
    fa = tmp_path / "c.fa"
    fa.write_bytes(b">c\nACGTACGTACGTACGTACGT\n")
    fq = tmp_path / "r.fq"
    fq.write_bytes(b"@r\n" + b"ACGT" * 300 + b"\n+\n" + b"I" * 1200 + b"\n")
    out = tmp_path / "r.tsv"
    cmd = [EXE, "-i", str(fq), "-x", "ont", "-o", str(tmp_path / "o.fq")] + [a.format(fa=fa, out=out) for a in args]
    pr = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=60)
    assert pr.returncode != 0
    assert msg in pr.stderr.decode()
    assert not (tmp_path / "o.fq").exists() and not out.exists()


# ---- GPU -------------------------------------------------------------------------------------------
_SETS = {}


def _set(name):
    if name not in _SETS:
        if name == "small":  # prefilter path (<= 2^17 keys)
            a = synth.make_contaminant(LAMBDA_LEN)
            b = synth.make_contaminant(6_000, seed=synth.SEED0 + 201)
            c = synth.make_contaminant(20_000, seed=synth.SEED0 + 202)
            _SETS[name] = [a[:20000].lower(), b, a[20000:30000] + b"NNRY" + a[30000:], b, rev_comp(c[:5000]), c]
        else:  # table only: a 5 Mb record plus small ones
            big = synth.make_contaminant(5_000_000, seed=synth.SEED0 + 102)
            s1 = synth.make_contaminant(LAMBDA_LEN)
            s2 = synth.make_contaminant(6_000, seed=synth.SEED0 + 201)
            _SETS[name] = [s1, big, s2, big[:3000]]
    return _SETS[name]


@pytest.mark.gpu
@pytest.mark.parametrize("set_name,k", [("small", 11), ("small", 17), ("small", 31), ("large", 17)])
def test_gpu_record_kmers(set_name, k):
    from tgsfilter_b200.engine import FilterEngine
    cset = _set(set_name)
    with FilterEngine(synth.config_params(1)) as eng:
        n, rk = eng.set_contaminants_labelled(cset, k=k)
        assert n == eng.set_contaminants(cset, k=k)
    o_n, o_rk = clo.labels(cset, k)
    assert n == o_n and np.array_equal(rk, o_rk) and int(rk.sum()) == n


def _classify_pieces(cset, rng, k):
    recs = [r for r in cset if len(r) > 2000]
    out = []
    for i in range(60):
        g = recs[i % len(recs)]
        L = int(rng.integers(k, 6000))
        if i % 3 == 0:
            out.append(synth.contaminant_read(g, L, 0.05, rng).tobytes())
        elif i % 3 == 1:
            h = recs[(i + 1) % len(recs)]
            out.append(synth.contaminant_read(g, L, 0.08, rng).tobytes() + synth.make_contaminant(300, seed=i)
                       + synth.contaminant_read(h, L // 2 + k, 0.02, rng).tobytes())
        else:
            out.append(synth.make_contaminant(L, seed=900 + i))
    out += [_tie(recs[1], recs[0], 50, k), _tie(recs[0], recs[1], 50, k), b"ACG", b""]
    out.append(synth.contaminant_read(recs[0], 520_000, 0.04, rng).tobytes())
    out.append(synth.contaminant_read(recs[1], 260_000, 0.10, rng).tobytes() + synth.make_contaminant(260_000, seed=7))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("set_name,k", [("small", 17), ("small", 11), ("large", 21)])
def test_gpu_classify_matches_oracle(set_name, k):
    from tgsfilter_b200.engine import FilterEngine
    cset = _set(set_name)
    rng = np.random.default_rng(k)
    pieces = _classify_pieces(cset, rng, k)
    with FilterEngine(synth.config_params(1)) as eng:
        eng.set_contaminants_labelled(cset, k=k, min_frac=0.05)
        got = eng.contam_classify(pieces)
        reads, bases = eng.contam_record_stats()
    want = clo.classify(cset, k, 0.05, pieces)
    for f in want.dtype.names:
        assert np.array_equal(got[f], want[f]), f
    assert (got["record"] >= 0).sum() > 20 and got["contam"].sum() > 10
    assert not reads.any() and not bases.any()  # classify touches no tally


@pytest.mark.gpu
def test_gpu_classify_more_records_than_the_shared_table():
    """One piece made of 5 000 records of 40 b: more distinct labels than one pass of the shared table holds, so the
    labels are split over several passes."""
    from tgsfilter_b200.engine import FilterEngine
    g = synth.make_contaminant(5000 * 40, seed=4242)
    cset = [g[i * 40:(i + 1) * 40] for i in range(5000)]
    # record 4321 gets two copies, so it wins
    pieces = [g, g[:100_000] + b"N" + cset[4321] + b"N" + cset[4321], g[::-1], cset[17] + b"N" + cset[3]]
    with FilterEngine(synth.config_params(1)) as eng:
        _, rk = eng.set_contaminants_labelled(cset, k=17)
        got = eng.contam_classify(pieces)
    want = clo.classify(cset, 17, 0.05, pieces)
    assert np.array_equal(rk, clo.labels(cset, 17)[1])
    for f in want.dtype.names:
        assert np.array_equal(got[f], want[f]), f
    assert int(got["record"][1]) == 4321 and int(got["record"][3]) == 3


def _run_pipeline(params, batches, cset, k, path, labelled):
    from tgsfilter_b200.engine import FilterEngine
    out = []
    with FilterEngine(params) as eng:
        if labelled:
            eng.set_contaminants_labelled(cset, k=k)
        else:
            eng.set_contaminants(cset, k=k)
        keep = []
        for batch in batches:  # every batch submitted before the first collect: two slots in flight
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
                keep.append((d_b, d_q, d_o))
                eng.submit_device(d_b.data_ptr(), None if d_q is None else d_q.data_ptr(), d_o.data_ptr(),
                                  batch.n_reads, batch.n_bases, keep=(d_b, d_q, d_o))
        for _ in batches:
            out.append(eng.collect())
        cnt = eng.counters().flat
        stats = eng.contam_record_stats() if labelled else None
    return out, cnt, stats


def _planted_batch(cfg, n, cset, seed):
    batch = synth.make_config(cfg, n, max_len=200_000)
    recs = [r for r in cset if len(r) > 2000]
    for j, g in enumerate(recs[:3]):
        batch, _, _ = synth.mix_contaminants(batch, g, 0.05, 0.04, chimeras=0.02, seed=seed + j)
    return batch


@pytest.mark.gpu
@pytest.mark.parametrize("cfg,n,k,set_name,path", [
    (1, 200, 17, "small", "submit"),
    (2, 300, 11, "small", "packed"),
    (3, 60, 31, "large", "device"),
    (4, 200, 17, "large", "packed"),
    (2, 300, 31, "small", "device"),
])
def test_gpu_pipeline_tallies(cfg, n, k, set_name, path):
    cset = _set(set_name)
    batches = [_planted_batch(cfg, n, cset, 10 * cfg), _planted_batch(cfg, n // 2, cset, 10 * cfg + 5)]
    params = synth.config_params(cfg)
    lab, cnt, (reads, bases) = _run_pipeline(params, batches, cset, k, path, True)
    plain, cnt0, _ = _run_pipeline(params, batches, cset, k, path, False)
    assert np.array_equal(cnt, cnt0)
    want_r = np.zeros(len(cset) + 1, dtype=np.uint64)
    want_b = np.zeros(len(cset) + 1, dtype=np.uint64)
    n_contam = contam_bases = 0
    for (r, p), (r0, p0), batch in zip(lab, plain, batches):
        assert np.array_equal(r, r0) and np.array_equal(p, p0)
        c = p[p["status"] == _capi.PIECE_CONTAM]
        n_contam += len(c)
        contam_bases += int(c["len"].sum())
        tr, tb = clo.tallies(batch, p, cset, k)
        want_r += tr
        want_b += tb
    assert n_contam > 10
    assert np.array_equal(reads, want_r) and np.array_equal(bases, want_b)
    assert int(reads.sum()) == n_contam and int(bases.sum()) == contam_bases
    # the pieces themselves equal the oracle's
    _, o_pieces, _ = contam_oracle.run(params, batches[0], (cset, k, 0.05))
    assert np.array_equal(lab[0][1], o_pieces)


@pytest.mark.gpu
def test_gpu_pool_overflow_batch_is_tallied_once():
    """A batch that overflows the region pool re-runs the tail; its contaminant pieces are tallied once.  Counter
    resets zero the tallies; a replacing set resets them; a plain set turns attribution off."""
    from tgsfilter_b200.engine import FilterEngine
    rng = np.random.default_rng(8)
    genome = synth.make_contaminant(5000, seed=5)
    seqs, quals = [], []
    for _ in range(600):  # the middle locations of the AC repeat overflow the pool; the tail is a contaminant piece
        L = int(rng.integers(2000, 4000))
        s = int(rng.integers(0, 3000))
        seqs.append((b"AC" * (L // 2 + 1))[:L] + genome[s:s + 1500])
        quals.append(bytes([50] * (L + 1500)))
    batch = synth.pack_reads(seqs, quals)
    params = FilterParams(min_len=100, min_q=1.0, head_trim=0, tail_trim=0, mid_match_len=10,
                          extra_len=0, adapters=[b"ACACACACACACACACACACAC"]).apply_read_type("ont")
    cset = [genome, b"AC" * 200, b"GT" * 100]
    with FilterEngine(params) as eng:
        eng.set_contaminants_labelled(cset, k=17)
        reads_res, pieces = eng.run(batch)
        assert int(reads_res["n_mid"].sum()) > 65536
        reads, bases = eng.contam_record_stats()
        c = pieces[pieces["status"] == _capi.PIECE_CONTAM]
        assert len(c) > 100
        assert int(reads.sum()) == len(c) and int(bases.sum()) == int(c["len"].sum())
        tr, tb = clo.tallies(batch, pieces, cset, 17)
        assert np.array_equal(reads, tr) and np.array_equal(bases, tb)
        with pytest.raises(_capi.TgsfError) as e:
            eng.contam_record_stats(n_records=2)
        assert e.value.code == _capi.TGSF_ERR_INVALID
        eng.submit(batch)
        with pytest.raises(_capi.TgsfError) as e:
            eng.contam_classify([b"ACGT" * 10])
        assert e.value.code == _capi.TGSF_ERR_STATE
        eng.collect()
        assert int(eng.contam_record_stats()[0].sum()) == 2 * len(c)
        eng.reset_counters()
        assert not any(x.any() for x in eng.contam_record_stats())
        eng.run(batch)
        eng.set_contaminants_labelled(cset, k=17)
        assert not any(x.any() for x in eng.contam_record_stats())
        eng.set_contaminants(cset, k=17)
        for call in (lambda: eng.contam_record_stats(), lambda: eng.contam_classify([b"ACGT" * 10])):
            with pytest.raises(_capi.TgsfError) as e:
                call()
            assert e.value.code in (_capi.TGSF_ERR_INVALID, _capi.TGSF_ERR_STATE)


# ---- CLI on the GPU ----------------------------------------------------------------------------------
def _fastq_records(data: bytes):
    lines = data.split(b"\n")
    return sorted(b"\n".join(lines[i:i + 4]) for i in range(0, len(lines) - 3, 4))


def _info(stderr: bytes):
    return [ln for ln in stderr.decode().splitlines() if ln.startswith("INFO:") and "written to" not in ln]


def _cli(d, fq, args, env=None, out_name="o.fq"):
    out = d / out_name
    pr = subprocess.run([EXE, "-i", str(fq), "-o", str(out), "-x", "ont", "-5", "0", "-3", "0", "-q", "10"] + args,
                        stdout=subprocess.PIPE, stderr=subprocess.PIPE, env={**os.environ, **(env or {})}, timeout=600)
    assert pr.returncode == 0, pr.stderr.decode()[-2000:]
    return out.read_bytes(), pr.stderr


@pytest.mark.gpu
def test_cli_contam_report(tmp_path):
    a = synth.make_contaminant(LAMBDA_LEN)
    b = synth.make_contaminant(8_000, seed=synth.SEED0 + 301)
    c = synth.make_contaminant(30_000, seed=synth.SEED0 + 302)
    batch = synth.make_config(2, 3000)
    batch, _, _ = synth.mix_contaminants(batch, a, 0.04, 0.04, chimeras=0.02, seed=1)
    batch, _, _ = synth.mix_contaminants(batch, c, 0.02, 0.04, seed=2)
    fq = tmp_path / "reads.fq"
    fq.write_bytes(batch.to_fastq())
    fa = tmp_path / "panel.fa"
    cset = [a, b, c]
    fa.write_bytes(b">lambda control\n" + a + b"\n>spike\tin\r\n" + b.lower() + b"\n>ecoli-like\n"
                   + b"\n".join(c[i:i + 60] for i in range(0, len(c), 60)) + b"\n")
    ad = tmp_path / "ad.fa"
    ad.write_bytes(b">ad\n" + ADAPTER_LIB[8] + b"\n")
    base = ["-a", str(ad), "--contam", str(fa)]
    out0, err0 = _cli(tmp_path, fq, base, out_name="o0.fq")
    rep = tmp_path / "r.tsv"
    out1, err1 = _cli(tmp_path, fq, base + ["--contam-report", str(rep)], out_name="o1.fq")
    assert out1 == out0 and _info(err1) == _info(err0)
    params = FilterParams(min_q=10.0, head_trim=0, tail_trim=0,
                          adapters=[ADAPTER_LIB[8], rev_comp(ADAPTER_LIB[8])]).apply_read_type("ont")
    _, o_pieces, _ = contam_oracle.run(params, batch, (cset, 17, 0.05))
    assert _fastq_records(out1) == sorted(t.rstrip(b"\n") for t, _, _ in
                                          records.format_records(batch, o_pieces, fastq=True))
    tr, tb = clo.tallies(batch, o_pieces, cset, 17)
    _, rk = clo.labels(cset, 17)
    lines = rep.read_text().splitlines()
    assert lines[0] == "#record\tname\tlength\tunique_kmers\treads\tbases"
    names = ["lambda", "spike", "ecoli-like"]
    want = [f"{i}\t{names[i]}\t{len(cset[i])}\t{rk[i]}\t{tr[i]}\t{tb[i]}" for i in range(3)]
    want.append(f"*\tshared\t.\t{rk[3]}\t{tr[3]}\t{tb[3]}")
    assert lines[1:] == want
    assert tr[0] > 50 and tr[2] > 20
    contam = o_pieces[o_pieces["status"] == _capi.PIECE_CONTAM]
    assert [ln for ln in _info(err1) if "as contaminant" in ln] == [
        f"INFO: {int(tr.sum())} reads were discarded with {int(tb.sum())} bases as contaminant."]
    assert int(tr.sum()) == len(contam)
    rep2 = tmp_path / "r2.tsv"
    out2, err2 = _cli(tmp_path, fq, base + ["--contam-report", str(rep2), "--gpus", "2"],
                      env={"TGSF_SHARE_DEVICES": "1", "TGSF_BATCH_MB": "4"}, out_name="o2.fq")
    assert rep2.read_text() == rep.read_text()
    assert _fastq_records(out2) == _fastq_records(out1) and _info(err2) == _info(err1)

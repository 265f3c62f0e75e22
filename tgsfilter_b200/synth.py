"""Synthetic long-read generators for the five BASELINE.json configs (SURVEY.md §8(d)).

Deterministic in (config, n_reads): seed = 20261017 + config index.  Bases are uniform uppercase
ACGT; each read draws a mean quality from N(mu, sigma) and per-base qualities
clip(round(N(mean, 5)), 1, 60), Phred+33.  Planted features per config follow the table in
SURVEY.md §8(d).  ``ReadBatch`` is the packed varlen layout the C-ABI consumes: concatenated base
bytes, concatenated quality bytes and an offsets array (n+1, uint64).
"""
from __future__ import annotations

import dataclasses
from typing import List, Optional

import numpy as np

from .params import ADAPTER_LIB, FilterParams

SEED0 = 20261017
_ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


@dataclasses.dataclass
class ReadBatch:
    bases: np.ndarray             # uint8, concatenated
    quals: Optional[np.ndarray]   # uint8, concatenated (None for FASTA input)
    offsets: np.ndarray           # uint64, n+1
    names: Optional[List[bytes]] = None

    @property
    def n_reads(self) -> int:
        return len(self.offsets) - 1

    @property
    def n_bases(self) -> int:
        return int(self.offsets[-1])

    def read(self, i: int):
        s, e = int(self.offsets[i]), int(self.offsets[i + 1])
        return self.bases[s:e], (self.quals[s:e] if self.quals is not None else None)

    def name(self, i: int) -> bytes:
        return self.names[i] if self.names is not None else b"read%d" % i

    def to_fastq(self) -> bytes:
        out = []
        for i in range(self.n_reads):
            b, q = self.read(i)
            out.append(b"@" + self.name(i) + b"\n" + b.tobytes() + b"\n+\n" + q.tobytes() + b"\n")
        return b"".join(out)

    def to_fasta(self) -> bytes:
        out = []
        for i in range(self.n_reads):
            b, _ = self.read(i)
            out.append(b">" + self.name(i) + b"\n" + b.tobytes() + b"\n")
        return b"".join(out)

    def slice(self, lo: int, hi: int) -> "ReadBatch":
        s, e = int(self.offsets[lo]), int(self.offsets[hi])
        return ReadBatch(self.bases[s:e], None if self.quals is None else self.quals[s:e],
                         (self.offsets[lo:hi + 1] - self.offsets[lo]).astype(np.uint64),
                         None if self.names is None else self.names[lo:hi])


def write_fastq_to(f, bases: np.ndarray, quals: np.ndarray, offsets: np.ndarray, prefix: bytes = b"read") -> int:
    """Concatenated arrays -> 4-line FASTQ records ``@<prefix><i>`` on an open binary file.  The per-base
    copies happen inside ``write``; the Python loop only runs once per read.  Returns the bytes written."""
    mb, mq = memoryview(bases), memoryview(quals)
    off = np.asarray(offsets).astype(np.int64).tolist()
    written = 0
    for i in range(len(off) - 1):
        s, e = off[i], off[i + 1]
        written += f.write(b"@%s%d\n" % (prefix, i))
        written += f.write(mb[s:e])
        written += f.write(b"\n+\n")
        written += f.write(mq[s:e])
        written += f.write(b"\n")
    return written


def write_fastq(path: str, bases: np.ndarray, quals: np.ndarray, offsets: np.ndarray,
                prefix: bytes = b"read") -> int:
    with open(path, "wb", buffering=1 << 24) as f:
        return write_fastq_to(f, bases, quals, offsets, prefix)


def pack_reads(seqs: List[bytes], quals: Optional[List[bytes]] = None,
               names: Optional[List[bytes]] = None) -> ReadBatch:
    """The batch packer: list of reads -> concatenated arrays + offsets."""
    lens = np.fromiter((len(s) for s in seqs), dtype=np.uint64, count=len(seqs))
    offsets = np.zeros(len(seqs) + 1, dtype=np.uint64)
    np.cumsum(lens, out=offsets[1:])
    bases = np.frombuffer(b"".join(seqs), dtype=np.uint8).copy()
    q = None
    if quals is not None:
        q = np.frombuffer(b"".join(quals), dtype=np.uint8).copy()
        assert len(q) == len(bases)
    return ReadBatch(bases, q, offsets, names)


def mutate(seq: bytes, err: float, rng: np.random.Generator) -> bytes:
    """Copy of seq with substitution / insertion / deletion errors at total rate err."""
    out = bytearray()
    for ch in seq:
        r = rng.random()
        if r < err / 3:
            out.append(int(_ACGT[rng.integers(0, 4)]))  # substitution (may be silent)
        elif r < 2 * err / 3:
            out.append(ch)
            out.append(int(_ACGT[rng.integers(0, 4)]))  # insertion
        elif r < err:
            continue  # deletion
        else:
            out.append(ch)
    return bytes(out)


def _lengths(config: int, n: int, rng: np.random.Generator) -> np.ndarray:
    if config in (1, 5):
        L = np.clip(rng.normal(15000, 2000, n), 1000, 30000)
    elif config == 2:
        L = np.maximum(rng.lognormal(9.819, 0.7, n), 200)
    elif config == 3:
        L = np.clip(rng.lognormal(10.873, 0.8, n), 200, 1_000_000)
    elif config == 4:
        L = np.maximum(rng.lognormal(8.9, 0.75, n), 200)  # N50 ~15 kb, mean ~10 kb
    else:
        raise ValueError(config)
    return L.astype(np.int64)


_QUAL = {1: (30, 4), 2: (14, 4), 3: (14, 4), 4: (10, 3), 5: (30, 4)}


def make_config(config: int, n_reads: int, *, with_names: bool = True,
                max_len: Optional[int] = None) -> ReadBatch:
    """Synthetic batch for BASELINE config 1..5, scaled to n_reads reads."""
    rng = np.random.default_rng(SEED0 + config)
    lens = _lengths(config, n_reads, rng)
    if max_len is not None:
        lens = np.minimum(lens, max_len)
    offsets = np.zeros(n_reads + 1, dtype=np.uint64)
    np.cumsum(lens, out=offsets[1:])
    total = int(offsets[-1])
    bases = _ACGT[rng.integers(0, 4, total, dtype=np.uint8)]
    mu, sigma = _QUAL[config]
    mean_q = rng.normal(mu, sigma, n_reads)
    if config in (1, 5):
        low = rng.random(n_reads) < 0.05
        mean_q[low] = rng.normal(15, 4, int(low.sum()))
    q = np.repeat(mean_q.astype(np.float32), lens) + rng.normal(0, 5, total).astype(np.float32)
    quals = (np.clip(np.rint(q), 1, 60) + 33).astype(np.uint8)
    del q

    def plant(read: int, pos: int, seq: bytes):
        s, e = int(offsets[read]), int(offsets[read + 1])
        pos = max(0, min(pos, e - s - len(seq)))
        if e - s < len(seq):
            return
        bases[s + pos:s + pos + len(seq)] = np.frombuffer(seq, dtype=np.uint8)

    if config in (1, 5):
        ad = ADAPTER_LIB[0]
        u = rng.random(n_reads)
        for r in np.nonzero(u < 0.033)[0]:
            m = mutate(ad, 0.03, rng)
            L = int(lens[r])
            if u[r] < 0.015:
                plant(r, 0, m)
            elif u[r] < 0.030:
                plant(r, L - len(m), m)
            else:
                plant(r, int(rng.integers(300, max(301, L - 300))), m)
    if config == 5:
        # 30 % of reads carry a 6-12 kb tandem repeat (unit 50-500 bp, 1 % error)
        for r in np.nonzero(rng.random(n_reads) < 0.30)[0]:
            L = int(lens[r])
            unit = _ACGT[rng.integers(0, 4, int(rng.integers(50, 501)))].tobytes()
            span = int(min(rng.integers(6000, 12001), L - 200))
            if span <= len(unit):
                continue
            rep = (unit * (span // len(unit) + 1))[:span]
            rep = mutate(rep, 0.01, rng)[:span]
            plant(r, int(rng.integers(100, max(101, L - span - 50))), rep)
    if config in (2, 3):
        ad = ADAPTER_LIB[8]
        u = rng.random(n_reads)
        for r in np.nonzero(u < 0.80)[0]:
            lead = _ACGT[rng.integers(0, 4, int(rng.integers(0, 31)))].tobytes()
            plant(r, 0, lead + mutate(ad, 0.10, rng))
        v = rng.random(n_reads)
        frac_mid, err_mid = (0.01, 0.10) if config == 2 else (0.10, 0.05)
        for r in np.nonzero(v < frac_mid)[0]:
            L = int(lens[r])
            if L < 1000:
                continue
            plant(r, int(rng.integers(400, L - 400)), mutate(ad, err_mid, rng))
            if config == 3 and v[r] < 0.001 * 10:  # 1 % of all reads: a second copy
                plant(r, int(rng.integers(400, L - 400)), mutate(ad, err_mid, rng))
    if config == 4:
        # first 12 bases composition-biased (70 % A/T) so that -b 1 trims
        for r in range(n_reads):
            s = int(offsets[r])
            k = int(min(12, lens[r]))
            at = rng.random(k) < 0.70
            pick = np.where(at, rng.integers(0, 2, k) * 3, rng.integers(1, 3, k))  # A/T vs C/G
            bases[s:s + k] = _ACGT[pick]
    names = None
    if with_names:
        names = []
        for i in range(n_reads):
            if i % 7 == 3:
                names.append(b"read%d runid=%08x ch=%d" % (i, (i * 2654435761) & 0xffffffff, i % 512))
            else:
                names.append(b"read%d" % i)
    return ReadBatch(bases, quals, offsets, names)


def config_params(config: int) -> FilterParams:
    """Resolved FilterParams the reference would run the main pass with for each config when the
    adapter set falls back to the read-type default (T.cpp:3115-3125); tests that exercise the
    pre-pass resolve head/tail trims and adapters through tgsfilter_b200.prepass instead."""
    from .params import rev_comp
    if config in (1, 5):
        p = FilterParams(min_q=20.0, adapters=[ADAPTER_LIB[0], ADAPTER_LIB[1]]).apply_read_type("hifi")
        if config == 5:
            p.kmer, p.min_repeat = 11, 5000
    elif config in (2, 3):
        p = FilterParams(min_q=10.0, adapters=[ADAPTER_LIB[8], rev_comp(ADAPTER_LIB[8])]).apply_read_type("ont")
        if config == 3:
            p.mid_match_len, p.extra_len = 35, 50
    elif config == 4:
        p = FilterParams(min_q=7.0, max_q=15.0, bc_len=150,
                         adapters=[ADAPTER_LIB[0], ADAPTER_LIB[1]]).apply_read_type("clr")
    else:
        raise ValueError(config)
    p.head_trim = p.tail_trim = 0
    return p


# ---- contaminant sets (tgsf_set_contaminants) --------------------------------------------------------
def make_contaminant(length: int, seed: int = SEED0 + 100) -> bytes:
    """A random uppercase contaminant genome of ``length`` bases (e.g. 48_502 for a lambda-sized set)."""
    return _ACGT[np.random.default_rng(seed).integers(0, 4, length, dtype=np.uint8)].tobytes()


_COMP = np.zeros(256, dtype=np.uint8)
_COMP[np.frombuffer(b"ACGT", dtype=np.uint8)] = np.frombuffer(b"TGCA", dtype=np.uint8)


def mutate_array(seq: np.ndarray, err: float, rng: np.random.Generator) -> np.ndarray:
    """``mutate`` on a uint8 array, vectorised: substitutions, insertions and deletions at err / 3 each."""
    r = rng.random(len(seq))
    sub = r < err / 3
    ins = (r >= err / 3) & (r < 2 * err / 3)
    keep = (r >= err) | sub | ins  # err * 2/3 <= r < err: deleted
    out = seq.copy()
    out[sub] = _ACGT[rng.integers(0, 4, int(sub.sum()), dtype=np.uint8)]
    reps = keep.astype(np.int64) + ins  # an insertion takes a second slot after its base
    res = np.repeat(out, reps)
    # the second slot of every insertion becomes a random base
    ins_pos = np.cumsum(reps)[ins] - 1
    res[ins_pos] = _ACGT[rng.integers(0, 4, len(ins_pos), dtype=np.uint8)]
    return res


def contaminant_read(genome: bytes, length: int, err: float, rng: np.random.Generator) -> np.ndarray:
    """``length`` bases drawn from a random position and strand of the (circular) genome, with errors at
    rate ``err``."""
    g = np.frombuffer(genome, dtype=np.uint8)
    want = length + length // 8 + 64  # room for net deletions
    start = int(rng.integers(0, len(g)))
    seg = np.take(g, np.arange(start, start + want) % len(g))
    if rng.random() < 0.5:
        seg = _COMP[seg[::-1]]
    out = mutate_array(seg, err, rng)
    while len(out) < length:  # pragma: no cover - only at extreme deletion rates
        out = np.concatenate([out, mutate_array(seg, err, rng)])
    return out[:length]


def mix_contaminants(batch: ReadBatch, genome: bytes, frac: float, err: float, *, chimeras: float = 0.0,
                     chimera_share=(0.3, 0.6), chimera_err: Optional[float] = None, seed: int = SEED0 + 101):
    """Copy of a ``make_config`` batch in which a fraction ``frac`` of the reads is replaced by reads drawn
    from ``genome`` (same lengths, so qualities and offsets stay), and a further fraction ``chimeras`` carries
    one contaminant segment covering a share in ``chimera_share`` of the read at error rate ``chimera_err``
    (default ``err``).  Returns (batch, planted read indices, chimera read indices)."""
    rng = np.random.default_rng(seed)
    bases = batch.bases.copy()
    u = rng.random(batch.n_reads)
    planted = np.nonzero(u < frac)[0]
    chim = np.nonzero((u >= frac) & (u < frac + chimeras))[0]
    off = batch.offsets.astype(np.int64)
    for r in planted:
        s, e = int(off[r]), int(off[r + 1])
        bases[s:e] = contaminant_read(genome, e - s, err, rng)
    cerr = err if chimera_err is None else chimera_err
    for r in chim:
        s, e = int(off[r]), int(off[r + 1])
        n = int(round((e - s) * rng.uniform(*chimera_share)))
        if n < 1:
            continue
        pos = s + int(rng.integers(0, e - s - n + 1))
        bases[pos:pos + n] = contaminant_read(genome, n, cerr, rng)
    return ReadBatch(bases, batch.quals, batch.offsets, batch.names), planted, chim

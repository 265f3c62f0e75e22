"""Pre-pass host logic around tgsf_prepass: what GetFilterParameterTask (T.cpp:869-1216) and the
parameter resolution in main (T.cpp:3058-3126) decide before the main pass.

The counting (CheckBaseContent's histogram, T.cpp:1080-1095) and the 22-adapter x sampled-ends
edlib loop (adapterSearch, T.cpp:1156-1176) run on the GPU; the 150x4x10-integer decision loop
(T.cpp:1097-1134), Get_qType (T.cpp:1042-1077) and the adapter selection rules stay on the host
and are evaluated with float32 arithmetic exactly as the reference's C++ expressions.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _capi
from .params import ADAPTER_LIB, FilterParams, rev_comp, rev_comp_rows

f32 = np.float32


def sample_ends(batch, params: FilterParams, ad_num: int = 100000, bc_num: int = 100000):
    """read_fastx of the pre-pass (T.cpp:949-982): first max(-N,-n) reads with
    len >= max(-l, 2*checkLen); returns (ends5p, ends3p revcomp'd, minQ, maxQ, checkLen)."""
    check_len = max(params.end_len, params.bc_len, 100)  # T.cpp:897-904
    min_len = max(params.min_len, 2 * check_len)
    max_seq = max(ad_num, bc_num)
    lens = np.diff(batch.offsets.astype(np.int64))
    idx = np.nonzero(lens >= min_len)[0][:max_seq]
    starts = batch.offsets[idx].astype(np.int64)
    ends = batch.offsets[idx + 1].astype(np.int64)
    cols = np.arange(check_len, dtype=np.int64)
    e5 = batch.bases[starts[:, None] + cols[None, :]]
    e3 = rev_comp_rows(batch.bases[(ends - check_len)[:, None] + cols[None, :]])
    min_q, max_q = 255, 0
    if batch.quals is not None and len(idx):
        q = batch.quals[starts[:, None] + cols[None, :]].view(np.int8)
        min_q, max_q = int(q.min()), int(q.max())
    return np.ascontiguousarray(e5), np.ascontiguousarray(e3), min_q, max_q, check_len


def get_qtype(min_q: int, max_q: int) -> int:
    """Get_qType, T.cpp:1043-1053."""
    if 33 <= min_q <= 78 and 33 <= max_q <= 127:
        return 33
    if 64 <= min_q <= 108 and 64 <= max_q <= 127:
        return 64
    return 33 if min_q < 55 else 64


def default_min_q(params_min_q: float, max_q_phred: int, read_type: str) -> float:
    """T.cpp:1060-1076 (the -q given case only validates)."""
    if params_min_q >= 0:
        return params_min_q
    if max_q_phred > 10 and read_type == "clr":
        return 10.0
    if max_q_phred > 20 and read_type == "hifi":
        return 20.0
    if max_q_phred > 10 and read_type == "ont":
        return 10.0
    return 0.0


def base_content_trim(bases_num: np.ndarray, seq_num: int, end_bias: float) -> int:
    """Decision loop of CheckBaseContent, T.cpp:1097-1134."""
    check_len = bases_num.shape[0]
    max_diff = int(f32(seq_num) * f32(end_bias) / f32(100))
    bn = bases_num.astype(np.int64)
    trim = 0
    for i in range(1, check_len - 1):
        l = min(i, 5)
        r = min(check_len - i - 1, 5)
        left = bool((np.abs(bn[i][None, :] - bn[i - l:i]) > max_diff).any())
        right = bool((np.abs(bn[i + 1:i + r + 1] - bn[i][None, :]) > max_diff).any())
        if left and right:
            trim = i + 1
    return trim


def device_prepass(ends5p: np.ndarray, ends3p: np.ndarray, lib: Optional[Sequence[bytes]],
                   mid_sim: float, device: int = 0):
    """tgsf_prepass: returns (basesNum5p, basesNum3p [row_len][4] int32, maps5p, maps3p int64)."""
    so = _capi.load()
    n, row = ends5p.shape
    e5 = np.ascontiguousarray(ends5p, dtype=np.uint8)
    e3 = np.ascontiguousarray(ends3p, dtype=np.uint8)
    c5 = np.zeros((row, 4), dtype=np.int32)
    c3 = np.zeros((row, 4), dtype=np.int32)
    if lib is not None:
        seqs = (C.c_char_p * len(lib))(*lib)
        lens = (C.c_int32 * len(lib))(*[len(a) for a in lib])
        m5 = np.zeros(len(lib), dtype=np.int64)
        m3 = np.zeros(len(lib), dtype=np.int64)
        rc = so.tgsf_prepass(device, e5.ctypes.data, e3.ctypes.data, n, row,
                             C.cast(seqs, C.POINTER(C.c_char_p)), C.cast(lens, C.POINTER(C.c_int32)),
                             len(lib), mid_sim, c5.ctypes.data, c3.ctypes.data, m5.ctypes.data,
                             m3.ctypes.data)
    else:
        m5 = m3 = None
        rc = so.tgsf_prepass(device, e5.ctypes.data, e3.ctypes.data, n, row, None, None, 0, mid_sim,
                             c5.ctypes.data, c3.ctypes.data, None, None)
    _capi.check(rc, "tgsf_prepass")
    return c5, c3, m5, m3


def device_end_kmers(rows: np.ndarray, k: int, split: int, device: int = 0) -> Tuple[np.ndarray, np.ndarray]:
    """tgsf_end_kmer_counts: ([4^k] u32 outer, [4^k] u32 inner) counts of the valid k-mer windows of rows [n][row_len]
    that start before / at or after column split."""
    so = _capi.load()
    r = np.ascontiguousarray(rows, dtype=np.uint8)
    n, row_len = r.shape
    outer = np.zeros(1 << (2 * k), dtype=np.uint32) if 1 <= k <= 13 else np.zeros(1, dtype=np.uint32)
    inner = np.zeros_like(outer)
    _capi.check(so.tgsf_end_kmer_counts(device, r.ctypes.data, n, row_len, k, split, outer.ctypes.data,
                                        inner.ctypes.data), "tgsf_end_kmer_counts")
    return outer, inner


# De novo adapter assembly (--adapter-denovo, an extension): the constants src/TGSFilter.cpp names in assemble_adapter
DENOVO_K = 12
DENOVO_SUPPORT = 100      # a seed occurs in at least 1 / DENOVO_SUPPORT of the rows (and at least DENOVO_MIN_SEED times)
DENOVO_MIN_SEED = 20
DENOVO_ENRICH = 4         # a seed's outer-half count is at least DENOVO_ENRICH x (inner-half count + 1)
DENOVO_MAX_RUN = 4        # longest run of one base in a seed
DENOVO_MIN_LEN = 20
DENOVO_MAX_LEN = 100
_BASES = b"ACGT"


def denovo_split(row_len: int, k: int = DENOVO_K) -> int:
    """s = (c - k + 1) / 2: windows j < s are the outer half of a row."""
    return max(0, row_len - k + 1) // 2


def _seed_ok(code: int, k: int) -> bool:
    s = [(code >> (2 * (k - 1 - i))) & 3 for i in range(k)]
    run = longest = 1
    for i in range(1, k):
        run = run + 1 if s[i] == s[i - 1] else 1
        longest = max(longest, run)
    return len(set(s)) >= 3 and longest <= DENOVO_MAX_RUN


def assemble_adapter(O: np.ndarray, I: np.ndarray, n: int, k: int = DENOVO_K, row_len: int = 0) -> bytes:
    """The assembly on the host from the outer / inner k-mer counts of n rows of row_len bases: the seed is the most
    frequent outer k-mer that has at least 3 distinct bases, no run of one base longer than 4, an outer count of at
    least max(20, ceil(n / 100)) and at least 4 x (inner count + 1) (ties: smallest code).  It is extended to the
    right, then to the left, one base at a time by the neighbour with the largest total count (A, C, G, T order wins a
    tie) until that count is below half the seed's, the k-mer is already in the path, or the path has 100 bases.
    Returns b"" when no k-mer qualifies or the path is shorter than 20 bases."""
    if not O.shape == I.shape == (1 << (2 * k),):
        raise ValueError(f"count tables of {O.shape} / {I.shape} entries, want 4^{k}")
    if n == 0 or row_len < k:
        return b""
    o = O.astype(np.int64)
    i_ = I.astype(np.int64)
    support = max(DENOVO_MIN_SEED, -(-n // DENOVO_SUPPORT))
    cand = np.nonzero((o >= support) & (o >= DENOVO_ENRICH * (i_ + 1)))[0]
    cand = cand[np.lexsort((cand, -o[cand]))]  # largest count first, then smallest code
    seed = next((int(x) for x in cand if _seed_ok(int(x), k)), None)
    if seed is None:
        return b""
    tot = o + i_
    cut = int(tot[seed])
    mask = (1 << (2 * k)) - 1
    path = [(seed >> (2 * (k - 1 - i))) & 3 for i in range(k)]
    seen = {seed}
    for right in (True, False):
        cur = seed if right else None
        while len(path) < DENOVO_MAX_LEN:
            if right:
                nxt = [((cur << 2) | b) & mask for b in range(4)]
            else:
                cur = 0
                for v in path[:k - 1]:
                    cur = (cur << 2) | v
                nxt = [(b << (2 * (k - 1))) | cur for b in range(4)]
            b = max(range(4), key=lambda j: (tot[nxt[j]], -j))
            y = nxt[b]
            if 2 * int(tot[y]) < cut or y in seen:
                break
            seen.add(y)
            if right:
                path.append(b)
                cur = y
            else:
                path.insert(0, b)
    if len(path) < DENOVO_MIN_LEN:
        return b""
    return bytes(_BASES[v] for v in path)


@dataclasses.dataclass
class PrepassResult:
    trim5p: int
    trim3p: int
    adapter5p: bytes
    adapter3p: bytes
    dep5p: float
    dep3p: float
    adapters: List[bytes]
    log: List[str]


def _pick(maps: np.ndarray, lib: Sequence[bytes], min_sim: f32) -> Tuple[bytes, f32]:
    """Tail of adapterSearch (T.cpp:1178-1208): best library adapter by sum(mlen), kept when the
    mean depth sum/len >= 2*minSim."""
    hit = np.nonzero(maps > 0)[0]
    if hit.size == 0:
        return b"", f32(0)
    best = int(hit[np.argmax(maps[hit])])
    mean_dep = f32(int(maps[best])) / f32(len(lib[best]))
    if mean_dep >= f32(2) * min_sim:
        return lib[best], mean_dep
    return b"", f32(0)


def denovo_adapters(ends5p: np.ndarray, ends3p: np.ndarray, run: Tuple[bool, bool], min_sim: f32,
                    device: int = 0) -> List[Tuple[bytes, f32]]:
    """--adapter-denovo for the ends flagged in run: assembles a candidate from each end's rows and scores the
    candidates with the library search (tgsf_prepass, lib = the candidates).  A candidate is accepted when its mean
    depth reaches 2 x min_sim and n / 100; returns (adapter, mean depth) per end, (b"", 0) when none is accepted."""
    n, row_len = ends5p.shape
    cands = [b"", b""]
    for e, rows in enumerate((ends5p, ends3p)):
        if run[e]:
            O, I = device_end_kmers(rows, DENOVO_K, denovo_split(row_len), device)
            cands[e] = assemble_adapter(O, I, n, DENOVO_K, row_len)
    out = [(b"", f32(0)), (b"", f32(0))]
    lib = [c for c in cands if c]
    if not lib:
        return out
    _, _, m5, m3 = device_prepass(ends5p, ends3p, lib, float(min_sim), device)
    for e, maps in enumerate((m5, m3)):
        if cands[e]:
            mean_dep = f32(int(maps[lib.index(cands[e])])) / f32(len(cands[e]))
            if mean_dep >= f32(2) * min_sim and mean_dep >= f32(n) / f32(100):
                out[e] = (cands[e], mean_dep)
    return out


def resolve(c5, c3, m5, m3, *, n: int, end_bias: float, mid_sim: float, bc_len: int, read_type: str,
            lib: Sequence[bytes] = ADAPTER_LIB, head_trim: int = -1, tail_trim: int = -1,
            adapter_file: Optional[Sequence[bytes]] = None, denovo: bool = False,
            ends: Optional[Tuple[np.ndarray, np.ndarray]] = None, device: int = 0) -> PrepassResult:
    """Everything main() derives from the pre-pass (T.cpp:3063-3126).  denovo (--adapter-denovo) assembles an adapter
    on the GPU for each end without a library pick from that end's sampled rows, ends = (ends5p, ends3p)."""
    if denovo and (adapter_file is not None or ends is None):
        raise ValueError("denovo needs the sampled ends and cannot be combined with an adapter file")
    log = []
    t5 = base_content_trim(c5, n, end_bias) if head_trim < 0 else head_trim
    t3 = base_content_trim(c3, n, end_bias) if tail_trim < 0 else tail_trim
    # the reference clamps trim5p to BCLen before each thread stores its result (T.cpp:1136-1144): a race;
    # resolved in thread-creation order (5' thread first, so the 3' thread's clamp sees the 5' result)
    if head_trim < 0 and tail_trim < 0 and t5 > bc_len:
        t5 = bc_len
    log.append(f"INFO: trim 5' end length: {t5}")
    log.append(f"INFO: trim 3' end length: {t3}")
    a5 = a3 = b""
    d5 = d3 = f32(0)
    adapters: List[bytes] = []
    if adapter_file is not None:  # Get_adapters, T.cpp:2923-2942
        for a in adapter_file:
            for s in (a, rev_comp(a)):
                if s not in adapters:
                    adapters.append(s)
    else:
        min_sim = f32(mid_sim)
        if float(min_sim) < 0.9:  # float compared with the double literal 0.9, T.cpp:1152
            min_sim = f32(0.9)
        a5, d5 = _pick(m5, lib, min_sim)
        a3, d3 = _pick(m3, lib, min_sim)
        if denovo:
            run = (not a5, not a3)
            found = denovo_adapters(ends[0], ends[1], run, min_sim, device)
            for e, name in enumerate(("5'", "3'")):
                if run[e]:
                    log.append(f"INFO: de novo {name} adapter: " + found[e][0].decode())
                    log.append(f"INFO: mean depth of de novo {name} adapter: {float(found[e][1]):g}")
            if run[0]:
                a5, d5 = found[0]
            if run[1]:
                a3, d3 = found[1]
        if d5 > f32(5) * d3:  # T.cpp:3086-3092
            a3, d3 = b"", f32(0)
        elif d3 > f32(5) * d5:
            a5, d5 = b"", f32(0)
        log.append("INFO: 5' adapter: " + a5.decode())
        log.append("INFO: 3' adapter: " + a3.decode())
        for a in (a5, a3):
            if a:
                for s in (a, rev_comp(a)):
                    if s not in adapters:
                        adapters.append(s)
        if not a5 and not a3:  # T.cpp:3115-3125
            if read_type in ("hifi", "clr"):
                adapters = [lib[0], lib[1]]
                log.append("INFO: set PacBio blunt adapter to trim: " + lib[0].decode())
            elif read_type == "ont":
                adapters = [lib[8], lib[9]]
                log.append("INFO: set NanoPore rapid adapter to trim: " + lib[8].decode())
    return PrepassResult(t5, t3, a5, a3, float(d5), float(d3), adapters, log)


def run_prepass(batch, params: FilterParams, read_type: str, *, end_bias: float = 1.0,
                ad_num: int = 100000, bc_num: int = 100000, device: int = 0,
                adapter_file: Optional[Sequence[bytes]] = None,
                denovo: bool = False) -> Tuple[FilterParams, PrepassResult]:
    """Pre-pass over a packed batch: resolves qtype, MinQ, Head/TailTrim and the adapter set and
    returns the FilterParams the main pass runs with (denovo: --adapter-denovo)."""
    e5, e3, min_q, max_q, _ = sample_ends(batch, params, ad_num, bc_num)
    p = dataclasses.replace(params)
    if batch.quals is not None:
        p.qtype = get_qtype(min_q, max_q)
        p.min_q = default_min_q(params.min_q, max_q - p.qtype, read_type)
    else:
        p.qtype = 0
    lib = None if adapter_file is not None else ADAPTER_LIB
    c5, c3, m5, m3 = device_prepass(e5, e3, lib, p.mid_sim, device)
    res = resolve(c5, c3, m5, m3, n=e5.shape[0], end_bias=end_bias, mid_sim=p.mid_sim,
                  bc_len=p.bc_len, read_type=read_type, head_trim=params.head_trim,
                  tail_trim=params.tail_trim, adapter_file=adapter_file, denovo=denovo, ends=(e5, e3),
                  device=device)
    p.head_trim, p.tail_trim, p.adapters = res.trim5p, res.trim3p, res.adapters
    return p, res

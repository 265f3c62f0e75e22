"""ctypes binding of tests/contam_label_oracle.c: the CPU restatement of the contaminant screen's per-record
attribution.  For a whole batch it composes with contam_oracle.run, whose pieces give the statuses and coordinates.
Test infrastructure only; the library is compiled once per process into a temporary directory."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

import contam_oracle
from tgsfilter_b200 import _capi

HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    d = tempfile.mkdtemp(prefix="contam_label_oracle_")
    atexit.register(shutil.rmtree, d, True)
    so = os.path.join(d, "libcontam_label_oracle.so")
    subprocess.run([os.environ.get("CC", "gcc"), "-O2", "-std=c11", "-fPIC", "-shared", "-o", so,
                    os.path.join(HERE, "contam_label_oracle.c")], check=True)
    lib = C.CDLL(so)
    lib.tgsfo_contam_labels.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_void_p]
    lib.tgsfo_contam_labels.restype = C.c_uint64
    lib.tgsfo_contam_attribute.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p,
                                           C.c_uint32, C.c_void_p]
    _lib = lib
    return lib


def _arrays(seqs):
    recs = [s.encode() if isinstance(s, str) else bytes(s) for s in seqs]
    offs = np.zeros(len(recs) + 1, dtype=np.uint64)
    np.cumsum([len(r) for r in recs], out=offs[1:])
    return np.frombuffer(b"".join(recs) + b"\0", dtype=np.uint8), offs, len(recs)


def labels(cset, k: int):
    """(n_kmers, record_kmers u64[len(cset) + 1]) of a labelled set."""
    buf, offs, n = _arrays(cset)
    rk = np.zeros(n + 1, dtype=np.uint64)
    nk = load().tgsfo_contam_labels(buf.ctypes.data, offs.ctypes.data, n, k, rk.ctypes.data)
    return int(nk), rk


def attribute(cset, k: int, pieces) -> np.ndarray:
    """(hits, record, record_hits) of every stand-alone piece (bytes) against the set, as an int32 array [n, 3]."""
    cbuf, coffs, cn = _arrays(cset)
    pbuf, poffs, pn = _arrays(pieces)
    out = np.zeros((max(pn, 1), 3), dtype=np.int32)
    if pn:
        load().tgsfo_contam_attribute(cbuf.ctypes.data, coffs.ctypes.data, cn, k, pbuf.ctypes.data,
                                      poffs.ctypes.data, pn, out.ctypes.data)
    return out[:pn]


def classify(cset, k: int, min_frac: float, pieces) -> np.ndarray:
    """What tgsf_contam_classify returns: CONTAM_CLASS_DTYPE rows, contam from the screen's threshold."""
    a = attribute(cset, k, pieces)
    out = np.zeros(len(pieces), dtype=_capi.CONTAM_CLASS_DTYPE)
    if len(pieces):
        out["hits"], out["record"], out["record_hits"] = a[:, 0], a[:, 1], a[:, 2]
    ppm = int(np.round(np.float64(np.float32(min_frac)) * 1e6))
    for i, s in enumerate(pieces):
        windows = len(s) - k + 1
        out["contam"][i] = int(windows >= 1 and int(out["hits"][i]) * 1_000_000 >= ppm * windows)
    return out


def tallies(batch, pieces, cset, k: int):
    """(reads, bases) u64[len(cset) + 1] of the TGSF_PIECE_CONTAM pieces of a pipeline run (contam_oracle.run)."""
    n = len(cset)
    reads = np.zeros(n + 1, dtype=np.uint64)
    bases = np.zeros(n + 1, dtype=np.uint64)
    sel = pieces[pieces["status"] == _capi.PIECE_CONTAM]
    seqs = []
    for p in sel:
        s = int(batch.offsets[int(p["read"])]) + int(p["start"])
        seqs.append(batch.bases[s:s + int(p["len"])].tobytes())
    a = attribute(cset, k, seqs)
    for (hits, rec, _), p in zip(a, sel):
        assert hits >= 1 and rec >= 0
        reads[rec] += 1
        bases[rec] += int(p["len"])
    return reads, bases


def run(params, batch, contam):
    """contam_oracle.run plus the tallies: returns (reads, pieces, counters, (tally_reads, tally_bases))."""
    reads, pieces, cnt = contam_oracle.run(params, batch, contam)
    return reads, pieces, cnt, tallies(batch, pieces, contam[0], contam[1])

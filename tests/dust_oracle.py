"""ctypes binding of tests/dust_oracle.c: the CPU restatement of the low-complexity (DUST) screen on top of the pinned
oracle.  Test infrastructure only; the library is compiled once per process into a temporary directory."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

import contam_oracle
import oracle_lib
from tgsfilter_b200 import _capi
from tgsfilter_b200.params import FilterParams

HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    d = tempfile.mkdtemp(prefix="dust_oracle_")
    atexit.register(shutil.rmtree, d, True)
    so = os.path.join(d, "libdust_oracle.so")
    subprocess.run([os.environ.get("CC", "gcc"), "-O2", "-std=c11", "-fPIC", "-shared", "-o", so,
                    os.path.join(HERE, "dust_oracle.c"), "-lm"], check=True)
    lib = C.CDLL(so)
    lib.tgsfo_dust_score.argtypes = [C.c_void_p, C.c_int32]
    lib.tgsfo_dust_score.restype = C.c_int
    lib.tgsfo_dust_masked.argtypes = [C.c_void_p, C.c_int32, C.c_int32]
    lib.tgsfo_dust_masked.restype = C.c_uint32
    lib.tgsfo_run_dust.argtypes = [C.POINTER(_capi.Params), C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                   C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_float,
                                   C.c_int32, C.c_float]
    _lib = lib
    return lib


def masked(seqs, level: int = 7) -> np.ndarray:
    """The oracle's M per piece."""
    lib = load()
    out = np.zeros(len(seqs), dtype=np.uint32)
    for i, s in enumerate(seqs):
        buf = np.frombuffer(bytes(s) + b"\0", dtype=np.uint8)
        out[i] = lib.tgsfo_dust_masked(buf.ctypes.data, len(s), level)
    return out


def scores(s: bytes) -> np.ndarray:
    """S of every window of s (-1 for an invalid window)."""
    lib = load()
    buf = np.frombuffer(bytes(s) + b"\0", dtype=np.uint8)
    return np.array([lib.tgsfo_dust_score(buf.ctypes.data, j) for j in range(len(s) - 63)], dtype=np.int32)


def run(params: FilterParams, batch, level: int = 7, min_frac: float = 0.5, contam=None, foldback: bool = False):
    """oracle_lib.run with the DUST screen on, after the optional contaminant set = (seqs, k, min_frac) and the
    optional fold-back screen.  Returns (reads, pieces, counters, fold-back stats[4] or None)."""
    lib = load()
    p, _keep = params.to_c()
    L = oracle_lib.layout(params)
    if contam is not None:
        cbuf, coffs, cn = contam_oracle._set_arrays(contam[0])
        cargs = (cbuf.ctypes.data, coffs.ctypes.data, cn, contam[1], contam[2])
    else:
        cargs = (None, None, 0, 0, 0.0)
    n = batch.n_reads
    reads = np.zeros(max(n, 1), dtype=_capi.READ_RESULT_DTYPE)
    bases = np.ascontiguousarray(batch.bases)
    quals = None if batch.quals is None else np.ascontiguousarray(batch.quals)
    offs = np.ascontiguousarray(batch.offsets, dtype=np.uint64)
    cap = max(16, 4 * n)
    while True:
        pieces = np.zeros(cap, dtype=_capi.PIECE_DTYPE)
        npieces = C.c_uint32(0)
        cnt = np.zeros(L.n_u64, dtype=np.uint64)
        stats = np.zeros(4, dtype=np.uint64)
        rc = lib.tgsfo_run_dust(C.byref(p), bases.ctypes.data, None if quals is None else quals.ctypes.data,
                                offs.ctypes.data, n, reads.ctypes.data, pieces.ctypes.data, cap, C.byref(npieces),
                                cnt.ctypes.data, stats.ctypes.data if foldback else None, *cargs, level, min_frac)
        if rc == _capi.TGSF_ERR_CAPACITY and npieces.value > cap:
            cap = npieces.value
            continue
        assert rc == 0, rc
        return reads[:n], pieces[:npieces.value], cnt, (stats if foldback else None)

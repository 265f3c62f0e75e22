"""ctypes binding of tests/contam_oracle.c: the CPU restatement of the contaminant screen on top of the pinned
oracle.  Test infrastructure only; the library is compiled once per process into a temporary directory."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

import oracle_lib
from tgsfilter_b200 import _capi
from tgsfilter_b200.params import FilterParams

HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    d = tempfile.mkdtemp(prefix="contam_oracle_")
    atexit.register(shutil.rmtree, d, True)
    so = os.path.join(d, "libcontam_oracle.so")
    subprocess.run([os.environ.get("CC", "gcc"), "-O2", "-std=c11", "-fPIC", "-shared", "-o", so,
                    os.path.join(HERE, "contam_oracle.c"), "-lm"], check=True)
    lib = C.CDLL(so)
    lib.tgsfo_run_contam.argtypes = [C.POINTER(_capi.Params), C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                     C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_float]
    lib.tgsfo_contam_kmers.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_int]
    lib.tgsfo_contam_kmers.restype = C.c_uint64
    _lib = lib
    return lib


def _set_arrays(seqs):
    recs = [s.encode() if isinstance(s, str) else bytes(s) for s in seqs]
    offs = np.zeros(len(recs) + 1, dtype=np.uint64)
    np.cumsum([len(r) for r in recs], out=offs[1:])
    return np.frombuffer(b"".join(recs) + b"\0", dtype=np.uint8), offs, len(recs)


def contam_kmers(seqs, k: int) -> int:
    """Distinct canonical k-mers of a contaminant set (what tgsf_set_contaminants reports)."""
    buf, offs, n = _set_arrays(seqs)
    return int(load().tgsfo_contam_kmers(buf.ctypes.data, offs.ctypes.data, n, k))


def run(params: FilterParams, batch, contam):
    """oracle_lib.run with a contaminant set installed: contam = (seqs, k, min_frac).
    Returns (reads, pieces, counters)."""
    lib = load()
    p, _keep = params.to_c()
    L = oracle_lib.layout(params)
    cbuf, coffs, cn = _set_arrays(contam[0])
    n = batch.n_reads
    reads = np.zeros(n, dtype=_capi.READ_RESULT_DTYPE)
    bases = np.ascontiguousarray(batch.bases)
    quals = None if batch.quals is None else np.ascontiguousarray(batch.quals)
    offs = np.ascontiguousarray(batch.offsets, dtype=np.uint64)
    cap = max(16, 4 * n)
    while True:
        pieces = np.zeros(cap, dtype=_capi.PIECE_DTYPE)
        npieces = C.c_uint32(0)
        cnt = np.zeros(L.n_u64, dtype=np.uint64)
        rc = lib.tgsfo_run_contam(C.byref(p), bases.ctypes.data, None if quals is None else quals.ctypes.data,
                                  offs.ctypes.data, n, reads.ctypes.data, pieces.ctypes.data, cap, C.byref(npieces),
                                  cnt.ctypes.data, cbuf.ctypes.data, coffs.ctypes.data, cn, contam[1], contam[2])
        if rc == _capi.TGSF_ERR_CAPACITY and npieces.value > cap:
            cap = npieces.value
            continue
        assert rc == 0, rc
        return reads, pieces[:npieces.value], cnt

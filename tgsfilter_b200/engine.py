"""Host-side driver of libtgsf_cuda: the batch-level replacement of TGSFilterTask's worker pool.

``FilterEngine`` owns one ``tgsf_ctx`` (one GPU).  ``submit`` enqueues the H2D copy, every kernel
and the D2H copy of a packed ``ReadBatch`` and returns immediately; ``collect`` retires the oldest
batch and returns numpy views of ``tgsf_read_result[n]`` and ``tgsf_piece[m]``.  Counters
(DropInfo, quality histograms, per-100 bp and 5'/3' tables: T.cpp:1796-1806) accumulate on the
device across batches and are read with ``counters()``.

There is no CPU path: constructing an engine without the built library or without a CUDA device
raises.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import numpy as np

from . import _capi
from .params import FilterParams


class Counters:
    """Named views into the flat uint64 counter block (tgsf_counter_layout)."""

    TABLES_BC = ("raw5p_cnt", "raw5p_qual", "raw3p_cnt", "raw3p_qual",
                 "clean5p_cnt", "clean5p_qual", "clean3p_cnt", "clean3p_qual")
    TABLES_BIN = ("raw_bin_cnt", "raw_bin_qual", "clean_bin_cnt", "clean_bin_qual")

    def __init__(self, flat: np.ndarray, layout: _capi.CounterLayout):
        self.flat = flat
        self.layout = layout
        L = layout
        self.drop_info = flat[L.drop_info:L.drop_info + _capi.DROPINFO_N]
        self.raw_hist = flat[L.raw_hist:L.raw_hist + _capi.QUAL_HIST_N]
        self.clean_hist = flat[L.clean_hist:L.clean_hist + _capi.QUAL_HIST_N]
        for name in self.TABLES_BC:
            off = getattr(L, name)
            setattr(self, name, flat[off:off + L.bc_len * 5].reshape(L.bc_len, 5))
        for name in self.TABLES_BIN:
            off = getattr(L, name)
            setattr(self, name, flat[off:off + L.max_bins * 5].reshape(L.max_bins, 5))


class FilterEngine:
    def __init__(self, params: FilterParams, device: int = 0):
        self._lib = _capi.load()
        self.params = params
        self.device = device
        p, self._keep = params.to_c()
        self._ctx = C.c_void_p()
        _capi.check(self._lib.tgsf_create(device, C.byref(p), C.byref(self._ctx)), "tgsf_create")
        self.layout = _capi.CounterLayout()
        _capi.check(self._lib.tgsf_counter_layout_get(self._ctx, C.byref(self.layout)),
                    "tgsf_counter_layout_get")
        self._inflight = []  # (n_reads, keep-alive host arrays)

    # -- lifecycle ------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx:
            self._lib.tgsf_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    # -- contaminant screen ---------------------------------------------------------------------
    def set_contaminants(self, seqs, k: int = 17, min_frac: float = 0.05) -> int:
        """tgsf_set_contaminants: screen every later batch against the canonical k-mers of ``seqs``
        (bytes / str records).  Returns the number of distinct canonical k-mers."""
        recs = [s.encode() if isinstance(s, str) else bytes(s) for s in seqs]
        offs = np.zeros(len(recs) + 1, dtype=np.uint64)
        np.cumsum([len(r) for r in recs], out=offs[1:])
        buf = np.frombuffer(b"".join(recs) + b"\0", dtype=np.uint8)
        n = C.c_uint64(0)
        _capi.check(self._lib.tgsf_set_contaminants(self._ctx, buf.ctypes.data, offs.ctypes.data, len(recs), k,
                                                     min_frac, C.byref(n)), "tgsf_set_contaminants")
        return int(n.value)

    # -- batches --------------------------------------------------------------------------------
    def submit(self, batch) -> None:
        bases = np.ascontiguousarray(batch.bases, dtype=np.uint8)
        quals = None if batch.quals is None else np.ascontiguousarray(batch.quals, dtype=np.uint8)
        offs = np.ascontiguousarray(batch.offsets, dtype=np.uint64)
        n = len(offs) - 1
        _capi.check(self._lib.tgsf_submit(
            self._ctx, bases.ctypes.data if bases.size else None,
            None if quals is None else (quals.ctypes.data if quals.size else bases.ctypes.data),
            offs.ctypes.data, n), "tgsf_submit")
        self._inflight.append((n, (bases, quals, offs)))

    def pack(self, batch):
        """tgsf_pack_bases on a ReadBatch: returns (packed, exc_pos, exc_byte) numpy arrays."""
        bases = np.ascontiguousarray(batch.bases, dtype=np.uint8)
        n = bases.size
        packed = np.zeros((n + 3) // 4 + 16, dtype=np.uint8)
        cap = 1024
        while True:
            pos = np.zeros(cap, dtype=np.uint64)
            val = np.zeros(cap, dtype=np.uint8)
            ne = C.c_uint64(0)
            rc = self._lib.tgsf_pack_bases(bases.ctypes.data if n else None, n, packed.ctypes.data,
                                           pos.ctypes.data, val.ctypes.data, cap, C.byref(ne))
            if rc == _capi.TGSF_ERR_CAPACITY:
                cap = int(ne.value)
                continue
            _capi.check(rc, "tgsf_pack_bases")
            return packed, pos[:ne.value], val[:ne.value]

    def submit_packed(self, batch, packed=None) -> None:
        """2-bit packed bases over PCIe (tgsf_submit_packed)."""
        if packed is None:
            packed = self.pack(batch)
        pk, pos, val = packed
        quals = None if batch.quals is None else np.ascontiguousarray(batch.quals, dtype=np.uint8)
        offs = np.ascontiguousarray(batch.offsets, dtype=np.uint64)
        n = len(offs) - 1
        _capi.check(self._lib.tgsf_submit_packed(
            self._ctx, pk.ctypes.data, None if quals is None else quals.ctypes.data, offs.ctypes.data, n,
            pos.ctypes.data if pos.size else None, val.ctypes.data if val.size else None, pos.size),
            "tgsf_submit_packed")
        self._inflight.append((n, (pk, pos, val, quals, offs)))

    def submit_packed_raw(self, packed_ptr: int, quals_ptr, offsets_ptr: int, n_reads: int,
                          exc_pos_ptr=None, exc_byte_ptr=None, n_exc: int = 0, keep=None) -> None:
        _capi.check(self._lib.tgsf_submit_packed(self._ctx, packed_ptr, quals_ptr, offsets_ptr, n_reads,
                                                 exc_pos_ptr, exc_byte_ptr, n_exc), "tgsf_submit_packed")
        self._inflight.append((n_reads, keep))

    def submit_raw(self, bases_ptr: int, quals_ptr: Optional[int], offsets_ptr: int, n_reads: int,
                   keep=None) -> None:
        """Host pointers (e.g. pinned torch tensors' data_ptr())."""
        _capi.check(self._lib.tgsf_submit(self._ctx, bases_ptr, quals_ptr, offsets_ptr, n_reads),
                    "tgsf_submit")
        self._inflight.append((n_reads, keep))

    def submit_device(self, d_bases: int, d_quals: Optional[int], d_offsets: int, n_reads: int,
                      n_bases: int, keep=None) -> None:
        """Device pointers of arrays already resident on this GPU."""
        _capi.check(self._lib.tgsf_submit_device(self._ctx, d_bases, d_quals, d_offsets, n_reads,
                                                 n_bases), "tgsf_submit_device")
        self._inflight.append((n_reads, keep))

    def collect(self, want_results: bool = True) -> Tuple[Optional[np.ndarray], Optional[np.ndarray]]:
        if not self._inflight:
            raise RuntimeError("collect() without an outstanding batch")
        n, _keep = self._inflight[0]
        npieces = C.c_uint32(0)
        if not want_results:
            rc = self._lib.tgsf_collect(self._ctx, None, 0, None, 0, C.byref(npieces))
            self._inflight.pop(0)
            _capi.check(rc, "tgsf_collect")
            return None, None
        reads = np.zeros(max(n, 1), dtype=_capi.READ_RESULT_DTYPE)
        cap = n + 4096
        pieces = np.zeros(cap, dtype=_capi.PIECE_DTYPE)
        rc = self._lib.tgsf_collect(self._ctx, reads.ctypes.data, n, pieces.ctypes.data, cap,
                                    C.byref(npieces))
        if rc == _capi.TGSF_ERR_CAPACITY and npieces.value > cap:
            cap = npieces.value
            pieces = np.zeros(cap, dtype=_capi.PIECE_DTYPE)
            rc = self._lib.tgsf_collect(self._ctx, reads.ctypes.data, n, pieces.ctypes.data, cap,
                                        C.byref(npieces))
        self._inflight.pop(0)
        _capi.check(rc, "tgsf_collect")
        return reads[:n], pieces[:npieces.value]

    def collect_gz(self):
        """Deflate blocks of the oldest outstanding batch (params.gz_blocks); call before collect().
        Returns (blob bytes as uint8 array, spans structured array with offset/bytes per piece)."""
        if not self._inflight:
            raise RuntimeError("collect_gz() without an outstanding batch")
        n, _keep = self._inflight[0]
        span_dtype = np.dtype([("offset", "<u8"), ("bytes", "<u4"), ("reserved", "<u4")])
        blob = np.zeros(1 << 20, dtype=np.uint8)
        spans = np.zeros(n + 4096, dtype=span_dtype)
        nb, ns = C.c_uint64(0), C.c_uint32(0)
        rc = self._lib.tgsf_collect_gz(self._ctx, blob.ctypes.data, blob.size, C.byref(nb), spans.ctypes.data,
                                       spans.size, C.byref(ns))
        if rc == _capi.TGSF_ERR_CAPACITY:
            blob = np.zeros(max(int(nb.value), 1), dtype=np.uint8)
            spans = np.zeros(max(int(ns.value), 1), dtype=span_dtype)
            rc = self._lib.tgsf_collect_gz(self._ctx, blob.ctypes.data, blob.size, C.byref(nb), spans.ctypes.data,
                                           spans.size, C.byref(ns))
        _capi.check(rc, "tgsf_collect_gz")
        return blob[:nb.value], spans[:ns.value]

    def run(self, batch):
        self.submit(batch)
        return self.collect()

    def last_timing(self) -> Tuple[float, float]:
        k, t = C.c_float(0), C.c_float(0)
        _capi.check(self._lib.tgsf_last_timing(self._ctx, C.byref(k), C.byref(t)), "tgsf_last_timing")
        return k.value, t.value

    def last_span(self) -> Tuple[float, float]:
        """[start, end] of the last collected batch's kernels on the device clock (ms since create)."""
        a, b = C.c_float(0), C.c_float(0)
        _capi.check(self._lib.tgsf_last_span(self._ctx, C.byref(a), C.byref(b)), "tgsf_last_span")
        return a.value, b.value

    def last_stage_ms(self) -> dict:
        arr = (C.c_float * _capi.N_STAGES)()
        _capi.check(self._lib.tgsf_last_stage_ms(self._ctx, arr, _capi.N_STAGES), "tgsf_last_stage_ms")
        return dict(zip(_capi.STAGE_NAMES, [float(x) for x in arr]))

    # -- counters -------------------------------------------------------------------------------
    def counters(self) -> Counters:
        # the block grows when a batch brings a read longer than every one before it: ask again
        _capi.check(self._lib.tgsf_counter_layout_get(self._ctx, C.byref(self.layout)), "tgsf_counter_layout_get")
        flat = np.zeros(self.layout.n_u64, dtype=np.uint64)
        _capi.check(self._lib.tgsf_counters(self._ctx, flat.ctypes.data, flat.size), "tgsf_counters")
        return Counters(flat, self.layout)

    def reset_counters(self) -> None:
        _capi.check(self._lib.tgsf_counters_reset(self._ctx), "tgsf_counters_reset")

    def counters_device_ptr(self) -> Tuple[int, int]:
        p, n = C.c_void_p(), C.c_uint32(0)
        _capi.check(self._lib.tgsf_counters_device(self._ctx, C.byref(p), C.byref(n)),
                    "tgsf_counters_device")
        return p.value, n.value

    def launch_count(self) -> int:
        return int(self._lib.tgsf_launch_count(self._ctx))

    def launch_shape(self) -> Tuple[int, int]:
        """(SM count the grids are sized by, middle-scan chunk shift of the last collected batch)."""
        sm, shift = C.c_int32(0), C.c_int32(0)
        _capi.check(self._lib.tgsf_launch_shape(self._ctx, C.byref(sm), C.byref(shift)), "tgsf_launch_shape")
        return sm.value, shift.value

    def mid_run_shift(self) -> int:
        """log2 of the chunks per middle-scan run of the last collected batch."""
        rs = C.c_int32(0)
        _capi.check(self._lib.tgsf_mid_run_shift(self._ctx, C.byref(rs)), "tgsf_mid_run_shift")
        return rs.value


def align_hw(pairs, device: int = 0) -> np.ndarray:
    """tgsf_align_hw on [(query, target, k)]: edlib HW+PATH semantics, one result per pair."""
    lib = _capi.load()
    n = len(pairs)
    q_off = np.zeros(n + 1, dtype=np.uint32)
    t_off = np.zeros(n + 1, dtype=np.uint32)
    np.cumsum([len(p[0]) for p in pairs], out=q_off[1:])
    np.cumsum([len(p[1]) for p in pairs], out=t_off[1:])
    q = np.frombuffer(b"".join(p[0] for p in pairs) + b"\0", dtype=np.uint8).copy()
    t = np.frombuffer(b"".join(p[1] for p in pairs) + b"\0", dtype=np.uint8).copy()
    k = np.array([p[2] for p in pairs], dtype=np.int32)
    out = np.zeros(n, dtype=_capi.ALIGN_RESULT_DTYPE)
    _capi.check(lib.tgsf_align_hw(device, q.ctypes.data, q_off.ctypes.data, t.ctypes.data,
                                  t_off.ctypes.data, k.ctypes.data, n, out.ctypes.data),
                "tgsf_align_hw")
    return out

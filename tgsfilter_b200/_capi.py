"""ctypes binding of include/tgsf.h (libtgsf_cuda.so).

The library is the product: there is no CPU fallback.  Importing this module never touches the
GPU; ``load()`` raises ``RuntimeError`` when the shared library has not been built
(``python -c 'import __graft_entry__ as g; g.build()'``).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TGSF_LIB_PATH") or os.path.join(_HERE, "libtgsf_cuda.so")  # override: A/B builds

TGSF_OK = 0
TGSF_ERR_INVALID = 1
TGSF_ERR_CUDA = 2
TGSF_ERR_NOMEM = 3
TGSF_ERR_STATE = 4
TGSF_ERR_CAPACITY = 5

FLAG_FILTER = 1
FLAG_ONLY_QC = 2
FLAG_DISCARD_MID = 4
FLAG_GZ_BLOCKS = 8
FLAG_GZ_FASTA = 16

READ_EVALUATED, READ_LOWQ, READ_EMPTY = 0, 1, 2
PIECE_EMIT, PIECE_SHORT_REPEAT, PIECE_LOWQ, PIECE_QC_ONLY, PIECE_CONTAM = 0, 1, 2, 3, 4

N_STAGES = 7
STAGE_NAMES = ("raw_scan", "raw_final", "mid_scan", "resolve", "regions", "kmer", "clean")
DROPINFO_N = 17
QUAL_HIST_N = 256


class Params(C.Structure):
    """struct tgsf_params (subset of Para_A24, T.cpp:82-172)."""

    _fields_ = [
        ("min_len", C.c_int32),
        ("max_len", C.c_int32),
        ("min_q", C.c_float),
        ("max_q", C.c_float),
        ("bc_len", C.c_int32),
        ("head_trim", C.c_int32),
        ("tail_trim", C.c_int32),
        ("end_len", C.c_int32),
        ("end_match_len", C.c_int32),
        ("mid_match_len", C.c_int32),
        ("extra_len", C.c_int32),
        ("end_sim", C.c_float),
        ("mid_sim", C.c_float),
        ("kmer", C.c_int32),
        ("min_repeat", C.c_int32),
        ("qtype", C.c_int32),
        ("flags", C.c_uint32),
        ("n_adapters", C.c_int32),
        ("adapter_seq", C.POINTER(C.c_char_p)),
        ("adapter_len", C.POINTER(C.c_int32)),
        ("max_read_len", C.c_int32),
        ("n_slots", C.c_int32),
    ]


class ReadResult(C.Structure):
    _fields_ = [
        ("sum_q", C.c_uint64),
        ("status", C.c_int32),
        ("n_mid", C.c_int32),
        ("n_5p", C.c_int32),
        ("n_3p", C.c_int32),
        ("piece_begin", C.c_int32),
        ("n_pieces", C.c_int32),
    ]


class Piece(C.Structure):
    _fields_ = [
        ("sum_q", C.c_uint64),
        ("read", C.c_int32),
        ("start", C.c_int32),
        ("len", C.c_int32),
        ("repeat_len", C.c_int32),
        ("status", C.c_int32),
        ("contam_hits", C.c_int32),
    ]


class CounterLayout(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in (
        "n_u64", "bc_len", "max_bins", "drop_info", "raw_hist", "clean_hist",
        "raw5p_cnt", "raw5p_qual", "raw3p_cnt", "raw3p_qual",
        "clean5p_cnt", "clean5p_qual", "clean3p_cnt", "clean3p_qual",
        "raw_bin_cnt", "raw_bin_qual", "clean_bin_cnt", "clean_bin_qual")]


class AlignResult(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "edit_distance", "n_locations", "align_len",
        "first_start", "first_end", "last_start", "last_end")] + [("loc_hash", C.c_uint32)]


# numpy views of the result structs (same memory layout)
READ_RESULT_DTYPE = [("sum_q", "<u8"), ("status", "<i4"), ("n_mid", "<i4"), ("n_5p", "<i4"),
                     ("n_3p", "<i4"), ("piece_begin", "<i4"), ("n_pieces", "<i4")]
PIECE_DTYPE = [("sum_q", "<u8"), ("read", "<i4"), ("start", "<i4"), ("len", "<i4"),
               ("repeat_len", "<i4"), ("status", "<i4"), ("contam_hits", "<i4")]
ALIGN_RESULT_DTYPE = [("edit_distance", "<i4"), ("n_locations", "<i4"), ("align_len", "<i4"),
                      ("first_start", "<i4"), ("first_end", "<i4"), ("last_start", "<i4"),
                      ("last_end", "<i4"), ("loc_hash", "<u4")]

# every symbol include/tgsf.h declares; tests check the built library exports all of them
EXPORTED_SYMBOLS = (
    "tgsf_version", "tgsf_last_error", "tgsf_create", "tgsf_destroy", "tgsf_device_count", "tgsf_host_alloc",
    "tgsf_host_free", "tgsf_submit", "tgsf_submit_packed", "tgsf_pack_bases", "tgsf_submit_device", "tgsf_collect", "tgsf_collect_gz", "tgsf_last_timing", "tgsf_last_span", "tgsf_last_stage_ms",
    "tgsf_counter_layout_get", "tgsf_counters", "tgsf_counters_reset", "tgsf_counters_device",
    "tgsf_launch_count", "tgsf_launch_shape", "tgsf_mid_run_shift", "tgsf_allreduce", "tgsf_prepass", "tgsf_align_hw", "tgsf_set_contaminants",
    "tgsf_end_kmer_counts",
)

_lib = None


def load() -> C.CDLL:
    """Load libtgsf_cuda.so and declare its prototypes; raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with __graft_entry__.build() "
            "(nvcc, sm_100a). tgsfilter_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, u8p, u64p = C.c_void_p, C.c_void_p, C.c_void_p
    lib.tgsf_version.restype = C.c_char_p
    lib.tgsf_version.argtypes = []
    lib.tgsf_last_error.restype = C.c_char_p
    lib.tgsf_last_error.argtypes = []
    lib.tgsf_create.argtypes = [C.c_int, C.POINTER(Params), C.POINTER(vp)]
    lib.tgsf_destroy.argtypes = [vp]
    lib.tgsf_device_count.argtypes = [C.POINTER(C.c_int)]
    lib.tgsf_host_alloc.argtypes = [C.POINTER(vp), C.c_size_t]
    lib.tgsf_host_free.argtypes = [vp]
    lib.tgsf_submit.argtypes = [vp, u8p, u8p, u64p, C.c_uint32]
    lib.tgsf_submit_packed.argtypes = [vp, u8p, u8p, u64p, C.c_uint32, u64p, u8p, C.c_uint64]
    lib.tgsf_pack_bases.argtypes = [u8p, C.c_uint64, u8p, u64p, u8p, C.c_uint64, C.POINTER(C.c_uint64)]
    lib.tgsf_submit_device.argtypes = [vp, u8p, u8p, u64p, C.c_uint32, C.c_uint64]
    lib.tgsf_collect.argtypes = [vp, vp, C.c_uint32, vp, C.c_uint32, C.POINTER(C.c_uint32)]
    lib.tgsf_collect_gz.argtypes = [vp, vp, C.c_uint64, C.POINTER(C.c_uint64), vp, C.c_uint32, C.POINTER(C.c_uint32)]
    lib.tgsf_last_timing.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    lib.tgsf_last_span.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    lib.tgsf_last_stage_ms.argtypes = [vp, C.POINTER(C.c_float), C.c_int]
    lib.tgsf_counter_layout_get.argtypes = [vp, C.POINTER(CounterLayout)]
    lib.tgsf_counters.argtypes = [vp, u64p, C.c_uint32]
    lib.tgsf_counters_reset.argtypes = [vp]
    lib.tgsf_counters_device.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_uint32)]
    lib.tgsf_launch_count.restype = C.c_uint64
    lib.tgsf_launch_count.argtypes = [vp]
    lib.tgsf_launch_shape.argtypes = [vp, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    lib.tgsf_mid_run_shift.argtypes = [vp, C.POINTER(C.c_int32)]
    lib.tgsf_allreduce.argtypes = [C.POINTER(vp), C.c_int]
    lib.tgsf_prepass.argtypes = [C.c_int, u8p, u8p, C.c_uint32, C.c_uint32,
                                 C.POINTER(C.c_char_p), C.POINTER(C.c_int32), C.c_int32, C.c_float,
                                 vp, vp, vp, vp]
    lib.tgsf_align_hw.argtypes = [C.c_int, u8p, vp, u8p, vp, vp, C.c_uint32, vp]
    lib.tgsf_end_kmer_counts.argtypes = [C.c_int, u8p, C.c_uint32, C.c_uint32, C.c_int32, C.c_uint32, vp, vp]
    lib.tgsf_set_contaminants.argtypes = [vp, u8p, u64p, C.c_uint32, C.c_int32, C.c_float, C.POINTER(C.c_uint64)]
    for name in EXPORTED_SYMBOLS:
        fn = getattr(lib, name)
        if fn.restype is C.c_int and name not in ("tgsf_version", "tgsf_last_error",
                                                   "tgsf_launch_count"):
            fn.restype = C.c_int
    _lib = lib
    return lib


class TgsfError(RuntimeError):
    def __init__(self, code: int, where: str):
        msg = ""
        try:
            msg = load().tgsf_last_error().decode("utf-8", "replace")
        except Exception:  # pragma: no cover - only if the library vanished
            pass
        super().__init__(f"{where} failed with status {code}: {msg}")
        self.code = code


def check(code: int, where: str) -> None:
    if code != TGSF_OK:
        raise TgsfError(code, where)

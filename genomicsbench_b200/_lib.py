"""ctypes binding of libbsw_b200.so -- the C ABI declared in include/bsw.h.

Python is plumbing only (tests, bench.py, multi-process launch); all DP work happens in
the CUDA library.  There is deliberately no Python or CPU implementation of the hot path:
if the library (or a GPU) is missing, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "lib" / "libbsw_b200.so"

# SeqPair, 72 bytes: benchmarks/bsw/bandedSWA.h:91-100
SEQPAIR_DTYPE = np.dtype(
    {
        "names": ["idr", "idq", "id", "len1", "len2", "h0", "seqid", "regid",
                  "score", "tle", "gtle", "qle", "gscore", "max_off"],
        "formats": ["<i8", "<i8", "<i8"] + ["<i4"] * 11,
        "offsets": [0, 8, 16, 24, 28, 32, 36, 40, 44, 48, 52, 56, 60, 64],
        "itemsize": 72,
    }
)
RESULT_FIELDS = ("score", "qle", "tle", "gtle", "gscore", "max_off")

BSW_OK = 0
BSW_ERR_PARAM, BSW_ERR_DOMAIN, BSW_ERR_CUDA, BSW_ERR_NOMEM, BSW_ERR_STATE, BSW_ERR_IO = -1, -2, -3, -4, -5, -6
BSW_ZDROP_VECTOR, BSW_ZDROP_SCALAR = 0, 1
BSW_SHORT_PACKED16, BSW_SHORT_WIDE32 = 0, 1


class BswParams(C.Structure):
    _fields_ = [
        ("o_del", C.c_int32), ("e_del", C.c_int32), ("o_ins", C.c_int32), ("e_ins", C.c_int32),
        ("zdrop", C.c_int32), ("end_bonus", C.c_int32), ("match", C.c_int32), ("mismatch", C.c_int32),
        ("ambig", C.c_int32), ("zdrop_mode", C.c_int32), ("n_devices", C.c_int32),
        ("devices", C.c_int32 * 16), ("host_threads", C.c_int32), ("long_min_qlen", C.c_int32),
        ("short_variant", C.c_int32), ("tiny_batch", C.c_int32), ("warp_max_pairs", C.c_int32),
        ("reserved", C.c_int32 * 4),
    ]


class BswStats(C.Structure):
    _fields_ = [
        ("pairs", C.c_int64), ("cells_nominal", C.c_int64), ("cells_effective", C.c_int64),
        ("ms_sort", C.c_double), ("ms_pack", C.c_double), ("ms_h2d", C.c_double),
        ("ms_kernel", C.c_double), ("ms_d2h", C.c_double), ("ms_scatter", C.c_double),
        ("ms_total", C.c_double), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64),
        ("kernel_launches", C.c_int32), ("n_short", C.c_int32), ("n_long", C.c_int32),
        ("partitioned", C.c_int32), ("shards", C.c_int32), ("reserved", C.c_int32 * 3),
    ]

    def as_dict(self) -> dict:
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}


# include/bsw.h: bsw_seed (= mem_seed_t), bsw_chain, bsw_alnreg, bsw_chain_opt
SEED_DTYPE = np.dtype([("rbeg", "<i8"), ("qbeg", "<i4"), ("len", "<i4"), ("score", "<i4"), ("reserved", "<i4")])
CHAIN_DTYPE = np.dtype([("seed_first", "<i8"), ("n_seeds", "<i4"), ("l_query", "<i4"), ("query_off", "<i8"),
                        ("rmax0", "<i8"), ("rmax1", "<i8"), ("ref_off", "<i8"), ("same_read", "<i4"), ("reserved", "<i4")])
ALNREG_DTYPE = np.dtype([("rb", "<i8"), ("re", "<i8"), ("qb", "<i4"), ("qe", "<i4"), ("score", "<i4"), ("truesc", "<i4"),
                         ("w", "<i4"), ("seedcov", "<i4"), ("seedlen0", "<i4"), ("reserved", "<i4")])
ALNREG_FIELDS = ("rb", "re", "qb", "qe", "score", "truesc", "w", "seedcov", "seedlen0")
# include/bsw.h: bsw_reg_in (a region + where its read and reference bases are), bsw_aln (the alignment record)
REG_IN_DTYPE = np.dtype([("reg", ALNREG_DTYPE), ("query_off", "<i8"), ("ref_off", "<i8"), ("l_query", "<i4"),
                         ("reserved", "<i4")])
ALN_DTYPE = np.dtype([("pos", "<i8"), ("is_rev", "<i4"), ("n_cigar", "<i4"), ("NM", "<i4"), ("gscore", "<i4"), ("w", "<i4"),
                      ("reserved", "<i4")])


class BswChainOpt(C.Structure):
    _fields_ = [("w", C.c_int32), ("pen_clip5", C.c_int32), ("pen_clip3", C.c_int32), ("max_band_try", C.c_int32)]


class BswGenConfig(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64), ("n_pairs", C.c_int64),
        ("qlen_min", C.c_int32), ("qlen_max", C.c_int32),
        ("tail_min", C.c_int32), ("tail_max", C.c_int32),
        ("h0_min", C.c_int32), ("h0_max", C.c_int32),
        ("max_len1", C.c_int32), ("max_score8", C.c_int32),
        ("error_rate", C.c_double), ("n_rate", C.c_double),
        ("match", C.c_int32), ("reserved", C.c_int32 * 7),
    ]


# include/bsw.h: the packed host format
PAIR_DESC_DTYPE = np.dtype([("q_off", "<u4"), ("r_off", "<u4"), ("len2", "<u2"), ("len1", "<u2"), ("h0", "<u2"), ("flags", "<u2")])
OUTSCORE_DTYPE = np.dtype([("score", "<i4"), ("tle", "<i4"), ("gtle", "<i4"), ("qle", "<i4"), ("gscore", "<i4"), ("max_off", "<i4")])
SCORE16_DTYPE = np.dtype([("score", "<i2"), ("qle", "<i2"), ("tle", "<i2"), ("gtle", "<i2"), ("gscore", "<i2"), ("max_off", "<i2"),
                          ("reserved", "<i2", (2,))])
BSW_PAIR_RAW = 1
BSW_PACKED_MAX_QLEN = 824


class BswPackedBatch(C.Structure):
    _fields_ = [
        ("n_pairs", C.c_int64), ("desc", C.c_void_p),
        ("q2", C.c_void_p), ("q2_words", C.c_int64), ("r2", C.c_void_p), ("r2_words", C.c_int64),
        ("raw_q", C.c_void_p), ("raw_q_bytes", C.c_int64), ("raw_r", C.c_void_p), ("raw_r_bytes", C.c_int64),
        ("ordered", C.c_int32), ("reserved", C.c_int32 * 3),
    ]


ALLOC_FN = C.CFUNCTYPE(C.c_void_p, C.c_size_t)
RELEASE_FN = C.CFUNCTYPE(None, C.c_void_p)

# every symbol include/bsw.h declares: (name, restype, argtypes); HOST_ABI = the subset libbsw_host.so exports too
_P = C.c_void_p
_PB = C.POINTER(BswPackedBatch)
HOST_ABI_NAMES = {"bsw_bucket_order", "bsw_split_by_cost", "bsw_gen_named_config", "bsw_gen_bounds", "bsw_gen_pairs",
                  "bsw_count_pairs_file", "bsw_read_pairs_file", "bsw_write_pairs_file", "bsw_batch_from_pairs",
                  "bsw_batch_from_file", "bsw_batch_to_pairs", "bsw_batch_release", "bsw_batch_gen"}
ABI = [
    ("bsw_batch_from_pairs", C.c_int, [_P, _P, _P, C.c_int64, C.c_int32, _P, _P, _PB]),
    ("bsw_batch_from_file", C.c_int, [C.c_char_p, C.c_int64, C.c_int32, _P, _P, _PB]),
    ("bsw_batch_to_pairs", C.c_int, [_PB, _P, _P, C.c_int64, _P, C.c_int64]),
    ("bsw_batch_release", None, [_PB, _P]),
    ("bsw_batch_gen", C.c_int, [C.POINTER(BswGenConfig), C.c_int64, C.c_int64, C.c_int32, _P, _P, _PB]),
    ("bsw_extend_packed", C.c_int, [_P, _PB, C.c_int32, _P]),
    ("bsw_extend_packed16", C.c_int, [_P, _PB, C.c_int32, _P]),
    ("bsw_create", _P, [C.POINTER(BswParams), C.POINTER(C.c_int)]),
    ("bsw_destroy", None, [_P]),
    ("bsw_last_error", C.c_char_p, [_P]),
    ("bsw_default_params", None, [C.POINTER(BswParams)]),
    ("bsw_extend", C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_int32]),
    ("bsw_extend32", C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_int32]),
    ("bsw_extend_async", C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_int32, C.POINTER(C.c_int64)]),
    ("bsw_wait", C.c_int, [_P, C.c_int64, C.POINTER(C.c_int64)]),
    ("bsw_async_stats", C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    ("bsw_extend_retry", C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_int32, C.c_int32, _P, _P]),
    ("bsw_chain_window", C.c_int, [C.POINTER(BswParams), C.c_int32, C.c_int64, _P, C.c_int32, C.c_int32,
                                   C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    ("bsw_extend_chains", C.c_int, [_P, _P, C.c_int64, _P, _P, _P, _P, _P, _P]),
    ("bsw_global", C.c_int, [_P, _P, _P, _P, C.c_int64, _P, _P, _P, _P, C.c_int64, _P]),
    ("bsw_global32", C.c_int, [_P, _P, _P, _P, C.c_int64, _P, _P, _P, _P, C.c_int64, _P]),
    ("bsw_reg2aln", C.c_int, [_P, _P, C.c_int64, _P, _P, C.c_int64, C.c_int32, _P, _P, C.c_int64, _P, _P, C.c_int64, _P]),
    ("bsw_host_alloc", _P, [C.c_size_t]),
    ("bsw_host_free", None, [_P]),
    ("bsw_host_register", C.c_int, [_P, C.c_size_t]),
    ("bsw_host_unregister", C.c_int, [_P]),
    ("bsw_stage", C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_int32]),
    ("bsw_run_staged", C.c_int, [_P]),
    ("bsw_fetch", C.c_int, [_P, _P, C.c_int64]),
    ("bsw_get_stats", C.c_int, [_P, C.POINTER(BswStats)]),
    ("bsw_bucket_order", C.c_int, [_P, C.c_int64, _P]),
    ("bsw_split_by_cost", C.c_int, [_P, C.c_int64, C.c_int32, C.c_int32, _P]),
    ("bsw_gen_named_config", C.c_int, [C.c_int32, C.POINTER(BswGenConfig)]),
    ("bsw_gen_bounds", C.c_int, [C.POINTER(BswGenConfig), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    ("bsw_gen_pairs", C.c_int, [C.POINTER(BswGenConfig), C.c_int64, C.c_int64, _P, _P, _P,
                                C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    ("bsw_count_pairs_file", C.c_int64, [C.c_char_p]),
    ("bsw_read_pairs_file", C.c_int, [C.c_char_p, C.c_int64, _P, _P, C.c_int64, _P, C.c_int64,
                                      C.POINTER(C.c_int64)]),
    ("bsw_write_pairs_file", C.c_int, [C.c_char_p, _P, C.c_int64, _P, _P]),
    ("bsw_measure_int_peak", C.c_double, [_P]),
    ("bsw_version", C.c_char_p, []),
]

_lib = None


def load_library(path: os.PathLike | None = None) -> C.CDLL:
    """Loads libbsw_b200.so and types every exported entry point.  Raises if it is missing."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = Path(path) if path else LIB_PATH
    if not p.exists():
        raise RuntimeError(
            f"{p} not found: build it with `python -m genomicsbench_b200.build` "
            "(there is no Python/CPU fallback for the bsw hot path)")
    lib = C.CDLL(str(p))
    for name, restype, argtypes in ABI:
        fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    if path is None:
        _lib = lib
    return lib


_host_lib = None
HOST_LIB_PATH = PKG_DIR / "lib" / "libbsw_host.so"


def load_host_library() -> C.CDLL:
    """libbsw_host.so: generator, text format, packed-batch builders, bucketing -- no CUDA code, maps no CUDA
    library.  For tools that must stay off the GPU stack (bench.py --impl reference)."""
    global _host_lib
    if _host_lib is not None:
        return _host_lib
    if not HOST_LIB_PATH.exists():
        raise RuntimeError(f"{HOST_LIB_PATH} not found: build it with `python -m genomicsbench_b200.build`")
    lib = C.CDLL(str(HOST_LIB_PATH))
    for name, restype, argtypes in ABI:
        if name in HOST_ABI_NAMES:
            fn = getattr(lib, name)
            fn.restype = restype
            fn.argtypes = argtypes
    _host_lib = lib
    return lib


def ptr(a: np.ndarray) -> int:
    return a.ctypes.data

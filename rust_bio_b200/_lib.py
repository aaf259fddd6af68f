"""ctypes binding of rust_bio_b200/csrc/libb200align.so (C ABI: include/b200align.h).

There is no Python or CPU implementation of the alignment behind this module: if the shared
library is missing, or no sm_100 device is usable, the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# B2A_LIB_VARIANT: dev knob for A/B runs of differently built libraries (python -m rust_bio_b200.build with
# B2A_VARIANT=<name> writes csrc/libb200align_<name>.so)
_VARIANT = os.environ.get("B2A_LIB_VARIANT", "")
SO_PATH = os.path.join(HERE, "csrc", "libb200align%s.so" % (("_" + _VARIANT) if _VARIANT else ""))

MIN_SCORE = -858993459
MODE_CUSTOM, MODE_GLOBAL, MODE_SEMIGLOBAL, MODE_LOCAL = 0, 1, 2, 3
ERRORS = {-1: "B2A_E_INVALID", -2: "B2A_E_NO_DEVICE", -3: "B2A_E_CUDA", -4: "B2A_E_RANGE",
          -5: "B2A_E_CAPACITY", -6: "B2A_E_STATE", -7: "B2A_E_UNSUPPORTED"}

# every symbol include/b200align.h declares
ABI_SYMBOLS = [
    "b2a_engine_create", "b2a_engine_destroy", "b2a_last_error", "b2a_version",
    "b2a_engine_set_stream", "b2a_engine_set_traceback_budget", "b2a_engine_set_tuning",
    "b2a_engine_set_pipeline", "b2a_engine_set_walk", "b2a_engine_last_alphabet",
    "b2a_align_batch", "b2a_score_batch", "b2a_align_batch_banded", "b2a_align_batch_banded_hinted", "b2a_banded_band_ranges", "b2a_banded_strip_pairs", "b2a_batch_stage", "b2a_batch_run",
    "b2a_batch_fetch", "b2a_batch_records", "b2a_batch_records_into", "b2a_record_stride",
    "b2a_records_decode", "b2a_batch_compact_bytes", "b2a_batch_compact_into", "b2a_compact_decode",
    "b2a_batch_compact_fixed", "b2a_gathered_fetch", "b2a_align_batch_packed", "b2a_align_batch_banded_packed",
    "b2a_multi_create", "b2a_multi_destroy", "b2a_multi_device_count", "b2a_multi_last_error",
    "b2a_multi_exchange_kind", "b2a_multi_align_batch",
    "b2a_util_int32_peak",
]


class CScoring(C.Structure):
    _fields_ = [("gap_open", C.c_int32), ("gap_extend", C.c_int32),
                ("xclip_prefix", C.c_int32), ("xclip_suffix", C.c_int32),
                ("yclip_prefix", C.c_int32), ("yclip_suffix", C.c_int32),
                ("match_score", C.c_int32), ("mismatch_score", C.c_int32),
                ("has_match_scores", C.c_int32),
                ("table", C.c_void_p), ("alphabet", C.c_void_p), ("alphabet_len", C.c_uint32)]


class CPairs(C.Structure):
    _fields_ = [("seq_blob", C.c_void_p), ("x_off", C.c_void_p), ("x_len", C.c_void_p),
                ("y_off", C.c_void_p), ("y_len", C.c_void_p), ("blob_bytes", C.c_uint64),
                ("n_pairs", C.c_uint64)]


class CPackedPairs(C.Structure):
    """b2a_packed_pairs (include/b200align.h): BitEnc storage as the batch input"""
    _fields_ = [("blocks", C.c_void_p), ("x_block", C.c_void_p), ("x_len", C.c_void_p), ("y_block", C.c_void_p),
                ("y_len", C.c_void_p), ("n_blocks", C.c_uint64), ("n_pairs", C.c_uint64), ("width", C.c_uint32)]


class CBandHints(C.Structure):
    """b2a_band_hints (include/b200align.h)"""
    _fields_ = [("match_off", C.c_void_p), ("match_xy", C.c_void_p), ("path_off", C.c_void_p),
                ("path_idx", C.c_void_p), ("allowed_mismatches", C.c_int32), ("use_lcskpp_union", C.c_int32)]


class CResults(C.Structure):
    _fields_ = [("score", C.c_void_p), ("xstart", C.c_void_p), ("xend", C.c_void_p),
                ("ystart", C.c_void_p), ("yend", C.c_void_p), ("ops_off", C.c_void_p),
                ("ops", C.c_void_p), ("ops_capacity", C.c_uint64), ("clip_len", C.c_void_p),
                ("status", C.c_void_p)]


class CScoreResults(C.Structure):
    """b2a_score_results (include/b200align.h)"""
    _fields_ = [("score", C.c_void_p), ("xend", C.c_void_p), ("yend", C.c_void_p), ("status", C.c_void_p)]


class CStats(C.Structure):
    _fields_ = [("cells", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("traceback_bytes", C.c_uint64), ("pack_ms", C.c_float), ("fill_ms", C.c_float),
                ("walk_ms", C.c_float), ("band_ms", C.c_float), ("kernel_launches", C.c_uint32),
                ("waves", C.c_uint32), ("fill_lanes_per_pair", C.c_uint32),
                ("fill_rows_per_lane", C.c_uint32)]

    def as_dict(self):
        return {f: getattr(self, f) for f, _ in self._fields_}


class B2AError(RuntimeError):
    def __init__(self, code, text):
        super().__init__(f"{ERRORS.get(code, code)}: {text}")
        self.code = code


_lib = None


def load():
    """Load libb200align.so; raises if it has not been built (python -m rust_bio_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise ImportError(f"{SO_PATH} is missing: build it with `python -m rust_bio_b200.build` "
                          "(there is no CPU fallback)")
    L = C.CDLL(SO_PATH)
    L.b2a_version.restype = C.c_char_p
    L.b2a_last_error.restype = C.c_char_p
    L.b2a_last_error.argtypes = [C.c_void_p]
    L.b2a_engine_create.argtypes = [C.POINTER(C.c_void_p), C.c_int32]
    L.b2a_engine_destroy.argtypes = [C.c_void_p]
    L.b2a_engine_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    L.b2a_engine_set_traceback_budget.argtypes = [C.c_void_p, C.c_uint64]
    L.b2a_engine_set_tuning.argtypes = [C.c_void_p, C.c_int32, C.c_int32]
    L.b2a_engine_set_pipeline.argtypes = [C.c_void_p, C.c_int32]
    L.b2a_engine_set_walk.argtypes = [C.c_void_p, C.c_int32]
    L.b2a_engine_last_alphabet.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint32)]
    L.b2a_align_batch.argtypes = [C.c_void_p, C.c_int32, C.POINTER(CScoring), C.POINTER(CPairs),
                                  C.POINTER(CResults), C.POINTER(CStats)]
    L.b2a_score_batch.argtypes = [C.c_void_p, C.c_int32, C.POINTER(CScoring), C.POINTER(CPairs),
                                  C.POINTER(CScoreResults), C.POINTER(CStats)]
    L.b2a_align_batch_banded.argtypes = [C.c_void_p, C.c_int32, C.POINTER(CScoring), C.c_uint32,
                                         C.c_uint32, C.POINTER(CPairs), C.POINTER(CResults),
                                         C.POINTER(CStats)]
    L.b2a_align_batch_banded_hinted.argtypes = [C.c_void_p, C.c_int32, C.POINTER(CScoring), C.c_uint32,
                                                C.c_uint32, C.POINTER(CPairs), C.POINTER(CBandHints),
                                                C.POINTER(CResults), C.POINTER(CStats)]
    L.b2a_banded_band_ranges.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64]
    L.b2a_banded_strip_pairs.argtypes = [C.c_void_p, C.c_void_p]
    L.b2a_batch_stage.argtypes = [C.c_void_p, C.c_int32, C.POINTER(CScoring), C.POINTER(CPairs)]
    L.b2a_batch_run.argtypes = [C.c_void_p]
    L.b2a_batch_fetch.argtypes = [C.c_void_p, C.POINTER(CResults), C.POINTER(CStats)]
    L.b2a_batch_records.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint32),
                                    C.POINTER(C.c_uint64)]
    L.b2a_batch_records_into.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint32)]
    L.b2a_record_stride.argtypes = [C.c_uint32, C.c_uint32]
    L.b2a_record_stride.restype = C.c_uint32
    L.b2a_records_decode.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.POINTER(CResults)]
    L.b2a_batch_compact_bytes.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
    L.b2a_batch_compact_into.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
    L.b2a_compact_decode.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(CResults),
                                     C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.b2a_batch_compact_fixed.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
    L.b2a_gathered_fetch.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.POINTER(CResults),
                                     C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.b2a_align_batch_packed.argtypes = [C.c_void_p, C.c_int32, C.POINTER(CScoring), C.POINTER(CPackedPairs),
                                         C.POINTER(CResults), C.POINTER(CStats)]
    L.b2a_align_batch_banded_packed.argtypes = [C.c_void_p, C.c_int32, C.POINTER(CScoring), C.c_uint32, C.c_uint32,
                                                C.POINTER(CPackedPairs), C.POINTER(CResults), C.POINTER(CStats)]
    L.b2a_multi_create.argtypes = [C.POINTER(C.c_void_p), C.c_void_p, C.c_int32]
    L.b2a_multi_destroy.argtypes = [C.c_void_p]
    L.b2a_multi_device_count.argtypes = [C.c_void_p]
    L.b2a_multi_last_error.argtypes = [C.c_void_p]
    L.b2a_multi_last_error.restype = C.c_char_p
    L.b2a_multi_exchange_kind.argtypes = [C.c_void_p]
    L.b2a_multi_exchange_kind.restype = C.c_char_p
    L.b2a_multi_align_batch.argtypes = [C.c_void_p, C.c_int32, C.POINTER(CScoring), C.POINTER(CPairs),
                                        C.POINTER(CResults), C.POINTER(CStats)]
    L.b2a_util_int32_peak.argtypes = [C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                      C.POINTER(C.c_float)]
    for name in ABI_SYMBOLS:
        fn = getattr(L, name)
        if fn.restype is C.c_int:
            fn.restype = C.c_int32
    _lib = L
    return L

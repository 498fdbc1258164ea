"""ctypes binding of the C ABI declared in include/vbq_b200.h.

There is no CPU fallback: if libvbq_b200.so is missing or a call fails, this module raises."""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libvbq_b200.so")

OK = 0
FLAG_LOGVAR = 1
FLAG_NO_PRUNE = 2
FLAG_FAST = 4
FLAG_ACCUMULATE_TOTALS = 8
FLAG_NO_SWEEP = 16
FLAG_REFERENCE_WALK = 32
FLAG_RESERVE_SM = 64
FLAG_BRACKET_WALK = 128
FLAG_WORKSPACE_ZEROED = 256
FLAG_NO_TMA = 512
FLAG_TABLE_STABLE = 1024
FLAG_NEIGHBOUR_EVERY_DEPTH = 2048
GROUP = 16
TOTALS = 4
PRIOR_PARAMS = 43
MAX_DEPTH = 20
RANS_SHARED_MAX_PLANES = 64
SCORE_DOT = 0
SCORE_COSINE = 1


class VbqError(RuntimeError):
    def __init__(self, status, what, detail):
        super().__init__("vbq_b200: %s (status %d): %s" % (what, status, detail))
        self.status = status


_p = C.c_void_p
_ll = C.c_longlong
_i = C.c_int
_u = C.c_uint

# name -> (restype, argtypes); must list every symbol of include/vbq_b200.h (tests/test_abi.py checks this)
SIGNATURES = {
    "vbq_version": (_i, []),
    "vbq_status_string": (C.c_char_p, [_i]),
    "vbq_last_error": (C.c_char_p, []),
    "vbq_learned_cdf": (_i, [_p, _i, _p, _ll, _p, _p]),
    "vbq_learned_inverse_cdf": (_i, [_p, _i, _p, _ll, _p, _p]),
    "vbq_gaussian_inverse_cdf": (_i, [_p, _p, _i, _p, _ll, _p, _p]),
    "vbq_build_code_points_learned": (_i, [_p, _i, _i, _p, _p]),
    "vbq_build_code_points_gaussian": (_i, [_p, _p, _i, _i, _p, _p]),
    "vbq_packed_table_floats": (_ll, [_i, _i]),
    "vbq_pack_code_points": (_i, [_p, _i, _i, _p, _p]),
    "vbq_quantize_workspace_bytes": (_ll, [_i]),
    "vbq_quantize": (_i, [_p, _p, _ll, _i, _p, _p, _i, _p, _p, _i, _i, _p,
                          _p, _p, _p, _p, _p, _p, _p, _ll, _u, _p]),
    "vbq_quantize_hp": (_i, [_p, _p, _ll, _i, _p, _p, _i, _p, _p, _p, _i, _i, _p,
                             _p, _p, _p, _p, _p, _p, _p, _ll, _u, _p]),
    "vbq_quantize_peer": (_i, [_p, _p, _ll, _i, _p, _p, _i, _p, _p, _p, _i, _i, _p,
                               _p, _p, _p, _p, _p, _p, _p, _ll, _u, _p, _p, C.c_ulonglong, _p, C.c_ulonglong, _p]),
    "vbq_peer_push": (_i, [_p, C.c_ulonglong, _i, _p, _p]),
    "vbq_peer_ctx_create": (_i, [_i, _i, _i, C.POINTER(C.c_void_p)]),
    "vbq_peer_ctx_handle": (_i, [_p, _p]),
    "vbq_peer_ctx_connect": (_i, [_p, _p]),
    "vbq_peer_ctx_destroy": (_i, [_p]),
    "vbq_peer_collect": (_i, [_p, C.c_ulonglong, _i, _p, _p]),
    "vbq_host_ctx_create": (_i, [_i, _i, _i, _ll, _u, C.POINTER(C.c_void_p)]),
    "vbq_host_ctx_destroy": (_i, [_p]),
    "vbq_quantize_host": (_i, [_p, _p, _p, _ll, _p, _p, _p, _p, _i, _p, _p, _p, _p, _p, _p, _p, _u]),
    "vbq_compress_coordinates_f64": (_i, [_p, _p, _ll, _p, _i, _p, C.c_double, _i, _p, _p, _p, _p]),
    "vbq_intervals": (_i, [_p, _ll, _i, _p, _i, _p, _p, _p]),
    "vbq_argmax_candidates": (_i, [_p, _p, _i, _i, _p, _p, _p, _p, _i, _i, _ll, _p, _p, _p, _p]),
    "vbq_selftest_divide": (_i, [_p, _p, _ll, _p, _p]),
    "vbq_selftest_span_cuts": (_i, [_ll, _i, _i, _p]),
    "vbq_packed_index_words": (_ll, [_ll, _i]),
    "vbq_pack_indices": (_i, [_p, _ll, _i, _p, _p]),
    "vbq_unpack_indices": (_i, [_p, _ll, _i, _p, _p]),
    "vbq_symbol_histogram": (_i, [_p, _ll, _i, _i, _p, _p]),
    "vbq_rans_workspace_bytes": (_ll, [_i, _i, _ll, _i, _ll]),
    "vbq_rans_payload_bound": (_ll, [_i, _i, _ll, _i, _ll]),
    "vbq_rans_encode": (_i, [_p, _i, _i, _ll, _i, _ll, _i, _i, _p, _p, _ll, _p, _p, _p, _ll, _p]),
    "vbq_rans_decode": (_i, [_p, _ll, _p, _i, _i, _ll, _i, _ll, _i, _i, _p, _p, _p, _p, _p, _p]),
    "vbq_rans_decode_batch": (_i, [_p, _ll, _p, _p, _i, _i, _i, _p, _ll, _p, _ll, _i, _p, _ll, _p, _p, _p, _p]),
    "vbq_rans_encode_batch_workspace_bytes": (_ll, [_ll, _ll]),
    "vbq_rans_encode_batch": (_i, [_p, _ll, _p, _p, _i, _i, _i, _p, _ll, _p, _ll, _p, _i, _ll, _p, _ll, _p, _p, _p,
                                   _ll, _p]),
    "vbq_rans_shared_workspace_bytes": (_ll, [_i, _ll, _p]),
    "vbq_rans_shared_payload_bound": (_ll, [_i, _ll, _p]),
    "vbq_rans_shared_encode": (_i, [_p, _i, _ll, _p, _i, _i, _p, _p, _ll, _p, _p, _p, _ll, _p]),
    "vbq_rans_shared_decode": (_i, [_p, _ll, _p, _i, _ll, _p, _i, _i, _p, _p, _p, _p, _p, _p]),
    "vbq_rans_shared_checkpoint_count": (_ll, [_ll, _ll, _ll]),
    "vbq_rans_shared_checkpoints": (_i, [_p, _ll, _p, _ll, _ll, _i, _i, _p, _ll, _p, _p, _p, _p]),
    "vbq_rans_shared_decode_rows": (_i, [_p, _ll, _p, _ll, _ll, _i, _i, _p, _ll, _p, _p, _p, _ll, _p, _ll, _ll,
                                         _p, _p, _p, _p, _p]),
    "vbq_rans_shared_score_max_queries": (_i, [_ll]),
    "vbq_rans_shared_row_scores": (_i, [_p, _ll, _p, _ll, _ll, _i, _i, _p, _ll, _p, _p, _ll, _ll, _ll, _p, _i, _i, _p,
                                        _p, _p, _p]),
    "vbq_score_ranks": (_i, [_p, _ll, _ll, _ll, _p, _ll, _i, _p, _p, _p, _p]),
    "vbq_pair_scores": (_i, [_p, _ll, _ll, _p, _ll, _p, _p, _ll, _i, _p, _p]),
}

_lib = None


def load():
    """Load libvbq_b200.so (once).  Raises ImportError with build instructions when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "vbq_b200: %s not found. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `python -m vbq_b200.build`. There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status, what):
    if status != OK:
        lib = load()
        raise VbqError(status, what, "%s: %s" % (lib.vbq_status_string(status).decode(),
                                                  lib.vbq_last_error().decode()))

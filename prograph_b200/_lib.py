"""ctypes binding of libprograph_b200.so (declared in include/prograph_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, this
module raises.  Build it with ``python -c "import __graft_entry__ as g; g.build()"``
or ``make -C prograph_b200/csrc``.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libprograph_b200.so")

# pgStatus
OK, ERR_INVALID, ERR_UNSUPPORTED, ERR_CUDA, ERR_RANGE = 0, -1, -2, -3, -4
# pgDtype
U8, I16, I32, I64, F16, F32, F64 = range(7)
# pgCmp
LT, LE, EQ, NE, GE, GT = range(6)
# pgWeight
W_I64, W_SIM_F32, W_I32, W_FLAG_U8 = range(4)
# flag bit of the threshold kernels' `guard`: eps is a python float (PG_EPS_FLOAT)
EPS_FLOAT = 4


class Unsupported(RuntimeError):
    """The fused kernels do not cover this configuration (the caller switches to the
    tile kernels; never to the CPU)."""


_vp, _i, _i64, _sz, _dbl = C.c_void_p, C.c_int, C.c_int64, C.c_size_t, C.c_double
_pi, _pi64, _pdbl = C.POINTER(C.c_int), C.POINTER(C.c_int64), C.POINTER(C.c_double)

# name -> (restype, argtypes); the single source for the "exports every symbol" test
SIGNATURES = {
    "pg_version": (_i, []),
    "pg_last_error": (C.c_char_p, []),
    "pg_device_info": (_i, [_pi, _pi, _pi]),
    "pg_packed_words": (_i, [_i]),
    "pg_packed_rows": (_i64, [_i64]),
    "pg_packed_bytes": (_sz, [_i64, _i, _i]),
    "pg_pack_tokens": (_i, [_vp, _i, _i64, _i, _i64, _vp, _i, _i, _vp, _vp]),
    "pg_pack_chars": (_i, [_vp, _i64, _i, _i64, _vp, _vp, _i, _i, _vp]),
    "pg_sweep_workspace_bytes": (_sz, [_i64, _i64, _i, _i]),
    "pg_eps_workspace_bytes": (_sz, [_i64, _i64, _i]),
    "pg_eps_workspace_bytes_capture": (_sz, [_i64, _i64, _i, _i]),
    "pg_eps_count_workspace_bytes": (_sz, [_i64, _i64, _i]),
    "pg_hamming_knn": (_i, [_vp, _i64, _i64, _i64, _vp, _i64, _i, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "pg_knn_sym_workspace_bytes": (_sz, [_i64, _i]),
    "pg_hamming_knn_boot": (_i, [_vp, _i64, _i64, _i64, _i64, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "pg_hamming_knn_sym": (_i, [_vp, _i64, _i, _i, _i, _i, _i, _i, _i64, _vp, _vp, _sz, _vp]),
    "pg_hamming_eps_sym": (_i, [_vp, _i64, _i, _i, _vp, _i, _i, _i, _i, _vp, _i64, _vp, _vp, _sz, _vp]),
    "pg_edge_keys_to_csr": (_i, [_vp, _i64, _vp, _i64, _i, _i64, _i, _vp, _vp, _vp, _vp]),
    "pg_knn_sym_band": (_i, [_i64, _i, _i64, _i, _i, _pi64, _pi64]),
    "pg_knn_lists_finalize": (_i, [_vp, _i, _i64, _i64, _i64, _i, _i, _i, _i, _vp, _vp, _vp]),
    "pg_knn_lists_merge": (_i, [_vp, _i, _i64, _i64, _i64, _i, _i, _i, _vp, _vp]),
    "pg_knn_sym_status": (_i, [_vp, _i64, _i, _vp]),
    "pg_knn_sym_plan": (_i, [_i64, _i, _i, _i64, _i, _i, _i, _i, _vp, _i64, _pi64]),
    "pg_hamming_eps_count": (_i, [_vp, _i64, _i64, _i64, _vp, _i64, _i, _i, _vp, _i, _vp, _vp, _sz, _vp]),
    "pg_hamming_eps_fill": (_i, [_vp, _i64, _i64, _i64, _vp, _i64, _i, _i, _vp, _i, _vp, _i, _vp, _vp, _vp, _sz, _vp]),
    "pg_hamming_eps_count_capture": (_i, [_vp, _i64, _i64, _i64, _vp, _i64, _i, _i, _vp, _i, _i, _vp, _vp, _sz, _vp]),
    "pg_hamming_eps_fill_capture": (_i, [_vp, _i64, _i64, _i64, _vp, _i64, _i, _i, _vp, _i, _i, _vp, _i, _vp, _vp, _vp, _sz,
                                         _vp]),
    "pg_hamming_tile": (_i, [_vp, _i64, _vp, _i64, _i64, _i64, _i, _i, _i, _vp, _i64, _vp]),
    "pg_hamming_flags_tile": (_i, [_vp, _i64, _vp, _i64, _i64, _i64, _i, _i, _i, _i, _vp, _i64, _vp]),
    "pg_flags_or_rows": (_i, [_vp, _i64, _i64, _i64, _vp, _vp, _vp]),
    "pg_exclusive_scan_i64": (_i, [_vp, _i64, _vp, _vp]),
    "pg_knn_extend_merge": (_i, [_vp, _vp, _i, _vp, _vp, _i, _i64, _i64, _i, _i, _vp, _vp, _vp]),
    "pg_csr_append": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i, _vp, _vp, _vp, _vp]),
    "pg_minkowski_tile": (_i, [_vp, _i64, _vp, _i64, _i64, _i64, _i, _i, _dbl, _i, _vp, _i64, _vp]),
    "pg_hamming_values_tile": (_i, [_vp, _i64, _vp, _i64, _i64, _i64, _i, _i, _i, _vp, _i64, _vp]),
    "pg_gemm_width": (_i, [_i]),
    "pg_gemm_rows": (_i64, [_i64]),
    "pg_gemm_pack": (_i, [_vp, _i, _i64, _i, _i64, _vp, _vp, _i, _i, _vp, _vp]),
    "pg_minkowski2_gemm_tile": (_i, [_vp, _vp, _i64, _vp, _vp, _i64, _i, _i, _i, _vp, _i64, _vp]),
    "pg_minkowski2_gemm_knn": (_i, [_vp, _vp, _i64, _vp, _vp, _i64, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "pg_minkowski2_gemm_eps_count": (_i, [_vp, _vp, _i64, _vp, _vp, _i64, _i, _i, _i, _vp, _vp, _vp]),
    "pg_minkowski2_gemm_eps_fill": (_i, [_vp, _vp, _i64, _vp, _vp, _i64, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "pg_tile_topk": (_i, [_vp, _i, _i64, _i64, _i64, _i, _i, _i, _vp, _vp, _vp]),
    "pg_tile_threshold_count": (_i, [_vp, _i, _i64, _i64, _i64, _i, _dbl, _i, _i, _vp, _vp]),
    "pg_tile_threshold_fill": (_i, [_vp, _i, _i64, _i64, _i64, _i, _dbl, _i, _i, _vp, _vp, _vp, _vp]),
    "pg_mutant_bits": (_i, [_vp, _i64, _i, _i, _vp, _vp, _vp]),
    "pg_mutant_bool": (_i, [_vp, _i64, _i, _i, _i, _vp, _vp, _vp]),
    "pg_mutant_any": (_i, [_vp, _i64, _i, _vp, _vp]),
    "pg_varying_columns": (_i, [_vp, _i64, _i, _i, _vp, _vp]),
    "pg_compact_columns": (_i, [_vp, _i64, _i, _i, _vp, _vp, _i, _vp]),
    "pg_select_rows": (_i, [_vp, _i64, _i, _vp, _i, _vp, _vp, _i, _vp, _vp]),
    "pg_flag_indices": (_i, [_vp, _i64, _vp, _vp, _vp]),
    "pg_distance_hist": (_i, [_vp, _i64, _i, _vp, _vp]),
    "pg_measure_int_peak": (_i, [_i, _i, _pdbl, _pdbl]),
    "pg_measure_i8_mma_peak": (_i, [_i, _pdbl, _pdbl]),
    "pg_launch_count": (_i64, [_i]),
    "pg_time_sweeps": (_i, [_i]),
    "pg_sweep_time": (_i, [_pdbl, _pi64, _i]),
    "pg_sweep_times": (_i, [_pdbl, _i64, _pi64, _i]),
}

_lib = None


def load():
    """Load the shared library (once).  Raises ImportError with build instructions if it
    is absent -- the product path never degrades to a CPU implementation."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build the CUDA library first "
            "(python -c 'import __graft_entry__ as g; g.build()' or make -C prograph_b200/csrc). "
            "prograph_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    msg = load().pg_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc):
    """Map a pgStatus onto the exception types the reference raises (SURVEY.md §8b)."""
    if rc == OK:
        return
    msg = last_error()
    if rc == ERR_INVALID:
        raise ValueError(msg)
    if rc == ERR_UNSUPPORTED:
        raise Unsupported(msg)
    if rc == ERR_RANGE:
        raise OverflowError(msg)
    raise RuntimeError(f"prograph_b200 CUDA error: {msg}")

"""ctypes binding of include/aadp.h.  Fails loudly when the native library is missing:
there is no Python/CPU fallback for any compute entry point."""
import ctypes as C
import os

from . import build as _build

_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if os.environ.get("AADP_LIB"):  # A/B measurements: an alternative build of the same library
        path = os.environ["AADP_LIB"]
    elif _build.needs_build():
        try:
            _build.build()
        except Exception as e:  # no nvcc on the box: use the shipped .so if there is one
            if not os.path.exists(path):
                raise RuntimeError(
                    "libaadp.so is missing and could not be built (%s); "
                    "alignment_algos_b200 has no CPU fallback" % e)
    L = C.CDLL(path)
    vp, i32, i64, f32, u32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_uint32
    cp = C.c_char_p
    L.aadp_create.restype = vp
    L.aadp_create.argtypes = [C.c_int]
    L.aadp_destroy.restype = None
    L.aadp_destroy.argtypes = [vp]
    L.aadp_last_error.restype = cp
    L.aadp_version.restype = cp
    L.aadp_set_stream.argtypes = [vp, vp]
    L.aadp_synchronize.argtypes = [vp]
    L.aadp_set_option.argtypes = [vp, cp, C.c_int]
    L.aadp_set_scoring.argtypes = [vp, vp, C.c_int, f32, f32, C.c_int, u32]
    L.aadp_set_profile_scoring.argtypes = [vp, vp, vp, i64, C.c_int, f32, f32, C.c_int, u32]
    L.aadp_fill_pair.argtypes = [vp, vp, C.c_int, vp, C.c_int, C.c_int, f32] + [vp] * 8
    L.aadp_fill_batch.argtypes = [vp, vp, vp, i64, vp, vp, i64, u32, f32, vp, vp, vp, vp]
    L.aadp_fill_batch_submit.argtypes = [vp, vp, vp, i64, vp, vp, i64, u32, f32, vp, vp, vp, vp]
    L.aadp_fill_batch_wait.argtypes = [vp]
    L.aadp_upload_batch.argtypes = [vp, vp, vp, i64, vp, vp, i64, u32]
    L.aadp_run_batch.argtypes = [vp, u32, f32, vp, vp, vp, vp]
    L.aadp_batch_resident_bytes.restype = i64
    L.aadp_batch_resident_bytes.argtypes = [vp, u32]
    L.aadp_last_launch_count.restype = i64
    L.aadp_last_launch_count.argtypes = [vp]
    L.aadp_last_h2d_bytes.restype = i64
    L.aadp_last_h2d_bytes.argtypes = [vp]
    L.aadp_last_d2h_bytes.restype = i64
    L.aadp_last_d2h_bytes.argtypes = [vp]
    L.aadp_last_cell_updates.restype = C.c_double
    L.aadp_last_cell_updates.argtypes = [vp]
    L.aadp_set_profiling.argtypes = [vp, C.c_int]
    L.aadp_profile_count.argtypes = [vp]
    L.aadp_profile_get.argtypes = [vp, C.c_int, vp, C.c_int, vp, vp]
    L.aadp_batch_fetch_pair.argtypes = [vp, i64] + [vp] * 7
    L.aadp_batch_optimal.argtypes = [vp, i64, C.c_int, vp, i32, vp, vp]
    L.aadp_tb_row_bytes.restype = i64
    L.aadp_tb_row_bytes.argtypes = [C.c_int]
    L.aadp_batch_tb_bytes.restype = i64
    L.aadp_batch_tb_bytes.argtypes = [vp, i64]
    L.aadp_batch_fetch_tb.argtypes = [vp, i64, C.c_int, vp, i64, vp]
    L.aadp_decode_cell.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, u32, vp, C.c_int, C.c_int, vp, vp]
    L.aadp_batch_optimal_all.argtypes = [vp, C.c_int, vp, vp, i64, vp, vp]
    L.aadp_batch_optimal_all_compact.argtypes = [vp, C.c_int, vp, vp, i64, vp, vp]
    L.aadp_fill_subpair.argtypes = [vp, vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp]
    L.aadp_fill_subpair_batch.argtypes = [vp, vp, vp, i64, vp, vp, vp, i64, C.c_int, vp, vp, vp, i64, vp, vp]
    L.aadp_fill_pair_general.argtypes = [vp, vp, C.c_int, C.c_int, f32, f32, C.c_int, u32, C.c_int, vp, vp, vp, vp]
    L.aadp_fill_pair_tabulated.argtypes = [vp, vp, C.c_int, C.c_int, vp, vp, C.c_int, u32, C.c_int, vp, vp, vp]
    L.aadp_batch_near_optimal.argtypes = [vp, vp, i64, f32, i32, vp, vp, vp, vp, vp, vp, i64, vp]
    L.aadp_batch_near_optimal_constrained.argtypes = [vp, vp, i64, vp, vp, f32, i32, vp, vp, vp, vp, vp, vp, i64, vp]
    L.aadp_batch_near_optimal_pruned.argtypes = [vp, i64, C.c_int, vp, f32, u32, u32, f32, u32, i32, vp, vp, vp, vp, vp, i64, vp]
    L.aadp_fill_batch_tabulated.argtypes = [vp, i64, vp, vp, vp, vp, vp, vp, vp, vp, C.c_int, u32, C.c_int, vp, vp, vp, vp, i64, vp, vp]
    L.aadp_upload_sequences.argtypes = [vp, vp, vp, i64]
    L.aadp_cross_run.argtypes = [vp, vp, i64, vp, i64, vp]
    L.aadp_cross_scores.argtypes = [vp, vp, vp, i64, vp, i64, vp, i64, vp]
    L.aadp_last_cross_cell_updates.restype = C.c_double
    L.aadp_last_cross_cell_updates.argtypes = [vp]
    _lib = L
    return L


EXPORTS = [
    "aadp_create", "aadp_destroy", "aadp_last_error", "aadp_version", "aadp_set_stream",
    "aadp_synchronize", "aadp_set_option", "aadp_set_scoring", "aadp_set_profile_scoring", "aadp_fill_pair", "aadp_fill_batch",
    "aadp_upload_batch", "aadp_run_batch", "aadp_batch_resident_bytes", "aadp_last_launch_count",
    "aadp_last_h2d_bytes", "aadp_last_d2h_bytes", "aadp_last_cell_updates", "aadp_set_profiling", "aadp_profile_count", "aadp_profile_get",
    "aadp_batch_fetch_pair", "aadp_batch_optimal", "aadp_tb_row_bytes", "aadp_batch_tb_bytes",
    "aadp_batch_fetch_tb", "aadp_decode_cell", "aadp_upload_sequences", "aadp_cross_run", "aadp_cross_scores",
    "aadp_last_cross_cell_updates", "aadp_batch_optimal_all", "aadp_fill_subpair", "aadp_fill_pair_general",
    "aadp_fill_subpair_batch", "aadp_fill_pair_tabulated", "aadp_fill_batch_tabulated", "aadp_fill_batch_submit", "aadp_fill_batch_wait", "aadp_batch_near_optimal", "aadp_batch_near_optimal_constrained",
    "aadp_batch_near_optimal_pruned", "aadp_batch_optimal_all_compact",
]

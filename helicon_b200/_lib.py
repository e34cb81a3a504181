"""ctypes binding of libhelicon_b200.so (include/helicon_b200.h).

The product path has NO CPU fallback: if the shared library is missing or no
CUDA device is visible, the entry points raise ``HeliconB200Error``.
"""

from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhelicon_b200.so")


class HeliconB200Error(RuntimeError):
    pass


HB2_FLAG_TIE_XY = 1
HB2_FLAG_TIE_Z = 2
HB2_FLAG_BOUNDED = 4
HB2_FLAG_NO_ROWS = 8
HB2_FLAG_TIE_Z_EXACT = 16
HB2_FLAG_NOT_CONVERGED = 32


class Geometry(C.Structure):
    _fields_ = [
        ("ny", C.c_int32), ("nx", C.c_int32), ("scale2d_to_3d", C.c_double), ("D2", C.c_int32), ("L2", C.c_int32),
        ("D3", C.c_int32), ("rmin", C.c_double), ("rmax", C.c_int32), ("interpolation", C.c_int32),
    ]


class Candidate(C.Structure):
    _fields_ = [
        ("view_begin", C.c_int32), ("view_count", C.c_int32), ("pair_begin", C.c_int32), ("pair_count", C.c_int32),
        ("min_sym_pairs", C.c_int64), ("positive", C.c_int32), ("flags_in", C.c_uint32),
    ]


class View(C.Structure):
    _fields_ = [("angle", C.c_int32), ("col_begin", C.c_int32), ("tie", C.c_int32), ("tie_slot0", C.c_int32),
                ("dup_of", C.c_int32), ("mult", C.c_int32)]


class Pair(C.Structure):
    _fields_ = [("ci", C.c_double), ("si", C.c_double), ("zi", C.c_double), ("cj", C.c_double), ("sj", C.c_double), ("zj", C.c_double)]


class SolveOptions(C.Structure):
    _fields_ = [
        ("max_iter", C.c_int32), ("atol", C.c_double), ("btol", C.c_double), ("conlim", C.c_double),
        ("check_every", C.c_int32), ("clip_pred", C.c_int32), ("trf_max_iter", C.c_int32), ("trf_tol", C.c_double),
        ("fixed_iters", C.c_int32), ("profile", C.c_int32), ("norm_mode", C.c_int32),
    ]


class ModelOptions(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("alpha", C.c_double), ("l1_ratio", C.c_double), ("gap_factor", C.c_double),
        ("max_iter", C.c_int32), ("check_every", C.c_int32), ("clip_pred", C.c_int32), ("power_start", C.c_void_p),
    ]


MODEL_ENET, MODEL_RIDGE = 0, 1

# score_metric names of lsq_reconstruct / search_grid -> HB2_METRIC_* (cosine is the solve's own score)
METRICS = {"ssim": 1, "ms_ssim": 2, "mutual_information": 3, "composite": 4}


class SymmParams(C.Structure):
    _fields_ = [
        ("nz0", C.c_int32), ("ny0", C.c_int32), ("nx0", C.c_int32), ("nz", C.c_int32), ("ny", C.c_int32), ("nx", C.c_int32),
        ("oz", C.c_int32), ("oy", C.c_int32), ("ox", C.c_int32), ("nz1", C.c_int32), ("ny1", C.c_int32), ("nx1", C.c_int32),
        ("apix", C.c_double), ("new_apix", C.c_double), ("csym", C.c_int32), ("n_ent", C.c_int32),
        ("zs0", C.c_int32), ("zs1", C.c_int32),
    ]


class ExplicitGeometry(C.Structure):
    _fields_ = [("interpolation", C.c_int32), ("dy_pixel", C.c_double), ("rot_yx", C.c_double * 9)]


class Result(C.Structure):
    _fields_ = [
        ("score", C.c_float), ("itn", C.c_int32), ("istop", C.c_int32), ("trf_nit", C.c_int32), ("flags", C.c_uint32),
        ("n_data_rows", C.c_int32), ("n_sym_rows", C.c_int32), ("normr", C.c_float), ("normar", C.c_float),
        ("normA", C.c_float), ("normx", C.c_float),
    ]


CANDIDATE_DTYPE = np.dtype(
    [("view_begin", "<i4"), ("view_count", "<i4"), ("pair_begin", "<i4"), ("pair_count", "<i4"),
     ("min_sym_pairs", "<i8"), ("positive", "<i4"), ("flags_in", "<u4")], align=True)
VIEW_DTYPE = np.dtype([("angle", "<i4"), ("col_begin", "<i4"), ("tie", "<i4"), ("tie_slot0", "<i4"), ("dup_of", "<i4"),
                       ("mult", "<i4")], align=True)
PAIR_DTYPE = np.dtype([("ci", "<f8"), ("si", "<f8"), ("zi", "<f8"), ("cj", "<f8"), ("sj", "<f8"), ("zj", "<f8")], align=True)
RESULT_DTYPE = np.dtype(
    [("score", "<f4"), ("itn", "<i4"), ("istop", "<i4"), ("trf_nit", "<i4"), ("flags", "<u4"), ("n_data_rows", "<i4"),
     ("n_sym_rows", "<i4"), ("normr", "<f4"), ("normar", "<f4"), ("normA", "<f4"), ("normx", "<f4")], align=True)
assert CANDIDATE_DTYPE.itemsize == C.sizeof(Candidate)
assert VIEW_DTYPE.itemsize == C.sizeof(View)
assert PAIR_DTYPE.itemsize == C.sizeof(Pair)
assert RESULT_DTYPE.itemsize == C.sizeof(Result)

# every symbol include/helicon_b200.h declares
EXPORTS = [
    "hb2_last_error", "hb2_device_count", "hb2_build_info", "hb2_problem_create", "hb2_problem_destroy",
    "hb2_problem_ndisk", "hb2_problem_rank_table", "hb2_batch_begin", "hb2_batch_ray_valid", "hb2_batch_angle_map",
    "hb2_batch_create", "hb2_batch_destroy", "hb2_batch_sym_rows", "hb2_batch_sym_order", "hb2_batch_rows_padded", "hb2_batch_rhs",
    "hb2_batch_apply_forward", "hb2_batch_apply_adjoint", "hb2_batch_solve", "hb2_batch_get_x", "hb2_batch_timing",
    "hb2_lsmr_scalar_step", "hb2_batch_trf_trace", "hb2_stream_create", "hb2_stream_destroy", "hb2_device_trim", "hb2_helical_symmetrize", "hb2_batch_set_ties",
    "hb2_batch_set_pixel_masks", "hb2_batch_add_exact_maps", "hb2_batch_explicit_rows", "hb2_batch_explicit_export", "hb2_batch_explicit_sym_rows",
    "hb2_batch_explicit_sym_export", "hb2_batch_explicit_pixel_mask",
    "hb2_batch_bilinear_maps", "hb2_batch_bilinear_ray_valid", "hb2_batch_bilinear_views", "hb2_batch_bilinear_sym_rows",
    "hb2_batch_bilinear_sym_export",
    "hb2_scoremap_create", "hb2_scoremap_destroy", "hb2_scoremap_device_ptr", "hb2_batch_scatter_scores",
    "hb2_scoremap_merge", "hb2_scoremap_topk", "hb2_scoremap_read", "hb2_scoremap_restore",
    "hb2_batch_set_real_rows", "hb2_batch_solve_model", "hb2_batch_model_info", "hb2_batch_apply_all",
    "hb2_batch_set_pixel_rows", "hb2_batch_score_metric",
]

_lib = None


def load():
    """Load the shared library (built by ``__graft_entry__.build()``); raise loudly if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise HeliconB200Error(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
            "helicon_b200 has no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    P = C.POINTER
    lib.hb2_last_error.restype = C.c_char_p
    lib.hb2_build_info.restype = C.c_char_p
    lib.hb2_device_count.restype = C.c_int
    lib.hb2_stream_create.argtypes = [C.c_int, P(vp)]
    lib.hb2_stream_destroy.argtypes = [C.c_int, vp]
    lib.hb2_device_trim.argtypes = [C.c_int]
    lib.hb2_problem_create.argtypes = [P(vp), vp, P(Geometry), C.c_int, vp]
    lib.hb2_problem_destroy.argtypes = [vp]
    lib.hb2_problem_destroy.restype = None
    lib.hb2_problem_ndisk.argtypes = [vp]
    lib.hb2_problem_rank_table.argtypes = [vp, vp]
    lib.hb2_batch_begin.argtypes = [P(vp), vp, i32, i32, i32, vp, vp, vp, vp]
    lib.hb2_batch_ray_valid.argtypes = [vp, vp]
    lib.hb2_batch_angle_map.argtypes = [vp, i32, vp]
    lib.hb2_batch_set_ties.argtypes = [vp, i32, i32, vp, vp, vp]
    lib.hb2_batch_add_exact_maps.argtypes = [vp, i32, vp, vp, vp]
    lib.hb2_batch_explicit_rows.argtypes = [vp, P(ExplicitGeometry), i32, vp, vp, vp, vp, i64, P(i32), vp, P(i64), P(i64)]
    lib.hb2_batch_explicit_sym_rows.argtypes = [vp, i32, vp, i64, P(i64)]
    lib.hb2_batch_explicit_sym_export.argtypes = [vp, vp, vp]
    lib.hb2_batch_explicit_pixel_mask.argtypes = [vp, vp]
    lib.hb2_batch_explicit_export.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.hb2_batch_set_pixel_masks.argtypes = [vp, i32, vp, vp]
    lib.hb2_batch_bilinear_maps.argtypes = [vp, i32, vp, i32, vp, vp, i32, vp, vp, vp]
    lib.hb2_batch_bilinear_ray_valid.argtypes = [vp, vp]
    lib.hb2_batch_bilinear_views.argtypes = [vp, i32, vp, vp, vp, i32, vp]
    lib.hb2_batch_bilinear_sym_rows.argtypes = [vp, i32, i32, vp, i64, P(i64)]
    lib.hb2_batch_bilinear_sym_export.argtypes = [vp, i32, vp, vp]
    lib.hb2_batch_create.argtypes = [vp, i32, vp, i32, vp, i32, vp, i32, vp]
    lib.hb2_batch_destroy.argtypes = [vp]
    lib.hb2_batch_destroy.restype = None
    lib.hb2_batch_sym_rows.argtypes = [vp, i32, P(i32), vp, vp, i64]
    lib.hb2_batch_sym_order.argtypes = [vp, i32, vp, i64]
    lib.hb2_batch_rows_padded.argtypes = [vp, i32, P(i64)]
    lib.hb2_batch_rows_padded.restype = i64
    lib.hb2_batch_rhs.argtypes = [vp, i32, vp]
    lib.hb2_batch_apply_forward.argtypes = [vp, i32, vp, vp]
    lib.hb2_batch_apply_adjoint.argtypes = [vp, i32, vp, vp]
    lib.hb2_batch_solve.argtypes = [vp, P(SolveOptions), vp]
    lib.hb2_batch_get_x.argtypes = [vp, i32, vp]
    lib.hb2_batch_timing.argtypes = [vp, vp]
    lib.hb2_batch_trf_trace.argtypes = [vp, i32, vp, i32]
    lib.hb2_batch_set_real_rows.argtypes = [vp, i32, vp, i64]
    lib.hb2_batch_solve_model.argtypes = [vp, P(ModelOptions), vp]
    lib.hb2_batch_model_info.argtypes = [vp, i32, vp]
    lib.hb2_batch_apply_all.argtypes = [vp, i32, vp, vp]
    lib.hb2_batch_set_pixel_rows.argtypes = [vp, i32, vp, i32, i32]
    lib.hb2_batch_score_metric.argtypes = [vp, i32, i32, vp, vp]
    lib.hb2_helical_symmetrize.argtypes = [vp, P(SymmParams), vp, vp, vp, vp, vp, vp, i32, vp, vp, vp, vp, C.c_int, vp]
    lib.hb2_lsmr_scalar_step.argtypes = [vp, C.c_int, C.c_float, C.c_float, f64, f64, f64, f64, C.c_int, P(C.c_float), P(C.c_float), P(C.c_float), vp]
    lib.hb2_scoremap_create.argtypes = [P(vp), i64, C.c_int]
    lib.hb2_scoremap_destroy.argtypes = [vp]
    lib.hb2_scoremap_destroy.restype = None
    lib.hb2_scoremap_device_ptr.argtypes = [vp]
    lib.hb2_scoremap_device_ptr.restype = vp
    lib.hb2_batch_scatter_scores.argtypes = [vp, vp, vp, vp]
    lib.hb2_scoremap_merge.argtypes = [vp, vp, i32, vp]
    lib.hb2_scoremap_restore.argtypes = [vp, i64, vp, vp, vp, vp]
    lib.hb2_scoremap_topk.argtypes = [vp, i32, vp, vp, vp]
    lib.hb2_scoremap_read.argtypes = [vp, vp, vp, vp, vp]
    _lib = lib
    return lib


def check(rc):
    if rc < 0:
        raise HeliconB200Error(f"helicon_b200 error {rc}: {load().hb2_last_error().decode()}")
    return rc


def require_gpu():
    lib = load()
    if lib.hb2_device_count() <= 0:
        raise HeliconB200Error("no CUDA device visible: helicon_b200 runs only on the GPU (no CPU fallback)")
    return lib


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)

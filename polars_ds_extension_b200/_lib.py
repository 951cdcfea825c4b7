"""ctypes bindings of libpds_b200 (include/pdsb.h).  The library is the product; this module only loads it.

There is no CPU fallback: if the shared library is missing or a CUDA device is not usable, calls raise.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "_polars_ds_b200.so"
_lib = None


class PdsbError(RuntimeError):
    """Error reported by libpds_b200 (message = pdsb_last_error())."""


class SolveOpts(C.Structure):
    _fields_ = [
        ("p", C.c_int), ("t", C.c_int), ("add_bias", C.c_int), ("method", C.c_int), ("solver", C.c_int),
        ("positive", C.c_int), ("max_iter", C.c_int), ("f32_gate", C.c_int),
        ("l1_reg", C.c_double), ("l2_reg", C.c_double), ("tol", C.c_double), ("singular_x_tol", C.c_double),
    ]


class Matrix(C.Structure):
    """pdsb_matrix: a host float64 view, strides in elements."""
    _fields_ = [("data", C.c_void_p), ("n_rows", C.c_int64), ("n_cols", C.c_int64),
                ("row_stride", C.c_int64), ("col_stride", C.c_int64)]


MODEL_LR, MODEL_ELASTIC_NET, MODEL_ONLINE_LR = range(3)
METHOD_LSTSQ, METHOD_CD, METHOD_NNLS, METHOD_RCOND, METHOD_INV = range(5)
SOLVER_QR, SOLVER_SVD, SOLVER_CHOLESKEY = range(3)
# enum pdsb_glm_family, by the names the reference's GLM class accepts (py_glm.rs / glm_solvers.rs GLMFamily::from)
GLM_FAMILIES = {"gaussian": 0, "normal": 0, "poisson": 1, "binomial": 2, "logistic": 2, "gamma": 3}


def lib() -> C.CDLL:
    """Load (once) the in-tree shared library; raise loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise PdsbError(
            f"{LIB_PATH} is missing: build it with `python -m polars_ds_extension_b200.build` "
            "(there is no CPU fallback)."
        )
    L = C.CDLL(str(LIB_PATH))
    vp, i64, dbl, ci = C.c_void_p, C.c_int64, C.c_double, C.c_int
    L.pdsb_last_error.restype = C.c_char_p
    L.pdsb_version.restype = ci
    L.pdsb_kernel_launch_count.restype = i64
    L.pdsb_last_moments_path.restype = ci
    L.pdsb_set_moments_path.argtypes = [ci]
    L.pdsb_student_t_sf.restype = dbl
    L.pdsb_student_t_sf.argtypes = [dbl, dbl]
    L.pdsb_student_t_ppf.restype = dbl
    L.pdsb_student_t_ppf.argtypes = [dbl, dbl]
    for sfx in ("f32", "f64"):
        getattr(L, f"pdsb_dev_moments_{sfx}").argtypes = [vp, i64, vp, i64, vp, vp, i64, ci, ci, vp, vp]
        getattr(L, f"pdsb_dev_predict_{sfx}").argtypes = [vp, i64, vp, i64, vp, vp, i64, ci, ci, ci, vp, vp, vp, vp,
                                                         i64, vp, vp, vp]
        getattr(L, f"pdsb_dev_grouped_lin_reg_{sfx}").argtypes = [vp, i64, vp, vp, i64, i64, ci, C.POINTER(SolveOpts),
                                                                 vp, vp, vp]
        getattr(L, f"pdsb_dev_online_lin_reg_{sfx}").argtypes = [vp, i64, vp, i64, ci, ci, i64, i64, ci, dbl, vp, vp,
                                                                vp, vp]
        getattr(L, f"pdsb_dev_recursive_shard_{sfx}").argtypes = [vp, i64, vp, i64, ci, ci, i64, ci, dbl, vp, i64, vp,
                                                                 vp, vp, vp]
        getattr(L, f"pdsb_dev_report_{sfx}").argtypes = [vp, i64, vp, vp, vp, i64, ci, ci, ci, dbl, vp, vp]
    L.pdsb_dev_solve.argtypes = [vp, C.POINTER(SolveOpts), vp, vp, vp, vp]
    L.pdsb_frame_elems.restype = C.c_size_t
    L.pdsb_frame_elems.argtypes = [i64, ci]
    L.pdsb_dev_frame_from_colmajor_f32.argtypes = [vp, i64, i64, ci, vp, vp]
    L.pdsb_dev_moments_frame_f32.argtypes = [vp, i64, ci, ci, ci, ci, ci, vp, vp, vp]
    L.pdsb_dev_predict_frame_f32.argtypes = [vp, i64, ci, ci, ci, ci, ci, ci, vp, vp, vp, vp, vp, i64, vp, vp, vp]
    L.pdsb_set_tc_variant.argtypes = [ci]
    mp = C.POINTER(Matrix)
    L.pdsb_model_fit.argtypes = [ci, mp, mp, ci, C.c_char_p, dbl, dbl, dbl, i64, vp, vp]
    L.pdsb_model_predict.argtypes = [mp, vp, ci, ci, vp]
    L.pdsb_glm_fit.argtypes = [mp, mp, ci, ci, i64, dbl, vp, vp]
    L.pdsb_glm_predict.argtypes = [mp, vp, ci, ci, ci, ci, vp]
    L.pdsb_dev_glm_f64.argtypes = [vp, i64, vp, i64, ci, ci, ci, i64, dbl, vp, vp, vp]
    L.pdsb_online_lr_new.restype = vp
    L.pdsb_online_lr_new.argtypes = [ci, ci]
    L.pdsb_online_lr_free.argtypes = [vp]
    L.pdsb_online_lr_free.restype = None
    L.pdsb_online_lr_set.argtypes = [vp, vp, vp]
    L.pdsb_online_lr_update.argtypes = [vp, vp, dbl, dbl]
    L.pdsb_online_lr_get.argtypes = [vp, vp, vp]
    L.pdsb_set_devices.argtypes = [C.POINTER(ci), ci]
    L.pdsb_comm_unique_id.argtypes = [vp]
    L.pdsb_comm_init_rank.argtypes = [ci, ci, vp]
    L.pdsb_comm_destroy.restype = None
    L.pdsb_dev_allreduce_f64.argtypes = [vp, i64, vp]
    L.pdsb_last_staged_bytes.restype = i64
    L.pdsb_plugin_live_results.restype = i64
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != 0:
        raise PdsbError(lib().pdsb_last_error().decode("utf-8", "replace"))

"""ctypes binding of include/sparselm_b200.h (the C-ABI drop-in boundary).

The library is loaded from sparselm_b200/lib (built in-tree by ``_build.build``).
There is no CPU fallback: if the shared object is missing or no CUDA device is
present, the functions below raise.
"""

from __future__ import annotations

import ctypes
import os

from . import _build

SLM_MAX_FOLDS = 16
SLM_STAT_MAX, SLM_STAT_MAPE, SLM_STAT_MEDIAN = 1 << 2, 1 << 3, 1 << 4

c_i32, c_i64, c_dbl, c_vp, c_sz = (
    ctypes.c_int32, ctypes.c_int64, ctypes.c_double, ctypes.c_void_p, ctypes.c_size_t,
)


class SlmBatch(ctypes.Structure):
    """Mirror of ``struct slm_batch``."""

    _fields_ = [
        ("n_folds", c_i32),
        ("n_groups", c_i32),
        ("p", c_i64),
        ("pa", c_i64),
        ("ldz", c_i64),
        ("G_dev", c_vp),
        ("g_stride", c_i64),
        ("gptr_dev", c_vp),
        ("K", c_i32 * SLM_MAX_FOLDS),
        ("n_obs", c_dbl * SLM_MAX_FOLDS),
        ("lipschitz", c_dbl * SLM_MAX_FOLDS),
        ("lam1_dev", c_vp),
        ("W1_dev", c_vp),
        ("W2_dev", c_vp),
        ("D2_dev", c_vp),
        ("B_dev", c_vp),
        ("skip_dev", c_vp),
        ("work_dev", c_vp),
        ("work_bytes", c_sz),
        ("tol", c_dbl),
        ("floor_rel", c_dbl),
        ("max_iter", c_i32),
        ("check_every", c_i32),
        ("gap_dev", c_vp),
        ("primal_dev", c_vp),
        ("n_iter_dev", c_vp),
        ("status_dev", c_vp),
        ("lipschitz_dev", c_vp),
        ("iters_run", c_i32),
        ("n_unconverged", c_i32),
        ("max_group", c_i32),
    ]


# every symbol include/sparselm_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "slm_version": (ctypes.c_int, []),
    "slm_create": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(c_vp)]),
    "slm_destroy": (None, [c_vp]),
    "slm_set_option": (ctypes.c_int, [c_vp, ctypes.c_char_p, ctypes.c_int]),
    "slm_last_error": (ctypes.c_char_p, [c_vp]),
    "slm_sm_count": (ctypes.c_int, [c_vp]),
    "slm_launch_count": (c_i64, [c_vp]),
    "slm_tma_launch_count": (c_i64, [c_vp]),
    "slm_timing_enable": (ctypes.c_int, [c_vp, ctypes.c_int]),
    "slm_timing_read": (ctypes.c_int, [c_vp, ctypes.c_int, ctypes.POINTER(c_dbl), ctypes.POINTER(c_i64), ctypes.POINTER(c_dbl)]),
    "slm_timing_reset": (ctypes.c_int, [c_vp]),
    "slm_padded_cols": (c_i64, [c_i64]),
    "slm_pack_design": (ctypes.c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp]),
    "slm_gram_blocks": (ctypes.c_int, [c_vp, c_vp, c_i64, ctypes.POINTER(c_i64), ctypes.c_int, c_vp, c_vp]),
    "slm_gram_block_add": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_vp]),
    "slm_gram_rows_update": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, ctypes.c_int, ctypes.POINTER(c_i64), c_vp, c_vp, c_i64,
                                            ctypes.c_int, ctypes.c_int, c_vp]),
    "slm_gram_complement": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int, c_i64, c_vp, c_vp]),
    "slm_tri_size": (c_i64, [c_i64]),
    "slm_tri_pack": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, ctypes.c_int, c_vp, c_vp]),
    "slm_tri_unpack": (ctypes.c_int, [c_vp, c_vp, c_i64, ctypes.c_int, c_vp, c_i64, c_vp]),
    "slm_tri_complement": (ctypes.c_int, [c_vp, c_vp, c_i64, ctypes.c_int, c_vp, c_i64, c_vp]),
    "slm_gram_allreduce": (ctypes.c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, ctypes.c_int, c_vp, c_vp]),
    "slm_allreduce_sum": (ctypes.c_int, [c_vp, c_vp, c_vp, c_i64, c_vp]),
    "slm_gather_results": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "slm_tma_probe": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_i32, c_i32, ctypes.POINTER(c_i32), c_vp, c_vp]),
    "slm_gram_center": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_vp]),
    "slm_gram_gather": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp]),
    "slm_lipschitz_workspace": (c_sz, [c_i64, ctypes.c_int]),
    "slm_lipschitz": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, ctypes.c_int, ctypes.c_int, c_vp, ctypes.POINTER(c_dbl), c_vp]),
    "slm_lipschitz_dev": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, ctypes.c_int, ctypes.c_int, c_vp, c_vp, c_vp]),
    "slm_solve_workspace": (c_sz, [c_i64, c_i64, ctypes.c_int, ctypes.c_int]),
    "slm_solve_batch": (ctypes.c_int, [c_vp, ctypes.POINTER(SlmBatch), c_vp]),
    "slm_adaptive_update": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_dbl, c_vp, c_vp, c_vp, c_vp]),
    "slm_fold_back": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i32, c_vp, c_vp]),
    "slm_cv_score": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_i64, c_vp, c_i64, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp]),
    "slm_cv_score_many": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp]),
    "slm_cv_score_rows": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp]),
    "slm_cv_score_stats": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32,
                                          c_i32, c_vp, c_vp, c_vp, c_vp]),
    "slm_support_counts": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int, c_i64, c_i64, ctypes.c_int, c_dbl, c_vp, c_vp, c_vp]),
    "slm_group_support_counts": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int, c_i64, c_i64, ctypes.c_int, c_dbl, c_vp, c_i32,
                                                c_vp, c_vp, c_vp]),
    "slm_gram_scale": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, ctypes.c_int, c_vp, c_i64, ctypes.POINTER(c_i64),
                                      c_vp]),
    "slm_intercepts": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_i32, c_vp, c_vp]),
    "slm_gram_apply": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, ctypes.c_int, ctypes.POINTER(c_i32), c_vp, c_i64, c_vp, c_vp]),
    "slm_newton_workspace": (c_sz, [c_i64, c_i32, c_i32, ctypes.c_int]),
    "slm_newton_step": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, ctypes.c_int, c_i32, ctypes.POINTER(c_i32), c_vp, c_vp,
                                       c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_sz, c_vp, c_vp]),
    "slm_newton_step_l1": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, ctypes.c_int, c_i32, ctypes.POINTER(c_i32), c_vp,
                                          c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_sz, c_vp, c_vp]),
    "slm_gram_cg_workspace": (c_sz, [c_i64]),
    "slm_gram_cg": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_dbl, c_i32, c_vp, c_sz, c_vp, ctypes.POINTER(c_i32), ctypes.POINTER(c_dbl), c_vp]),
    "slm_rowsparse_workspace": (c_sz, [c_i64, c_i64, ctypes.c_int]),
    "slm_gram_apply_rowsparse": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, ctypes.c_int, ctypes.POINTER(c_i32), c_vp, c_i64, c_vp, ctypes.c_int, c_vp, c_sz, c_vp]),
    "slm_apply_stats": (ctypes.c_int, [c_vp, ctypes.POINTER(c_dbl), ctypes.POINTER(c_dbl)]),
    "slm_group_whiten_factors": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "slm_gram_whiten": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_i32, c_vp, c_vp, c_dbl, c_vp, c_vp, c_vp]),
    "slm_coef_unwhiten": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i64, c_i32, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp]),
}

_lib = None


def lib_path() -> str:
    # SLM_B200_LIB: an alternative build of the same ABI (tuning variants); the default is the in-tree build
    return os.environ.get("SLM_B200_LIB") or _build.LIB_PATH


def load():
    """dlopen the engine and set prototypes. Raises if the .so is missing."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise RuntimeError(
            f"sparselm_b200 CUDA engine not built ({path} missing): run "
            "`python -c 'import __graft_entry__ as g; g.build()'` -- there is no CPU fallback"
        )
    lib = ctypes.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library diverge
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib

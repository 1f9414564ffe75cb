"""ctypes binding of libsco_b200.so (the C ABI of include/sco_b200.h).

There is no fallback: if the shared library is missing or cannot be loaded the
import of anything that needs the engine raises.
"""
import ctypes
import os

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SCO_B200_LIB", os.path.join(PKG, "libsco_b200.so"))  # override: A/B runs of two builds

MAX_BLOCKS = 16
MAX_GROUPS = 8
MAX_OBJ_BLOCKS = 4

c_i32, c_i64, c_dbl, c_vp = ctypes.c_int32, ctypes.c_int64, ctypes.c_double, ctypes.c_void_p


class CField(ctypes.Structure):
    _fields_ = [("off", c_i64), ("shared", c_i32), ("pad_", c_i32)]


class CBlock(ctypes.Structure):
    _fields_ = [("family", c_i32), ("cnt_type", c_i32), ("m", c_i32), ("group_mask", c_i32),
                ("jw", c_i32), ("n_in", c_i32), ("ipar", c_i32 * 8), ("par", CField), ("val", CField),
                ("cols", c_vp)]


class CObjBlock(ctypes.Structure):
    _fields_ = [("m", c_i32), ("n_in", c_i32), ("n_instr", c_i32), ("flags", c_i32), ("prog", CField),
                ("cols", c_vp)]


class CStructure(ctypes.Structure):
    _fields_ = [("n", c_i32), ("m_lin", c_i32), ("n_blocks", c_i32), ("n_groups", c_i32),
                ("stride", c_i64), ("shared_len", c_i64),
                ("Q", CField), ("q", CField), ("c", CField), ("lin_l", CField), ("lin_u", CField),
                ("lin_rowptr", c_vp), ("lin_col", c_vp), ("lin_val", c_vp), ("shared", c_vp),
                ("group_overlap", c_vp), ("blocks", CBlock * MAX_BLOCKS),
                ("obj_prog", CField), ("obj_prog_len", c_i32), ("obj_prog_flags", c_i32),
                ("qa", CField), ("lb0", CField), ("ub0", CField),
                ("n_obj_blocks", c_i32), ("obj_blocks", CObjBlock * MAX_OBJ_BLOCKS)]


class CBatchIO(ctypes.Structure):
    _fields_ = [("d_params", c_vp), ("d_x0", c_vp), ("d_x_out", c_vp), ("d_verdict", c_vp), ("d_merit", c_vp),
                ("d_objective", c_vp), ("d_max_vio", c_vp), ("d_stats", c_vp), ("d_nonconverged", c_vp),
                ("d_order", c_vp), ("d_x_warm", c_vp), ("d_y_warm", c_vp)]


class CSettings(ctypes.Structure):
    _fields_ = [
        ("improve_ratio_threshold", c_dbl), ("min_trust_region_size", c_dbl),
        ("min_approx_improve", c_dbl), ("trust_shrink_ratio", c_dbl), ("trust_expand_ratio", c_dbl),
        ("cnt_tolerance", c_dbl), ("merit_coeff_increase_ratio", c_dbl),
        ("initial_trust_region_size", c_dbl), ("initial_penalty_coeff", c_dbl),
        ("max_merit_coeff_increases", c_i32), ("max_sqp_iters", c_i32),
        ("osqp_eps_abs", c_dbl), ("osqp_eps_rel", c_dbl), ("osqp_rho", c_dbl), ("osqp_sigma", c_dbl),
        ("osqp_alpha", c_dbl), ("osqp_eps_prim_inf", c_dbl), ("osqp_eps_dual_inf", c_dbl),
        ("osqp_max_iter", c_i32), ("osqp_scaling", c_i32), ("osqp_check_termination", c_i32),
        ("osqp_adaptive_rho", c_i32), ("osqp_adaptive_rho_interval", c_i32),
        ("compound_penalty", c_i32), ("freeze_sparsity", c_i32), ("duplicate_rows", c_i32),
        ("threads_per_problem", c_i32), ("force_generic", c_i32), ("aff_obj_quirk", c_i32),
        ("warm_start", c_i32), ("pad_", c_i32),
    ]


EXPORTS = ["sco_last_error", "sco_default_settings", "sco_create", "sco_destroy", "sco_query",
           "sco_solve_batch", "sco_solve_batch_ordered", "sco_solve_batch_io", "sco_solve_batch_host",
           "sco_solve_batch_host_async", "sco_solve_batch_host_groups", "sco_convexify", "sco_convexify_model", "sco_qp_solve",
           "sco_qp_solve_w", "sco_merit", "sco_probe_fp64"]

_lib = None


def load():
    """Loads the shared library; raises if it is missing (no CPU fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "sco_py_b200: %s not found. Build it with `python -m sco_py_b200.build` (needs nvcc); "
            "the engine has no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    lib.sco_last_error.restype = ctypes.c_char_p
    lib.sco_default_settings.restype = None
    for name in EXPORTS[2:]:
        getattr(lib, name).restype = ctypes.c_int
    lib.sco_create.argtypes = [ctypes.POINTER(CStructure), ctypes.c_int, ctypes.POINTER(c_vp)]
    lib.sco_destroy.argtypes = [c_vp]
    lib.sco_query.argtypes = [c_vp, ctypes.POINTER(c_i64)]
    lib.sco_solve_batch.argtypes = [c_vp, c_i64, c_vp, c_vp, ctypes.POINTER(CSettings), c_vp, c_vp,
                                    c_vp, c_vp, c_vp, c_vp, c_vp]
    lib.sco_solve_batch_ordered.argtypes = [c_vp, c_i64, c_vp, c_vp, ctypes.POINTER(CSettings), c_vp, c_vp,
                                            c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]
    lib.sco_solve_batch_io.argtypes = [c_vp, c_i64, ctypes.POINTER(CBatchIO), ctypes.POINTER(CSettings), c_vp]
    lib.sco_solve_batch_host_groups.argtypes = [c_vp, c_i64, c_vp, c_vp, ctypes.POINTER(CSettings), c_vp,
                                                c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]
    lib.sco_qp_solve_w.argtypes = [c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                   ctypes.c_int, ctypes.c_int, ctypes.POINTER(CSettings), c_vp, c_vp,
                                   c_vp, c_vp]
    lib.sco_solve_batch_host.argtypes = [c_vp, c_i64, c_vp, c_vp, ctypes.POINTER(CSettings), c_vp,
                                         c_vp, c_vp, c_vp, c_vp, c_vp]
    lib.sco_solve_batch_host_async.argtypes = [c_vp, c_i64, c_vp, c_vp, ctypes.POINTER(CSettings), c_vp,
                                               c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]
    lib.sco_convexify.argtypes = [c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]
    lib.sco_convexify_model.argtypes = [c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]
    lib.sco_qp_solve.argtypes = [c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                 ctypes.c_int, ctypes.c_int, ctypes.POINTER(CSettings), c_vp, c_vp,
                                 c_vp, c_vp]
    lib.sco_merit.argtypes = [c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                              c_vp]
    lib.sco_probe_fp64.argtypes = [ctypes.c_int, ctypes.POINTER(c_dbl)]
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise RuntimeError("sco_b200 error %d: %s" % (rc, load().sco_last_error().decode()))

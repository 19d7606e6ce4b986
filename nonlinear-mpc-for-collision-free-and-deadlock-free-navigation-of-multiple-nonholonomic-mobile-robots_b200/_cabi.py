"""ctypes binding of libnmpc_b200.so (include/nmpc_b200.h).  No fallback: a missing library or a
missing CUDA device raises -- the product path never runs on the CPU."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "lib", "libnmpc_b200.so")      # built by __graft_entry__.build()
NSTATS = 11      # NMPC_NSTATS (the last column counts filter evictions)
NTRACE = 8
STATUS = {0: "SOLVED", 1: "ACCEPTABLE", 2: "MAX_ITER", 3: "INFEASIBLE", 4: "NUMERICAL"}
SYMBOLS = ["nmpc_default_opts", "nmpc_last_error", "nmpc_create", "nmpc_destroy", "nmpc_n", "nmpc_mg", "nmpc_np",
           "nmpc_nnz_jac", "nmpc_nnz_hess", "nmpc_workspace_bytes", "nmpc_workspace_bytes_batched_bounds", "nmpc_solve",
           "nmpc_solve_trace", "nmpc_solve_host", "nmpc_shift",
           "nmpc_plant", "nmpc_eval", "nmpc_jac_pattern", "nmpc_hess_pattern", "nmpc_launch_count", "nmpc_probe_fp64",
           "nmpc_debug_block_profile", "nmpc_set_order", "nmpc_create_obstacles", "nmpc_create_ocp",
           "nmpc_default_tuning", "nmpc_create_tuned", "nmpc_probe_dmma", "nmpc_create_moving_obstacles",
           "nmpc_create_tracking", "nmpc_create_tracking_obstacles", "nmpc_solution_vjp", "nmpc_solution_jvp",
           "nmpc_sensitivity_workspace_bytes"]


class Desc(C.Structure):
    _fields_ = [("Nr", C.c_int), ("N", C.c_int), ("T", C.c_double), ("Q", C.c_double * 3), ("R", C.c_double * 2)]


class Opts(C.Structure):
    _fields_ = [("tol", C.c_double), ("max_iter", C.c_int), ("acceptable_tol", C.c_double),
                ("acceptable_iter", C.c_int), ("acceptable_obj_change_tol", C.c_double),
                ("dual_inf_tol", C.c_double), ("constr_viol_tol", C.c_double), ("compl_inf_tol", C.c_double),
                ("mu_init", C.c_double), ("kappa_mu", C.c_double), ("theta_mu", C.c_double),
                ("barrier_tol_factor", C.c_double), ("tau_min", C.c_double), ("bound_push", C.c_double),
                ("bound_frac", C.c_double), ("bound_relax_factor", C.c_double),
                ("bound_mult_init_val", C.c_double), ("constr_mult_init_max", C.c_double),
                ("kappa_sigma", C.c_double), ("kappa_d", C.c_double), ("nlp_scaling_max_gradient", C.c_double),
                ("max_soc", C.c_int), ("max_resto_iter", C.c_int)]


class Tuning(C.Structure):
    """nmpc_tuning: launch tuning, no effect on results (include/nmpc_b200.h)."""
    _fields_ = [("convoy", C.c_int), ("ctas_per_sm", C.c_int), ("force_block_path", C.c_int), ("thread_min_batch", C.c_int)]


class NmpcError(RuntimeError):
    pass


_LIB = None


def lib():
    """Load libnmpc_b200.so and declare the prototypes of every symbol of include/nmpc_b200.h."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise NmpcError("libnmpc_b200.so is not built (run __graft_entry__.build()); there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    vp, dp, ip, H = C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p   # raw addresses (device or host)
    L.nmpc_default_opts.argtypes = [C.POINTER(Opts)]
    L.nmpc_default_opts.restype = None
    L.nmpc_last_error.restype = C.c_char_p
    L.nmpc_create.argtypes = [C.POINTER(Desc), C.POINTER(Opts), C.POINTER(H)]
    L.nmpc_create_obstacles.argtypes = [C.POINTER(Desc), C.POINTER(Opts), C.c_int, vp, C.POINTER(H)]
    L.nmpc_default_tuning.argtypes = [C.POINTER(Tuning)]
    L.nmpc_default_tuning.restype = None
    L.nmpc_create_tuned.argtypes = [C.POINTER(Desc), C.POINTER(Opts), C.POINTER(Tuning), C.c_int, vp, C.POINTER(H)]
    L.nmpc_create_moving_obstacles.argtypes = [C.POINTER(Desc), C.POINTER(Opts), C.POINTER(Tuning), C.c_int, C.POINTER(H)]
    L.nmpc_create_tracking.argtypes = [C.POINTER(Desc), C.POINTER(Opts), C.POINTER(Tuning), C.POINTER(H)]
    L.nmpc_create_tracking_obstacles.argtypes = [C.POINTER(Desc), C.POINTER(Opts), C.POINTER(Tuning), C.c_int, C.POINTER(H)]
    L.nmpc_create_ocp.argtypes = [C.c_int, C.c_int, C.c_double, C.c_int, C.POINTER(Opts), C.POINTER(H)]
    L.nmpc_destroy.argtypes = [H]
    L.nmpc_destroy.restype = None
    for fn in ("nmpc_n", "nmpc_mg", "nmpc_np", "nmpc_nnz_jac", "nmpc_nnz_hess"):
        getattr(L, fn).argtypes = [H]
    L.nmpc_workspace_bytes.argtypes = [H, C.c_int]
    L.nmpc_workspace_bytes.restype = C.c_size_t
    L.nmpc_workspace_bytes_batched_bounds.argtypes = [H, C.c_int]
    L.nmpc_workspace_bytes_batched_bounds.restype = C.c_size_t
    L.nmpc_solve.argtypes = [H, C.c_int] + [dp] * 6 + [C.c_int] + [dp] * 5 + [ip, ip, dp, vp, C.c_size_t, vp]
    L.nmpc_solve_trace.argtypes = [H, C.c_int] + [dp] * 6 + [C.c_int] + [dp] * 5 + [ip, ip, dp, dp, C.c_int, vp, C.c_size_t, vp]
    L.nmpc_solve_host.argtypes = [H, C.c_int] + [dp] * 6 + [C.c_int] + [dp] * 5 + [ip, ip, dp]
    L.nmpc_shift.argtypes = [H, C.c_int, dp, dp, vp]
    L.nmpc_plant.argtypes = [H, C.c_int, dp, dp, dp, vp]
    L.nmpc_eval.argtypes = [H, C.c_int] + [dp] * 8 + [vp]
    L.nmpc_jac_pattern.argtypes = [H, vp, vp]
    L.nmpc_hess_pattern.argtypes = [H, vp, vp]
    L.nmpc_launch_count.argtypes = [H]
    L.nmpc_probe_fp64.argtypes = [C.POINTER(C.c_double)]
    L.nmpc_debug_block_profile.argtypes = [C.POINTER(C.c_longlong), C.c_int]
    L.nmpc_set_order.argtypes = [H, vp, C.c_int]
    L.nmpc_solution_vjp.argtypes = [H, C.c_int] + [dp] * 8 + [C.c_int, dp, dp, ip, vp, C.c_size_t, vp]
    L.nmpc_solution_jvp.argtypes = [H, C.c_int] + [dp] * 8 + [C.c_int, dp, dp, ip, vp, C.c_size_t, vp]
    L.nmpc_sensitivity_workspace_bytes.argtypes = [H, C.c_int, C.c_int]
    L.nmpc_sensitivity_workspace_bytes.restype = C.c_size_t
    L.nmpc_probe_dmma.argtypes = [C.POINTER(C.c_double)]
    L.nmpc_launch_count.restype = C.c_longlong
    _LIB = L
    return L


def check(rc):
    if rc != 0:
        raise NmpcError("nmpc error %d: %s" % (rc, lib().nmpc_last_error().decode()))


def default_tuning(**kw):
    t = Tuning()
    lib().nmpc_default_tuning(C.byref(t))
    for k, v in kw.items():
        if k not in {f[0] for f in Tuning._fields_}:
            raise ValueError("unknown tuning key %r" % (k,))
        setattr(t, k, int(v))
    return t


def default_opts(**kw):
    o = Opts()
    lib().nmpc_default_opts(C.byref(o))
    names = {f[0] for f in Opts._fields_}
    for k, v in kw.items():
        if k in names:
            setattr(o, k, v)
    return o

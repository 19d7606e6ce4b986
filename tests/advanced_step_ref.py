"""References for advanced-step NMPC (nmpc_solution_x0_jacobian / nmpc_advanced_step) -- TEST INFRASTRUCTURE ONLY.

* emu_sens_x0: the product's WarpSolver::sensitivity_x0 through the CPU fibre emulation (tests/emul/emul_sens_x0.cpp, built
  into a temporary directory; nothing is written into the tree).
* advanced_step: the feedback correction in NumPy, as include/nmpc_b200.h states it.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from oracle.oracle_lib import Desc, Opts, lib as _orc_lib
from tests import sensitivity_ref as SR
from tests.tracking_ref import TrackingNLP

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_TMP = None
_LIBS = {}


def _emul_lib(tracking):
    global _TMP
    key = bool(tracking)
    if key in _LIBS:
        return _LIBS[key]
    if _TMP is None:
        _TMP = tempfile.mkdtemp(prefix="nmpc_sens_x0_")
    so = os.path.join(_TMP, "libnmpc_emul_sens_x0_%d.so" % int(key))
    subprocess.check_call(["g++", "-O2", "-mavx2", "-mfma", "-fPIC", "-shared", "-std=c++17", "-x", "c++", "-Wno-unknown-pragmas",
                           "-DSENS_TRK=%d" % int(key), "-I" + os.path.join(_ROOT, "tests", "emul"), "-I" + SR._PKG_CSRC,
                           "-I" + os.path.join(_ROOT, "include"), "-o", so, os.path.join(_ROOT, "tests", "emul", "emul_sens_x0.cpp"),
                           "-lm"])
    L = C.CDLL(so)
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
    L.emu_sens_x0.argtypes = [C.POINTER(Desc), C.POINTER(Opts), C.c_int] + [dp] * 8 + [C.c_int, dp, ip, C.c_int]
    _LIBS[key] = L
    return L


def emu_sens_x0(nlp, x, lam_x, lam_g, p, bounds, lane_rev=0, **opts):
    """Batched as sensitivity_ref.emu_sens; returns (jac [B, 3Nr, n], status, rc)."""
    L = _emul_lib(isinstance(nlp, TrackingNLP))
    f64 = lambda a: np.ascontiguousarray(np.atleast_2d(np.asarray(a, dtype=np.float64)))
    x, lam_x, lam_g, p = map(f64, (x, lam_x, lam_g, p))
    lbx, ubx, lbg, ubg = (np.ascontiguousarray(np.asarray(b, np.float64)) for b in bounds)
    B, ns = x.shape[0], 3 * nlp.Nr
    d = Desc(nlp.Nr, nlp.N, nlp.T, (C.c_double * 3)(*nlp.Q), (C.c_double * 2)(*nlp.R))
    o = Opts()
    _orc_lib().orc_default_opts(C.byref(o))
    for k, v in opts.items():
        setattr(o, k, v)
    jac = np.full((B, ns, nlp.n), -7.0)
    st = np.full(B, -99, np.int32)
    dptr = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    rc = L.emu_sens_x0(C.byref(d), C.byref(o), B, dptr(x), dptr(lam_x), dptr(lam_g), dptr(p), dptr(lbx), dptr(ubx), dptr(lbg),
                       dptr(ubg), 1 if lbx.ndim == 2 else 0, dptr(jac), st.ctypes.data_as(C.POINTER(C.c_int)), int(lane_rev))
    return jac, st, rc


def advanced_step(x, jac, status, p, x0m, lbx, ubx):
    """x_corr = x + jac' (x0m - p[:, :ns]) summed over j in order, clamped into [min(lb, x), max(ub, x)] where a bound is finite;
    X_0 = x0m; instances with status != 0 keep x."""
    x, jac, p, x0m = (np.asarray(a, np.float64) for a in (x, jac, p, x0m))
    B, ns, n = jac.shape
    lbx, ubx = np.broadcast_to(lbx, (B, n)), np.broadcast_to(ubx, (B, n))
    dlt = x0m - p[:, :ns]
    s = np.zeros((B, n))
    for j in range(ns):
        s = s + jac[:, j] * dlt[:, j:j + 1]
    xc = x + s
    xc = np.where(np.isfinite(lbx), np.maximum(xc, np.minimum(lbx, x)), xc)
    xc = np.where(np.isfinite(ubx), np.minimum(xc, np.maximum(ubx, x)), xc)
    xc = np.where((np.asarray(status) != 0)[:, None], x, xc)
    xc[:, :ns] = x0m
    return xc

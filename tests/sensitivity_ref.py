"""References for the parametric sensitivities (nmpc_solution_vjp / nmpc_solution_jvp) -- TEST INFRASTRUCTURE ONLY.

* sigma_vjp / sigma_jvp: the dense Sigma-condensed KKT solve in NumPy float64, from the NLP restatements (hess_lag, jac_g) and
  the interior-point weights rebuilt from a returned point, as include/nmpc_b200.h states them:
      K = [[W + Sx, J'], [J, -Ss^-1]],   reverse: K [a; b] = [x_bar; 0],  p_bar = -Lxp' a - Gp' b
                                         forward: K [x_dot; .] = -[Lxp p_dot; Gp p_dot]
  with Lxp = d(grad f)/dp and Gp = dg/dp (both exact: grad f and g are affine in p).
* refined_solve (refined=True): the same system unreduced, with iterative refinement -- the accurate answer where large
  weights cost the condensed solve digits.
* active_vjp / active_jvp: the active-set implicit-function derivative (active bounds fixed, active rows as equalities).
* emu_sens: the product's WarpSolver::sensitivity through the CPU fibre emulation (tests/emul/emul_sens.cpp, built into a
  temporary directory; nothing is written into the tree).
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from oracle.nlp_numpy import UnicycleNLP
from oracle.oracle_lib import Desc, Opts, lib as _orc_lib
from tests.tracking_ref import TrackingNLP

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_PKG_CSRC = os.path.join(_ROOT, "nonlinear-mpc-for-collision-free-and-deadlock-free-navigation-of-multiple-nonholonomic-mobile-robots_b200",
                         "csrc")
_TMP = None
_LIBS = {}


def nlp_for(Nr, N, T, tracking, Q=(1.0, 5.0, 0.1), R=(0.5, 0.05)):
    return (TrackingNLP if tracking else UnicycleNLP)(Nr, N, T, Q, R)


def n_params(nlp):
    return nlp.ns + nlp.N * (nlp.ns + nlp.nc) if isinstance(nlp, TrackingNLP) else 2 * nlp.ns


def param_jacobians(nlp):
    """(Lxp [n, np], Gp [mg, np]) = (d grad f / dp, dg / dp)."""
    ns, nc, N = nlp.ns, nlp.nc, nlp.N
    Lxp, Gp = np.zeros((nlp.n, n_params(nlp))), np.zeros((nlp.mg, n_params(nlp)))
    Gp[:ns, :ns] = -np.eye(ns)
    for k in range(N):
        for i in range(nlp.Nr):
            for c in range(3):
                col = ns + k * (ns + nc) + 3 * i + c if isinstance(nlp, TrackingNLP) else ns + 3 * i + c
                Lxp[nlp.ix(k, i, c), col] = -2.0 * nlp.Q[c]
            if isinstance(nlp, TrackingNLP):
                for c in range(2):
                    Lxp[nlp.iu(k, i, c), ns + k * (ns + nc) + ns + 2 * i + c] = -2.0 * nlp.R[c]
    return Lxp, Gp


def _relax(b, f, sign):
    return b + sign * f * np.maximum(1.0, np.abs(b))


def _weights(v, lam, lo, hi, relax):
    """|lam| / distance to the relaxed bound it pushes against (0 without a finite bound on that side)."""
    fl, fu = np.isfinite(lo), np.isfinite(hi)
    dl = np.where(fl, v - _relax(np.where(fl, lo, 0.0), relax, -1), 1.0)
    du = np.where(fu, _relax(np.where(fu, hi, 0.0), relax, 1) - v, 1.0)
    return np.where(fl, np.maximum(-lam, 0.0) / dl, 0.0) + np.where(fu, np.maximum(lam, 0.0) / du, 0.0)


def _rows(nlp, lbg, ubg):
    dummy = np.zeros(nlp.mg, bool)
    dummy[nlp.ns:nlp.blk] = True
    eq = (lbg == ubg) & ~dummy
    ineq = ~eq & ~dummy & (np.isfinite(lbg) | np.isfinite(ubg))
    return eq, ineq


def kkt_parts(nlp, x, lam_x, lam_g, p, lbx, ubx, lbg, ubg, relax=1e-8):
    W = nlp.hess_lag(x, p, lam_g)
    J = nlp.jac_g(x, p)
    eq, ineq = _rows(nlp, lbg, ubg)
    Sx = _weights(x, lam_x, lbx, ubx, relax)
    Ss = np.where(ineq, _weights(nlp.g(x, p), lam_g, lbg, ubg, relax), 0.0)
    return W, J, Sx, Ss, eq, ineq


def sigma_solve(parts, rx, rg):
    """K [dx; y] = [rx; rg] for K = [[W + Sx, J'], [J, -Ss^-1]] on the equality and inequality rows (Ss = 0: y = 0)."""
    W, J, Sx, Ss, eq, ineq = parts
    JE, JI = J[eq], J[ineq]
    H = W + np.diag(Sx) + JI.T @ (Ss[ineq][:, None] * JI)
    r = rx + JI.T @ (Ss[ineq] * rg[ineq])
    nE = JE.shape[0]
    K = np.block([[H, JE.T], [JE, np.zeros((nE, nE))]])
    sol = np.linalg.solve(K, np.concatenate([r, rg[eq]]))
    dx = sol[: H.shape[0]]
    y = np.zeros(J.shape[0])
    y[eq] = sol[H.shape[0]:]
    y[ineq] = Ss[ineq] * (JI @ dx - rg[ineq])
    return dx, y


def refined_solve(parts, rx, rg, steps=3):
    """The same system, unreduced ([[W + Sx, JE', JI'], [JE, 0, 0], [JI, 0, -Ss^-1]] on the rows with Ss > 0) and improved by
    iterative refinement: accurate where the condensed form loses digits (weights Ss, Sx of 1e10..1e12 on active rows and
    bounds, condensed into the Hessian as Ss JI'JI)."""
    W, J, Sx, Ss, eq, ineq = parts
    act = ineq & (Ss > 0)
    JE, JI = J[eq], J[act]
    n, mE, mI = W.shape[0], JE.shape[0], JI.shape[0]
    K = np.block([[W + np.diag(Sx), JE.T, JI.T], [JE, np.zeros((mE, mE)), np.zeros((mE, mI))],
                  [JI, np.zeros((mI, mE)), -np.diag(1.0 / Ss[act])]])
    rhs = np.concatenate([rx, rg[eq], rg[act]])
    sol = np.linalg.solve(K, rhs)
    for _ in range(steps):
        sol += np.linalg.solve(K, rhs - K @ sol)
    y = np.zeros(J.shape[0])
    y[eq], y[act] = sol[n: n + mE], sol[n + mE:]
    return sol[:n], y


def max_weight(parts):
    """Largest interior-point weight of the point (Sx or Ss): the conditioning of the condensed factorisation."""
    return float(max(parts[2].max(initial=0.0), parts[3].max(initial=0.0)))


def reduced_hessian_min_eig(parts):
    """Smallest eigenvalue of the condensed Hessian on the null space of the equality rows (> 0: the inertia is right)."""
    W, J, Sx, Ss, eq, ineq = parts
    JI = J[ineq]
    H = W + np.diag(Sx) + JI.T @ (Ss[ineq][:, None] * JI)
    _, s, vt = np.linalg.svd(J[eq])
    Z = vt[int(np.sum(s > 1e-12 * s.max())):].T
    return float(np.linalg.eigvalsh(Z.T @ H @ Z).min())


def sigma_vjp(nlp, sol, p, bounds, x_bar, relax=1e-8, refined=False):
    """refined: the unreduced system with iterative refinement (refined_solve) instead of the condensed dense solve."""
    parts = kkt_parts(nlp, sol["x"], sol["lam_x"], sol["lam_g"], p, *bounds, relax=relax)
    Lxp, Gp = param_jacobians(nlp)
    a, b = (refined_solve if refined else sigma_solve)(parts, np.asarray(x_bar, float), np.zeros(nlp.mg))
    return -Lxp.T @ a - Gp.T @ b


def sigma_jvp(nlp, sol, p, bounds, p_dot, relax=1e-8, refined=False):
    parts = kkt_parts(nlp, sol["x"], sol["lam_x"], sol["lam_g"], p, *bounds, relax=relax)
    Lxp, Gp = param_jacobians(nlp)
    return (refined_solve if refined else sigma_solve)(parts, -Lxp @ p_dot, -Gp @ p_dot)[0]


def _active_system(nlp, sol, p, bounds, thr):
    lbx, ubx, lbg, ubg = bounds
    x, lam_x, lam_g = sol["x"], sol["lam_x"], sol["lam_g"]
    eq, ineq = _rows(nlp, lbg, ubg)
    rows = eq | (ineq & (np.abs(lam_g) > thr))
    fixed = np.abs(lam_x) > thr
    W, J = nlp.hess_lag(x, p, lam_g), nlp.jac_g(x, p)
    A = np.vstack([J[rows], np.eye(nlp.n)[fixed]])
    m = A.shape[0]
    return np.block([[W, A.T], [A, np.zeros((m, m))]]), rows, fixed


def active_jvp(nlp, sol, p, bounds, p_dot, thr=1e-6):
    K, rows, fixed = _active_system(nlp, sol, p, bounds, thr)
    Lxp, Gp = param_jacobians(nlp)
    rhs = np.concatenate([-Lxp @ p_dot, -(Gp @ p_dot)[rows], np.zeros(int(fixed.sum()))])
    return np.linalg.solve(K, rhs)[: nlp.n]


def active_vjp(nlp, sol, p, bounds, x_bar, thr=1e-6):
    K, rows, fixed = _active_system(nlp, sol, p, bounds, thr)
    Lxp, Gp = param_jacobians(nlp)
    s = np.linalg.solve(K, np.concatenate([x_bar, np.zeros(K.shape[0] - nlp.n)]))
    return -Lxp.T @ s[: nlp.n] - Gp[rows].T @ s[nlp.n: nlp.n + int(rows.sum())]


def strict_active_set(nlp, sol, p, bounds, thr=1e-4, relax=1e-8):
    """Every finite bound of every variable and inequality row is clearly active (|lam| > thr) or clearly inactive
    (distance > thr): the active set does not change under small perturbations of p."""
    lbx, ubx, lbg, ubg = bounds
    eq, ineq = _rows(nlp, lbg, ubg)

    def ok(v, lam, lo, hi):
        for b, side, lm in ((lo, -1, np.maximum(-lam, 0.0)), (hi, 1, np.maximum(lam, 0.0))):
            f = np.isfinite(b)
            gap = np.where(f, side * (_relax(np.where(f, b, 0.0), relax, side) - v), np.inf)
            if np.any(f & (lm <= thr) & (gap <= thr)):
                return False
        return True
    g = nlp.g(sol["x"], p)
    return ok(sol["x"], sol["lam_x"], lbx, ubx) and ok(g[ineq], sol["lam_g"][ineq], lbg[ineq], ubg[ineq])


# ---- the emulated device pass ---------------------------------------------------------------------------------------------
def _emul_lib(tracking):
    global _TMP
    key = bool(tracking)
    if key in _LIBS:
        return _LIBS[key]
    if _TMP is None:
        _TMP = tempfile.mkdtemp(prefix="nmpc_sens_")
    so = os.path.join(_TMP, "libnmpc_emul_sens_%d.so" % int(key))
    subprocess.check_call(["g++", "-O2", "-mavx2", "-mfma", "-fPIC", "-shared", "-std=c++17", "-x", "c++", "-Wno-unknown-pragmas",
                           "-DSENS_TRK=%d" % int(key), "-I" + os.path.join(_ROOT, "tests", "emul"), "-I" + _PKG_CSRC,
                           "-I" + os.path.join(_ROOT, "include"), "-o", so, os.path.join(_ROOT, "tests", "emul", "emul_sens.cpp"), "-lm"])
    L = C.CDLL(so)
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
    L.emu_sens.argtypes = [C.POINTER(Desc), C.POINTER(Opts), C.c_int] + [dp] * 8 + [C.c_int, dp, dp, ip, C.c_int, C.c_int]
    _LIBS[key] = L
    return L


def emu_sens(nlp, x, lam_x, lam_g, p, bounds, seed, reverse, lane_rev=0, **opts):
    """Batched: x, lam_x [B, n], lam_g [B, mg], p [B, np], seed [B, n] (reverse) or [B, np]; bounds shared ([n] / [mg]) or
    per instance ([B, .]).  Returns (out, status, rc)."""
    tracking = isinstance(nlp, TrackingNLP)
    L = _emul_lib(tracking)
    f64 = lambda a: np.ascontiguousarray(np.atleast_2d(np.asarray(a, dtype=np.float64)))
    x, lam_x, lam_g, p, seed = map(f64, (x, lam_x, lam_g, p, seed))
    lbx, ubx, lbg, ubg = (np.ascontiguousarray(np.asarray(b, np.float64)) for b in bounds)
    B = x.shape[0]
    d = Desc(nlp.Nr, nlp.N, nlp.T, (C.c_double * 3)(*nlp.Q), (C.c_double * 2)(*nlp.R))
    o = Opts()
    _orc_lib().orc_default_opts(C.byref(o))
    for k, v in opts.items():
        setattr(o, k, v)
    out = np.full((B, n_params(nlp) if reverse else nlp.n), -7.0)
    st = np.full(B, -99, np.int32)
    dptr = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    rc = L.emu_sens(C.byref(d), C.byref(o), B, dptr(x), dptr(lam_x), dptr(lam_g), dptr(p), dptr(lbx), dptr(ubx), dptr(lbg),
                    dptr(ubg), 1 if lbx.ndim == 2 else 0, dptr(seed), dptr(out), st.ctypes.data_as(C.POINTER(C.c_int)),
                    int(reverse), int(lane_rev))
    return out, st, rc

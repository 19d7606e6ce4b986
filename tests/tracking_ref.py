"""Trajectory-tracking references for tests/test_tracking.py -- TEST INFRASTRUCTURE ONLY.

The references of the centralized family minimise the distance to one setpoint xs (p = [x0bar; xs]).  The tracking variant
(p = [x0bar; Z], Z [N][5 Nr], Z[k] = [xr_k; ur_k], cost sum_k (X_k - xr_k)'Q(X_k - xr_k) + (U_k - ur_k)'R(U_k - ur_k)) is
derived from them here, so that it runs the very same restated IPOPT and the very same device source:
  * TrackingOracle: oracle/nmpc_oracle.c compiled with the cost and its gradient reading Z[k] of the instance's p;
  * tracking_emu_solve: tests/emul/emul_solver.cpp compiled with the tracking instantiation of the product's warp solver;
  * TrackingNLP: oracle/nlp_numpy.py's NumPy restatement with f / grad_f on Z (the SLSQP check).
The sources are rewritten by exact substitutions that must each match, and compiled into a temporary directory (nothing is
written into the tree); a change of the underlying source that breaks a substitution fails the tests loudly.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
from scipy.optimize import minimize

from oracle import oracle_lib
from oracle.nlp_numpy import UnicycleNLP

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_PKG_CSRC = os.path.join(_ROOT, "nonlinear-mpc-for-collision-free-and-deadlock-free-navigation-of-multiple-nonholonomic-mobile-robots_b200",
                         "csrc")
_TMP = None
_LIBS = {}

# oracle: xs (= p + ns) is read at stage k as xs + k nz, and the controls are measured from ur_k = xs + k nz + ns
_XR, _XRD = "xs[(size_t)k * D.nz + 3 * i + c]", "xs[(size_t)k * D->nz + 3 * i + c]"
_UR, _URD = "xs[(size_t)k * D.nz + D.ns + 2 * i + c]", "xs[(size_t)k * D->nz + D->ns + 2 * i + c]"
_ORACLE_SUBS = [
    # orc_eval
    ("double e = w[IX(&D, k, i, c)] - xs[3 * i + c];", "double e = w[IX(&D, k, i, c)] - %s;" % _XR, 1),
    ("double u = w[IU(&D, k, i, c)];", "double u = w[IU(&D, k, i, c)] - %s;" % _UR, 1),
    # eval_obj
    ("double e = zk[3 * i + c] - xs[3 * i + c]; acc += D->Q[c] * e * e;",
     "double e = zk[3 * i + c] - %s; acc += D->Q[c] * e * e;" % _XRD, 1),
    ("double u = zk[D->ns + 2 * i + c]; acc += D->R[c] * u * u;",
     "double u = zk[D->ns + 2 * i + c] - %s; acc += D->R[c] * u * u;" % _URD, 1),
    # eval_grad
    ("gk[3 * i + c] = 2 * D->Q[c] * (zk[3 * i + c] - xs[3 * i + c]);", "gk[3 * i + c] = 2 * D->Q[c] * (zk[3 * i + c] - %s);" % _XRD, 1),
    ("gk[D->ns + 2 * i + c] = 2 * D->R[c] * zk[D->ns + 2 * i + c];",
     "gk[D->ns + 2 * i + c] = 2 * D->R[c] * (zk[D->ns + 2 * i + c] - %s);" % _URD, 1),
    # orc_solve_batch: the stride of p
    ("np = 6 * d->Nr;", "np = 3 * d->Nr + 5 * d->Nr * d->N;", 1),
]
# emulation: the product's tracking instantiation and parameter block
_EMU_SUBS = [
    ("    WarpSolver<NR> s(*job.P, job.sm, job.ws);", "    WarpSolver<NR, false, true> s(*job.P, job.sm, job.ws);", 1),
    ("WarpSolver<NR, NR <= 4>::", "WarpSolver<NR, false, true>::", 2),
    ("P.nobs = nobs; P.family = family; P.obs = obs;",
     "P.nobs = nobs; P.family = family; P.obs = obs; P.np = 3 * Nr + 5 * Nr * N;", 1),
]


def _rewrite(src, subs, dst):
    s = open(src).read()
    for a, b, n in subs:
        if s.count(a) != n:
            raise RuntimeError("%s: expected %d occurrence(s) of %r, found %d" % (src, n, a, s.count(a)))
        s = s.replace(a, b)
    with open(dst, "w") as fh:
        fh.write(s)


def _build(kind):
    global _TMP
    if kind in _LIBS:
        return _LIBS[kind]
    if _TMP is None:
        _TMP = tempfile.mkdtemp(prefix="nmpc_tracking_")
    if kind == "oracle":
        src = os.path.join(_TMP, "nmpc_oracle_tracking.c")
        _rewrite(os.path.join(_ROOT, "oracle", "nmpc_oracle.c"), _ORACLE_SUBS, src)
        so = os.path.join(_TMP, "liboracle_tracking.so")
        cmd = ["gcc", "-O3", "-mavx2", "-mfma", "-fopenmp", "-fPIC", "-Wall", "-Wno-unused-variable", "-std=gnu11",
               "-I" + os.path.join(_ROOT, "oracle"), "-shared", "-o", so, src, "-lm"]
        ref = oracle_lib.lib()
    else:
        src = os.path.join(_TMP, "emul_solver_tracking.cpp")
        _rewrite(os.path.join(_ROOT, "tests", "emul", "emul_solver.cpp"), _EMU_SUBS, src)
        so = os.path.join(_TMP, "libnmpc_emul_tracking.so")
        cmd = ["g++", "-O2", "-mavx2", "-mfma", "-fPIC", "-shared", "-std=c++17", "-x", "c++", "-Wno-unknown-pragmas",
               "-I" + os.path.join(_ROOT, "tests", "emul"), "-I" + _PKG_CSRC, "-I" + os.path.join(_ROOT, "include"),
               "-o", so, src, "-lm"]
        from tests.emul import emul_lib
        ref = emul_lib.lib()
    subprocess.check_call(cmd)
    L = C.CDLL(so)
    for name in dir(ref):      # same prototypes as the unmodified library
        if name.startswith(("orc_", "emu_")):
            fn = getattr(ref, name)
            getattr(L, name).argtypes, getattr(L, name).restype = fn.argtypes, fn.restype
    _LIBS[kind] = L
    return L


class TrackingOracle(oracle_lib.Oracle):
    """The C oracle tracking p = [x0bar; Z[N][5 Nr]] (np = 3 Nr + 5 Nr N)."""

    def __init__(self, Nr, N, T, **kw):
        super().__init__(Nr, N, T, **kw)
        self.L = _build("oracle")
        self.np_ = 3 * self.Nr + 5 * self.Nr * self.N


def tracking_emu_solve(monkeypatch, Nr, N, T, x0, p, lbx, ubx, lbg, ubg, **kw):
    """tests.emul.emul_lib.emu_solve on the emulation built with the tracking instantiation."""
    from tests.emul import emul_lib
    monkeypatch.setattr(emul_lib, "_LIB", _build("emul"))
    return emul_lib.emu_solve(Nr, N, T, x0, p, lbx, ubx, lbg, ubg, **kw)


def constant_reference(N, xs):
    """Z = [xs; 0] at every stage: [..., N * 5 Nr] from xs [..., 3 Nr]."""
    xs = np.asarray(xs, float)
    Z = np.concatenate([xs, np.zeros(xs.shape[:-1] + (2 * xs.shape[-1] // 3,))], axis=-1)
    return np.tile(Z, N) if Z.ndim == 1 else np.tile(Z, (1, N))


class TrackingNLP(UnicycleNLP):
    """UnicycleNLP with the tracking cost: p = [x0bar; Z], Z[k] = [xr_k; ur_k]."""

    def ref(self, p):
        Z = np.asarray(p, float).reshape(-1)[self.ns:].reshape(self.N, self.ns + self.nc)
        return Z[:, :self.ns].reshape(self.N, self.Nr, 3), Z[:, self.ns:].reshape(self.N, self.Nr, 2)

    def f(self, w, p):
        X, U = self.split(w)
        xr, ur = self.ref(p)
        e, eu = X[: self.N] - xr, U - ur
        return float(np.sum(self.Q * e * e) + np.sum(self.R * eu * eu))

    def grad_f(self, w, p):
        X, U = self.split(w)
        xr, ur = self.ref(p)
        gX = np.zeros_like(X)
        gX[: self.N] = 2.0 * self.Q * (X[: self.N] - xr)
        gU = 2.0 * self.R * (U - ur)
        return np.concatenate([gX.reshape(-1), gU.reshape(-1)])

    def solve_slsqp(self, w0, p, lbx, ubx, lbg, ubg, tol=1e-12, maxiter=2000):
        """Independent solve: SLSQP on the same functions, equality rows (lbg == ubg) and one-sided inequality rows."""
        eq = np.where(lbg == ubg)[0]
        lo = np.where((lbg > -np.inf) & (lbg != ubg))[0]
        cons = [{"type": "eq", "fun": lambda w: self.g(w, p)[eq] - lbg[eq], "jac": lambda w: self.jac_g(w, p)[eq]}]
        if lo.size:
            cons.append({"type": "ineq", "fun": lambda w: self.g(w, p)[lo] - lbg[lo], "jac": lambda w: self.jac_g(w, p)[lo]})
        lb = np.where(np.isfinite(lbx), lbx, None)
        ub = np.where(np.isfinite(ubx), ubx, None)
        return minimize(lambda w: self.f(w, p), w0, jac=lambda w: self.grad_f(w, p), method="SLSQP", constraints=cons,
                        bounds=list(zip(lb, ub)), options={"ftol": tol, "maxiter": maxiter})


def line_reference(start, goal, N, T, steps=0, speed=0.15):
    """A feasible time-parameterised reference for robots driving straight from start to goal ([3 Nr] each, heading along the
    line) at `speed` (< v_max) and stopping there: rows [xr_t; ur_t] for t = 0..steps + N - 1, [steps + N, 5 Nr].  Each robot's
    heading is the line's and ur_t = ((s_{t+1} - s_t) / T, 0) for the arc length s_t, so the rows obey the Euler dynamics."""
    start, goal = np.asarray(start, float).reshape(-1, 3), np.asarray(goal, float).reshape(-1, 3)
    Nr, H = start.shape[0], steps + N
    d = goal[:, :2] - start[:, :2]
    L = np.linalg.norm(d, axis=1)
    head = np.arctan2(d[:, 1], d[:, 0])
    s_all = np.minimum(speed * np.arange(H + 1)[:, None] * T, L[None])                   # [H + 1, Nr]
    s = s_all[:H]
    xr = np.stack([start[None, :, 0] + s * np.cos(head)[None], start[None, :, 1] + s * np.sin(head)[None],
                   np.broadcast_to(head[None], s.shape)], axis=-1)
    ur = np.stack([np.diff(s_all, axis=0) / T, np.zeros_like(s)], axis=-1)
    return np.concatenate([xr.reshape(H, 3 * Nr), ur.reshape(H, 2 * Nr)], axis=1)


def rotation_reference(start, N, T, steps=0, omega=0.2, turn=np.pi):
    """Robots on a circle about the origin (start [3 Nr]: their positions; headings are replaced by the tangent) rotating the
    formation at the angular rate omega until it has turned by `turn`, then holding: rows [xr_t; ur_t], [steps + N, 5 Nr].
    While it turns, ur = (r omega, omega) for a robot at radius r; the last partial step and the hold use the rate that ends
    exactly at `turn`, and 0 afterwards."""
    start = np.asarray(start, float).reshape(-1, 3)
    Nr, H = start.shape[0], steps + N
    r = np.hypot(start[:, 0], start[:, 1])
    a0 = np.arctan2(start[:, 1], start[:, 0])
    sgn = np.sign(omega) if omega != 0 else 1.0
    ang = np.minimum(abs(omega) * np.arange(H + 1) * T, turn)[:, None] * sgn             # [H + 1, 1]
    a = a0[None] + ang[:H]
    xr = np.stack([r[None] * np.cos(a), r[None] * np.sin(a), a + sgn * np.pi / 2], axis=-1)
    w = np.diff(ang, axis=0) / T                                                           # [H, 1]
    ur = np.stack([r[None] * np.abs(w), np.broadcast_to(w, (H, Nr))], axis=-1)
    return np.concatenate([xr.reshape(H, 3 * Nr), ur.reshape(H, 2 * Nr)], axis=1)

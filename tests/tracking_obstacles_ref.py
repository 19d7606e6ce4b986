"""References of trajectory tracking among obstacles for tests/test_tracking_obstacles.py -- TEST INFRASTRUCTURE ONLY.

nmpc_create_tracking_obstacles is the moving-obstacle family (tests/obstacles_in_p.py) with the tracking cost of
tests/tracking_ref.py: p = [x0bar; Z; O], Z [N][5 Nr] with Z[k] = [xr_k; ur_k], O [N][n_obs][3].  Its references are derived
from those two modules' substitutions, applied together, so that they run the very same restated IPOPT and the very same
device source:
  * TrackingObstaclesOracle: oracle/nmpc_oracle.c with both sets of oracle substitutions.  The two rewrites of the stride
    `np = 6 * d->Nr;` conflict and are replaced by one with the combined stride, and the obstacle base p + 6 Nr moves to
    p + 3 Nr + 5 Nr N.  The tracking cost substitutions already cover the obstacle family (eval_obj / eval_grad serve both);
  * tracking_obstacles_emu_solve: tests/emul/emul_solver.cpp with the <NR, true, true> instantiation of the product's warp
    solver, its workspace sizing, and the parameter block with the obstacles in p after Z;
  * TrackingStageObstacleNLP: the one-robot StageObstacleNLP with the tracking f / grad_f (its SLSQP solve and the KKT
    certificate use them).
The sources are compiled into a temporary directory (nothing is written into the tree); a change of the underlying source that
breaks a substitution fails the tests loudly.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle_lib
from tests import obstacles_in_p, tracking_ref

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_TMP = None
_LIBS = {}

_NP_OLD = "np = 6 * d->Nr;"
_NP_NEW = "np = 3 * d->Nr + 5 * d->Nr * d->N + 3 * d->N * d->nobs;"
_OBS_BASE = ("C.D.obs = p + 6 * d->Nr;", "C.D.obs = p + 3 * d->Nr + 5 * d->Nr * d->N;")


def _oracle_subs():
    subs = [s for s in tracking_ref._ORACLE_SUBS if s[0] != _NP_OLD]
    for a, b, n in obstacles_in_p._ORACLE_SUBS:
        if a == _NP_OLD:
            continue
        if _OBS_BASE[0] in b:
            assert b.count(_OBS_BASE[0]) == 1
            b = b.replace(*_OBS_BASE)
        subs.append((a, b, n))
    assert len(subs) == len(tracking_ref._ORACLE_SUBS) + len(obstacles_in_p._ORACLE_SUBS) - 2
    assert any(_OBS_BASE[1] in b for _, b, _ in subs)
    return subs + [(_NP_OLD, _NP_NEW, 1)]


_EMU_SUBS = [
    ("        WarpSolver<(NR <= 4 ? NR : 1), true> s(*job.P, job.sm, job.ws);",
     "        WarpSolver<(NR <= 4 ? NR : 1), true, true> s(*job.P, job.sm, job.ws);", 1),
    ("WarpSolver<NR, NR <= 4>::", "WarpSolver<NR, NR <= 4, true>::", 2),
    ("P.nobs = nobs; P.family = family; P.obs = obs;",
     "P.nobs = nobs; P.family = family; P.obs = obs; P.obs_in_p = 1; P.np = 3 * Nr + 5 * Nr * N + 3 * N * nobs;", 1),
]


def _build(kind):
    global _TMP
    if kind in _LIBS:
        return _LIBS[kind]
    if _TMP is None:
        _TMP = tempfile.mkdtemp(prefix="nmpc_tracking_obstacles_")
    if kind == "oracle":
        src = os.path.join(_TMP, "nmpc_oracle_tracking_obstacles.c")
        tracking_ref._rewrite(os.path.join(_ROOT, "oracle", "nmpc_oracle.c"), _oracle_subs(), src)
        so = os.path.join(_TMP, "liboracle_tracking_obstacles.so")
        cmd = ["gcc", "-O3", "-mavx2", "-mfma", "-fopenmp", "-fPIC", "-Wall", "-Wno-unused-variable", "-std=gnu11",
               "-I" + os.path.join(_ROOT, "oracle"), "-shared", "-o", so, src, "-lm"]
        ref = oracle_lib.lib()
    else:
        src = os.path.join(_TMP, "emul_solver_tracking_obstacles.cpp")
        tracking_ref._rewrite(os.path.join(_ROOT, "tests", "emul", "emul_solver.cpp"), _EMU_SUBS, src)
        so = os.path.join(_TMP, "libnmpc_emul_tracking_obstacles.so")
        cmd = ["g++", "-O2", "-mavx2", "-mfma", "-fPIC", "-shared", "-std=c++17", "-x", "c++", "-Wno-unknown-pragmas",
               "-I" + os.path.join(_ROOT, "tests", "emul"), "-I" + tracking_ref._PKG_CSRC, "-I" + os.path.join(_ROOT, "include"),
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


class TrackingObstaclesOracle(oracle_lib.Oracle):
    """The C oracle with p = [x0bar; Z[N][5 Nr]; O[N][n_obs][3]] (np = 3 Nr + 5 Nr N + 3 N n_obs)."""

    def __init__(self, Nr, N, T, n_obs, **kw):
        super().__init__(Nr, N, T, **kw)
        self.L = _build("oracle")
        self.d.nobs = int(n_obs)
        self.nobs = int(n_obs)
        self.np_ = 3 * self.Nr + 5 * self.Nr * self.N + 3 * self.N * self.nobs
        self.mg = self.L.orc_mg(C.byref(self.d))


def tracking_obstacles_emu_solve(monkeypatch, Nr, N, T, x0, p, lbx, ubx, lbg, ubg, n_obs, **kw):
    """tests.emul.emul_lib.emu_solve on the emulation built with the <NR, true, true> instantiation."""
    from tests.emul import emul_lib
    monkeypatch.setattr(emul_lib, "_LIB", _build("emul"))
    return emul_lib.emu_solve(Nr, N, T, x0, p, lbx, ubx, lbg, ubg, obstacles=np.zeros((int(n_obs), 3)), **kw)


def pack(x0bar, Z, O):
    """p = [x0bar; Z; O] of one instance from x0bar [3 Nr], Z [N, 5 Nr] (or flat) and O [N, n_obs, 3] (or flat)."""
    return np.concatenate([np.ravel(x0bar), np.ravel(Z), np.ravel(O)]).astype(np.float64)


class TrackingStageObstacleNLP(obstacles_in_p.StageObstacleNLP):
    """One robot: StageObstacleNLP's rows (one obstacle table per stage, x0bar = p[0:3]) with the tracking cost on
    Z = p[3:3 + 5 N]."""

    def ref(self, p):
        Z = np.asarray(p, float).reshape(-1)[3:3 + 5 * self.N].reshape(self.N, 5)
        return Z[:, :3], Z[:, 3:]

    def f(self, w, p):
        X, U = self.split(w)
        xr, ur = self.ref(p)
        e, eu = X[:self.N] - xr, U - ur
        return float((self.Q * e * e).sum() + (self.R * eu * eu).sum())

    def grad_f(self, w, p):
        X, U = self.split(w)
        xr, ur = self.ref(p)
        gX = np.zeros_like(X)
        gX[:self.N] = 2.0 * self.Q * (X[:self.N] - xr)
        return np.concatenate([gX.ravel(), (2.0 * self.R * (U - ur)).ravel()])

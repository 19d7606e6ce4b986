"""Obstacles-in-p references for tests/test_moving_obstacles.py -- TEST INFRASTRUCTURE ONLY.

The references of the static-obstacle family read one obstacle table for every stage.  The variant with the tables in p
(p = [x0bar; xs; O], O [N][n_obs][3], row (k, i, o) on X_k against the stage-k table) is derived from them here, so that it runs
the very same restated IPOPT and the very same device source:
  * MovingOracle: oracle/nmpc_oracle.c compiled with the obstacle row reading the stage-k table of the instance's p;
  * moving_emu_solve: tests/emul/emul_solver.cpp compiled with NmpcSolveParams.obs_in_p set (the product's warp solver);
  * StageObstacleNLP: oracle/obstacle_nlp.py's NumPy restatement with one table per stage (the SLSQP check).
The sources are rewritten by exact substitutions that must each match, and compiled into a temporary directory (nothing is
written into the tree); a change of the underlying source that breaks a substitution fails the tests loudly.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle_lib
from oracle.obstacle_nlp import ObstacleNLP

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_PKG_CSRC = os.path.join(_ROOT, "nonlinear-mpc-for-collision-free-and-deadlock-free-navigation-of-multiple-nonholonomic-mobile-robots_b200",
                         "csrc")
_TMP = None
_LIBS = {}

# oracle: the obstacle row of stage k reads D->obs + k D->ostr, with D->obs = p + 6 Nr and D->ostr = 3 nobs
_ORACLE_SUBS = [
    ("    const double *obs;\n", "    const double *obs;\n    int ostr;\n", 1),
    ("static inline rowg_t row_geom(const dims_t *D, const double *zk, int q)\n{",
     "static inline rowg_t row_geom(const dims_t *D, const double *zk, int k, int q)\n{", 1),
    ("        r.i = e / D->nobs; r.j = -1;\n",
     "        r.i = e / D->nobs; r.j = -1;\n        const double *obs_k = D->obs + (size_t)k * D->ostr;\n", 1),
    ("double dx = zk[3 * r.i] - D->obs[3 * o], dy = zk[3 * r.i + 1] - D->obs[3 * o + 1];",
     "double dx = zk[3 * r.i] - obs_k[3 * o], dy = zk[3 * r.i + 1] - obs_k[3 * o + 1];", 1),
    ("r.dv = rho - D->obs[3 * o + 2];", "r.dv = rho - obs_k[3 * o + 2];", 1),
    ("D->nobs = d->obs ? d->nobs : 0; D->obs = d->obs;", "D->nobs = d->nobs; D->obs = NULL; D->ostr = 3 * d->nobs;", 1),
    ("if (d->obs && d->nobs > 0) return", "if (d->nobs > 0) return", 1),
    ("row_geom(D, zk, q)", "row_geom(D, zk, k, q)", 4),
    ("dims_init(&C.D, d); C.o = o; C.p = p;", "dims_init(&C.D, d); C.o = o; C.p = p; C.D.obs = p + 6 * d->Nr;", 1),
    ("np = 6 * d->Nr;", "np = 6 * d->Nr + 3 * d->N * d->nobs;", 1),
]
# emulation: the product's parameter block with the obstacles in p
_EMU_SUBS = [
    ("P.nobs = nobs; P.family = family; P.obs = obs;",
     "P.nobs = nobs; P.family = family; P.obs = obs; P.obs_in_p = 1; P.np = 6 * Nr + 3 * N * nobs;", 1),
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
        _TMP = tempfile.mkdtemp(prefix="nmpc_obs_in_p_")
    if kind == "oracle":
        src = os.path.join(_TMP, "nmpc_oracle_moving.c")
        _rewrite(os.path.join(_ROOT, "oracle", "nmpc_oracle.c"), _ORACLE_SUBS, src)
        so = os.path.join(_TMP, "liboracle_moving.so")
        cmd = ["gcc", "-O3", "-mavx2", "-mfma", "-fopenmp", "-fPIC", "-Wall", "-Wno-unused-variable", "-std=gnu11",
               "-I" + os.path.join(_ROOT, "oracle"), "-shared", "-o", so, src, "-lm"]
        ref = oracle_lib.lib()
    else:
        src = os.path.join(_TMP, "emul_solver_moving.cpp")
        _rewrite(os.path.join(_ROOT, "tests", "emul", "emul_solver.cpp"), _EMU_SUBS, src)
        so = os.path.join(_TMP, "libnmpc_emul_moving.so")
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


class MovingOracle(oracle_lib.Oracle):
    """The C oracle with n_obs obstacles per stage in p = [x0bar; xs; O[N][n_obs][3]] (np = 6 Nr + 3 N n_obs)."""

    def __init__(self, Nr, N, T, n_obs, **kw):
        super().__init__(Nr, N, T, **kw)
        self.L = _build("oracle")
        self.d.nobs = int(n_obs)
        self.nobs = int(n_obs)
        self.np_ = 6 * self.Nr + 3 * self.N * self.nobs
        self.mg = self.L.orc_mg(C.byref(self.d))


def moving_emu_solve(monkeypatch, Nr, N, T, x0, p, lbx, ubx, lbg, ubg, n_obs, **kw):
    """tests.emul.emul_lib.emu_solve on the emulation built with the obstacles in p."""
    from tests.emul import emul_lib
    monkeypatch.setattr(emul_lib, "_LIB", _build("emul"))
    return emul_lib.emu_solve(Nr, N, T, x0, p, lbx, ubx, lbg, ubg, obstacles=np.zeros((int(n_obs), 3)), **kw)


class StageObstacleNLP(ObstacleNLP):
    """ObstacleNLP with one obstacle table per stage: obstacles [N, n_obs, 3], row (k, o) on X_k against table k."""

    def __init__(self, N, T, obstacles, Q=(1.0, 5.0, 0.1), R=(0.5, 0.05)):
        O = np.asarray(obstacles, float).reshape(int(N), -1, 3)
        super().__init__(N, T, O[0], Q, R)
        self.obs_k = O

    def g(self, w, p):
        X, _ = self.split(w)
        out = ObstacleNLP.g(self, w, p)
        for k in range(self.N):
            o = 3 + k * self.blk
            out[o + 3:o + self.blk] = np.hypot(X[k, 0] - self.obs_k[k, :, 0], X[k, 1] - self.obs_k[k, :, 1]) - self.obs_k[k, :, 2]
        return out

    def jac_g(self, w, p):
        X, _ = self.split(w)
        J = ObstacleNLP.jac_g(self, w, p)
        for k in range(self.N):
            o, ix = 3 + k * self.blk, 3 * k
            dx, dy = X[k, 0] - self.obs_k[k, :, 0], X[k, 1] - self.obs_k[k, :, 1]
            rho = np.hypot(dx, dy)
            J[o + 3:o + self.blk, ix] = dx / rho
            J[o + 3:o + self.blk, ix + 1] = dy / rho
        return J

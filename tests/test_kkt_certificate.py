"""Multipliers (lam_x, lam_g) of every solver path checked with an independent KKT certificate (tests/kkt_certificate.py), over
bound structures the reference's bounds never produce:

  S0  reference bounds
  S1  pair rows dmin^2 <= d^2 <= dmax^2 with the upper bound active (robots must stay within range of each other)
  S2  pair rows with an upper bound only
  S3  one-sided state bounds: x lower-only, y upper-only, theta lower-only (each active for some robot)
  S4  v in [0, v_max]
  S5  a nonzero constant right-hand side on the x defect rows (a constant drift)
  S6  non-default Q / R and far goals: objective scaling df < 1, every returned multiplier divided by df
  S7  S0..S5 mixed per instance (bounds_batched)

The obstacle family (one robot) uses the same structures with its obstacle rows in place of the pair rows."""
import numpy as np
import pytest

from oracle.nlp_numpy import UnicycleNLP
from oracle.obstacle_nlp import ObstacleNLP
from oracle.oracle_lib import Oracle
from tests.emul.emul_lib import emu_solve
from tests.kkt_certificate import certify, derivatives, objective_scaling

STRUCTS = ["S0", "S1", "S2", "S3", "S4", "S5", "S6", "S7"]
Q6, R6 = (2.0, 8.0, 0.5), (1.0, 0.2)
INF = np.inf


# ---- instances and bound structures ------------------------------------------------------------------------------------
def ring_instances(Nr, B, seed, expand=False):
    """B perturbed rings: robots swap to the antipodal point (expand=False) or move out to twice the radius (expand=True)."""
    rng = np.random.default_rng(seed)
    r = max(0.8, 0.4 / np.sin(np.pi / max(Nr, 2)))
    a = np.arange(Nr) * 2 * np.pi / Nr + 0.3
    st = np.stack([r * np.cos(a), r * np.sin(a), (a + np.pi + np.pi) % (2 * np.pi) - np.pi], 1)
    if expand:
        goal = np.stack([2 * st[:, 0], 2 * st[:, 1], a], 1)
    else:
        goal = np.stack([-st[:, 0], -st[:, 1], st[:, 2]], 1)
    P = np.tile(np.concatenate([st.ravel(), goal.ravel()]), (B, 1))
    P[:, :3 * Nr] += 0.04 * rng.normal(size=(B, 3 * Nr))
    return P, r


class Central:
    """Bound structures of the centralized family (UnicycleNLP layout: block 0 = [X_0 rows; constant pair rows])."""

    def __init__(self, Nr, N, T):
        self.Nr, self.N, self.T = Nr, N, T
        self.ns, self.M = 3 * Nr, Nr * (Nr - 1) // 2
        self.blk, self.nX = self.ns + self.M, 3 * Nr * (N + 1)

    def reference(self):
        return UnicycleNLP(self.Nr, self.N, self.T).bounds(0.3, 0.22, 2.84)

    def pair_rows(self):
        m = np.zeros((self.N + 1, self.blk), bool)
        m[1:, self.ns:] = True      # block 0's pair rows are constants and keep the reference bounds
        return m.ravel()

    def upper_rows(self, P):
        """Pair rows and an upper bound d^2 <= dmax^2 that X_0 satisfies and the goals violate."""
        X0 = P[:, :3 * self.Nr].reshape(P.shape[0], self.Nr, 3)[:, :, :2]
        dmax = 1.05 * np.linalg.norm(X0[:, :, None] - X0[:, None], axis=-1).max()
        return self.pair_rows(), dmax ** 2

    def defect_rows(self, c):
        m = np.zeros((self.N + 1, self.blk), bool)
        m[1:, c:self.ns:3] = True
        return m.ravel()

    def build(self, S, P):
        """(P, lbx, ubx, lbg, ubg, Q, R): bounds [n]/[mg], or [B, .] where they depend on the instance."""
        B, Nr = P.shape[0], self.Nr
        lbx, ubx, lbg, ubg = (a.copy() for a in self.reference())
        Q, R = (1.0, 5.0, 0.1), (0.5, 0.05)
        if S in ("S1", "S2"):
            m, hi = self.upper_rows(P)
            ubg[m] = hi
            if S == "S2":
                lbg[m] = -INF
        elif S == "S3":
            lbx, ubx = np.tile(lbx, (B, 1)), np.tile(ubx, (B, 1))
            st, gl = P[:, :3 * Nr].reshape(B, Nr, 3), P[:, 3 * Nr:6 * Nr].reshape(B, Nr, 3)
            # x >= x0 - 0.05 (active for robots heading to smaller x), y <= y0 + 0.05, theta >= theta0 - 0.1
            lo_x = np.where(gl[..., 0] < st[..., 0], st[..., 0] - 0.05, st[..., 0] - 1.0)
            hi_y = np.where(gl[..., 1] > st[..., 1], st[..., 1] + 0.05, st[..., 1] + 1.0)
            lo_t = st[..., 2] - 0.1
            for b in range(B):
                X_lo = lbx[b, :self.nX].reshape(self.N + 1, Nr, 3)
                X_hi = ubx[b, :self.nX].reshape(self.N + 1, Nr, 3)
                X_lo[:, :, 0], X_hi[:, :, 0] = lo_x[b], INF
                X_lo[:, :, 1], X_hi[:, :, 1] = -INF, hi_y[b]
                X_lo[:, :, 2], X_hi[:, :, 2] = lo_t[b], INF
        elif S == "S4":
            lbx[self.nX::2] = 0.0
        elif S == "S5":
            m = self.defect_rows(0)
            lbg[m] = ubg[m] = 0.004
        elif S == "S6":
            Q, R = Q6, R6
            P = P.copy()
            for i in range(Nr):
                P[:, 3 * Nr + 3 * i:3 * Nr + 3 * i + 2] *= 40.0
        if lbx.ndim == 2:       # per-instance bounds: all four arrays are [B, .]
            lbg, ubg = np.tile(lbg, (B, 1)), np.tile(ubg, (B, 1))
        return P, lbx, ubx, lbg, ubg, Q, R

    def mixed(self, P):
        """S7: instance b gets structure S(b mod 6) (S0..S5); bounds [B, .]."""
        B = P.shape[0]
        parts = [self.build("S%d" % (b % 6), P[b:b + 1]) for b in range(B)]
        return (P,) + tuple(np.stack([np.broadcast_to(q[i], (1, q[i].shape[-1]))[0] for q in parts]) for i in (1, 2, 3, 4)) \
            + ((1.0, 5.0, 0.1), (0.5, 0.05))


class Obstacles(Central):
    """The same structures for the static-obstacle family, one robot (g = [X_0 - x0bar; per k: defect rows, obstacle rows]):
    the obstacle rows take the place of the pair rows (S1: the robot must stay within range of the first obstacle)."""

    def __init__(self, N, T, obs):
        self.Nr, self.N, self.T, self.obs = 1, N, T, np.asarray(obs, float).reshape(-1, 3)
        self.ns, self.M, self.nobs = 3, 0, self.obs.shape[0]
        self.blk, self.nX = 3 + self.nobs, 3 * (N + 1)

    def reference(self):
        return ObstacleNLP(self.N, self.T, self.obs).bounds(0.05, 0.2, np.pi / 4)

    def _rows(self, cols):
        m = np.zeros(self.N * self.blk, bool).reshape(self.N, self.blk)
        m[:, cols] = True
        return np.concatenate([np.zeros(3, bool), m.ravel()])

    def upper_rows(self, P):
        ox, oy, c = self.obs[0]
        d0 = np.hypot(P[:, 0] - ox, P[:, 1] - oy).max() - c
        return self._rows(slice(3, 4)), d0 + 0.08

    def defect_rows(self, c):
        return self._rows(slice(c, c + 1))


def structure(fam, S, P):
    return fam.mixed(P) if S == "S7" else fam.build(S, P)


def bound_row(a, b):
    return a[b] if a.ndim == 2 else a


# ---- the checker catches what it should --------------------------------------------------------------------------------
def _oracle_point(S="S1", Nr=2, N=10, T=0.3):
    fam = Central(Nr, N, T)
    P, lbx, ubx, lbg, ubg, Q, R = fam.build(S, ring_instances(Nr, 1, 3, expand=S in ("S1", "S2"))[0])
    o, nlp = Oracle(Nr, N, T, Q=Q, R=R), UnicycleNLP(Nr, N, T, Q=Q, R=R)
    lbx, ubx = bound_row(lbx, 0), bound_row(ubx, 0)
    w0 = o.cold_start(P[0, :3 * Nr])
    r = o.solve(w0, P[0], lbx, ubx, lbg, ubg)
    assert r["status"] == 0
    df = objective_scaling(nlp, w0, P[0])
    return nlp, r, (P[0], lbx, ubx, lbg, ubg), df


def test_certificate_accepts_the_oracle_and_rejects_broken_multipliers():
    nlp, r, (p, lbx, ubx, lbg, ubg), df = _oracle_point("S1")
    args = (p, lbx, ubx, lbg, ubg, df)
    m = certify(nlp, r["x"], r["lam_x"], r["lam_g"], *args)
    assert m["stat"] <= 1e-9
    # one active multiplier with its sign flipped (the largest pair-row multiplier: the upper bound dmax^2 is active)
    lg = r["lam_g"].copy()
    i = np.argmax(np.abs(lg) * Central(2, 10, 0.3).pair_rows())
    assert abs(lg[i]) > 1e-3 and lg[i] > 0
    lg[i] = -lg[i]
    with pytest.raises(AssertionError):
        certify(nlp, r["x"], r["lam_x"], lg, *args)
    # an active variable bound multiplier with its sign flipped
    lx = r["lam_x"].copy()
    j = np.argmax(np.abs(lx))
    assert abs(lx[j]) > 1e-3
    lx[j] = -lx[j]
    with pytest.raises(AssertionError):
        certify(nlp, r["x"], lx, r["lam_g"], *args)
    # lam_g off by a relative 1e-4
    with pytest.raises(AssertionError):
        certify(nlp, r["x"], r["lam_x"], r["lam_g"] * (1 + 1e-4), *args)
    # lam_x nonzero on a free variable (theta has no bounds in the reference structure)
    lx = r["lam_x"].copy()
    lx[2] = 1e-300
    with pytest.raises(AssertionError):
        certify(nlp, r["x"], lx, r["lam_g"], *args)


def test_certificate_rejects_multipliers_left_in_scaled_units():
    """df < 1: a solver that forgot to divide by df returns df * lam; the certificate must see it."""
    nlp, r, (p, lbx, ubx, lbg, ubg), df = _oracle_point("S6")
    assert df < 0.9
    certify(nlp, r["x"], r["lam_x"], r["lam_g"], p, lbx, ubx, lbg, ubg, df)
    with pytest.raises(AssertionError):
        certify(nlp, r["x"], df * r["lam_x"], df * r["lam_g"], p, lbx, ubx, lbg, ubg, df)


def test_certificate_needs_the_multipliers_of_fixed_variables():
    """Van der Pol: X_0 is fixed by lbx == ubx; its lam_x is -(grad f + J' lam_g) there, the cost's sensitivity to the
    initial state.  A solution with the fixed variables' multipliers zeroed is not a KKT point."""
    from oracle.vdp_nlp import VdpNLP
    nlp = VdpNLP()
    w0, lbw, ubw, lbg, ubg = nlp.demo_arrays()
    w = nlp.solve_slsqp(w0, lbw, ubw).x
    grad, g, J = derivatives(nlp, w, None)
    # multipliers from the active set: least squares on the free variables, then lam_x = -(grad + J' lam_g)
    act = (w - lbw <= 1e-7) | (ubw - w <= 1e-7)
    lam_g = np.linalg.lstsq(J[:, ~act].T, -grad[~act], rcond=None)[0]
    lam_x = -(grad + J.T @ lam_g)
    lam_x[~act] = 0.0
    df = objective_scaling(nlp, w0, None, lbw, ubw)
    certify(nlp, w, lam_x, lam_g, None, lbw, ubw, lbg, ubg, df, tol=1e-6)
    assert np.abs(lam_x[:2]).min() > 1e-3
    bad = lam_x.copy(); bad[:2] = 0.0
    with pytest.raises(AssertionError):
        certify(nlp, w, bad, lam_g, None, lbw, ubw, lbg, ubg, df, tol=1e-6)


# ---- CPU: the emulated warp kernel and the oracle over the structure matrix ---------------------------------------------
CPU_CASES = [(2, 10, 0.3), (3, 8, 0.3), (8, 5, 0.3)]


def _multiplier_close(a, b, rel):
    return np.abs(a - b).max() <= rel * max(1.0, np.abs(b).max())


@pytest.mark.parametrize("S", STRUCTS)
@pytest.mark.parametrize("Nr,N,T", CPU_CASES)
def test_emulated_kernel_multipliers_over_bound_structures(Nr, N, T, S):
    fam = Central(Nr, N, T)
    B = 6 if S == "S7" else 2
    P, lbx, ubx, lbg, ubg, Q, R = structure(fam, S, ring_instances(Nr, B, 10 * Nr + 1, expand=S in ("S1", "S2"))[0])
    o, nlp = Oracle(Nr, N, T, Q=Q, R=R), UnicycleNLP(Nr, N, T, Q=Q, R=R)
    w0 = np.stack([o.cold_start(q[:3 * Nr]) for q in P])
    ref = o.solve_batch(w0, P, lbx, ubx, lbg, ubg, want_duals=True)
    assert (ref["status"] == 0).all(), ref["status"]
    for rev in (0, 1):
        e = emu_solve(Nr, N, T, w0, P, lbx, ubx, lbg, ubg, Q=Q, R=R, reverse=rev)
        assert e["rc"] == 0 and (e["status"] == ref["status"]).all(), (e["status"], ref["status"])
        assert np.abs(e["iters"] - ref["iters"]).max() <= 2, (e["iters"], ref["iters"])
        for b in range(B):
            bnd = (bound_row(lbx, b), bound_row(ubx, b), bound_row(lbg, b), bound_row(ubg, b))
            df = objective_scaling(nlp, w0[b], P[b])
            if S == "S6":
                assert df < 1.0
            for k in ("x", "lam_x", "lam_g"):
                assert _multiplier_close(e[k][b], ref[k][b], 1e-7), (k, b, np.abs(e[k][b] - ref[k][b]).max())
            for out in (ref, e):
                certify(nlp, out["x"][b], out["lam_x"][b], out["lam_g"][b], P[b], *bnd, df)


OBS = np.array([[0.45, 0.5, 0.3], [1.0, 0.9, 0.2]])
OBS_P0 = np.array([0.0, 0.0, 0.6, 1.2, 1.3, 0.0])


def obstacle_instances(B, seed):
    rng = np.random.default_rng(seed)
    P = np.tile(OBS_P0, (B, 1))
    P[:, :3] += 0.05 * rng.normal(size=(B, 3))
    return P


@pytest.mark.parametrize("S", STRUCTS)
def test_emulated_kernel_multipliers_obstacle_family(S):
    N, T = 15, 0.3
    fam = Obstacles(N, T, OBS)
    B = 6 if S == "S7" else 2
    P, lbx, ubx, lbg, ubg, Q, R = structure(fam, S, obstacle_instances(B, 5))
    o, nlp = Oracle(1, N, T, Q=Q, R=R, obstacles=OBS), ObstacleNLP(N, T, OBS, Q=Q, R=R)
    w0 = np.stack([o.cold_start(q[:3]) for q in P])
    ref = o.solve_batch(w0, P, lbx, ubx, lbg, ubg, want_duals=True)
    assert (ref["status"] == 0).all(), ref["status"]
    e = emu_solve(1, N, T, w0, P, lbx, ubx, lbg, ubg, Q=Q, R=R, obstacles=OBS)
    assert e["rc"] == 0 and (e["status"] == ref["status"]).all() and np.abs(e["iters"] - ref["iters"]).max() <= 2
    for b in range(B):
        bnd = (bound_row(lbx, b), bound_row(ubx, b), bound_row(lbg, b), bound_row(ubg, b))
        for k in ("x", "lam_x", "lam_g"):
            assert _multiplier_close(e[k][b], ref[k][b], 1e-7), (k, b)
        for out in (ref, e):
            certify(nlp, out["x"][b], out["lam_x"][b], out["lam_g"][b], P[b], *bnd, objective_scaling(nlp, w0[b], P[b]))


# ---- GPU: every device path against its family's oracle, every solved instance certified ------------------------------
U_TOL, F_RTOL, VIOL = 1e-4, 1e-6, 1e-6       # north_star's primal tolerances
REPORT = {}                                  # path -> [max stationarity residual, max |dlam| / max(1, |lam_ref|)]


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    yield torch
    for path, (st, dl) in sorted(REPORT.items()):
        print("KKT %-22s max stationarity %.2e   max multiplier difference vs oracle %.2e" % (path, st, dl))


def _t(torch, a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda:0")


def _gpu_solve(torch, prob, w0, P, bnds):
    out = prob.solve(*[_t(torch, a) for a in (w0, P) + tuple(bnds)])
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def _check_gpu(path, out, ref, nlps, P, w0, bnds, nU, it_tol):
    """Status, primal agreement, iterations and multipliers against the oracle; the certificate and the self-report on every
    solved instance.  nlps: one NumPy NLP per instance (or one for all); nU: index where the controls start."""
    B = P.shape[0]
    assert (out["status"] == ref["status"]).all(), (out["status"], ref["status"])
    assert (out["status"] == 0).all(), out["status"]
    same = np.zeros(B, bool)
    rep = REPORT.setdefault(path, [0.0, 0.0])
    for b in range(B):
        nlp = nlps[b] if isinstance(nlps, list) else nlps
        bnd = [bound_row(a, b) for a in bnds]
        du = np.abs(out["x"][b] - ref["x"][b])[nU:].max()
        f_rel = abs(out["f"][b] - ref["f"][b]) / max(1.0, abs(ref["f"][b]))
        g = nlp.g(out["x"][b], P[b]) if not hasattr(nlp, "fg") else nlp.fg(out["x"][b])[1]
        viol = max(np.maximum(bnd[2] - g, 0).max(), np.maximum(g - bnd[3], 0).max())
        assert viol <= VIOL, (b, viol)
        same[b] = du <= U_TOL and f_rel <= F_RTOL
        if same[b]:
            assert abs(int(out["iters"][b]) - int(ref["iters"][b])) <= it_tol, (b, out["iters"], ref["iters"])
            for k in ("lam_x", "lam_g"):
                dl = np.abs(out[k][b] - ref[k][b]).max() / max(1.0, np.abs(ref[k][b]).max())
                assert dl <= 1e-5, (k, b, dl)
                rep[1] = max(rep[1], dl)
        m = certify(nlp, out["x"][b], out["lam_x"][b], out["lam_g"][b], P[b], *bnd, objective_scaling(nlp, w0[b], P[b]))
        rep[0] = max(rep[0], m["stat"])
        if out["stats"][b, 0] <= 1e-8:        # the kernel's own optimality error is what an independent measurement gives
            assert m["scaled_err"] <= 2e-8, (b, m["scaled_err"], out["stats"][b, 0])
    # a rounding-level fork into another local minimiser of these non-convex NLPs is possible; both are certified above
    assert same.sum() >= B - 1, same
    return same


CENTRAL_PATHS = [  # name, Nr, N, T, tuning, B, iteration tolerance
    ("warp-Nr2-N10", 2, 10, 0.3, None, 3, 3),
    ("warp-Nr6-N20", 6, 20, 0.3, None, 3, 3),
    ("team-Nr8", 8, 8, 0.3, None, 3, 3),
    ("block-Nr12", 12, 4, 0.3, None, 2, 5),
    ("block-Nr17", 17, 3, 0.3, None, 2, 5),
    ("forced-block-Nr3", 3, 8, 0.3, dict(force_block_path=1), 3, 5),
]


@pytest.mark.gpu
@pytest.mark.parametrize("S", STRUCTS)
@pytest.mark.parametrize("path,Nr,N,T,tuning,B,it_tol", CENTRAL_PATHS, ids=[c[0] for c in CENTRAL_PATHS])
def test_gpu_central_multipliers(pkg, torch_cuda, path, Nr, N, T, tuning, B, it_tol, S):
    fam = Central(Nr, N, T)
    B = 6 if S == "S7" else B
    P, lbx, ubx, lbg, ubg, Q, R = structure(fam, S, ring_instances(Nr, B, 7 * Nr + 2, expand=S in ("S1", "S2"))[0])
    prob, o = pkg.Problem(Nr, N, T, Q=Q, R=R, tuning=tuning), Oracle(Nr, N, T, Q=Q, R=R)
    w0 = prob.cold_start(P[:, :3 * Nr])
    out = _gpu_solve(torch_cuda, prob, w0, P, (lbx, ubx, lbg, ubg))
    ref = o.solve_batch(w0, P, lbx, ubx, lbg, ubg, want_duals=True)
    _check_gpu(path, out, ref, UnicycleNLP(Nr, N, T, Q=Q, R=R), P, w0, (lbx, ubx, lbg, ubg), fam.nX, it_tol)
    if S == "S7" and path.startswith(("block", "forced")):
        # per-instance bounds read through the block path's own layout: bit-identical to one call per instance
        for b in range(B):
            one = _gpu_solve(torch_cuda, prob, w0[b:b + 1], P[b:b + 1], (lbx[b], ubx[b], lbg[b], ubg[b]))
            for k in ("x", "lam_x", "lam_g", "iters", "status"):
                np.testing.assert_array_equal(one[k][0], out[k][b], err_msg=k)


OBS_PATHS = [("obstacles-warp", None), ("obstacles-forced-block", dict(force_block_path=1)),
             ("obstacles-thread", dict(thread_min_batch=1))]


@pytest.mark.gpu
@pytest.mark.parametrize("S", STRUCTS)
@pytest.mark.parametrize("path,tuning", OBS_PATHS, ids=[c[0] for c in OBS_PATHS])
def test_gpu_obstacle_multipliers(pkg, torch_cuda, path, tuning, S):
    N, T = 15, 0.3
    fam = Obstacles(N, T, OBS)
    B = 6 if S == "S7" else 3
    P, lbx, ubx, lbg, ubg, Q, R = structure(fam, S, obstacle_instances(B, 11))
    prob, o = pkg.Problem(1, N, T, Q=Q, R=R, obstacles=OBS, tuning=tuning), Oracle(1, N, T, Q=Q, R=R, obstacles=OBS)
    w0 = prob.cold_start(P[:, :3])
    out = _gpu_solve(torch_cuda, prob, w0, P, (lbx, ubx, lbg, ubg))
    ref = o.solve_batch(w0, P, lbx, ubx, lbg, ubg, want_duals=True)
    _check_gpu(path, out, ref, ObstacleNLP(N, T, OBS, Q=Q, R=R), P, w0, (lbx, ubx, lbg, ubg), fam.nX,
               5 if "block" in path else 3)


@pytest.mark.gpu
@pytest.mark.parametrize("S", STRUCTS)
def test_gpu_moving_obstacle_multipliers(pkg, torch_cuda, S):
    from tests.obstacles_in_p import MovingOracle, StageObstacleNLP
    N, T, B = 12, 0.3, (6 if S == "S7" else 3)
    fam = Obstacles(N, T, OBS)
    P6, lbx, ubx, lbg, ubg, Q, R = structure(fam, S, obstacle_instances(B, 13))
    # the obstacles drift by up to 2 cm per stage, each instance its own way (stage 0 is the static table above)
    rng = np.random.default_rng(14)
    O = np.tile(OBS, (B, N, 1, 1))
    O[..., :2] += np.arange(N)[None, :, None, None] * 0.02 * rng.uniform(-1, 1, (B, 1, len(OBS), 2))
    prob = pkg.Problem(1, N, T, Q=Q, R=R, moving_obstacles=len(OBS))
    o = MovingOracle(1, N, T, len(OBS), Q=Q, R=R)
    P = prob.params(P6[:, :3], P6[:, 3:6], obstacles=O)
    w0 = prob.cold_start(P[:, :3])
    out = _gpu_solve(torch_cuda, prob, w0, P, (lbx, ubx, lbg, ubg))
    ref = o.solve_batch(w0, P, lbx, ubx, lbg, ubg, want_duals=True)
    nlps = [StageObstacleNLP(N, T, O[b], Q=Q, R=R) for b in range(B)]
    _check_gpu("moving-obstacles-warp", out, ref, nlps, P, w0, (lbx, ubx, lbg, ubg), fam.nX, 3)


TRACK_PATHS = [("tracking-warp", None), ("tracking-forced-block", dict(force_block_path=1))]


@pytest.mark.gpu
@pytest.mark.parametrize("S", STRUCTS)
@pytest.mark.parametrize("path,tuning", TRACK_PATHS, ids=[c[0] for c in TRACK_PATHS])
def test_gpu_tracking_multipliers(pkg, torch_cuda, path, tuning, S):
    from tests.tracking_ref import TrackingNLP, TrackingOracle
    Nr, N, T = 3, 8, 0.3
    fam = Central(Nr, N, T)
    B = 6 if S == "S7" else 3
    P6, lbx, ubx, lbg, ubg, Q, R = structure(fam, S, ring_instances(Nr, B, 17, expand=S in ("S1", "S2"))[0])
    prob, o = pkg.Problem(Nr, N, T, Q=Q, R=R, tracking=True, tuning=tuning), TrackingOracle(Nr, N, T, Q=Q, R=R)
    # a reference that moves from the goal towards the start, with a nonzero control reference
    xr = P6[:, None, 3 * Nr:] + np.linspace(0, 0.3, N)[None, :, None] * (P6[:, None, :3 * Nr] - P6[:, None, 3 * Nr:])
    ur = np.tile(np.tile([0.05, 0.1], Nr), (B, N, 1))
    P = prob.params(P6[:, :3 * Nr], xr, uref=ur)
    w0 = prob.cold_start(P[:, :3 * Nr])
    out = _gpu_solve(torch_cuda, prob, w0, P, (lbx, ubx, lbg, ubg))
    ref = o.solve_batch(w0, P, lbx, ubx, lbg, ubg, want_duals=True)
    _check_gpu(path, out, ref, TrackingNLP(Nr, N, T, Q=Q, R=R), P, w0, (lbx, ubx, lbg, ubg), fam.nX,
               5 if "block" in path else 3)


@pytest.mark.gpu
@pytest.mark.parametrize("S", ["demo", "S5"])
def test_gpu_van_der_pol_multipliers(pkg, torch_cuda, S):
    """Thread path: the demo's bounds (X_0 fixed by lbx == ubx) and a nonzero right-hand side on the x1 shooting rows.  The
    fixed X_0's multipliers must be -(grad f + J' lam_g) there, or the certificate fails in those two components."""
    from scipy.optimize import minimize
    from oracle.vdp_nlp import VdpNLP
    ocp, nlp = pkg.SmallOcp("van_der_pol", N=20, T=10.0, rk_steps=4), VdpNLP()
    w0, lbw, ubw, lbg, ubg = ocp.demo_arrays()
    if S == "S5":
        lbg = lbg.copy(); lbg[0::2] = 0.01; ubg = lbg.copy()
    W0 = np.tile(w0, (4, 1)); W0[1:, 2:] += 0.05 * np.random.default_rng(3).normal(size=(3, nlp.n - 2))
    out = ocp.solve_host(W0, lbw, ubw, lbg, ubg)
    assert (out["status"] == 0).all(), out["status"]
    cons = [{"type": "eq", "fun": lambda w: nlp.fg(w)[1] - lbg}]
    ref = minimize(lambda w: nlp.fg(w)[0], out["x"][0], method="SLSQP", constraints=cons, bounds=list(zip(lbw, ubw)),
                   options={"ftol": 1e-13, "maxiter": 1000})
    rep = REPORT.setdefault("vdp-thread", [0.0, 0.0])
    df = objective_scaling(nlp, w0, None, lbw, ubw)
    for b in range(4):
        assert ref.fun >= out["f"][b] - 1e-8 and np.abs(ref.x - out["x"][b])[2::3].max() <= 1e-4
        m = certify(nlp, out["x"][b], out["lam_x"][b], out["lam_g"][b], None, lbw, ubw, lbg, ubg, df, tol=1e-6)
        rep[0] = max(rep[0], m["stat"])
        assert np.abs(out["lam_x"][b][:2]).min() > 1e-3     # the cost does depend on the initial state
        if out["stats"][b, 0] <= 1e-8:
            assert m["scaled_err"] <= 2e-8 + 1e-7, (m["scaled_err"], out["stats"][b, 0])


BAD_BOUNDS = ["lbx>ubx", "fixed-variable", "equality-ineq-row", "inequality-defect-row"]


def _bad(kind, lbx, ubx, lbg, ubg, ineq_row, defect_row, var):
    lbx, ubx, lbg, ubg = (a.copy() for a in (lbx, ubx, lbg, ubg))
    if kind == "lbx>ubx":
        lbx[var] = ubx[var] + 1.0
    elif kind == "fixed-variable":
        lbx[var] = ubx[var] = 0.1
    elif kind == "equality-ineq-row":
        ubg[ineq_row] = lbg[ineq_row]
    else:
        lbg[defect_row] = -1.0
    return lbx, ubx, lbg, ubg


@pytest.mark.gpu
@pytest.mark.parametrize("kind", BAD_BOUNDS)
def test_gpu_rejected_bounds_give_the_same_code_on_every_path(pkg, torch_cuda, kind):
    """One instance with a bound set that must be rejected, between two good ones: it gets the same status code on the warp,
    block and thread paths (obstacle family, one robot) and on the centralized family's warp and block paths, and the host
    entry point raises on every path.  (The warp and block paths reject the whole batch with that code; the thread path
    solves the other instances.)"""
    want = -2 if kind == "lbx>ubx" else -3
    N, T = 6, 0.3
    fam = Obstacles(N, T, OBS)
    P = obstacle_instances(3, 21)
    good = fam.reference()
    bad = _bad(kind, *good, ineq_row=3 + fam.blk + 3, defect_row=3 + fam.blk, var=fam.nX + 4)
    bnds = [np.stack([good[i], bad[i], good[i]]) for i in range(4)]
    cases = [(pkg.Problem(1, N, T, obstacles=OBS, tuning=tuning), P, 3, path) for path, tuning in OBS_PATHS]
    cfam = Central(2, N, T)
    Pc = ring_instances(2, 3, 22)[0]
    good = cfam.reference()
    bad = _bad(kind, *good, ineq_row=2 * cfam.blk + cfam.ns, defect_row=cfam.blk + 1, var=cfam.nX + 2)
    cbnds = [np.stack([good[i], bad[i], good[i]]) for i in range(4)]
    cases += [(pkg.Problem(2, N, T, tuning=tuning), Pc, 6, path)
              for path, tuning in (("central-warp", None), ("central-forced-block", dict(force_block_path=1)))]
    codes = {}
    for prob, PP, ns, path in cases:
        b4 = cbnds if path.startswith("central") else bnds
        w0 = prob.cold_start(PP[:, :ns])
        st = _gpu_solve(torch_cuda, prob, w0, PP, b4)["status"]
        codes[path] = st.tolist()
        assert st[1] == want and set(st[[0, 2]].tolist()) <= {0, want}, (path, st)
        with pytest.raises(pkg.NmpcError):
            prob.solve_host(w0, PP, *b4)

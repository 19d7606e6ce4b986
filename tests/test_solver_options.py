"""The IPOPT options (nmpc_opts, the keys the reference passes through nlpsol(..., opts)) checked iteration by iteration against
the C oracle, on the CPU emulation of the warp kernel and on every device path.

OPTION_CASES is one table of non-default option sets.  Every comparison runs each case on every start point of its
configuration, in one batch: a cold start, a warm start (the plant step and shift of an optimum, as in the closed loop) and,
with two or more robots, the infeasible instance with every robot at the origin.

test_every_option_case_acts is the evidence that a misread option fails those comparisons.  On every configuration a
comparison runs (ACT_CONFIGS), the oracle's run with the option must leave the default run on some start point by more than
ACT_GAP times the device comparison's tolerances.  divergence() measures exactly what the device comparison checks: status,
iteration count, stats counters, line-search count, mu and delta_w, and the continuous trace columns on every iteration.  A
(case, configuration) pair on which an option cannot act is listed in NOT_ACTING with its reason, and the test checks that
list in both directions.  The pairs that share a default (bound_push / bound_frac, constr_viol_tol / compl_inf_tol) run in
both orders, and the two orders must take different paths on every configuration.  test_device_check_rejects_misread_termination
feeds the device check the oracle's run with a termination tolerance ignored or a pair swapped, and requires it to fail.

  CPU  the emulated warp kernel (tests/emul) against the oracle: same status, iterations, stats counters 5-10, trace columns
       mu, delta_w and line-search count; theta, f, alpha, alpha_z within TR_RTOL; x, lam_x, lam_g within 1e-10.
  GPU  solve(..., trace=K) against Oracle.solve(trace=True) (check_device_instance): the same status, iteration count and
       stats counters 5-10; on every iteration the same line-search count, mu and delta_w within MU_RTOL, the continuous
       columns within GPU_TR_RTOL; a KKT certificate (tests/kkt_certificate.py) at the case's tol and bound_relax_factor
       for every solved instance.  The truncated solves (max_iter = k) compare x, f, g, lam_x and lam_g with the oracle's
       k-th iterate (max_iter = 0: the projected start point and the least-squares multipliers).
Every returned x lies within its bounds relaxed by the case's bound_relax_factor (not by the default 1e-8).

Measured on one B200 (1000 W power limit) over the whole table, per path: the largest trace difference in units of the
tolerance (GPU_TR_ATOL + GPU_TR_RTOL |ref|), the largest difference of a truncated iterate from the oracle's (relative to
max(1, |ref|)) and the largest stationarity residual of the certificate:
  warp Nr 1      1.7e-3   8.3e-16   3.0e-7        obstacles warp           2.9e-2   3.1e-14   2.8e-6
  warp Nr 2      4.8e-3   2.3e-14   2.4e-6        obstacles forced-block   2.9e-2   1.0e-13   2.8e-6
  warp Nr 6      5.7e-2   1.8e-14   3.8e-6        obstacles thread         1.7e-1   4.1e-14   2.8e-6
  team Nr 8      6.8e-3   7.5e-15   2.9e-7        moving obstacles warp    2.3e-3   1.5e-15   (no certificate: two robots)
  block Nr 12    2.2e-2   1.0e-14   1.4e-7        tracking warp            2.7e-3   1.1e-14   2.0e-11
  forced block   2.3e-3   2.0e-14   1.3e-8
Every status, iteration count and stats counter was the oracle's, and mu / delta_w agreed to MU_RTOL.  The six-robot warp path
runs N = 8: at N = 10 with kappa_sigma = 2 the cold start meets an inertia test whose pivot sits at rounding level, and the
emulation and the oracle already take different regularisations there.
"""
import numpy as np
import pytest

from oracle.nlp_numpy import UnicycleNLP
from oracle.obstacle_nlp import ObstacleNLP
from oracle.oracle_lib import Oracle
from tests.emul.emul_lib import emu_solve
from tests.kkt_certificate import certify, objective_scaling

ACCEPTABLE = dict(tol=1e-12, acceptable_tol=1e-4, acceptable_iter=2, acceptable_obj_change_tol=1e20)

# id, options
OPTION_CASES = [
    ("mu_init=1e-3", dict(mu_init=1e-3)),
    ("mu_init=1", dict(mu_init=1.0)),
    ("kappa_mu,theta_mu", dict(kappa_mu=0.5, theta_mu=1.2)),
    ("tau_min=0.9", dict(tau_min=0.9)),
    ("barrier_tol_factor=2", dict(barrier_tol_factor=2.0)),
    ("push>frac", dict(bound_push=0.05, bound_frac=0.002)),
    ("frac>push", dict(bound_push=0.002, bound_frac=0.05)),
    ("bound_mult_init_val=0.3", dict(bound_mult_init_val=0.3)),
    ("constr_mult_init_max=0", dict(constr_mult_init_max=0.0)),
    ("bound_relax_factor=0", dict(bound_relax_factor=0.0)),
    ("bound_relax_factor=1e-5", dict(bound_relax_factor=1e-5)),
    ("kappa_sigma=2", dict(kappa_sigma=2.0)),
    ("kappa_d=0", dict(kappa_d=0.0)),
    ("kappa_d=1e-2", dict(kappa_d=1e-2)),
    ("nlp_scaling_max_gradient=1", dict(nlp_scaling_max_gradient=1.0)),
    ("max_soc=0", dict(max_soc=0)),
    ("max_soc=1", dict(max_soc=1)),
    ("max_resto_iter=0", dict(max_resto_iter=0)),
    ("acceptable", ACCEPTABLE),
    ("acceptable,tiny_obj_change", dict(ACCEPTABLE, acceptable_obj_change_tol=1e-30)),
    ("tol=1e-5", dict(tol=1e-5)),
    ("viol<compl", dict(constr_viol_tol=1e-12, compl_inf_tol=1e-2)),
    ("compl<viol", dict(constr_viol_tol=1e-2, compl_inf_tol=1e-12)),
    ("dual_inf_tol=1e-9", dict(dual_inf_tol=1e-9)),
    ("dual_inf_tol=1e-12", dict(dual_inf_tol=1e-12)),
] + [("max_iter=%d" % k, dict(max_iter=k)) for k in (0, 1, 2, 3, 5, 8)]
CASE_IDS = [c[0] for c in OPTION_CASES]
OPTS = dict(OPTION_CASES)
SWAPPED = [("push>frac", "frac>push"), ("viol<compl", "compl<viol")]
_NO_ORIGIN = ("Nr1-N10", "obstacles", "moving")
# (case, compared configuration) pairs on which the option leaves every start point's run as it is, and why.
# test_every_option_case_acts asserts both directions: every pair not listed acts, every listed pair does not.
# (max_iter = k is exempt by rule where every default run of the configuration needs k iterations or fewer.)
NOT_ACTING = {
    **{("kappa_d=0", c): "one robot without obstacles: no pair rows, so no one-sided bound for kappa_d to damp"
       for c in ("Nr1-N10",)},
    **{("kappa_d=1e-2", c): "one robot without obstacles: no pair rows, so no one-sided bound for kappa_d to damp"
       for c in ("Nr1-N10",)},
    **{("max_soc=0", c): "no second-order correction in any default run of this configuration"
       for c in ("Nr8-N4", "Nr12-N4", "tracking", "moving")},
    **{("max_soc=1", c): "no default run here takes a second correction in a row (only Nr2-N10's warm start does)"
       for c in ("Nr1-N10", "Nr3-N6", "Nr6-N8", "Nr8-N4", "Nr12-N4", "obstacles", "tracking", "moving")},
    **{("max_resto_iter=0", c): "no infeasible start here (one robot, or no pair rows at block 0): no restoration phase runs"
       for c in _NO_ORIGIN},
    **{("viol<compl", c): "the default runs already stop at a point whose constraint violation is below 1e-12"
       for c in ("Nr8-N4", "Nr12-N4", "moving")},
    **{("dual_inf_tol=1e-9", c): "the default runs already stop with dinf / df <= 1e-9 (dual_inf_tol=1e-12 acts there)"
       for c in ("Nr1-N10", "Nr2-N10", "Nr3-N6", "Nr6-N8", "Nr8-N4", "Nr12-N4", "tracking", "moving")},
}
MAX_ITER = 200        # every solve below ends long before this unless the case truncates it

ACT_CONFIGS = ["Nr1-N10", "Nr2-N10", "Nr3-N6", "Nr6-N8", "Nr8-N4", "Nr12-N4", "obstacles", "tracking", "moving"]
ACT_GAP = 100.0       # acting: the trace leaves the default run's by more than 100 x the device comparison's tolerance
TR_RTOL, TR_ATOL = 1e-9, 1e-12       # emulation vs oracle, theta, f, alpha, alpha_z
GPU_TR_RTOL, GPU_TR_ATOL = 1e-9, 1e-12   # device vs oracle, the same columns (measured maxima: test_gpu_options_follow_the_oracle)
MU_RTOL = 1e-13       # device vs oracle, mu and delta_w: the device's pow() may differ from the host's in the last bit
X_TOL = 1e-10         # emulation vs oracle, x / lam_x / lam_g, relative to max(1, |ref|)
X_TOL_INFEASIBLE = 1e-8    # the same after a failed restoration (status 3): its last step is a rank-deficient projection
GPU_X_TOL = 1e-8      # device vs oracle on the truncated solves
DISCRETE, CONTINUOUS = [0, 6, 7], [2, 3, 4, 5]     # trace columns (ORC_TR_*): mu, delta_w, line searches / theta, f, alpha, alpha_z


def opts_of(case):
    return dict(dict(max_iter=MAX_ITER), **OPTS[case])


# ---- start points ------------------------------------------------------------------------------------------------------
def ring(Nr, jitter=0.02):
    """Nr robots on a ring swapping to the antipodes: p = [start; goal]."""
    a = np.arange(Nr) * 2 * np.pi / Nr + 0.3
    r = max(0.8, 0.4 / np.sin(np.pi / max(Nr, 2)))
    st = np.stack([r * np.cos(a), r * np.sin(a), (a + np.pi + np.pi) % (2 * np.pi) - np.pi], 1)
    gl = np.stack([-st[:, 0], -st[:, 1], st[:, 2]], 1)
    return np.concatenate([st.ravel() + jitter * np.sin(1.0 + np.arange(3 * Nr)), gl.ravel()])


P3 = np.array([-1, -1, 1.57, 0, -1, 1.57, 1, -1, 1.57, 1, 2, 0, 0, 1, 0, -1, 0.5, 0], float)


def centralized_p(Nr):
    return P3.copy() if Nr == 3 else ring(Nr)


def warm_from(orc, w0, p, bnds):
    """One closed-loop step: the default solve from (w0, p), its first control through the plant, the shifted optimum."""
    r = orc.solve(w0, p, *bnds)
    nX = orc.ns * (orc.N + 1)
    p2 = p.copy()
    p2[:orc.ns] = orc.plant(p[:orc.ns], r["x"][nX:nX + orc.nc])
    return orc.shift(r["x"]), p2


def origin_p(p):
    """Every robot at the origin: the block-0 pair rows d^2 = 0 < dmin^2 cannot be met."""
    q = p.copy()
    q[:len(q) // 2] = 0.0
    return q


def centralized_starts(Nr, N, T):
    """(W [B, n], P [B, np], names) for the centralized family: cold, warm and (Nr >= 2) origin."""
    orc = Oracle(Nr, N, T)
    bnds = orc.bounds(0.3, 0.22, 2.84)
    p = centralized_p(Nr)
    w0 = orc.cold_start(p[:3 * Nr])
    ww, pw = warm_from(orc, w0, p, bnds)
    W, P, names = [w0, ww], [p, pw], ["cold", "warm"]
    if Nr >= 2:
        po = origin_p(p)
        W.append(orc.cold_start(po[:3 * Nr])); P.append(po); names.append("origin")
    return np.stack(W), np.stack(P), names, bnds


# ---- comparing runs ----------------------------------------------------------------------------------------------------
def divergence(r, r0):
    """How far the oracle run r leaves the run r0, in units of the device comparison's tolerances: inf for a different status,
    iteration count, stats counter (5-10) or line-search count; otherwise the largest of |a - b| / (MU_RTOL |b|) over mu and
    delta_w and |a - b| / (GPU_TR_ATOL + GPU_TR_RTOL |b|) over the continuous trace columns, on every iteration."""
    if r["status"] != r0["status"] or r["iters"] != r0["iters"] or not np.array_equal(r["stats"][5:10], r0["stats"][5:10]):
        return np.inf
    m = r["iters"]
    a, b = r["trace"][:m], r0["trace"][:m]
    if not np.array_equal(a[:, 7], b[:, 7]):
        return np.inf
    dm = np.abs(a[:, [0, 6]] - b[:, [0, 6]])
    dm = np.where(dm > 0, dm / np.maximum(MU_RTOL * np.abs(b[:, [0, 6]]), 1e-300), 0.0)
    d = np.abs(a[:, CONTINUOUS] - b[:, CONTINUOUS]) / (GPU_TR_ATOL + GPU_TR_RTOL * np.abs(b[:, CONTINUOUS]))
    return float(max(dm.max(initial=0.0), d.max(initial=0.0)))


def relax_of(opts):
    return opts.get("bound_relax_factor", 1e-8)


def assert_within_relaxed_bounds(x, lbx, ubx, relax):
    """An interior-point iterate lies within the bounds relaxed by relax * max(1, |b|), whatever the status."""
    fl, fu = np.isfinite(lbx), np.isfinite(ubx)
    lo = np.where(fl, lbx - relax * np.maximum(1.0, np.abs(np.where(fl, lbx, 0.0))), -np.inf)
    hi = np.where(fu, ubx + relax * np.maximum(1.0, np.abs(np.where(fu, ubx, 0.0))), np.inf)
    assert (x >= lo).all() and (x <= hi).all(), (relax, (lo - x).max(), (x - hi).max())


def _rel(a, b):
    return np.abs(a - b).max(initial=0.0) / max(1.0, np.abs(b).max(initial=0.0))


def assert_follows(e, b, r, opts, what):
    """Emulated instance b of e against the oracle run r: the CPU tolerances of the module docstring."""
    assert (int(e["status"][b]), int(e["iters"][b])) == (r["status"], r["iters"]), (what, e["status"][b], e["iters"][b], r["status"], r["iters"])
    np.testing.assert_array_equal(e["stats"][b][5:11], r["stats"][5:11], err_msg=what)
    m = r["iters"]
    np.testing.assert_array_equal(e["trace"][b][:m, DISCRETE], r["trace"][:m, DISCRETE], err_msg=what)
    np.testing.assert_allclose(e["trace"][b][:m, CONTINUOUS], r["trace"][:m, CONTINUOUS], rtol=TR_RTOL, atol=TR_ATOL, err_msg=what)
    for k in ("x", "lam_x", "lam_g"):
        assert _rel(e[k][b], r[k]) <= (X_TOL_INFEASIBLE if r["status"] == 3 else X_TOL), (what, k, _rel(e[k][b], r[k]))


# ---- 2. CPU: the emulated warp kernel against the oracle over the whole matrix ---------------------------------------------
OBS = np.array([[0.45, 0.5, 0.3], [1.0, 0.9, 0.2]])
OBS_P0 = np.array([0.0, 0.0, 0.6, 1.2, 1.3, 0.0])


def obstacle_starts(N, T):
    orc = Oracle(1, N, T, obstacles=OBS)
    bnds = ObstacleNLP(N, T, OBS).bounds(0.05, 0.2, np.pi / 4)
    w0 = orc.cold_start(OBS_P0[:3])
    ww, pw = warm_from(orc, w0, OBS_P0, bnds)
    return np.stack([w0, ww]), np.stack([OBS_P0, pw]), ["cold", "warm"], bnds


def tracking_setup(Nr, N, T):
    from tests.test_tracking import _rotation_case
    from tests.tracking_ref import TrackingOracle
    orc = TrackingOracle(Nr, N, T)
    x0, Zt = _rotation_case(Nr, N, T, seed=Nr)
    p = np.concatenate([x0, Zt.ravel()])
    bnds = orc.bounds(0.3, 0.6, np.pi / 2)
    w0 = orc.cold_start(x0)
    ww, pw = warm_from(orc, w0, p, bnds)
    po = p.copy(); po[:3 * Nr] = 0.0
    return orc, np.stack([w0, ww, orc.cold_start(po[:3 * Nr])]), np.stack([p, pw, po]), ["cold", "warm", "origin"], bnds


def moving_setup(Nr, N, T):
    from tests.obstacles_in_p import MovingOracle
    from tests.test_moving_obstacles import _orc_bounds, _two_robot_case
    p6, O = _two_robot_case(N, T)
    orc = MovingOracle(Nr, N, T, O.shape[1])
    bnds = _orc_bounds(orc, O.shape[1], 0.05)
    p = np.concatenate([p6, O.ravel()])
    w0 = orc.cold_start(p6[:3 * Nr])
    ww, pw = warm_from(orc, w0, p, bnds)
    return orc, O, np.stack([w0, ww]), np.stack([p, pw]), ["cold", "warm"], bnds


_STARTS = {}


def _cached(key, fn, *a):
    if key not in _STARTS:
        _STARTS[key] = fn(*a)
    return _STARTS[key]


# ---- 1. the option matrix acts, on every configuration the comparisons below run -------------------------------------------
def act_config(name):
    """(oracle factory opts -> Oracle, W, P, start names, bounds) of a configuration that a comparison below runs."""
    if name.startswith("Nr"):
        Nr, N = (int(v) for v in name[2:].split("-N"))
        W, P, names, bnds = _cached(("central", Nr, N, 0.3), centralized_starts, Nr, N, 0.3)
        return (lambda o: Oracle(Nr, N, 0.3, **o)), W, P, names, bnds
    if name == "obstacles":
        W, P, names, bnds = _cached(("obstacles", 8, 0.3), obstacle_starts, 8, 0.3)
        return (lambda o: Oracle(1, 8, 0.3, obstacles=OBS, **o)), W, P, names, bnds
    if name == "tracking":
        from tests.tracking_ref import TrackingOracle
        _, W, P, names, bnds = _cached(("tracking", 2, 6, 0.2), tracking_setup, 2, 6, 0.2)
        return (lambda o: TrackingOracle(2, 6, 0.2, **o)), W, P, names, bnds
    from tests.obstacles_in_p import MovingOracle
    _, O, W, P, names, bnds = _cached(("moving", 2, 6, 0.3), moving_setup, 2, 6, 0.3)
    return (lambda o: MovingOracle(2, 6, 0.3, O.shape[1], **o)), W, P, names, bnds


_RUNS = {}


def oracle_runs(config, case):
    """The oracle's runs of one configuration's start points with the options of `case` (None: the defaults)."""
    if (config, case) not in _RUNS:
        mk, W, P, names, bnds = act_config(config)
        orc = mk(dict(max_iter=MAX_ITER) if case is None else opts_of(case))
        _RUNS[(config, case)] = [orc.solve(W[i], P[i], *bnds, trace=True) for i in range(len(W))]
    return _RUNS[(config, case)]


@pytest.mark.parametrize("config", ACT_CONFIGS)
@pytest.mark.parametrize("case", CASE_IDS)
def test_every_option_case_acts(case, config):
    """The evidence that a misread option fails the comparisons below: on every configuration a comparison runs, the oracle's
    run with the option leaves the default run on at least one start point by more than ACT_GAP x the device comparison's
    tolerances (divergence() measures exactly what test_gpu_options_follow_the_oracle compares), unless NOT_ACTING lists the
    pair with its reason; a listed pair must indeed not act."""
    assert TR_RTOL <= GPU_TR_RTOL and TR_ATOL <= GPU_TR_ATOL
    base, runs = oracle_runs(config, None), oracle_runs(config, case)
    div = [divergence(r, r0) for r, r0 in zip(runs, base)]
    if case.startswith("max_iter"):
        k = OPTS[case]["max_iter"]
        for r, r0, d in zip(runs, base, div):
            assert (d > ACT_GAP) == (r0["iters"] > k), (case, config, d, r0["iters"])
            if r0["iters"] > k:
                assert (r["status"], r["iters"]) == (2, k)
        return
    if (case, config) in NOT_ACTING:
        assert max(div) <= ACT_GAP, (case, config, div, "listed in NOT_ACTING but acts")
        return
    assert max(div) > ACT_GAP, (case, config, div)
    names = act_config(config)[3]
    if "origin" in names:
        r0 = base[names.index("origin")]
        assert r0["status"] == 3 and r0["stats"][6] >= 1     # the restoration phase runs there and fails
    if case == "acceptable":
        assert all(r["status"] == 1 for r, r0 in zip(runs, base) if r0["status"] == 0)
    if case == "acceptable,tiny_obj_change":
        assert all(r["status"] != 1 for r in runs)


@pytest.mark.parametrize("config", ACT_CONFIGS)
@pytest.mark.parametrize("a,b", SWAPPED)
def test_swapped_pairs_differ_from_each_other(a, b, config):
    """Options that share a default: on every compared configuration the two orders of a pair take different paths on some
    start point, so a kernel that reads one field for the other fails there."""
    d = [divergence(ra, rb) for ra, rb in zip(oracle_runs(config, a), oracle_runs(config, b))]
    assert max(d) > ACT_GAP, (a, b, config, d)


CPU_CENTRAL = [(1, 10, 0.3), (2, 10, 0.3), (3, 6, 0.3), (8, 4, 0.3)]


@pytest.mark.parametrize("case", CASE_IDS)
@pytest.mark.parametrize("Nr,N,T", CPU_CENTRAL, ids=["Nr%d" % c[0] for c in CPU_CENTRAL])
@pytest.mark.parametrize("reverse", [0, 1])
def test_emulated_kernel_options(Nr, N, T, reverse, case):
    opts = opts_of(case)
    W, P, names, bnds = _cached(("central", Nr, N, T), centralized_starts, Nr, N, T)
    e = emu_solve(Nr, N, T, W, P, *bnds, trace=True, reverse=reverse, **opts)
    assert e["rc"] == 0
    orc = Oracle(Nr, N, T, **opts)
    for b, name in enumerate(names):
        r = orc.solve(W[b], P[b], *bnds, trace=True)
        assert_follows(e, b, r, opts, (case, name))
        assert_within_relaxed_bounds(e["x"][b], bnds[0], bnds[1], relax_of(opts))


@pytest.mark.parametrize("case", CASE_IDS)
def test_emulated_kernel_options_obstacle_family(case):
    opts = opts_of(case)
    N, T = 8, 0.3
    W, P, names, bnds = _cached(("obstacles", N, T), obstacle_starts, N, T)
    e = emu_solve(1, N, T, W, P, *bnds, trace=True, obstacles=OBS, **opts)
    assert e["rc"] == 0
    orc = Oracle(1, N, T, obstacles=OBS, **opts)
    for b, name in enumerate(names):
        r = orc.solve(W[b], P[b], *bnds, trace=True)
        assert_follows(e, b, r, opts, (case, name))
        assert_within_relaxed_bounds(e["x"][b], bnds[0], bnds[1], relax_of(opts))


@pytest.mark.parametrize("case", CASE_IDS)
def test_emulated_kernel_options_tracking(case, monkeypatch):
    from tests.tracking_ref import TrackingOracle, tracking_emu_solve
    opts = opts_of(case)
    Nr, N, T = 2, 6, 0.2
    _, W, P, names, bnds = _cached(("tracking", Nr, N, T), tracking_setup, Nr, N, T)
    e = tracking_emu_solve(monkeypatch, Nr, N, T, W, P, *bnds, trace=True, reverse=1, **opts)
    assert e["rc"] == 0
    orc = TrackingOracle(Nr, N, T, **opts)
    for b, name in enumerate(names):
        assert_follows(e, b, orc.solve(W[b], P[b], *bnds, trace=True), opts, (case, name))


@pytest.mark.parametrize("case", CASE_IDS)
def test_emulated_kernel_options_moving_obstacles(case, monkeypatch):
    from tests.obstacles_in_p import MovingOracle, moving_emu_solve
    opts = opts_of(case)
    Nr, N, T = 2, 6, 0.3
    _, O, W, P, names, bnds = _cached(("moving", Nr, N, T), moving_setup, Nr, N, T)
    e = moving_emu_solve(monkeypatch, Nr, N, T, W, P, *bnds, O.shape[1], trace=True, **opts)
    assert e["rc"] == 0
    orc = MovingOracle(Nr, N, T, O.shape[1], **opts)
    for b, name in enumerate(names):
        assert_follows(e, b, orc.solve(W[b], P[b], *bnds, trace=True), opts, (case, name))


# ---- 3. GPU: the same matrix through the real kernels ----------------------------------------------------------------------
GPU_PATHS = [  # name, family, Nr, N, T, tuning
    ("warp-Nr1", "central", 1, 10, 0.3, None),
    ("warp-Nr2", "central", 2, 10, 0.3, None),
    ("warp-Nr6", "central", 6, 8, 0.3, None),
    ("team-Nr8", "central", 8, 4, 0.3, None),
    ("block-Nr12", "central", 12, 4, 0.3, None),
    ("forced-block-Nr3", "central", 3, 6, 0.3, dict(force_block_path=1)),
    ("obstacles-warp", "obstacles", 1, 8, 0.3, None),
    ("obstacles-forced-block", "obstacles", 1, 8, 0.3, dict(force_block_path=1)),
    ("obstacles-thread", "obstacles", 1, 8, 0.3, dict(thread_min_batch=1)),
    ("moving-obstacles-warp", "moving", 2, 6, 0.3, None),
    ("tracking-warp", "tracking", 2, 6, 0.2, None),
]
REPORT = {}     # path -> [max trace error / tolerance, max truncated-iterate difference, max stationarity residual]


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    yield torch
    for path, (tr, xd, st) in sorted(REPORT.items()):
        print("OPTIONS %-24s max trace |d| / (%.0e + %.0e |ref|) %.2e   max truncated-iterate diff %.2e   max stationarity %.2e"
              % (path, GPU_TR_ATOL, GPU_TR_RTOL, tr, xd, st))


def _t(torch, a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda:0")


def gpu_setup(pkg, family, Nr, N, T, tuning, opts):
    """(Problem, oracle, NumPy NLP per instance, W, P, bounds, names) for one path and option set."""
    if family == "central":
        W, P, names, bnds = _cached(("central", Nr, N, T), centralized_starts, Nr, N, T)
        return (pkg.Problem(Nr, N, T, tuning=tuning, **opts), Oracle(Nr, N, T, **opts), [UnicycleNLP(Nr, N, T)] * len(W),
                W, P, bnds, names)
    if family == "obstacles":
        W, P, names, bnds = _cached(("obstacles", N, T), obstacle_starts, N, T)
        return (pkg.Problem(1, N, T, obstacles=OBS, tuning=tuning, **opts), Oracle(1, N, T, obstacles=OBS, **opts),
                [ObstacleNLP(N, T, OBS)] * len(W), W, P, bnds, names)
    if family == "moving":
        from tests.obstacles_in_p import MovingOracle, StageObstacleNLP
        _, O, W, P, names, bnds = _cached(("moving", Nr, N, T), moving_setup, Nr, N, T)
        nlp = StageObstacleNLP(N, T, O) if Nr == 1 else None      # the certificate's NumPy restatement has one robot
        return (pkg.Problem(Nr, N, T, moving_obstacles=O.shape[1], tuning=tuning, **opts),
                MovingOracle(Nr, N, T, O.shape[1], **opts), [nlp] * len(W), W, P, bnds, names)
    from tests.tracking_ref import TrackingNLP, TrackingOracle
    _, W, P, names, bnds = _cached(("tracking", Nr, N, T), tracking_setup, Nr, N, T)
    return (pkg.Problem(Nr, N, T, tracking=True, tuning=tuning, **opts), TrackingOracle(Nr, N, T, **opts),
            [TrackingNLP(Nr, N, T)] * len(W), W, P, bnds, names)


def check_device_instance(out, b, r, opts, what, rep=None):
    """Instance b of a device solve against the oracle run r: the same status and iteration count, the same stats counters
    (5-10), on every iteration the same line-search count, mu and delta_w within MU_RTOL and theta, f, alpha, alpha_z within
    GPU_TR_RTOL / GPU_TR_ATOL -- exactly what divergence() measures -- and for a truncated solve the k-th iterate itself."""
    st, it = int(out["status"][b]), int(out["iters"][b])
    assert (st, it) == (r["status"], r["iters"]), (what, st, it, r["status"], r["iters"])
    np.testing.assert_array_equal(out["stats"][b][5:11], r["stats"][5:11], err_msg=str(what))
    a, ref = out["trace"][b][:it], r["trace"][:it]
    np.testing.assert_array_equal(a[:, 7], ref[:, 7], err_msg=str(what))
    np.testing.assert_allclose(a[:, [0, 6]], ref[:, [0, 6]], rtol=MU_RTOL, atol=0, err_msg=str(what))
    err = np.abs(a[:, CONTINUOUS] - ref[:, CONTINUOUS]) / (GPU_TR_ATOL + GPU_TR_RTOL * np.abs(ref[:, CONTINUOUS]))
    if rep is not None:
        rep[0] = max(rep[0], err.max(initial=0.0))
    assert err.max(initial=0.0) <= 1.0, (what, err.max())
    if "max_iter" in opts and opts["max_iter"] < MAX_ITER and r["status"] == 2:
        # the k-th iterate itself (k = 0: the projected start point and the least-squares multipliers)
        for k in ("x", "g", "lam_x", "lam_g"):
            d = _rel(out[k][b], r[k])
            if rep is not None:
                rep[1] = max(rep[1], d)
            assert d <= GPU_X_TOL, (what, k, d)
        assert abs(out["f"][b] - r["f"]) <= GPU_X_TOL * max(1.0, abs(r["f"])), what


def stand_in(runs, K):
    """Device-shaped outputs [B, ...] built from oracle runs (trace padded to K rows)."""
    out = {k: np.stack([r[k] for r in runs]) for k in ("x", "g", "lam_x", "lam_g")}
    out.update(f=np.array([r["f"] for r in runs]), status=np.array([r["status"] for r in runs]),
               iters=np.array([r["iters"] for r in runs]), stats=np.stack([r["stats"][:11] for r in runs]))
    out["trace"] = np.zeros((len(runs), K, 8))
    for b, r in enumerate(runs):
        out["trace"][b, :len(r["trace"])] = r["trace"][:K]
    return out


MISREADS = [  # termination case, what a misreading device path would run instead
    ("tol=1e-5", {}), ("viol<compl", OPTS["compl<viol"]), ("compl<viol", OPTS["viol<compl"]), ("viol<compl", {}),
    ("compl<viol", {}), ("dual_inf_tol=1e-12", {}), ("acceptable", dict(tol=1e-12)), ("acceptable,tiny_obj_change", ACCEPTABLE),
]


@pytest.mark.parametrize("case,instead", MISREADS, ids=["%s<-%s" % (c, ",".join("%s=%g" % kv for kv in i.items()) or "default")
                                                       for c, i in MISREADS])
def test_device_check_rejects_misread_termination(case, instead):
    """A device path that ignores a termination tolerance (runs the default) or reads one field of a pair for the other: the
    oracle's run with the misread options stands in for the device's output.  On every centralized configuration the GPU
    runs where that run leaves the case's (divergence > ACT_GAP), check_device_instance rejects it; the case's own run passes."""
    caught = []
    for config in [c for c in ACT_CONFIGS if c.startswith("Nr")]:
        mk, W, P, names, bnds = act_config(config)
        refs = oracle_runs(config, case)
        mis = [mk(dict(dict(max_iter=MAX_ITER), **instead)).solve(W[b], P[b], *bnds, trace=True) for b in range(len(W))]
        good, bad = stand_in(refs, MAX_ITER + 1), stand_in(mis, MAX_ITER + 1)
        for b in range(len(W)):
            check_device_instance(good, b, refs[b], opts_of(case), (case, config))
            if divergence(mis[b], refs[b]) > ACT_GAP:
                with pytest.raises(AssertionError):
                    check_device_instance(bad, b, refs[b], opts_of(case), (case, config))
                caught.append(config)
    assert caught, (case, instead)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASE_IDS)
@pytest.mark.parametrize("path,family,Nr,N,T,tuning", GPU_PATHS, ids=[c[0] for c in GPU_PATHS])
def test_gpu_options_follow_the_oracle(pkg, torch_cuda, path, family, Nr, N, T, tuning, case):
    opts = opts_of(case)
    prob, orc, nlps, W, P, bnds, names = gpu_setup(pkg, family, Nr, N, T, tuning, opts)
    out = prob.solve(*[_t(torch_cuda, a) for a in (W, P) + tuple(bnds)], trace=opts["max_iter"] + 1)
    torch_cuda.cuda.synchronize()
    out = {k: v.cpu().numpy() for k, v in out.items()}
    rep = REPORT.setdefault(path, [0.0, 0.0, 0.0])
    relax, tol = relax_of(opts), opts.get("tol", 1e-8)
    for b, name in enumerate(names):
        r = orc.solve(W[b], P[b], *bnds, trace=True)
        check_device_instance(out, b, r, opts, (path, case, name), rep)
        assert_within_relaxed_bounds(out["x"][b], bnds[0], bnds[1], relax)
        if int(out["status"][b]) == 0 and nlps[b] is not None:
            # the rows are met to the stopping tolerance, the variable bounds to the relaxation
            df = objective_scaling(nlps[b], W[b], P[b], max_gradient=opts.get("nlp_scaling_max_gradient", 100.0))
            cert = certify(nlps[b], out["x"][b], out["lam_x"][b], out["lam_g"][b], P[b], *bnds, df, relax=relax, tol=tol,
                           feas=max(relax, tol))
            rep[2] = max(rep[2], cert["stat"])


# the Van der Pol thread path has no IPM oracle: the status each option set implies, the certificate, and that it acts
VDP_CASES = CASE_IDS


@pytest.fixture(scope="module")
def vdp_default(pkg):
    ocp = pkg.SmallOcp("van_der_pol", N=20, T=10.0, rk_steps=4, max_iter=MAX_ITER)
    w0, lbw, ubw, lbg, ubg = ocp.demo_arrays()
    W0 = np.tile(w0, (3, 1)); W0[1:, 2:] += 0.05 * np.random.default_rng(3).normal(size=(2, len(w0) - 2))
    return W0, (lbw, ubw, lbg, ubg), ocp.solve_host(W0, lbw, ubw, lbg, ubg)


@pytest.mark.gpu
@pytest.mark.parametrize("case", VDP_CASES)
def test_gpu_van_der_pol_options(pkg, torch_cuda, vdp_default, case):
    from oracle.vdp_nlp import VdpNLP
    opts = opts_of(case)
    W0, (lbw, ubw, lbg, ubg), base = vdp_default
    assert (base["status"] == 0).all()
    out = pkg.SmallOcp("van_der_pol", N=20, T=10.0, rk_steps=4, **opts).solve_host(W0, lbw, ubw, lbg, ubg)
    nlp, relax, tol = VdpNLP(), relax_of(opts), opts.get("tol", 1e-8)
    print("VDP %-28s status %s iters %s (default %s)" % (case, out["status"], out["iters"], base["iters"]))
    if case == "acceptable":
        assert (out["status"] == 1).all(), out["status"]
    elif case.startswith("max_iter"):
        k = opts["max_iter"]
        assert (out["status"] == np.where(base["iters"] > k, 2, 0)).all() and (out["iters"] == np.minimum(base["iters"], k)).all()
    else:
        assert (out["status"] == 0).all(), out["status"]
    for b in range(len(W0)):
        assert_within_relaxed_bounds(out["x"][b], lbw, ubw, relax)
        if out["status"][b] == 0:
            df = objective_scaling(nlp, W0[b], None, lbw, ubw, max_gradient=opts.get("nlp_scaling_max_gradient", 100.0))
            certify(nlp, out["x"][b], out["lam_x"][b], out["lam_g"][b], None, lbw, ubw, lbg, ubg, df, relax=relax,
                    tol=max(tol, 1e-6), feas=max(relax, tol, 1e-6))
    if case in VDP_ACTS:
        assert (out["iters"] != base["iters"]).any(), (case, out["iters"], base["iters"])


# the cases that change the Van der Pol demo's iteration count (on a B200: 9 iterations by default).  The others leave it at 9:
# no SOC or restoration happens, its bounds are far from the start or fixed (push / frac, relax), its gradient is below 1
# (df = 1), kappa_d moves the path by less than it takes to change a count, and its stopping tests meet the others' at once.
VDP_ACTS = ["mu_init=1", "kappa_mu,theta_mu", "barrier_tol_factor=2", "bound_mult_init_val=0.3", "kappa_sigma=2", "acceptable",
            "acceptable,tiny_obj_change", "tol=1e-5", "viol<compl", "compl<viol"] + [c for c in CASE_IDS if c.startswith("max_iter")]


# ---- 4. small related checks ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_nlpsol_shim_forwards_options(pkg, torch_cuda):
    """nlpsol(..., {'ipopt': {...}}) is Problem(**options): bit-identical outputs; stats() reports the termination branch;
    keys outside nmpc_opts (print_level, mu_strategy) are accepted and ignored."""
    Nr, N, T = 3, 8, 0.3
    W, P, names, bnds = _cached(("central", Nr, N, T), centralized_starts, Nr, N, T)
    desc = {"family": "unicycle_centralized", "Nr": Nr, "N": N, "T": T}
    for kw, want, success in ((dict(mu_init=1e-3, max_iter=3), "MAX_ITER", False), (ACCEPTABLE, "ACCEPTABLE", True),
                              (dict(tol=1e-5), "SOLVED", True)):
        solver = pkg.nlpsol("solver", "ipopt", desc, {"print_time": 0, "ipopt": dict(kw, print_level=0, mu_strategy="monotone")})
        sol = solver(x0=W[0], p=P[0], lbx=bnds[0], ubx=bnds[1], lbg=bnds[2], ubg=bnds[3])
        ref = pkg.Problem(Nr, N, T, **kw).solve_host(W[:1], P[:1], *bnds)
        for k in ("x", "g", "lam_x", "lam_g"):
            np.testing.assert_array_equal(np.asarray(sol[k]).ravel(), ref[k][0], err_msg=k)
        st = solver.stats()
        assert (st["return_status"], st["success"], st["iter_count"]) == (want, success, int(ref["iters"][0])), st
    # a misspelt or foreign key changes nothing
    a = pkg.nlpsol("s", "ipopt", desc, {"ipopt": {"mu_strategy": "adaptive", "linear_solver": "ma57"}})(
        x0=W[1], p=P[1], lbx=bnds[0], ubx=bnds[1], lbg=bnds[2], ubg=bnds[3])
    b = pkg.Problem(Nr, N, T).solve_host(W[1:2], P[1:2], *bnds)
    np.testing.assert_array_equal(np.asarray(a["x"]).ravel(), b["x"][0])


@pytest.mark.gpu
def test_gpu_launch_tuning_changes_no_result(pkg, torch_cuda):
    """nmpc_tuning promises no effect on results.  ctas_per_sm = 1 and B = 700 > 148 SMs x 4 teams = 592 resident warp teams
    (Nr = 2), so the convoy runs and scratch slots are reused; the batch mixes solved instances, origin instances (INFEASIBLE)
    and instances that max_iter truncates.  convoy 0 / 1 / 2, one call per instance, trace on and want=() give the same bits."""
    torch = torch_cuda
    Nr, N, T, B = 2, 8, 0.3, 700
    rng = np.random.default_rng(5)
    base = ring(Nr)
    P = np.tile(base, (B, 1))
    P[:, :3 * Nr] += 0.3 * rng.normal(size=(B, 3 * Nr))
    P[::7, :3 * Nr] = 0.0                             # every robot at the origin: INFEASIBLE
    probe = Oracle(Nr, N, T)
    bnds = probe.bounds(0.3, 0.22, 2.84)
    W = np.stack([probe.cold_start(q[:3 * Nr]) for q in P])
    it = probe.solve_batch(W, P, *bnds)["iters"]
    max_iter = int(np.median(it[it > 0]))            # truncates the slower half
    args = [_t(torch, a) for a in (W, P) + tuple(bnds)]
    keys = ("x", "lam_g", "status", "iters")
    runs = {}
    for convoy in (0, 1, 2):
        prob = pkg.Problem(Nr, N, T, tuning=dict(convoy=convoy, ctas_per_sm=1), max_iter=max_iter)
        runs[convoy] = {k: v.cpu().numpy() for k, v in prob.solve(*args).items()}
    st = runs[0]["status"]
    assert (st == 0).any() and (st == 2).any() and (st == 3).sum() >= B // 7, np.bincount(st)
    for convoy in (1, 2):
        for k in keys:
            np.testing.assert_array_equal(runs[convoy][k], runs[0][k], err_msg="convoy %d %s" % (convoy, k))
    prob = pkg.Problem(Nr, N, T, tuning=dict(convoy=2, ctas_per_sm=1), max_iter=max_iter)
    tr = {k: v.cpu().numpy() for k, v in prob.solve(*args, trace=max_iter + 1).items()}
    bare = {k: v.cpu().numpy() for k, v in prob.solve(*args, want=()).items()}
    for k in keys:
        np.testing.assert_array_equal(tr[k], runs[0][k], err_msg="trace " + k)
    for k in ("x", "status", "iters"):
        np.testing.assert_array_equal(bare[k], runs[0][k], err_msg="want=() " + k)
    for b in range(B):
        one = {k: v.cpu().numpy() for k, v in prob.solve(*[a[b:b + 1] for a in args[:2]], *args[2:]).items()}
        for k in keys:
            np.testing.assert_array_equal(one[k][0], runs[0][k][b], err_msg="alone %d %s" % (b, k))

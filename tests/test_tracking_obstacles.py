"""Trajectory tracking among obstacles (nmpc_create_tracking_obstacles): the per-stage reference of nmpc_create_tracking and the
per-stage obstacle tables of nmpc_create_moving_obstacles in one p = [x0bar; Z; O].  CPU: the combined C oracle against the
moving-obstacle oracle on constant references, the NumPy restatement and SLSQP, and the product's <NR, true, true>
instantiation in the fibre emulation.  GPU: bitwise equivalence with the moving-obstacle handle on constant references,
time-varying references among per-instance obstacle fields against the combined oracle, traces, the KKT certificate, SLSQP,
the closed loop, the nlpsol shim, the error paths and run-to-run reproducibility."""
import numpy as np
import pytest

from tests.obstacles_in_p import MovingOracle
from tests.test_moving_obstacles import EQUIV, _field, _orc_bounds, _start_goal
from tests.tracking_obstacles_ref import (TrackingObstaclesOracle, TrackingStageObstacleNLP, pack,
                                          tracking_obstacles_emu_solve)
from tests.tracking_ref import constant_reference, line_reference


def _crossing(N=20, T=0.3, speed=0.2):
    """One robot following a line reference from (0, 0) to (2.4, 0) at `speed`; one obstacle (clearance 0.35) crossing the line
    upwards at x = 1.2 at 0.15 m/s, timed to reach the line when the reference does.  x0bar [3], Z [N, 5], O [N, 1, 3]."""
    start = np.array([0.0, 0.0, 0.0])
    Z = line_reference(start, [2.4, 0.0, 0.0], N, T, speed=speed)
    t = np.arange(N) * T
    O = np.stack([np.full(N, 1.2), 0.15 * (t - 1.2 / speed), np.full(N, 0.35)], axis=1)[:, None, :]
    return start, Z, O


def _two_robot_case(N=8, T=0.3):
    """Two robots swapping sides along line references, past two obstacles that drift across the horizon."""
    start = np.array([-1.0, -0.1, 0.0, 1.0, -0.1, np.pi])
    Z = line_reference(start, [1.0, 0.1, 0.0, -1.0, 0.1, np.pi], N, T, speed=0.15)
    t = np.arange(N) * T
    O = np.stack([np.stack([np.full(N, 0.1), 0.8 - 0.1 * t, np.full(N, 0.3)], 1),
                  np.stack([-0.3 + 0.05 * t, np.full(N, -0.9), np.full(N, 0.25)], 1)], axis=1)
    return start, Z, O


def _four_robot_case(N=6, T=0.3):
    """Four robots crossing a square along line references among six obstacles (6 pair rows + 4 x 6 obstacle rows = 30 lanes)."""
    ang = np.pi / 4 + np.pi / 2 * np.arange(4)
    head = ang + np.pi
    start = np.stack([1.2 * np.cos(ang), 1.2 * np.sin(ang), np.angle(np.exp(1j * head))], 1).ravel()
    goal = np.stack([-1.2 * np.cos(ang), -1.2 * np.sin(ang), np.angle(np.exp(1j * head))], 1).ravel()
    Z = line_reference(start, goal, N, T, speed=0.15)
    t = np.arange(N) * T
    # one obstacle just off each robot's line, 0.3 m ahead of its start, and two away from the lines
    off = 0.04 * np.stack([-np.sin(ang), np.cos(ang)], 1)
    c = np.concatenate([0.9 * np.stack([np.cos(ang), np.sin(ang)], 1) + off, [[0.0, 0.0], [1.3, 0.0]]])
    O = np.stack([c[None, :, 0] + 0.03 * t[:, None], c[None, :, 1] - 0.02 * t[:, None], np.full((N, 6), 0.2)], axis=-1)
    return start, Z, O


def _lines(Nr, B, rng, N, T):
    """B line references (antipodal swaps on a circle, jittered) and x0bar near their starts: x0bar [B, 3Nr], Z [B, N, 5Nr]."""
    P = _start_goal(Nr, B, rng)
    Z = np.stack([line_reference(P[b, :3 * Nr], P[b, 3 * Nr:], N, T, speed=rng.uniform(0.1, 0.18)) for b in range(B)])
    X0 = P[:, :3 * Nr] + 0.02 * rng.normal(size=(B, 3 * Nr))
    return X0, Z


def _moving_field(rng, B, nobs, N, T):
    """Per-instance obstacle fields drifting at up to 5 cm/s: [B, N, nobs, 3]."""
    F = _field(rng, B, nobs, N)
    F[..., :2] += np.arange(N)[None, :, None, None] * T * rng.uniform(-0.05, 0.05, size=(B, 1, nobs, 2))
    return F


# ---------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("Nr,nobs", [(1, 6), (2, 3)])
def test_oracle_constant_reference_is_the_moving_oracle(Nr, nobs):
    N, T = 10, 0.3
    rng = np.random.default_rng(Nr)
    P = _start_goal(Nr, 1, rng)[0]
    O = _moving_field(rng, 1, nobs, N, T)[0]
    mv, tr = MovingOracle(Nr, N, T, nobs), TrackingObstaclesOracle(Nr, N, T, nobs)
    assert (tr.n, tr.mg, tr.np_) == (mv.n, mv.mg, 3 * Nr + 5 * Nr * N + 3 * N * nobs)
    lbx, ubx, lbg, ubg = _orc_bounds(mv, nobs, 0.05)
    w0 = mv.cold_start(P[:3 * Nr])
    a = mv.solve(w0, np.concatenate([P, O.ravel()]), lbx, ubx, lbg, ubg, trace=True)
    b = tr.solve(w0, pack(P[:3 * Nr], constant_reference(N, P[3 * Nr:]), O), lbx, ubx, lbg, ubg, trace=True)
    assert a["status"] == 0
    for k in ("x", "g", "lam_x", "lam_g", "trace", "stats"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    assert (a["f"], a["status"], a["iters"]) == (b["f"], b["status"], b["iters"])


def test_numpy_cost_rows_and_derivatives_match_the_oracle():
    N, T = 20, 0.3
    x0, Z, O = _crossing(N, T)
    nlp, orc = TrackingStageObstacleNLP(N, T, O), TrackingObstaclesOracle(1, N, T, 1)
    p = pack(x0, Z, O)
    rng = np.random.default_rng(5)
    w = rng.normal(size=nlp.n)
    eps = 1e-6
    fd = np.array([(nlp.f(w + eps * e, p) - nlp.f(w - eps * e, p)) / (2 * eps) for e in np.eye(nlp.n)])
    np.testing.assert_allclose(nlp.grad_f(w, p), fd, atol=1e-6)
    Jfd = np.stack([(nlp.g(w + eps * e, p) - nlp.g(w - eps * e, p)) / (2 * eps) for e in np.eye(nlp.n)], axis=1)
    np.testing.assert_allclose(nlp.jac_g(w, p), Jfd, atol=1e-8)
    # the oracle's returned f and g at its solution are the NumPy ones (whose tables come from O, not from p: so the oracle
    # reads O at 3 + 5 N)
    lbx, ubx, lbg, ubg = nlp.bounds(0.05, 0.3, np.pi / 4)
    r = orc.solve(nlp.cold_start(x0), p, lbx, ubx, lbg, ubg)
    assert r["status"] == 0
    np.testing.assert_allclose(r["g"], nlp.g(r["x"], p), rtol=0, atol=1e-12)
    assert abs(r["f"] - nlp.f(r["x"], p)) <= 1e-12 * max(1.0, abs(r["f"]))
    # the control reference enters the cost: moving ur moves f
    p2 = p.copy()
    p2[3 + 3] += 0.1
    assert nlp.f(r["x"], p2) != nlp.f(r["x"], p)


def test_slsqp_confirms_the_oracle_on_a_crossing_obstacle():
    N, T = 20, 0.3
    x0, Z, O = _crossing(N, T)
    nlp, orc = TrackingStageObstacleNLP(N, T, O), TrackingObstaclesOracle(1, N, T, 1)
    lbx, ubx, lbg, ubg = nlp.bounds(0.05, 0.3, np.pi / 4)
    p = pack(x0, Z, O)
    r = orc.solve(nlp.cold_start(x0), p, lbx, ubx, lbg, ubg)
    assert r["status"] == 0
    g = nlp.g(r["x"], p)
    assert (g[lbg != ubg] < 0.05 + 1e-6).any(), "the crossing obstacle should be active"
    ref = nlp.solve_slsqp(nlp.cold_start(x0), p, lbx, ubx, lbg, ubg)
    if np.abs(ref.x - r["x"])[nlp.nX:].max() > 1e-4:      # SLSQP found another local minimum: polish from the oracle's point
        ref = nlp.solve_slsqp(r["x"], p, lbx, ubx, lbg, ubg)
        assert ref.fun >= r["f"] - 1e-9 * max(1.0, abs(r["f"]))
    assert np.abs(ref.x - r["x"])[nlp.nX:].max() <= 1e-4
    assert abs(ref.fun - r["f"]) <= 1e-6 * abs(r["f"])


EMU_CASES = {"one_robot_crossing": (1, 20, 0.3, _crossing),
             "two_robots_per_stage": (2, 8, 0.3, _two_robot_case),
             "four_robots_30_lanes": (4, 6, 0.3, _four_robot_case)}


@pytest.mark.parametrize("case", list(EMU_CASES))
@pytest.mark.parametrize("reverse", [0, 1])
def test_emulated_kernel_follows_the_oracle(case, reverse, monkeypatch):
    Nr, N, T, make = EMU_CASES[case]
    x0, Z, O = make(N, T)
    nobs = O.shape[1]
    assert Nr * (Nr - 1) // 2 + Nr * nobs <= 32
    orc = TrackingObstaclesOracle(Nr, N, T, nobs)
    lbx, ubx, lbg, ubg = _orc_bounds(orc, nobs, 0.05, v=0.3)
    p = pack(x0, Z, O)
    w0 = orc.cold_start(x0)
    r = orc.solve(w0, p, lbx, ubx, lbg, ubg, trace=True)
    e = tracking_obstacles_emu_solve(monkeypatch, Nr, N, T, w0, p, lbx, ubx, lbg, ubg, nobs, trace=True, reverse=reverse)
    assert e["rc"] == 0 and e["status"][0] == r["status"] == 0
    assert abs(int(e["iters"][0]) - r["iters"]) <= 2
    nX = 3 * Nr * (N + 1)
    assert np.abs(e["x"][0] - r["x"])[nX:].max() <= 1e-7
    assert abs(e["f"][0] - r["f"]) / r["f"] <= 1e-9
    np.testing.assert_allclose(e["g"][0], r["g"], atol=1e-8)
    np.testing.assert_allclose(e["lam_g"][0], r["lam_g"], atol=1e-5)
    m = min(int(e["iters"][0]), r["iters"]) - 3
    np.testing.assert_allclose(e["trace"][0][:m, [0, 6, 7]], r["trace"][:m, [0, 6, 7]], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(e["trace"][0][:m, [2, 3, 4, 5]], r["trace"][:m, [2, 3, 4, 5]], rtol=1e-5, atol=1e-9)


def test_params_packs_numpy():
    """Problem.params needs no device for NumPy input; the handle does, so call it on a stand-in with the same attributes."""
    import __graft_entry__ as ge
    Problem = ge.load_package().Problem
    fake = Problem.__new__(Problem)
    fake.ns, fake.nc, fake.N, fake.nobs, fake.moving, fake.tracking = 3, 2, 4, 2, True, True
    B = 5
    rng = np.random.default_rng(0)
    x0bar, xr, ur, O = rng.normal(size=(B, 3)), rng.normal(size=(B, 4, 3)), rng.normal(size=(B, 4, 2)), rng.normal(size=(B, 4, 2, 3))
    p = fake.params(x0bar, xr, obstacles=O, uref=ur)
    assert p.shape == (B, 3 + 5 * 4 + 3 * 4 * 2) and p.dtype == np.float64
    np.testing.assert_array_equal(p[:, :3], x0bar)
    Z = p[:, 3:23].reshape(B, 4, 5)
    np.testing.assert_array_equal(Z[:, :, :3], xr)
    np.testing.assert_array_equal(Z[:, :, 3:], ur)
    np.testing.assert_array_equal(p[:, 23:].reshape(B, 4, 2, 3), O)
    pc = fake.params(x0bar, xr[:, 0], O)                 # constant reference [B, 3Nr], uref defaults to zeros
    np.testing.assert_array_equal(pc[:, 3:23], constant_reference(4, xr[:, 0]))
    np.testing.assert_array_equal(pc[:, 23:], O.reshape(B, -1))
    for bad in (dict(obstacles=None), dict(obstacles=O[:, :3]), dict(obstacles=O, uref=ur[:, :2])):
        with pytest.raises(ValueError):
            fake.params(x0bar, xr, **bad)


# ---------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _t(torch, a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda:0")


def _np(out):
    return {k: v.cpu().numpy() for k, v in out.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("Nr,N,nobs,tuning,batched", EQUIV)
def test_gpu_constant_reference_is_bitwise_the_moving_obstacle_handle(pkg, torch_cuda, Nr, N, nobs, tuning, batched):
    torch = torch_cuda
    rng = np.random.default_rng(Nr * 100 + nobs)
    B, T = 64, 0.3
    mv = pkg.Problem(Nr, N, T, moving_obstacles=nobs, tuning=tuning)
    tr = pkg.Problem(Nr, N, T, tracking_obstacles=nobs, tuning=tuning)
    assert (tr.n, tr.mg, tr.np_) == (mv.n, mv.mg, 3 * Nr + 5 * Nr * N + 3 * N * nobs)
    P = _start_goal(Nr, B, rng)
    O = _moving_field(rng, B, nobs, N, T)
    lbx, ubx, lbg, ubg = mv.bounds_obstacles(0.05, 0.2, np.pi / 4, dmin=0.3)
    assert all(np.array_equal(a, b) for a, b in zip((lbx, ubx, lbg, ubg), tr.bounds_obstacles(0.05, 0.2, np.pi / 4, dmin=0.3)))
    if batched:
        lbx, ubx, lbg, ubg = (np.tile(a, (B, 1)) for a in (lbx, ubx, lbg, ubg))
        lbg[:, -Nr * nobs:] += 0.01 * rng.uniform(size=(B, 1))
    x0 = mv.cold_start(P[:, :3 * Nr])
    bnd = [_t(torch, a) for a in (lbx, ubx, lbg, ubg)]
    a = mv.solve(_t(torch, x0), mv.params(_t(torch, P[:, :3 * Nr]), _t(torch, P[:, 3 * Nr:]), _t(torch, O)), *bnd)
    pt = tr.params(_t(torch, P[:, :3 * Nr]), _t(torch, P[:, 3 * Nr:]), obstacles=_t(torch, O))
    b = tr.solve(_t(torch, x0), pt, *bnd)
    torch.cuda.synchronize()
    assert (a["status"] == 0).double().mean().item() >= 0.9
    for k in ("x", "f", "g", "lam_x", "lam_g", "status", "iters"):
        assert torch.equal(a[k], b[k]), k


PATHS = [(1, 6, None), (2, 3, None), (2, 3, dict(force_block_path=1))]


@pytest.mark.gpu
@pytest.mark.parametrize("Nr,nobs,tuning", PATHS)
def test_gpu_time_varying_references_among_obstacles_match_the_oracle(pkg, torch_cuda, Nr, nobs, tuning):
    torch = torch_cuda
    rng = np.random.default_rng(17 + Nr)
    B, N, T, margin = 256, 12, 0.3, 0.05
    prob = pkg.Problem(Nr, N, T, tracking_obstacles=nobs, tuning=tuning)
    orc = TrackingObstaclesOracle(Nr, N, T, nobs)
    X0, Z = _lines(Nr, B, rng, N, T)
    p = prob.params(X0, Z[..., :3 * Nr], obstacles=_moving_field(rng, B, nobs, N, T), uref=Z[..., 3 * Nr:])
    lbx, ubx, lbg, ubg = prob.bounds_obstacles(margin, 0.2, np.pi / 4, dmin=0.3)
    x0 = prob.cold_start(X0)
    out = _np(prob.solve(_t(torch, x0), _t(torch, p), *(_t(torch, a) for a in (lbx, ubx, lbg, ubg))))
    ref = orc.solve_batch(x0, p, lbx, ubx, lbg, ubg)
    x, f, g, st, it = out["x"], out["f"], out["g"], out["status"], out["iters"]
    nX = 3 * Nr * (N + 1)
    ineq = lbg != ubg
    viol = np.maximum(np.abs(g[:, ~ineq]).max(1), np.maximum(lbg[ineq][None] - g[:, ineq], 0).max(1))
    ok = ((np.abs(x - ref["x"])[:, nX:].max(1) <= 1e-4) & (np.abs(f - ref["f"]) <= 1e-6 * np.maximum(1.0, np.abs(ref["f"])))
          & (viol <= 1e-6) & (st == ref["status"]) & (np.abs(it - ref["iters"]) <= 3))
    assert ok.mean() >= 0.99, (ok.mean(), np.nonzero(~ok)[0][:10])
    assert (st == 0).mean() >= 0.9


@pytest.mark.gpu
@pytest.mark.parametrize("Nr,nobs,tuning", PATHS)
def test_gpu_trace_follows_the_oracle(pkg, torch_cuda, Nr, nobs, tuning):
    """solve(trace=K) on a few instances: the same status, iteration count and line-search counts as the oracle, mu and
    delta_w to the last bits, theta, f, alpha and alpha_z to 1e-9 relative."""
    torch = torch_cuda
    rng = np.random.default_rng(29 + Nr)
    B, N, T = 4, 12, 0.3
    prob = pkg.Problem(Nr, N, T, tracking_obstacles=nobs, tuning=tuning)
    orc = TrackingObstaclesOracle(Nr, N, T, nobs)
    X0, Z = _lines(Nr, B, rng, N, T)
    p = prob.params(X0, Z[..., :3 * Nr], obstacles=_moving_field(rng, B, nobs, N, T), uref=Z[..., 3 * Nr:])
    lbx, ubx, lbg, ubg = prob.bounds_obstacles(0.05, 0.2, np.pi / 4, dmin=0.3)
    x0 = prob.cold_start(X0)
    K = int(prob.opts.max_iter) + 1
    out = _np(prob.solve(_t(torch, x0), _t(torch, p), *(_t(torch, a) for a in (lbx, ubx, lbg, ubg)), trace=K))
    for b in range(B):
        r = orc.solve(x0[b], p[b], lbx, ubx, lbg, ubg, trace=True)
        it = int(out["iters"][b])
        assert (int(out["status"][b]), it) == (r["status"], r["iters"]), b
        a, ref = out["trace"][b][:it], r["trace"][:it]
        np.testing.assert_array_equal(a[:, 7], ref[:, 7])
        np.testing.assert_allclose(a[:, [0, 6]], ref[:, [0, 6]], rtol=1e-13, atol=0)
        np.testing.assert_allclose(a[:, [2, 3, 4, 5]], ref[:, [2, 3, 4, 5]], rtol=1e-9, atol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("tuning", [None, dict(force_block_path=1)], ids=["warp", "forced-block"])
def test_gpu_kkt_certificate_one_robot(pkg, torch_cuda, tuning):
    from tests.kkt_certificate import certify, objective_scaling
    torch = torch_cuda
    N, T, nobs, B = 12, 0.3, 4, 4
    rng = np.random.default_rng(41)
    prob = pkg.Problem(1, N, T, tracking_obstacles=nobs, tuning=tuning)
    X0, Z = _lines(1, B, rng, N, T)
    O = _moving_field(rng, B, nobs, N, T)
    p = prob.params(X0, Z[..., :3], obstacles=O, uref=Z[..., 3:])
    lbx, ubx, lbg, ubg = prob.bounds_obstacles(0.05, 0.2, np.pi / 4)
    x0 = prob.cold_start(X0)
    out = _np(prob.solve(_t(torch, x0), _t(torch, p), *(_t(torch, a) for a in (lbx, ubx, lbg, ubg))))
    assert (out["status"] == 0).all(), out["status"]
    for b in range(B):
        nlp = TrackingStageObstacleNLP(N, T, O[b])
        m = certify(nlp, out["x"][b], out["lam_x"][b], out["lam_g"][b], p[b], lbx, ubx, lbg, ubg,
                    objective_scaling(nlp, x0[b], p[b]))
        if out["stats"][b, 0] <= 1e-8:
            assert m["scaled_err"] <= 2e-8, (b, m["scaled_err"], out["stats"][b, 0])


@pytest.mark.gpu
@pytest.mark.parametrize("tuning", [None, dict(force_block_path=1)], ids=["warp", "forced-block"])
def test_gpu_crossing_obstacle_matches_slsqp(pkg, torch_cuda, tuning):
    torch = torch_cuda
    N, T = 20, 0.3
    x0, Z, O = _crossing(N, T)
    nlp = TrackingStageObstacleNLP(N, T, O)
    lbx, ubx, lbg, ubg = nlp.bounds(0.05, 0.3, np.pi / 4)
    prob = pkg.Problem(1, N, T, tracking_obstacles=1, tuning=tuning)
    p = prob.params(x0[None], Z[None, :, :3], obstacles=O[None], uref=Z[None, :, 3:])
    np.testing.assert_array_equal(p[0], pack(x0, Z, O))
    out = prob.solve(_t(torch, prob.cold_start(x0[None])), _t(torch, p), *(_t(torch, a) for a in (lbx, ubx, lbg, ubg)))
    x, f = out["x"].cpu().numpy()[0], float(out["f"].cpu().numpy()[0])
    assert int(out["status"][0]) == 0
    np.testing.assert_allclose(out["g"].cpu().numpy()[0], nlp.g(x, p[0]), atol=1e-10)
    ref = nlp.solve_slsqp(nlp.cold_start(x0), p[0], lbx, ubx, lbg, ubg)
    if np.abs(ref.x - x)[nlp.nX:].max() > 1e-4:
        ref = nlp.solve_slsqp(x, p[0], lbx, ubx, lbg, ubg)
        assert ref.fun >= f - 1e-9 * max(1.0, abs(f))
    assert np.abs(ref.x - x)[nlp.nX:].max() <= 1e-4
    assert abs(ref.fun - f) <= 1e-6 * abs(f)


def _closed_loop_case(steps, N, T, B=4):
    """B robots following the line (0, 0) -> (3.6, 0) at 0.15 m/s from slightly different poses; an obstacle (clearance
    0.35) crosses the line upwards at x = 0.9 when the reference is there (t = 6 s) at a per-instance speed, and a second one
    (clearance 0.25) drifts along y = 0.8 towards the start.  P [B, 3], reference [steps + N, B, 5], obstacles
    [steps + N, B, 2, 3]."""
    P = np.array([[0.0, 0.0, 0.0], [0.0, 0.1, 0.2], [0.05, -0.1, -0.2], [0.0, 0.0, 0.1]])[:B]
    ref = np.repeat(line_reference([0.0, 0.0, 0.0], [3.6, 0.0, 0.0], N, T, steps, speed=0.15)[:, None], B, axis=1)
    tt = np.arange(steps + N)[:, None] * T
    vy = np.array([0.15, 0.10, 0.12, 0.18])[None, :B]
    ob = np.zeros((steps + N, B, 2, 3))
    ob[..., 0, 0], ob[..., 0, 1], ob[..., 0, 2] = 0.9, vy * (tt - 6.0), 0.35
    ob[..., 1, 0], ob[..., 1, 1], ob[..., 1, 2] = 3.0 - 0.05 * tt, 0.8, 0.25
    return P, ref, ob


@pytest.mark.gpu
def test_gpu_closed_loop_tracks_a_line_past_moving_obstacles(pkg, torch_cuda):
    torch = torch_cuda
    N, T, steps, B, margin = 20, 0.3, 40, 4, 0.05
    prob = pkg.Problem(1, N, T, tracking_obstacles=2)
    orc = TrackingObstaclesOracle(1, N, T, 2)
    lbx, ubx, lbg, ubg = prob.bounds_obstacles(margin, 0.3, np.pi / 4)
    P, ref, ob = _closed_loop_case(steps, N, T, B)
    res = pkg.closed_loop(prob, _t(torch, P), *(_t(torch, a) for a in (lbx, ubx, lbg, ubg)), steps,
                          reference=_t(torch, ref), obstacles=_t(torch, ob))
    status, u = res["status"].cpu().numpy(), res["u"].cpu().numpy()
    assert (status <= 1).all(), status
    assert res["active"].all().item()
    # the oracle's closed loop: same plant, same shift warm start, same reference and obstacle windows
    state = P.copy()
    x0 = np.stack([orc.cold_start(P[b]) for b in range(B)])
    for t in range(steps):
        for b in range(B):
            r = orc.solve(x0[b], pack(state[b], ref[t:t + N, b], ob[t:t + N, b]), lbx, ubx, lbg, ubg)
            u0 = r["x"][3 * (N + 1):3 * (N + 1) + 2]
            assert np.abs(u[t, b] - u0).max() <= 1e-4, (t, b, u[t, b], u0)
            state[b] = orc.plant(state[b], u0)
            x0[b] = orc.shift(r["x"])
    np.testing.assert_allclose(res["traj"].cpu().numpy()[-1], state, atol=1e-4)
    assert (res["min_clearance"].cpu().numpy() >= margin - 1e-6).all(), res["min_clearance"]
    err = res["track_err"].cpu().numpy()
    assert err.shape == (steps + 1, B)
    # the crossing obstacle holds the robots back (the oracle's loop: up to 0.5 m behind at t = 6.3 s); once it has passed they
    # catch up, and from t = 10.8 s every robot is within 5 cm of its reference (oracle: 2.7 cm, and 5 mm at t = 12 s)
    assert err[15:30].max() >= 0.3, err[15:30].max()
    assert err[36:].max() <= 0.05, err[36:].max()
    assert err[-1].max() <= 0.01, err[-1]


@pytest.mark.gpu
def test_gpu_nlpsol_shim_tracking_obstacles(pkg, torch_cuda):
    N, T = 20, 0.3
    x0, Z, O = _crossing(N, T)
    nlp = TrackingStageObstacleNLP(N, T, O)
    solver = pkg.nlpsol("solver", "ipopt", {"family": "unicycle_tracking_obstacles", "Nr": 1, "N": N, "T": T, "n_obs": 1},
                        {"print_time": 0, "ipopt": {"max_iter": 2000, "print_level": 0}})
    lbx, ubx, lbg, ubg = nlp.bounds(0.05, 0.3, np.pi / 4)
    p = pack(x0, Z, O)
    sol = solver(x0=nlp.cold_start(x0), p=p, lbx=lbx, ubx=ubx, lbg=lbg, ubg=ubg)
    assert solver.stats()["success"]
    w = np.asarray(sol["x"].full()).ravel()
    lam_g = np.asarray(sol["lam_g"].full()).ravel()
    np.testing.assert_allclose(np.asarray(sol["g"].full()).ravel(), nlp.g(w, p), atol=1e-10)

    def lagr(pv):   # f + lam_g' g at the solution, as a function of all of p (reference and obstacle blocks)
        n2 = TrackingStageObstacleNLP(N, T, pv[3 + 5 * N:].reshape(N, 1, 3))
        return n2.f(w, pv) + lam_g @ n2.g(w, pv)
    eps = 1e-6
    fd = np.array([(lagr(p + eps * e) - lagr(p - eps * e)) / (2 * eps) for e in np.eye(p.size)])
    lam_p = np.asarray(sol["lam_p"].full()).ravel()
    assert lam_p.shape == p.shape
    np.testing.assert_allclose(lam_p, fd, atol=1e-6)
    assert np.abs(lam_p[3:3 + 5 * N]).max() > 1e-3, "the reference block should carry a multiplier"
    assert np.abs(lam_p[3 + 5 * N:]).max() > 1e-3, "the obstacle block should carry a multiplier"


@pytest.mark.gpu
def test_gpu_errors(pkg, torch_cuda):
    torch = torch_cuda
    from nmpc_b200._cabi import NmpcError
    for bad in (0, 33):
        with pytest.raises(NmpcError):
            pkg.Problem(1, 10, 0.3, tracking_obstacles=bad)
    for kw in (dict(tracking=True), dict(moving_obstacles=2), dict(obstacles=[[1.0, 1.0, 0.3]])):
        with pytest.raises(ValueError):
            pkg.Problem(1, 10, 0.3, tracking_obstacles=2, **kw)
    prob = pkg.Problem(1, 10, 0.3, tracking_obstacles=2)
    assert prob.tracking and prob.moving and prob.np_ == 3 + 5 * 10 + 3 * 10 * 2
    lbx, ubx, lbg, ubg = prob.bounds_obstacles(0.05, 0.2, np.pi / 4)
    bnd = [_t(torch, a) for a in (lbx, ubx, lbg, ubg)]
    P = np.array([[0.0, 0.0, 0.0, 1.0, 0.0, 0.0]])
    x0 = prob.cold_start(P[:, :3])
    for width in (6 + 3 * 10 * 2, 3 + 5 * 10, 6):     # the moving-obstacle, the tracking and the plain p
        with pytest.raises(ValueError):
            prob.solve(_t(torch, x0), _t(torch, np.zeros((1, width))), *bnd)
        with pytest.raises(ValueError):
            prob.solve_host(x0, np.zeros((1, width)), lbx, ubx, lbg, ubg)
    steps = 3
    ref, ob = _t(torch, np.zeros((steps + 10, 1, 5))), _t(torch, np.zeros((steps + 10, 1, 2, 3)))
    with pytest.raises(ValueError):
        pkg.closed_loop(prob, _t(torch, P), *bnd, steps, reference=ref)
    with pytest.raises(ValueError):
        pkg.closed_loop(prob, _t(torch, P), *bnd, steps, obstacles=ob)
    with pytest.raises(ValueError):
        pkg.closed_loop(prob, _t(torch, P), *bnd, steps)
    with pytest.raises(ValueError):      # wrong shapes
        pkg.closed_loop(prob, _t(torch, P), *bnd, steps, reference=ref[:, :, :3], obstacles=ob)
    with pytest.raises(ValueError):
        pkg.closed_loop(prob, _t(torch, P), *bnd, steps, reference=ref, obstacles=ob[:, :, :1])
    mv = pkg.Problem(1, 10, 0.3, moving_obstacles=2)
    with pytest.raises(ValueError):      # reference= on the moving-obstacle handle
        pkg.closed_loop(mv, _t(torch, P), *bnd, steps, reference=ref, obstacles=ob)
    with pytest.raises(NmpcError):
        prob.eval(_t(torch, x0), _t(torch, np.zeros((1, prob.np_))))
    with pytest.raises(NmpcError):
        prob.jac_pattern()
    with pytest.raises(NmpcError):
        prob.hess_pattern()


@pytest.mark.gpu
@pytest.mark.parametrize("Nr,nobs,tuning", PATHS + [(4, 7, None)], ids=["warp-1x6", "warp-2x3", "forced-block-2x3", "block-4x7"])
def test_gpu_bitwise_reproducible(pkg, torch_cuda, Nr, nobs, tuning):
    torch = torch_cuda
    rng = np.random.default_rng(53 + Nr)
    B, N, T = 96, 10, 0.3
    prob = pkg.Problem(Nr, N, T, tracking_obstacles=nobs, tuning=tuning)
    X0, Z = _lines(Nr, B, rng, N, T)
    p = _t(torch, prob.params(X0, Z[..., :3 * Nr], obstacles=_moving_field(rng, B, nobs, N, T), uref=Z[..., 3 * Nr:]))
    bnd = [_t(torch, a) for a in prob.bounds_obstacles(0.05, 0.2, np.pi / 4, dmin=0.3)]
    x0 = _t(torch, prob.cold_start(X0))
    a = prob.solve(x0, p, *bnd)
    b = prob.solve(x0, p, *bnd)
    torch.cuda.synchronize()
    assert (a["status"] <= 1).double().mean().item() >= 0.9
    for k in ("x", "f", "g", "lam_x", "lam_g", "status", "iters", "stats"):
        assert torch.equal(a[k], b[k]), k

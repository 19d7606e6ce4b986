"""Obstacles carried in p (nmpc_create_moving_obstacles): per-instance and per-stage obstacle tables for the static-obstacle
family.  CPU: the C oracle's obstacles-in-p mode against its static mode and against the NumPy restatement / SLSQP, and the
product's device source in the fibre emulation.  GPU: bitwise equivalence with the static handle on a repeated table,
per-instance layouts against the oracle, moving obstacles (SLSQP, closed loop), the nlpsol shim and the error paths."""
import numpy as np
import pytest

from oracle.oracle_lib import Oracle
from tests.obstacles_in_p import MovingOracle, StageObstacleNLP, moving_emu_solve

THIRD = [(-0.6, 3.3, 0.2), (0.6, 3.3, 0.125), (0.0, 2.3, 0.15), (1.0, 2.3, 0.15), (-0.6, 1.3, 0.2), (0.6, 1.3, 0.175)]
OBS6 = np.array([[x, y, r + 0.15] for x, y, r in THIRD])


def _repeat(obs, N, B=None):
    """[n_obs, 3] -> the O block [N * n_obs * 3] (one copy per stage); [B, ...] when B is given."""
    O = np.tile(np.asarray(obs, float).ravel(), N)
    return O if B is None else np.tile(O, (B, 1))


def _crossing(N=20, T=0.3):
    """One robot driving from (0, 0) to (2.4, 0); one obstacle (clearance 0.35) crossing its path upwards at 0.15 m/s, timed to
    meet it halfway.  O [N, 1, 3]."""
    t = np.arange(N) * T
    O = np.stack([np.full(N, 1.2), -0.9 + 0.15 * t, np.full(N, 0.35)], axis=1)[:, None, :]
    p6 = np.array([0.0, 0.0, 0.0, 2.4, 0.0, 0.0])
    return p6, O


def _two_robot_case(N=8, T=0.3):
    """Two robots swapping sides past two obstacles that drift across the horizon."""
    p6 = np.array([-1.0, -0.1, 0.0, 1.0, 0.1, np.pi, 1.0, -0.1, 0.0, -1.0, 0.1, np.pi])
    t = np.arange(N) * T
    O = np.stack([np.stack([np.full(N, 0.1), 0.8 - 0.1 * t, np.full(N, 0.3)], 1),
                  np.stack([-0.3 + 0.05 * t, np.full(N, -0.9), np.full(N, 0.25)], 1)], axis=1)
    return p6, O


def _orc_bounds(orc, nobs, margin, dmin=0.3, v=0.2, w=np.pi / 4):
    """bounds_obstacles of the product, restated for the oracle's dimensions."""
    inf, ns, N = np.inf, orc.ns, orc.N
    lbx = np.concatenate([np.tile([-10.0, -10.0, -2 * np.pi], orc.Nr * (N + 1)), np.tile([-v, -w], orc.Nr * N)])
    blk_lo = np.concatenate([np.zeros(ns), np.full(orc.M, dmin * dmin), np.full(orc.Nr * nobs, margin)])
    blk_hi = np.concatenate([np.zeros(ns), np.full(orc.M + orc.Nr * nobs, inf)])
    return lbx, -lbx, np.concatenate([np.zeros(ns), np.tile(blk_lo, N)]), np.concatenate([np.zeros(ns), np.tile(blk_hi, N)])


# ---------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("Nr", [1, 2])
def test_oracle_repeated_table_is_the_static_oracle(Nr):
    N, T = 10, 0.3
    obs = OBS6[:3] if Nr == 1 else np.array([[0.0, 0.9, 0.3], [0.2, -0.8, 0.25]])
    p6 = np.array([0.0, 0.6, 1.57, 0.1, 3.9, 1.57]) if Nr == 1 else _two_robot_case(N, T)[0]
    st, mv = Oracle(Nr, N, T, obstacles=obs), MovingOracle(Nr, N, T, len(obs))
    assert (mv.n, mv.mg, mv.np_) == (st.n, st.mg, 6 * Nr + 3 * N * len(obs))
    lbx, ubx, lbg, ubg = _orc_bounds(st, len(obs), 0.1)
    w0 = st.cold_start(p6[:3 * Nr])
    a = st.solve(w0, p6, lbx, ubx, lbg, ubg, trace=True)
    b = mv.solve(w0, np.concatenate([p6, _repeat(obs, N)]), lbx, ubx, lbg, ubg, trace=True)
    assert a["status"] == 0
    for k in ("x", "g", "lam_x", "lam_g", "trace", "stats"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    assert (a["f"], a["status"], a["iters"]) == (b["f"], b["status"], b["iters"])


def test_numpy_per_stage_rows_and_derivatives():
    N, T = 20, 0.3
    p6, O = _crossing(N, T)
    nlp = StageObstacleNLP(N, T, O)
    assert nlp.no == 1 and nlp.mg == 3 + N * 4
    rng = np.random.default_rng(3)
    w = rng.normal(size=nlp.n)
    eps = 1e-6
    Jfd = np.stack([(nlp.g(w + eps * e, p6) - nlp.g(w - eps * e, p6)) / (2 * eps) for e in np.eye(nlp.n)], axis=1)
    np.testing.assert_allclose(nlp.jac_g(w, p6), Jfd, atol=1e-8)
    X, _ = nlp.split(w)
    g = nlp.g(w, p6)
    for k in (0, 7, N - 1):       # row (k, o) on X_k against the stage-k obstacle
        assert g[3 + k * 4 + 3] == pytest.approx(np.hypot(X[k, 0] - O[k, 0, 0], X[k, 1] - O[k, 0, 1]) - O[k, 0, 2], abs=1e-14)
    # the C oracle evaluates the same rows at its solution
    orc = MovingOracle(1, N, T, 1)
    lbx, ubx, lbg, ubg = nlp.bounds(0.05, 0.2, np.pi / 4)
    p = np.concatenate([p6, O.ravel()])
    r = orc.solve(nlp.cold_start(p6[:3]), p, lbx, ubx, lbg, ubg)
    assert r["status"] == 0
    np.testing.assert_allclose(r["g"], nlp.g(r["x"], p6), atol=1e-12)
    assert abs(r["f"] - nlp.f(r["x"], p6)) <= 1e-10 * max(1.0, abs(r["f"]))


def test_slsqp_confirms_the_oracle_on_a_crossing_obstacle():
    N, T = 20, 0.3
    p6, O = _crossing(N, T)
    nlp, orc = StageObstacleNLP(N, T, O), MovingOracle(1, N, T, 1)
    lbx, ubx, lbg, ubg = nlp.bounds(0.05, 0.2, np.pi / 4)
    r = orc.solve(nlp.cold_start(p6[:3]), np.concatenate([p6, O.ravel()]), lbx, ubx, lbg, ubg)
    assert r["status"] == 0
    g = nlp.g(r["x"], p6)
    assert (g[lbg != ubg] < 0.05 + 1e-6).any(), "the moving obstacle should be active"
    ref = nlp.solve_slsqp(nlp.cold_start(p6[:3]), p6, lbx, ubx, lbg, ubg)
    if np.abs(ref.x - r["x"])[nlp.nX:].max() > 1e-4:      # SLSQP found another local minimum: polish from the oracle's point
        ref = nlp.solve_slsqp(r["x"], p6, lbx, ubx, lbg, ubg)
        assert ref.fun >= r["f"] - 1e-9 * max(1.0, abs(r["f"]))
    assert np.abs(ref.x - r["x"])[nlp.nX:].max() <= 1e-4
    assert abs(ref.fun - r["f"]) <= 1e-6 * abs(r["f"])


@pytest.mark.parametrize("case", ["one_robot_crossing", "two_robots_per_stage"])
@pytest.mark.parametrize("reverse", [0, 1])
def test_emulated_kernel_follows_the_oracle_with_obstacles_in_p(case, reverse, monkeypatch):
    if case == "one_robot_crossing":
        Nr, N, T = 1, 20, 0.3
        p6, O = _crossing(N, T)
    else:
        Nr, N, T = 2, 8, 0.3
        p6, O = _two_robot_case(N, T)
    orc = MovingOracle(Nr, N, T, O.shape[1])
    lbx, ubx, lbg, ubg = _orc_bounds(orc, O.shape[1], 0.05)
    p = np.concatenate([p6, O.ravel()])
    w0 = orc.cold_start(p6[:3 * Nr])
    r = orc.solve(w0, p, lbx, ubx, lbg, ubg, trace=True)
    e = moving_emu_solve(monkeypatch, Nr, N, T, w0, p, lbx, ubx, lbg, ubg, O.shape[1], trace=True, reverse=reverse)
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
    fake.ns, fake.N, fake.nobs, fake.moving = 3, 4, 2, True
    B = 5
    rng = np.random.default_rng(0)
    x0bar, xs, O = rng.normal(size=(B, 3)), rng.normal(size=(B, 3)), rng.normal(size=(B, 4, 2, 3))
    p = fake.params(x0bar, xs, O)
    assert p.shape == (B, 6 + 3 * 4 * 2) and p.dtype == np.float64
    np.testing.assert_array_equal(p[:, :3], x0bar)
    np.testing.assert_array_equal(p[:, 3:6], xs)
    np.testing.assert_array_equal(p[:, 6:].reshape(B, 4, 2, 3), O)
    with pytest.raises(ValueError):
        fake.params(x0bar, xs, O[:, :3])
    with pytest.raises(ValueError):
        fake.params(x0bar, xs)


# ---------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _t(torch, a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda:0")


def _start_goal(Nr, B, rng):
    """B start/goal pairs for Nr robots on a circle of radius 1.6 (antipodal swaps, jittered)."""
    ang = 2 * np.pi * np.arange(Nr) / Nr + 0.3
    head = np.angle(np.exp(1j * (ang + np.pi)))      # facing the centre, inside the +-2 pi box of bounds_obstacles
    st = np.stack([1.6 * np.cos(ang), 1.6 * np.sin(ang), head], 1).ravel()
    gl = np.stack([-1.6 * np.cos(ang), -1.6 * np.sin(ang), head], 1).ravel()
    P = np.tile(np.concatenate([st, gl]), (B, 1))
    P[:, 0:3 * Nr:3] += 0.05 * rng.normal(size=(B, Nr)); P[:, 1:3 * Nr:3] += 0.05 * rng.normal(size=(B, Nr))
    return P


def _field(rng, B, nobs, N=None):
    """Random obstacle fields inside the circle, away from the start poses: [B, nobs, 3] (or [B, N, nobs, 3] repeated)."""
    r, a = 0.9 * np.sqrt(rng.uniform(size=(B, nobs))), rng.uniform(0, 2 * np.pi, size=(B, nobs))
    F = np.stack([r * np.cos(a), r * np.sin(a), rng.uniform(0.15, 0.3, size=(B, nobs))], -1)
    return F if N is None else np.repeat(F[:, None], N, axis=1)


EQUIV = [  # (Nr, N, n_obs, tuning, batched bounds)
    (1, 20, 6, None, False), (1, 20, 6, None, True), (2, 10, 3, None, False), (4, 8, 2, None, True),
    (2, 10, 3, dict(force_block_path=1), False), (2, 10, 3, dict(force_block_path=1), True),
    (4, 8, 7, None, False),       # 6 pair rows + 28 obstacle rows > 32 lanes: the dense-block path
]


@pytest.mark.gpu
@pytest.mark.parametrize("Nr,N,nobs,tuning,batched", EQUIV)
def test_gpu_repeated_table_is_bitwise_the_static_handle(pkg, torch_cuda, Nr, N, nobs, tuning, batched):
    torch = torch_cuda
    rng = np.random.default_rng(Nr * 100 + nobs)
    B, T = 64, 0.3
    obs = _field(rng, 1, nobs)[0]
    st = pkg.Problem(Nr, N, T, obstacles=obs, tuning=tuning)
    mv = pkg.Problem(Nr, N, T, moving_obstacles=nobs, tuning=tuning)
    assert (mv.n, mv.mg, mv.np_) == (st.n, st.mg, 6 * Nr + 3 * N * nobs)
    P = _start_goal(Nr, B, rng)
    lbx, ubx, lbg, ubg = st.bounds_obstacles(0.05, 0.2, np.pi / 4, dmin=0.3)
    if batched:
        lbx, ubx, lbg, ubg = (np.tile(a, (B, 1)) for a in (lbx, ubx, lbg, ubg))
        lbg[:, -Nr * nobs:] += 0.01 * rng.uniform(size=(B, 1))
    x0 = st.cold_start(P[:, :3 * Nr])
    bnd = [_t(torch, a) for a in (lbx, ubx, lbg, ubg)]
    a = st.solve(_t(torch, x0), _t(torch, P), *bnd)
    pm = mv.params(_t(torch, P[:, :3 * Nr]), _t(torch, P[:, 3 * Nr:]), _t(torch, np.tile(obs, (B, N, 1, 1))))
    b = mv.solve(_t(torch, x0), pm, *bnd)
    torch.cuda.synchronize()
    assert (a["status"] == 0).double().mean().item() >= 0.9
    for k in ("x", "f", "g", "lam_x", "lam_g", "status", "iters"):
        assert torch.equal(a[k], b[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("Nr,nobs,tuning", [(1, 6, None), (2, 3, None), (2, 3, dict(force_block_path=1))])
def test_gpu_per_instance_layouts_match_the_oracle(pkg, torch_cuda, Nr, nobs, tuning):
    torch = torch_cuda
    rng = np.random.default_rng(7 + Nr)
    B, N, T, margin = 256, 12, 0.3, 0.05
    prob = pkg.Problem(Nr, N, T, moving_obstacles=nobs, tuning=tuning)
    orc = MovingOracle(Nr, N, T, nobs)
    P6 = _start_goal(Nr, B, rng)
    p = prob.params(P6[:, :3 * Nr], P6[:, 3 * Nr:], _field(rng, B, nobs, N))
    lbx, ubx, lbg, ubg = prob.bounds_obstacles(margin, 0.2, np.pi / 4, dmin=0.3)
    x0 = prob.cold_start(P6[:, :3 * Nr])
    out = prob.solve(_t(torch, x0), _t(torch, p), *(_t(torch, a) for a in (lbx, ubx, lbg, ubg)))
    ref = orc.solve_batch(x0, p, lbx, ubx, lbg, ubg)
    x, f, g = (out[k].cpu().numpy() for k in ("x", "f", "g"))
    st, it = out["status"].cpu().numpy(), out["iters"].cpu().numpy()
    nX = 3 * Nr * (N + 1)
    ineq = lbg != ubg
    viol = np.maximum(np.abs(g[:, ~ineq]).max(1), np.maximum(lbg[ineq][None] - g[:, ineq], 0).max(1))
    ok = ((np.abs(x - ref["x"])[:, nX:].max(1) <= 1e-4) & (np.abs(f - ref["f"]) <= 1e-6 * np.maximum(1.0, np.abs(ref["f"])))
          & (viol <= 1e-6) & (st == ref["status"]) & (np.abs(it - ref["iters"]) <= 3))
    assert ok.mean() >= 0.99, (ok.mean(), np.nonzero(~ok)[0][:10])
    assert (st == 0).mean() >= 0.9


@pytest.mark.gpu
def test_gpu_crossing_obstacle_matches_slsqp(pkg, torch_cuda):
    torch = torch_cuda
    N, T = 20, 0.3
    p6, O = _crossing(N, T)
    nlp = StageObstacleNLP(N, T, O)
    lbx, ubx, lbg, ubg = nlp.bounds(0.05, 0.2, np.pi / 4)
    for tuning in (None, dict(force_block_path=1)):
        prob = pkg.Problem(1, N, T, moving_obstacles=1, tuning=tuning)
        p = prob.params(p6[None, :3], p6[None, 3:], O[None])
        out = prob.solve(_t(torch, prob.cold_start(p6[None, :3])), _t(torch, p), *(_t(torch, a) for a in (lbx, ubx, lbg, ubg)))
        x, f = out["x"].cpu().numpy()[0], float(out["f"].cpu().numpy()[0])
        assert int(out["status"][0]) == 0
        np.testing.assert_allclose(out["g"].cpu().numpy()[0], nlp.g(x, p6), atol=1e-10)
        ref = nlp.solve_slsqp(nlp.cold_start(p6[:3]), p6, lbx, ubx, lbg, ubg)
        if np.abs(ref.x - x)[nlp.nX:].max() > 1e-4:
            ref = nlp.solve_slsqp(x, p6, lbx, ubx, lbg, ubg)
            assert ref.fun >= f - 1e-9 * max(1.0, abs(f))
        assert np.abs(ref.x - x)[nlp.nX:].max() <= 1e-4
        assert abs(ref.fun - f) <= 1e-6 * abs(f)


@pytest.mark.gpu
def test_gpu_closed_loop_with_moving_obstacles_matches_the_oracle(pkg, torch_cuda):
    torch = torch_cuda
    N, T, steps, B, margin = 20, 0.3, 40, 4, 0.05
    prob = pkg.Problem(1, N, T, moving_obstacles=2)
    orc = MovingOracle(1, N, T, 2)
    lbx, ubx, lbg, ubg = prob.bounds_obstacles(margin, 0.2, np.pi / 4)
    P = np.array([[0.0, 0.0, 0.0, 2.4, 0.0, 0.0], [0.0, 0.2, 0.3, 2.4, -0.2, 0.0],
                  [0.1, -0.1, -0.2, 2.2, 0.3, 0.0], [0.0, 0.0, 0.1, 2.4, 0.1, 0.0]])
    # known trajectories: one obstacle crossing upwards, one drifting towards the start; time t = index * T
    tt = np.arange(steps + N)[:, None] * T
    vy = np.array([0.15, 0.10, 0.12, 0.18])[None]
    ob = np.zeros((steps + N, B, 2, 3))
    ob[..., 0, 0], ob[..., 0, 1], ob[..., 0, 2] = 1.2, -0.9 + vy * tt, 0.35
    ob[..., 1, 0], ob[..., 1, 1], ob[..., 1, 2] = 3.0 - 0.05 * tt, 0.8, 0.25
    res = pkg.closed_loop(prob, _t(torch, P), *(_t(torch, a) for a in (lbx, ubx, lbg, ubg)), steps, obstacles=_t(torch, ob))
    status = res["status"].cpu().numpy()
    u = res["u"].cpu().numpy()
    active = res["active"].cpu().numpy()
    # oracle closed loop: same plant, same shift warm start, same obstacle windows
    state = P[:, :3].copy()
    x0 = np.stack([orc.cold_start(P[b, :3]) for b in range(B)])
    for t in range(steps):
        for b in range(B):
            act = active[t, b]
            p = np.concatenate([state[b], P[b, 3:], ob[t:t + N, b].ravel()])
            r = orc.solve(x0[b], p, lbx, ubx, lbg, ubg)
            u0 = r["x"][3 * (N + 1):3 * (N + 1) + 2]
            if act:
                assert np.abs(u[t, b] - u0).max() <= 1e-4, (t, b, u[t, b], u0)
                state[b] = orc.plant(state[b], u0)
            x0[b] = orc.shift(r["x"])
    solved = (status <= 1).all(axis=0)
    assert solved.all(), status
    assert (res["min_clearance"].cpu().numpy()[solved] >= margin - 1e-6).all(), res["min_clearance"]
    np.testing.assert_allclose(res["traj"].cpu().numpy()[-1], state, atol=1e-4)


@pytest.mark.gpu
def test_gpu_nlpsol_shim_with_obstacles_in_p(pkg, torch_cuda):
    N, T = 20, 0.3
    p6, O = _crossing(N, T)
    nlp = StageObstacleNLP(N, T, O)
    solver = pkg.nlpsol("solver", "ipopt", {"family": "unicycle_moving_obstacles", "Nr": 1, "N": N, "T": T, "n_obs": 1},
                        {"print_time": 0, "ipopt": {"max_iter": 2000, "print_level": 0}})
    lbx, ubx, lbg, ubg = nlp.bounds(0.05, 0.2, np.pi / 4)
    p = np.concatenate([p6, O.ravel()])
    sol = solver(x0=nlp.cold_start(p6[:3]), p=p, lbx=lbx, ubx=ubx, lbg=lbg, ubg=ubg)
    assert solver.stats()["success"]
    w = np.asarray(sol["x"].full()).ravel()
    lam_g = np.asarray(sol["lam_g"].full()).ravel()
    np.testing.assert_allclose(np.asarray(sol["g"].full()).ravel(), nlp.g(w, p6), atol=1e-10)

    def lagr(pv):   # f + lam_g' g at the solution, as a function of p (obstacle block included)
        n2 = StageObstacleNLP(N, T, pv[6:].reshape(N, 1, 3))
        return n2.f(w, pv[:6]) + lam_g @ n2.g(w, pv[:6])
    eps = 1e-6
    fd = np.array([(lagr(p + eps * e) - lagr(p - eps * e)) / (2 * eps) for e in np.eye(p.size)])
    lam_p = np.asarray(sol["lam_p"].full()).ravel()
    assert lam_p.shape == p.shape
    np.testing.assert_allclose(lam_p, fd, atol=1e-6)
    assert np.abs(lam_p[6:]).max() > 1e-3, "the obstacle block should carry a multiplier"


@pytest.mark.gpu
def test_gpu_errors(pkg, torch_cuda):
    torch = torch_cuda
    from nmpc_b200._cabi import NmpcError
    for bad in (0, 33):
        with pytest.raises(NmpcError):
            pkg.Problem(1, 10, 0.3, moving_obstacles=bad)
    with pytest.raises(ValueError):
        pkg.Problem(1, 10, 0.3, obstacles=OBS6, moving_obstacles=6)
    prob = pkg.Problem(1, 10, 0.3, moving_obstacles=2)
    assert prob.np_ == 6 + 3 * 10 * 2
    lbx, ubx, lbg, ubg = prob.bounds_obstacles(0.05, 0.2, np.pi / 4)
    P = np.array([[0.0, 0.0, 0.0, 1.0, 0.0, 0.0]])
    x0 = prob.cold_start(P[:, :3])
    with pytest.raises(ValueError):      # p without the obstacle block
        prob.solve(_t(torch, x0), _t(torch, P), *(_t(torch, a) for a in (lbx, ubx, lbg, ubg)))
    with pytest.raises(ValueError):
        prob.solve_host(x0, P, lbx, ubx, lbg, ubg)
    with pytest.raises(NmpcError):
        prob.eval(_t(torch, x0), _t(torch, np.zeros((1, prob.np_))))
    with pytest.raises(NmpcError):
        prob.jac_pattern()
    with pytest.raises(NmpcError):
        prob.hess_pattern()

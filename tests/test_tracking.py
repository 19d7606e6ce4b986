"""Trajectory tracking (nmpc_create_tracking): a per-instance, per-stage state and control reference Z[k] = [xr_k; ur_k] in p for
the centralized family.  CPU: the derived C oracle against the setpoint oracle, the NumPy restatement and SLSQP, and the
product's tracking instantiation in the fibre emulation.  GPU: bitwise equivalence with nmpc_create on constant references,
time-varying references against the derived oracle, nmpc_eval, the closed loop, the nlpsol shim and the error paths."""
import numpy as np
import pytest

from oracle.oracle_lib import Oracle
from tests.tracking_ref import (TrackingNLP, TrackingOracle, constant_reference, line_reference, rotation_reference,
                                tracking_emu_solve)


def _circle(Nr, radius=1.6, phase=0.3):
    """Nr robots evenly on a circle, facing the centre: [3 Nr]."""
    ang = 2 * np.pi * np.arange(Nr) / Nr + phase
    return np.stack([radius * np.cos(ang), radius * np.sin(ang), np.angle(np.exp(1j * (ang + np.pi)))], 1).ravel()


def _swap(Nr, radius=1.6):
    """Start / goal of the antipodal swap on a circle: p6 = [start; goal]."""
    st = _circle(Nr, radius)
    gl = st.copy()
    gl[0::3], gl[1::3] = -st[0::3], -st[1::3]
    return np.concatenate([st, gl])


def _rotation_case(Nr, N, T, steps=0, radius=None, omega=0.2, jitter=0.03, seed=0):
    """x0bar near the start of a rotating-formation reference, and the reference rows [steps + N, 5 Nr]."""
    radius = radius or (1.0 if Nr == 1 else max(1.0, 0.35 * Nr))
    Zt = rotation_reference(_circle(Nr, radius), N, T, steps, omega)
    x0 = Zt[0, :3 * Nr] + jitter * np.sin(1.0 + seed + 2.0 * np.arange(3 * Nr))
    return x0, Zt


def _bounds(orc_or_prob, dmin=0.3, v=0.6, w=np.pi / 2):
    return orc_or_prob.bounds(dmin, v, w)


# ---------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("Nr", [1, 2, 6])
def test_oracle_constant_reference_is_the_setpoint_oracle(Nr, hexagon_p):
    N, T = 10, 0.2
    p6 = hexagon_p if Nr == 6 else _swap(Nr)
    st, tr = Oracle(Nr, N, T), TrackingOracle(Nr, N, T)
    assert (tr.n, tr.mg, tr.np_) == (st.n, st.mg, 3 * Nr + 5 * Nr * N)
    lbx, ubx, lbg, ubg = _bounds(st, dmin=0.3 if Nr < 6 else 0.4, v=0.2, w=np.pi / 4)
    w0 = st.cold_start(p6[:3 * Nr] + 0.02 * np.sin(1.0 + 2.0 * np.arange(3 * Nr)))
    a = st.solve(w0, p6, lbx, ubx, lbg, ubg, trace=True)
    b = tr.solve(w0, np.concatenate([p6[:3 * Nr], constant_reference(N, p6[3 * Nr:])]), lbx, ubx, lbg, ubg, trace=True)
    assert a["status"] == 0
    for k in ("x", "g", "lam_x", "lam_g", "trace", "stats"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    assert (a["f"], a["status"], a["iters"]) == (b["f"], b["status"], b["iters"])


@pytest.mark.parametrize("Nr", [1, 2])
def test_numpy_cost_and_gradient_match_the_oracle(Nr):
    N, T = 8, 0.3
    rng = np.random.default_rng(11 + Nr)
    nlp, orc = TrackingNLP(Nr, N, T), TrackingOracle(Nr, N, T)
    for _ in range(3):
        w = rng.normal(size=nlp.n)
        p = rng.normal(size=orc.np_)
        e = orc.eval(w, p, want_jac=False, want_hess=False)
        f, gf = nlp.f(w, p), nlp.grad_f(w, p)
        assert abs(e["f"] - f) <= 1e-13 * max(1.0, abs(f))
        np.testing.assert_allclose(e["grad"], gf, rtol=1e-13, atol=1e-13)
        eps = 1e-6
        fd = np.array([(nlp.f(w + eps * d, p) - nlp.f(w - eps * d, p)) / (2 * eps) for d in np.eye(nlp.n)])
        np.testing.assert_allclose(gf, fd, atol=1e-6)
        # the control reference enters the cost: moving ur moves f
        p2 = p.copy()
        p2[3 * Nr + 3 * Nr] += 0.1
        assert nlp.f(w, p2) != f


@pytest.mark.parametrize("Nr", [1, 2])
def test_slsqp_confirms_the_oracle_on_a_time_varying_reference(Nr):
    N, T = 10, 0.3
    nlp, orc = TrackingNLP(Nr, N, T), TrackingOracle(Nr, N, T)
    if Nr == 1:
        start, goal = np.array([0.0, 0.0, 0.3]), np.array([1.5, 0.6, 0.0])
        x0 = start
        Zt = line_reference(start, goal, N, T)
    else:
        x0, Zt = _rotation_case(Nr, N, T)
    p = np.concatenate([x0, Zt.ravel()])
    lbx, ubx, lbg, ubg = nlp.bounds(0.3, 0.6, np.pi / 2)
    r = orc.solve(nlp.cold_start(x0), p, lbx, ubx, lbg, ubg)
    assert r["status"] == 0
    assert abs(r["f"] - nlp.f(r["x"], p)) <= 1e-10 * max(1.0, abs(r["f"]))
    ref = nlp.solve_slsqp(nlp.cold_start(x0), p, lbx, ubx, lbg, ubg)
    if np.abs(ref.x - r["x"])[nlp.ns * (N + 1):].max() > 1e-4:     # SLSQP found another local minimum: polish from the oracle's
        ref = nlp.solve_slsqp(r["x"], p, lbx, ubx, lbg, ubg)
        assert ref.fun >= r["f"] - 1e-9 * max(1.0, abs(r["f"]))
    assert np.abs(ref.x - r["x"])[nlp.ns * (N + 1):].max() <= 1e-4
    assert abs(ref.fun - r["f"]) <= 1e-6 * abs(r["f"])


@pytest.mark.parametrize("Nr", [1, 2, 6, 8])
@pytest.mark.parametrize("reverse", [0, 1])
def test_emulated_tracking_kernel_follows_the_oracle(Nr, reverse, monkeypatch):
    N, T = 8, 0.2
    orc = TrackingOracle(Nr, N, T)
    x0, Zt = _rotation_case(Nr, N, T, seed=Nr)
    p = np.concatenate([x0, Zt.ravel()])
    lbx, ubx, lbg, ubg = _bounds(orc)
    w0 = orc.cold_start(x0)
    r = orc.solve(w0, p, lbx, ubx, lbg, ubg, trace=True)
    e = tracking_emu_solve(monkeypatch, Nr, N, T, w0, p, lbx, ubx, lbg, ubg, trace=True, reverse=reverse)
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
    fake.ns, fake.nc, fake.N, fake.nobs, fake.moving, fake.tracking = 6, 4, 3, 0, False, True
    B = 5
    rng = np.random.default_rng(0)
    x0bar, xr, ur = rng.normal(size=(B, 6)), rng.normal(size=(B, 3, 6)), rng.normal(size=(B, 3, 4))
    p = fake.params(x0bar, xr, uref=ur)
    assert p.shape == (B, 6 + 10 * 3) and p.dtype == np.float64
    np.testing.assert_array_equal(p[:, :6], x0bar)
    Z = p[:, 6:].reshape(B, 3, 10)
    np.testing.assert_array_equal(Z[:, :, :6], xr)
    np.testing.assert_array_equal(Z[:, :, 6:], ur)
    pc = fake.params(x0bar, xr[:, 0])                   # constant reference, uref defaults to zeros
    np.testing.assert_array_equal(pc[:, 6:], constant_reference(3, xr[:, 0]))
    with pytest.raises(ValueError):
        fake.params(x0bar, xr, uref=ur[:, :2])
    with pytest.raises(ValueError):
        fake.params(x0bar, xr, np.zeros((B, 3, 1, 3)))
    fake.tracking = False
    with pytest.raises(ValueError):
        fake.params(x0bar, xr[:, 0], uref=ur)


# ---------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _t(torch, a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda:0")


def _swaps(Nr, B, rng):
    """B jittered antipodal swaps on a circle big enough for Nr robots: [B, 6 Nr]."""
    P = np.tile(_swap(Nr, radius=max(1.6, 0.3 * Nr)), (B, 1))
    P[:, 0:3 * Nr:3] += 0.05 * rng.normal(size=(B, Nr)); P[:, 1:3 * Nr:3] += 0.05 * rng.normal(size=(B, Nr))
    return P


EQUIV = [  # (Nr, N, tuning): warp path one warp, six robots, the two-warp team, the dense-block path, the forced block path
    (1, 20, None), (6, 20, None), (8, 12, None), (12, 10, None), (6, 12, dict(force_block_path=1)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("batched", [False, True])
@pytest.mark.parametrize("Nr,N,tuning", EQUIV)
def test_gpu_constant_reference_is_bitwise_nmpc_create(pkg, torch_cuda, Nr, N, tuning, batched):
    torch = torch_cuda
    rng = np.random.default_rng(Nr * 10 + N)
    B, T = 64, 0.2
    st = pkg.Problem(Nr, N, T, tuning=tuning)
    tr = pkg.Problem(Nr, N, T, tuning=tuning, tracking=True)
    assert (tr.n, tr.mg, tr.np_, tr.nnz_jac, tr.nnz_hess) == (st.n, st.mg, 3 * Nr + 5 * Nr * N, st.nnz_jac, st.nnz_hess)
    P = _swaps(Nr, B, rng)
    lbx, ubx, lbg, ubg = st.bounds(0.3, 0.6, np.pi / 2)
    if batched:
        lbx, ubx, lbg, ubg = (np.tile(a, (B, 1)) for a in (lbx, ubx, lbg, ubg))
        ubx[:, -2 * Nr * N::2] -= 0.1 * rng.uniform(size=(B, 1))
    x0 = st.cold_start(P[:, :3 * Nr])
    bnd = [_t(torch, a) for a in (lbx, ubx, lbg, ubg)]
    a = st.solve(_t(torch, x0), _t(torch, P), *bnd)
    pt = tr.params(_t(torch, P[:, :3 * Nr]), _t(torch, P[:, 3 * Nr:]))
    b = tr.solve(_t(torch, x0), pt, *bnd)
    torch.cuda.synchronize()
    assert (a["status"] == 0).double().mean().item() >= 0.9
    for k in ("x", "f", "g", "lam_x", "lam_g", "status", "iters", "stats"):
        assert torch.equal(a[k], b[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("Nr,B,N,tuning,dit", [(6, 256, 12, None, 3), (16, 8, 8, None, 5)])
def test_gpu_time_varying_references_match_the_oracle(pkg, torch_cuda, Nr, B, N, tuning, dit):
    torch = torch_cuda
    rng = np.random.default_rng(5 + Nr)
    T = 0.2
    prob = pkg.Problem(Nr, N, T, tuning=tuning, tracking=True)
    orc = TrackingOracle(Nr, N, T)
    X0, Zs = [], []
    for b in range(B):      # rotating formations: per-instance radius, rate, direction and start offset
        Zt = rotation_reference(_circle(Nr, max(1.0, 0.35 * Nr) * rng.uniform(0.9, 1.1), rng.uniform(0, 2 * np.pi)), N, T,
                                omega=rng.choice([-1, 1]) * rng.uniform(0.1, 0.3))
        X0.append(Zt[0, :3 * Nr] + 0.05 * rng.normal(size=3 * Nr))
        Zs.append(Zt)
    X0, Zs = np.array(X0), np.array(Zs)
    p = prob.params(X0, Zs[:, :, :3 * Nr], uref=Zs[:, :, 3 * Nr:])
    lbx, ubx, lbg, ubg = _bounds(prob)
    x0 = prob.cold_start(X0)
    out = prob.solve(_t(torch, x0), _t(torch, p), *(_t(torch, a) for a in (lbx, ubx, lbg, ubg)))
    ref = orc.solve_batch(x0, p, lbx, ubx, lbg, ubg)
    x, f, g = (out[k].cpu().numpy() for k in ("x", "f", "g"))
    st, it = out["status"].cpu().numpy(), out["iters"].cpu().numpy()
    nX = 3 * Nr * (N + 1)
    ineq = lbg != ubg
    viol = np.maximum(np.abs(g[:, ~ineq]).max(1), np.maximum(lbg[ineq][None] - g[:, ineq], 0).max(1))
    ok = ((np.abs(x - ref["x"])[:, nX:].max(1) <= 1e-4) & (np.abs(f - ref["f"]) <= 1e-6 * np.maximum(1.0, np.abs(ref["f"])))
          & (viol <= 1e-6) & (st == ref["status"]) & (np.abs(it - ref["iters"]) <= dit))
    assert ok.mean() >= (0.99 if B >= 100 else 1.0), (ok.mean(), np.nonzero(~ok)[0][:10])
    assert (st == 0).mean() >= 0.9


@pytest.mark.gpu
@pytest.mark.parametrize("Nr,N", [(2, 10), (6, 20), (12, 10)])
def test_gpu_eval_tracking(pkg, torch_cuda, Nr, N):
    torch = torch_cuda
    rng = np.random.default_rng(21 + Nr)
    B, T = 16, 0.2
    st, tr = pkg.Problem(Nr, N, T), pkg.Problem(Nr, N, T, tracking=True)
    nlp = TrackingNLP(Nr, N, T)
    for a, b in zip(st.jac_pattern() + st.hess_pattern(), tr.jac_pattern() + tr.hess_pattern()):
        np.testing.assert_array_equal(a, b)
    w = rng.normal(size=(B, tr.n))
    lam = rng.normal(size=(B, tr.mg))
    # time-varying reference: NumPy restatement
    p = rng.normal(size=(B, tr.np_))
    o = tr.eval(_t(torch, w), _t(torch, p), _t(torch, lam))
    for b in range(B):
        f = nlp.f(w[b], p[b])
        assert abs(o["f"][b].item() - f) <= 1e-12 * max(1.0, abs(f))
        np.testing.assert_allclose(o["grad"][b].cpu().numpy(), nlp.grad_f(w[b], p[b]), rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(o["g"][b].cpu().numpy(), nlp.g(w[b], p[b]), rtol=1e-12, atol=1e-12)
    # constant reference: bitwise the regular handle's evaluation
    P6 = rng.normal(size=(B, 6 * Nr))
    a = st.eval(_t(torch, w), _t(torch, P6), _t(torch, lam))
    c = tr.eval(_t(torch, w), tr.params(_t(torch, P6[:, :3 * Nr]), _t(torch, P6[:, 3 * Nr:])), _t(torch, lam))
    torch.cuda.synchronize()
    for k in ("f", "grad", "g", "jac", "hess"):
        assert torch.equal(a[k], c[k]), k


@pytest.mark.gpu
def test_gpu_closed_loop_tracks_rotating_formations(pkg, torch_cuda):
    torch = torch_cuda
    Nr, N, T, steps, B, dmin = 6, 12, 0.2, 40, 512, 0.3
    prob = pkg.Problem(Nr, N, T, tracking=True)
    rng = np.random.default_rng(3)
    refs, P = [], []
    for b in range(B):
        Zt = rotation_reference(_circle(Nr, rng.uniform(1.4, 1.8), rng.uniform(0, 2 * np.pi)), N, T, steps,
                                omega=rng.choice([-1, 1]) * rng.uniform(0.1, 0.3))
        refs.append(Zt)
        P.append(Zt[0, :3 * Nr] + 0.05 * rng.normal(size=3 * Nr))
    ref, P = np.stack(refs, axis=1), np.array(P)                    # [steps + N, B, 5 Nr], [B, 3 Nr]
    lbx, ubx, lbg, ubg = prob.bounds(dmin, 0.6, np.pi / 2)
    bnd = [_t(torch, a) for a in (lbx, ubx, lbg, ubg)]
    res = pkg.closed_loop(prob, _t(torch, P), *bnd, steps, reference=_t(torch, ref))
    status = res["status"].cpu().numpy()
    assert (status <= 1).all(), np.unique(status, return_counts=True)
    assert res["active"].all().item()
    assert (res["min_dist"].cpu().numpy() >= dmin - 1e-6).all()
    err = res["track_err"].cpu().numpy()
    assert err.shape == (steps + 1, B)
    # after a transient of 2 s every robot follows its formation within 10 cm (measured on a B200: 8.1 cm at most), and at the
    # end of the 8 s typically within a few millimetres
    assert err[10:].max() <= 0.1, err[10:].max()
    assert np.median(err[-1]) <= 0.02, np.median(err[-1])
    # the first steps of two instances against the derived oracle's closed loop (same plant, same shift warm start)
    orc = TrackingOracle(Nr, N, T)
    u = res["u"].cpu().numpy()
    for b in range(2):
        state = P[b].copy()
        x0 = orc.cold_start(state)
        for t in range(steps):
            r = orc.solve(x0, np.concatenate([state, ref[t:t + N, b].ravel()]), lbx, ubx, lbg, ubg)
            u0 = r["x"][3 * Nr * (N + 1):3 * Nr * (N + 1) + 2 * Nr]
            assert np.abs(u[t, b] - u0).max() <= 1e-4, (t, b)
            state = orc.plant(state, u0)
            x0 = orc.shift(r["x"])


@pytest.mark.gpu
def test_gpu_nlpsol_shim_tracking(pkg, torch_cuda):
    Nr, N, T = 2, 10, 0.2
    nlp = TrackingNLP(Nr, N, T)
    solver = pkg.nlpsol("solver", "ipopt", {"family": "unicycle_tracking", "Nr": Nr, "N": N, "T": T},
                        {"print_time": 0, "ipopt": {"max_iter": 2000, "print_level": 0}})
    x0, Zt = _rotation_case(Nr, N, T)
    p = np.concatenate([x0, Zt.ravel()])
    lbx, ubx, lbg, ubg = nlp.bounds(0.3, 0.6, np.pi / 2)
    sol = solver(x0=nlp.cold_start(x0), p=p, lbx=lbx, ubx=ubx, lbg=lbg, ubg=ubg)
    assert solver.stats()["success"]
    w = np.asarray(sol["x"].full()).ravel()
    lam_g = np.asarray(sol["lam_g"].full()).ravel()
    np.testing.assert_allclose(np.asarray(sol["g"].full()).ravel(), nlp.g(w, p), atol=1e-10)

    def lagr(pv):   # f + lam_g' g at the solution, as a function of p
        return nlp.f(w, pv) + lam_g @ nlp.g(w, pv)
    eps = 1e-6
    fd = np.array([(lagr(p + eps * e) - lagr(p - eps * e)) / (2 * eps) for e in np.eye(p.size)])
    lam_p = np.asarray(sol["lam_p"].full()).ravel()
    assert lam_p.shape == p.shape
    np.testing.assert_allclose(lam_p, fd, atol=1e-6)
    assert np.abs(lam_p[3 * Nr:]).max() > 1e-3, "the reference block should carry a multiplier"


@pytest.mark.gpu
def test_gpu_errors(pkg, torch_cuda):
    torch = torch_cuda
    with pytest.raises(ValueError):
        pkg.Problem(1, 10, 0.3, tracking=True, obstacles=[[1.0, 1.0, 0.3]])
    with pytest.raises(ValueError):
        pkg.Problem(1, 10, 0.3, tracking=True, moving_obstacles=2)
    prob = pkg.Problem(2, 10, 0.3, tracking=True)
    assert prob.np_ == 6 + 10 * 10
    lbx, ubx, lbg, ubg = prob.bounds(0.3, 0.6, np.pi / 2)
    P = _swap(2)[None]
    x0 = prob.cold_start(P[:, :6])
    bnd = [_t(torch, a) for a in (lbx, ubx, lbg, ubg)]
    with pytest.raises(ValueError):      # p = [x0bar; xs]: the regular width
        prob.solve(_t(torch, x0), _t(torch, P), *bnd)
    with pytest.raises(ValueError):
        prob.solve_host(x0, P, lbx, ubx, lbg, ubg)
    with pytest.raises(ValueError):      # a tracking problem needs reference=
        pkg.closed_loop(prob, _t(torch, P), *bnd, 3)
    with pytest.raises(ValueError):      # reference of the wrong shape
        pkg.closed_loop(prob, _t(torch, P), *bnd, 3, reference=_t(torch, np.zeros((3, 1, 10))))
    reg = pkg.Problem(2, 10, 0.3)
    with pytest.raises(ValueError):      # reference= on a regular problem
        pkg.closed_loop(reg, _t(torch, P), *bnd, 3, reference=_t(torch, np.zeros((13, 1, 10))))

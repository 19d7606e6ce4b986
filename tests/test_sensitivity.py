"""Parametric sensitivities of returned solutions (nmpc_solution_vjp / nmpc_solution_jvp, Problem.solution_vjp / solution_jvp /
solve_differentiable).  CPU: the NumPy Sigma-condensed reference against the active-set implicit-function derivative and
central differences of oracle re-solves; the product's sensitivity pass in the fibre emulation against the reference.  GPU: the
device pass on the GPU solver's own outputs against the reference and against central differences of GPU re-solves, the
adjoint identity, tracking against setpoint handles, the autograd function and the error paths."""
import numpy as np
import pytest

from oracle.oracle_lib import Oracle
from oracle.nlp_numpy import synthetic_instances
from tests import sensitivity_ref as SR
from tests.tracking_ref import TrackingOracle, rotation_reference


def _circle(Nr, radius, phase=0.3):
    ang = 2 * np.pi * np.arange(Nr) / Nr + phase
    return np.stack([radius * np.cos(ang), radius * np.sin(ang), np.angle(np.exp(1j * (ang + np.pi)))], 1).ravel()


def _swap(Nr, radius=None):
    """Antipodal swap on a circle: p = [start; goal]."""
    st = _circle(Nr, radius or max(1.0, 0.3 * Nr))
    gl = st.copy()
    gl[0::3], gl[1::3] = -st[0::3], -st[1::3]
    return np.concatenate([st, gl])


def _jitter(P, Nr, scale, seed):
    rng = np.random.default_rng(seed)
    P = np.atleast_2d(P).copy()
    P[:, :3 * Nr] += scale * rng.normal(size=P[:, :3 * Nr].shape)
    return P


def _tracking_params(Nr, N, T, B, seed):
    """B instances near a rotating-formation reference with per-instance phases: p = [x0bar; Z] [B, 3 Nr + 5 Nr N]."""
    rng = np.random.default_rng(seed)
    P = []
    for b in range(B):
        Zt = rotation_reference(_circle(Nr, max(1.0, 0.35 * Nr), phase=rng.uniform(0, 2 * np.pi)), N, T, 0, omega=0.2)
        P.append(np.concatenate([Zt[0, :3 * Nr] + 0.03 * rng.normal(size=3 * Nr), Zt[:N].reshape(-1)]))
    return np.array(P)


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


# (Nr, N, T, tracking, dmin, v_max): the configurations of the CPU tests
CPU_CASES = {"1": (1, 10, 0.1, False, 0.25, 0.22), "2": (2, 10, 0.1, False, 0.25, 0.22), "6": (6, 10, 0.1, False, 0.4, 0.22),
             "8": (8, 6, 0.1, False, 0.4, 0.3), "2trk": (2, 10, 0.2, True, 0.3, 0.6), "6trk": (6, 8, 0.2, True, 0.3, 0.6),
             "8trk": (8, 6, 0.2, True, 0.3, 0.6)}


def _cpu_case(key, hexagon_p, B=3, tol=1e-11):
    """Oracle solutions of B instances of a configuration: (nlp, oracle, P [B, np], bounds, [solution dicts])."""
    Nr, N, T, trk, dmin, vmax = CPU_CASES[key]
    orc = (TrackingOracle if trk else Oracle)(Nr, N, T, tol=tol, acceptable_tol=tol)
    if trk:
        P = _tracking_params(Nr, N, T, B, seed=Nr)
    else:
        P = _jitter(np.tile(hexagon_p if Nr == 6 else _swap(Nr), (B, 1)), Nr, 0.03, seed=Nr)
        P[0] = hexagon_p if Nr == 6 else _swap(Nr)
    bounds = orc.bounds(dmin, vmax, np.pi / 2 if trk else 2.84)
    sols = [orc.solve(orc.cold_start(p[:3 * Nr]), p, *bounds) for p in P]
    return SR.nlp_for(Nr, N, T, trk), orc, P, bounds, sols


# ---------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("key", ["1", "2", "6", "2trk"])
def test_reference_matches_active_set_derivative_and_central_differences(key, hexagon_p):
    nlp, orc, P, bounds, sols = _cpu_case(key, hexagon_p)
    rng = np.random.default_rng(5)
    strict = 0
    for p, sol in zip(P, sols):
        assert sol["status"] == 0
        if not SR.strict_active_set(nlp, sol, p, bounds):
            continue
        strict += 1
        x_bar, p_dot = rng.normal(size=nlp.n), rng.normal(size=SR.n_params(nlp))
        pb, xd = SR.sigma_vjp(nlp, sol, p, bounds, x_bar), SR.sigma_jvp(nlp, sol, p, bounds, p_dot)
        assert _rel(SR.active_vjp(nlp, sol, p, bounds, x_bar), pb) <= 1e-6
        assert _rel(SR.active_jvp(nlp, sol, p, bounds, p_dot), xd) <= 1e-6
        eps = 1e-4
        sp, sm = orc.solve(sol["x"], p + eps * p_dot, *bounds), orc.solve(sol["x"], p - eps * p_dot, *bounds)
        assert sp["status"] == 0 and sm["status"] == 0
        assert _rel((sp["x"] - sm["x"]) / (2 * eps), xd) <= 1e-5
        assert abs(x_bar @ xd - pb @ p_dot) <= 1e-10 * (np.abs(x_bar) @ np.abs(xd))
    assert strict >= 1


@pytest.mark.parametrize("key", ["1", "2", "6", "8", "2trk", "6trk", "8trk"])
@pytest.mark.parametrize("lane_rev", [0, 1])
def test_emulated_pass_matches_the_reference(key, lane_rev, hexagon_p):
    nlp, _, P, bounds, sols = _cpu_case(key, hexagon_p, B=2)
    X, LX, LG = (np.array([s[k] for s in sols]) for k in ("x", "lam_x", "lam_g"))
    rng = np.random.default_rng(7)
    x_bar, p_dot = rng.normal(size=(len(P), nlp.n)), rng.normal(size=(len(P), SR.n_params(nlp)))
    pb, st, rc = SR.emu_sens(nlp, X, LX, LG, P, bounds, x_bar, 1, lane_rev)
    assert rc == 0 and np.all(st == 0)
    xd, st, rc = SR.emu_sens(nlp, X, LX, LG, P, bounds, p_dot, 0, lane_rev)
    assert rc == 0 and np.all(st == 0)
    for b, sol in enumerate(sols):
        assert _rel(pb[b], SR.sigma_vjp(nlp, sol, P[b], bounds, x_bar[b])) <= 1e-10
        assert _rel(xd[b], SR.sigma_jvp(nlp, sol, P[b], bounds, p_dot[b])) <= 1e-10
        assert abs(x_bar[b] @ xd[b] - pb[b] @ p_dot[b]) <= 1e-10 * (np.abs(x_bar[b]) @ np.abs(xd[b]))


def test_emulated_per_instance_bounds_equal_shared_bounds(hexagon_p):
    nlp, _, P, bounds, sols = _cpu_case("2", hexagon_p, B=2)
    X, LX, LG = (np.array([s[k] for s in sols]) for k in ("x", "lam_x", "lam_g"))
    x_bar = np.random.default_rng(3).normal(size=(len(P), nlp.n))
    a = SR.emu_sens(nlp, X, LX, LG, P, bounds, x_bar, 1)
    b = SR.emu_sens(nlp, X, LX, LG, P, [np.tile(v, (len(P), 1)) for v in bounds], x_bar, 1)
    np.testing.assert_array_equal(a[0], b[0])
    np.testing.assert_array_equal(a[1], b[1])


@pytest.mark.parametrize("key", ["2", "2trk"])
def test_emulated_wrong_inertia_gives_status_1_and_nan(key, hexagon_p):
    nlp, _, P, bounds, sols = _cpu_case(key, hexagon_p, B=1)
    sol = dict(sols[0])
    sol["lam_g"] = -40.0 * sol["lam_g"]                   # the Lagrangian's curvature turned negative
    parts = SR.kkt_parts(nlp, sol["x"], sol["lam_x"], sol["lam_g"], P[0], *bounds)
    assert SR.reduced_hessian_min_eig(parts) < 0          # the input really has the wrong inertia
    for reverse, seed in ((1, np.ones(nlp.n)), (0, np.ones(SR.n_params(nlp)))):
        out, st, rc = SR.emu_sens(nlp, sol["x"], sol["lam_x"], sol["lam_g"], P[0], bounds, seed, reverse)
        assert rc == 0 and st[0] == 1 and np.all(np.isnan(out))


def test_emulated_rejected_bounds_give_the_error_code_and_nan(hexagon_p):
    nlp, _, P, bounds, sols = _cpu_case("2", hexagon_p, B=1)
    lbx = bounds[0].copy()
    lbx[0] = bounds[1][0] + 1.0                            # lb > ub
    out, st, rc = SR.emu_sens(nlp, sols[0]["x"], sols[0]["lam_x"], sols[0]["lam_g"], P[0], (lbx,) + tuple(bounds[1:]),
                              np.ones(nlp.n), 1)
    assert rc == -2 and st[0] == -2 and np.all(np.isnan(out))


# ---------------------------------------------------------------------------------------------- GPU
def _torch():
    import torch
    return torch


def _t(a):
    torch = _torch()
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda:0")


def _gpu_solutions(pkg, Nr, N, T, P, dmin, vmax, wmax=2.84, tracking=False, **opts):
    prob = pkg.Problem(Nr, N, T, tracking=tracking, **opts)
    bounds = prob.bounds(dmin, vmax, wmax)
    x0 = prob.cold_start(P[:, :3 * Nr])
    out = prob.solve(_t(x0), _t(P), *map(_t, bounds))
    return prob, bounds, out


def _np(out):
    return {k: v.cpu().numpy() for k, v in out.items()}


def _tolerance(parts, rtol=1e-8):
    """rtol, widened by the conditioning that the interior-point weights give the condensed factorisation: with a weight w
    (|lam| / distance to a relaxed bound, up to ~4e12 on active rows and bounds at tol = 1e-8) the stage-wise sweep, like any
    condensed solve in double precision, keeps about eps * w / 100 relative (measured in the emulation: 1e-6 at w = 2.4e12,
    4.5e-7 at 1e12, 1e-14 without active rows)."""
    return rtol + 1e-2 * np.finfo(float).eps * SR.max_weight(parts)


def _check_against_reference(prob, P, bounds, out, tracking, rtol=1e-8, seed=0):
    torch = _torch()
    nlp = SR.nlp_for(prob.Nr, prob.N, prob.T, tracking)
    B = P.shape[0]
    rng = np.random.default_rng(seed)
    x_bar, p_dot = rng.normal(size=(B, prob.n)), rng.normal(size=(B, prob.np_))
    tb = list(map(_t, bounds))
    pb, st1 = prob.solution_vjp(out, _t(P), *tb, _t(x_bar))
    xd, st2 = prob.solution_jvp(out, _t(P), *tb, _t(p_dot))
    torch.cuda.synchronize()
    o, pb, xd = _np(out), pb.cpu().numpy(), xd.cpu().numpy()
    assert np.all(st1.cpu().numpy() == 0) and np.all(st2.cpu().numpy() == 0)
    for b in range(B):
        sol = dict(x=o["x"][b], lam_x=o["lam_x"][b], lam_g=o["lam_g"][b])
        tol = _tolerance(SR.kkt_parts(nlp, sol["x"], sol["lam_x"], sol["lam_g"], P[b], *bounds), rtol)
        err = max(_rel(pb[b], SR.sigma_vjp(nlp, sol, P[b], bounds, x_bar[b], refined=True)),
                  _rel(xd[b], SR.sigma_jvp(nlp, sol, P[b], bounds, p_dot[b], refined=True)))
        assert err <= tol, (b, err, tol)
        assert abs(x_bar[b] @ xd[b] - pb[b] @ p_dot[b]) <= 1e-10 * (np.abs(x_bar[b]) @ np.abs(xd[b]))
    return pb, xd


@pytest.mark.gpu
def test_gpu_six_robots_hexagon_and_synthetic_instances(pkg, hexagon_p):
    P = np.concatenate([hexagon_p[None], synthetic_instances(95, 6, seed=20261021)])
    prob, bounds, out = _gpu_solutions(pkg, 6, 20, 0.1, P, 0.4, 0.22)
    assert np.all(out["status"].cpu().numpy() <= 1)
    _check_against_reference(prob, P, bounds, out, False)


@pytest.mark.gpu
@pytest.mark.parametrize("Nr", [1, 2, 8, 10])
def test_gpu_robot_counts(pkg, Nr):
    P = _jitter(np.tile(_swap(Nr), (6, 1)), Nr, 0.05, seed=Nr)
    prob, bounds, out = _gpu_solutions(pkg, Nr, 10, 0.1, P, 0.3, 0.3)
    _check_against_reference(prob, P, bounds, out, False)


@pytest.mark.gpu
def test_gpu_tracking_time_varying_references(pkg):
    Nr, N, T = 3, 10, 0.2
    P = _tracking_params(Nr, N, T, 64, seed=11)
    prob, bounds, out = _gpu_solutions(pkg, Nr, N, T, P, 0.3, 0.6, np.pi / 2, tracking=True)
    _check_against_reference(prob, P, bounds, out, True)


@pytest.mark.gpu
@pytest.mark.parametrize("tracking", [False, True])
def test_gpu_against_central_differences_of_resolves(pkg, hexagon_p, tracking):
    torch = _torch()
    if tracking:
        Nr, N, T = 2, 10, 0.2
        P, dmin, vmax, wmax = _tracking_params(Nr, N, T, 8, seed=3), 0.3, 0.6, np.pi / 2
    else:
        Nr, N, T = 6, 10, 0.1
        P, dmin, vmax, wmax = _jitter(np.tile(hexagon_p, (8, 1)), 6, 0.03, seed=4), 0.4, 0.22, 2.84
    prob, bounds, out = _gpu_solutions(pkg, Nr, N, T, P, dmin, vmax, wmax, tracking=tracking, tol=1e-10, acceptable_tol=1e-10)
    nlp, o = SR.nlp_for(Nr, N, T, tracking), _np(out)
    strict = np.array([SR.strict_active_set(nlp, dict(x=o["x"][b], lam_x=o["lam_x"][b], lam_g=o["lam_g"][b]), P[b], bounds)
                       for b in range(len(P))]) & (o["status"] == 0)
    assert strict.sum() >= 2
    p_dot = np.random.default_rng(9).normal(size=P.shape)
    xd, st = prob.solution_jvp(out, _t(P), *map(_t, bounds), _t(p_dot))
    eps, tb = 1e-4, list(map(_t, bounds))
    xp = prob.solve(out["x"].clone(), _t(P + eps * p_dot), *tb)
    xm = prob.solve(out["x"].clone(), _t(P - eps * p_dot), *tb)
    fd = ((xp["x"] - xm["x"]) / (2 * eps)).cpu().numpy()
    xd = xd.cpu().numpy()
    for b in np.nonzero(strict)[0]:
        assert _rel(fd[b], xd[b]) <= 1e-5, (b, _rel(fd[b], xd[b]))


@pytest.mark.gpu
def test_gpu_tracking_constant_reference_matches_the_setpoint_handle(pkg):
    torch = _torch()
    Nr, N, T = 2, 10, 0.1
    P = _jitter(np.tile(_swap(Nr), (4, 1)), Nr, 0.05, seed=2)
    sp, bounds, out = _gpu_solutions(pkg, Nr, N, T, P, 0.3, 0.3)
    Pt = np.concatenate([P[:, :3 * Nr], np.tile(np.concatenate([P[:, 3 * Nr:], np.zeros((len(P), 2 * Nr))], 1), (1, N))], 1)
    tr, _, out_t = _gpu_solutions(pkg, Nr, N, T, Pt, 0.3, 0.3, tracking=True)
    for k in ("x", "lam_x", "lam_g"):
        assert torch.equal(out[k], out_t[k])
    x_bar = _t(np.random.default_rng(1).normal(size=(len(P), sp.n)))
    pb, _ = sp.solution_vjp(out, _t(P), *map(_t, bounds), x_bar)
    pbt, _ = tr.solution_vjp(out_t, _t(Pt), *map(_t, bounds), x_bar)
    pb, pbt = pb.cpu().numpy(), pbt.cpu().numpy()
    ns = 3 * Nr
    assert np.abs(pb[:, :ns] - pbt[:, :ns]).max() <= 1e-12 * np.abs(pb).max()
    sum_xr = pbt[:, ns:].reshape(len(P), N, 5 * Nr)[:, :, :ns].sum(1)
    assert np.abs(pb[:, ns:] - sum_xr).max() <= 1e-12 * np.abs(pb).max()


@pytest.mark.gpu
def test_gpu_solve_differentiable_backward(pkg):
    torch = _torch()
    Nr, N, T = 2, 10, 0.1
    P = _jitter(np.tile(_swap(Nr), (4, 1)), Nr, 0.05, seed=6)
    prob = pkg.Problem(Nr, N, T, tol=1e-10, acceptable_tol=1e-10)
    bounds = list(map(_t, prob.bounds(0.3, 0.3, 2.84)))
    x0 = _t(prob.cold_start(P[:, :3 * Nr]))
    W = _t(np.random.default_rng(2).normal(size=(len(P), prob.n)))
    p = _t(P).requires_grad_(True)

    def loss_of(pp):
        x = prob.solve_differentiable(x0, pp, *bounds)
        return (W * x).sum() + 0.5 * (x ** 2).sum(), x

    loss, x = loss_of(p)
    loss.backward()
    out = prob.solve(x0, _t(P), *bounds)
    direct, st = prob.solution_vjp(out, _t(P), *bounds, (W + out["x"]).contiguous())
    assert torch.equal(p.grad, direct) and bool((st == 0).all())
    d = np.random.default_rng(3).normal(size=P.shape)
    eps = 1e-4
    with torch.no_grad():
        lp, lm = loss_of(_t(P + eps * d))[0].item(), loss_of(_t(P - eps * d))[0].item()
    fd, an = (lp - lm) / (2 * eps), float((p.grad.cpu().numpy() * d).sum())
    assert abs(fd - an) <= 1e-5 * max(abs(an), 1.0), (fd, an)


@pytest.mark.gpu
def test_gpu_reproducible_and_independent_of_bounds_batched(pkg, hexagon_p):
    torch = _torch()
    P = _jitter(np.tile(hexagon_p, (16, 1)), 6, 0.03, seed=8)
    prob, bounds, out = _gpu_solutions(pkg, 6, 10, 0.1, P, 0.4, 0.22)
    x_bar = _t(np.random.default_rng(4).normal(size=(len(P), prob.n)))
    a, sa = prob.solution_vjp(out, _t(P), *map(_t, bounds), x_bar)
    b, sb = prob.solution_vjp(out, _t(P), *map(_t, bounds), x_bar)
    c, sc = prob.solution_vjp(out, _t(P), *[_t(np.tile(v, (len(P), 1))) for v in bounds], x_bar)
    assert torch.equal(a, b) and torch.equal(a, c) and torch.equal(sa, sc)


@pytest.mark.gpu
def test_gpu_wrong_inertia_gives_status_1_and_nan(pkg):
    torch = _torch()
    Nr, N, T = 2, 10, 0.1
    P = _swap(Nr)[None]
    prob, bounds, out = _gpu_solutions(pkg, Nr, N, T, P, 0.25, 0.22)
    bad = dict(out)
    bad["lam_g"] = (-40.0 * out["lam_g"]).contiguous()
    nlp = SR.nlp_for(Nr, N, T, False)
    o = _np(bad)
    assert SR.reduced_hessian_min_eig(SR.kkt_parts(nlp, o["x"][0], o["lam_x"][0], o["lam_g"][0], P[0], *bounds)) < 0
    pb, st = prob.solution_vjp(bad, _t(P), *map(_t, bounds), torch.ones_like(out["x"]))
    xd, st2 = prob.solution_jvp(bad, _t(P), *map(_t, bounds), _t(np.ones_like(P)))
    assert st.item() == 1 and st2.item() == 1 and bool(torch.isnan(pb).all()) and bool(torch.isnan(xd).all())


@pytest.mark.gpu
def test_gpu_error_paths(pkg):
    import ctypes as C
    torch = _torch()
    cabi = pkg._cabi
    L = cabi.lib()
    # unsupported handles: obstacle families, 11 robots (dense blocks), the small-OCP family
    unsupported = [pkg.Problem(1, 5, 0.1, obstacles=[[0.0, 0.0, 0.3]]), pkg.Problem(1, 5, 0.1, moving_obstacles=2),
                   pkg.Problem(1, 5, 0.1, tracking_obstacles=2), pkg.Problem(11, 3, 0.1), pkg.SmallOcp()]
    dummy = torch.zeros(64, dtype=torch.float64, device="cuda:0")
    for prob in unsupported:
        assert L.nmpc_sensitivity_workspace_bytes(prob.h, 1, 0) == 0
        for fn in (L.nmpc_solution_vjp, L.nmpc_solution_jvp):
            args = [prob.h, 1] + [dummy.data_ptr()] * 8 + [0, dummy.data_ptr(), dummy.data_ptr(), None, dummy.data_ptr(), 512, None]
            assert fn(*args) == -3, L.nmpc_last_error()
    # a supported handle, also on the forced dense-block path
    for tuning in (None, dict(force_block_path=1)):
        Nr, N, T = 2, 10, 0.1
        P = _swap(Nr)[None]
        prob = pkg.Problem(Nr, N, T, tuning=tuning)
        bounds = list(map(_t, prob.bounds(0.25, 0.22, 2.84)))
        out = prob.solve(_t(prob.cold_start(P[:, :3 * Nr])), _t(P), *bounds)
        xb = torch.ones_like(out["x"])
        pb, st = prob.solution_vjp(out, _t(P), *bounds, xb)
        assert st.item() == 0 and bool(torch.isfinite(pb).all())
        need = L.nmpc_sensitivity_workspace_bytes(prob.h, 1, 0)
        ws = torch.empty(need, dtype=torch.uint8, device="cuda:0")
        res = torch.empty_like(pb)
        ptrs = [out["x"].data_ptr(), out["lam_x"].data_ptr(), out["lam_g"].data_ptr(), _t(P).data_ptr()] + [b.data_ptr() for b in bounds]
        base = lambda: [prob.h, 1] + ptrs + [0, xb.data_ptr(), res.data_ptr(), None, ws.data_ptr(), need, None]
        assert L.nmpc_solution_vjp(*base()) == 0
        a = base(); a[2] = None                                   # NULL x
        assert L.nmpc_solution_vjp(*a) == -1
        a = base(); a[1] = 0                                      # B = 0
        assert L.nmpc_solution_vjp(*a) == -1
        a = base(); a[-2] = need - 8                              # small workspace
        assert L.nmpc_solution_vjp(*a) == -1
        if torch.cuda.device_count() > 1:                         # wrong device current
            with torch.cuda.device(1):
                assert L.nmpc_solution_vjp(*base()) == -1
        torch.cuda.synchronize()
    with pytest.raises(cabi.NmpcError):
        prob = unsupported[0]
        o = dict(x=torch.zeros((1, prob.n), dtype=torch.float64, device="cuda:0"))
        o["lam_x"], o["lam_g"] = torch.zeros_like(o["x"]), torch.zeros((1, prob.mg), dtype=torch.float64, device="cuda:0")
        bnd = [torch.zeros(prob.n, dtype=torch.float64, device="cuda:0")] * 2 + [torch.zeros(prob.mg, dtype=torch.float64, device="cuda:0")] * 2
        prob.solution_vjp(o, torch.zeros((1, prob.np_), dtype=torch.float64, device="cuda:0"), *bnd, o["x"])

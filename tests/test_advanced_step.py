"""Advanced-step NMPC (nmpc_solution_x0_jacobian / nmpc_advanced_step, Problem.solution_x0_jacobian / advanced_step,
closed_loop(disturbance=, advanced_step=)).  CPU: the product's Jacobian pass in the fibre emulation against the emulated
forward-mode pass column by column and against the NumPy reference.  GPU: the device pass against nmpc_solution_jvp, the
refined reference and central differences of re-solves; the feedback kernel against NumPy; closed loops without and with
disturbances against today's loop and against the ideal controller; reproducibility and the error paths."""
import numpy as np
import pytest

from oracle.nlp_numpy import synthetic_instances
from tests import advanced_step_ref as AR
from tests import sensitivity_ref as SR
from tests.test_sensitivity import _circle, _cpu_case, _jitter, _rel, _swap, _tracking_params
from tests.tracking_ref import rotation_reference


def _unit(B, ncols, j):
    e = np.zeros((B, ncols))
    e[:, j] = 1.0
    return e


# ---------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("key", ["1", "2", "6", "8", "2trk", "6trk", "8trk"])
@pytest.mark.parametrize("lane_rev", [0, 1])
def test_emulated_x0_pass_equals_the_emulated_jvp_and_the_reference(key, lane_rev, hexagon_p):
    nlp, _, P, bounds, sols = _cpu_case(key, hexagon_p, B=2)
    X, LX, LG = (np.array([s[k] for s in sols]) for k in ("x", "lam_x", "lam_g"))
    B, ns = len(P), 3 * nlp.Nr
    jac, st, rc = AR.emu_sens_x0(nlp, X, LX, LG, P, bounds, lane_rev)
    assert rc == 0 and np.all(st == 0)
    for j in range(ns):
        xd, st2, rc2 = SR.emu_sens(nlp, X, LX, LG, P, bounds, _unit(B, SR.n_params(nlp), j), 0, lane_rev)
        assert rc2 == 0 and np.all(st2 == 0)
        assert np.array_equal(jac[:, j], xd), j
        for b, sol in enumerate(sols):
            assert _rel(jac[b, j], SR.sigma_jvp(nlp, sol, P[b], bounds, _unit(1, SR.n_params(nlp), j)[0])) <= 1e-10
    np.testing.assert_array_equal(jac[:, :, :ns], np.broadcast_to(np.eye(ns), (B, ns, ns)))


@pytest.mark.parametrize("key", ["2", "2trk"])
def test_emulated_wrong_inertia_gives_status_1_and_nan(key, hexagon_p):
    nlp, _, P, bounds, sols = _cpu_case(key, hexagon_p, B=1)
    sol = dict(sols[0])
    sol["lam_g"] = -40.0 * sol["lam_g"]                   # the Lagrangian's curvature turned negative
    assert SR.reduced_hessian_min_eig(SR.kkt_parts(nlp, sol["x"], sol["lam_x"], sol["lam_g"], P[0], *bounds)) < 0
    jac, st, rc = AR.emu_sens_x0(nlp, sol["x"], sol["lam_x"], sol["lam_g"], P[0], bounds)
    assert rc == 0 and st[0] == 1 and np.all(np.isnan(jac))


def test_emulated_rejected_bounds_give_the_error_code_and_nan(hexagon_p):
    nlp, _, P, bounds, sols = _cpu_case("2", hexagon_p, B=1)
    lbx = bounds[0].copy()
    lbx[0] = bounds[1][0] + 1.0                            # lb > ub
    jac, st, rc = AR.emu_sens_x0(nlp, sols[0]["x"], sols[0]["lam_x"], sols[0]["lam_g"], P[0], (lbx,) + tuple(bounds[1:]))
    assert rc == -2 and st[0] == -2 and np.all(np.isnan(jac))


def test_numpy_feedback_reference_rules():
    rng = np.random.default_rng(0)
    B, ns, n = 3, 2, 6
    x, jac, p = rng.normal(size=(B, n)), rng.normal(size=(B, ns, n)), rng.normal(size=(B, 4))
    lbx, ubx = np.full(n, -np.inf), np.full(n, np.inf)
    lbx[4], ubx[4] = x[:, 4].min() - 1e-9, x[:, 4].max() + 1e-9
    np.testing.assert_array_equal(AR.advanced_step(x, jac, np.zeros(B), p, p[:, :ns], lbx, ubx)[:, ns:], x[:, ns:])
    xc = AR.advanced_step(x, jac, np.array([0, 1, 0]), p, p[:, :ns] + 1.0, lbx, ubx)
    np.testing.assert_array_equal(xc[1, ns:], x[1, ns:])
    assert np.all(xc[:, :ns] == p[:, :ns] + 1.0) and np.all(xc[:, 4] >= lbx[4]) and np.all(xc[:, 4] <= ubx[4])


# ---------------------------------------------------------------------------------------------- GPU
def _torch():
    import torch
    return torch


def _t(a):
    torch = _torch()
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda:0")


def _gpu_solutions(pkg, Nr, N, T, P, dmin, vmax, wmax=2.84, tracking=False, tuning=None, **opts):
    prob = pkg.Problem(Nr, N, T, tracking=tracking, tuning=tuning, **opts)
    bounds = prob.bounds(dmin, vmax, wmax)
    out = prob.solve(_t(prob.cold_start(P[:, :3 * Nr])), _t(P), *map(_t, bounds))
    return prob, bounds, out


def _tolerance(parts, rtol=1e-8):
    """The rule of test_sensitivity.py: rtol, widened by the conditioning that the interior-point weights w (|lam| / distance
    to a relaxed bound, up to ~4e12) give the condensed factorisation, about eps * w / 100 relative."""
    return rtol + 1e-2 * np.finfo(float).eps * SR.max_weight(parts)


def _check_jacobian(prob, P, bounds, out, tracking, n_ref=0):
    """jac equals solution_jvp(e_j) bit for bit; the first n_ref instances also against the refined NumPy reference."""
    torch = _torch()
    tP, tb = _t(P), list(map(_t, bounds))
    jac, st = prob.solution_x0_jacobian(out, tP, *tb)
    B, ns = P.shape[0], prob.ns
    assert tuple(jac.shape) == (B, ns, prob.n) and bool((st == 0).all())
    for j in range(ns):
        xd, st2 = prob.solution_jvp(out, tP, *tb, _t(_unit(B, prob.np_, j)))
        assert torch.equal(jac[:, j], xd) and torch.equal(st, st2), j
    nlp, o, J = SR.nlp_for(prob.Nr, prob.N, prob.T, tracking), {k: v.cpu().numpy() for k, v in out.items()}, jac.cpu().numpy()
    for b in range(n_ref):
        sol = dict(x=o["x"][b], lam_x=o["lam_x"][b], lam_g=o["lam_g"][b])
        tol = _tolerance(SR.kkt_parts(nlp, sol["x"], sol["lam_x"], sol["lam_g"], P[b], *bounds))
        for j in range(ns):
            err = _rel(J[b, j], SR.sigma_jvp(nlp, sol, P[b], bounds, _unit(1, prob.np_, j)[0], refined=True))
            assert err <= tol, (b, j, err, tol)
    return jac, st


@pytest.mark.gpu
def test_gpu_six_robots_hexagon_and_synthetic_instances(pkg, hexagon_p):
    P = np.concatenate([hexagon_p[None], synthetic_instances(95, 6, seed=20261021)])
    prob, bounds, out = _gpu_solutions(pkg, 6, 20, 0.1, P, 0.4, 0.22)
    _check_jacobian(prob, P, bounds, out, False, n_ref=6)


@pytest.mark.gpu
@pytest.mark.parametrize("Nr", [1, 2, 8, 10])
def test_gpu_robot_counts(pkg, Nr):
    P = _jitter(np.tile(_swap(Nr), (6, 1)), Nr, 0.05, seed=Nr)
    prob, bounds, out = _gpu_solutions(pkg, Nr, 10, 0.1, P, 0.3, 0.3)
    _check_jacobian(prob, P, bounds, out, False, n_ref=2)


@pytest.mark.gpu
def test_gpu_tracking_time_varying_references(pkg):
    Nr, N, T = 3, 10, 0.2
    P = _tracking_params(Nr, N, T, 64, seed=11)
    prob, bounds, out = _gpu_solutions(pkg, Nr, N, T, P, 0.3, 0.6, np.pi / 2, tracking=True)
    _check_jacobian(prob, P, bounds, out, True, n_ref=4)


@pytest.mark.gpu
def test_gpu_handle_on_the_dense_block_path(pkg):
    Nr = 2
    P = _jitter(np.tile(_swap(Nr), (8, 1)), Nr, 0.05, seed=12)
    prob, bounds, out = _gpu_solutions(pkg, Nr, 10, 0.1, P, 0.3, 0.3, tuning=dict(force_block_path=1))
    _check_jacobian(prob, P, bounds, out, False, n_ref=2)


@pytest.mark.gpu
def test_gpu_against_central_differences_of_resolves(pkg, hexagon_p):
    Nr, N, T = 6, 10, 0.1
    P = _jitter(np.tile(hexagon_p, (8, 1)), 6, 0.03, seed=4)
    prob, bounds, out = _gpu_solutions(pkg, Nr, N, T, P, 0.4, 0.22, tol=1e-10, acceptable_tol=1e-10)
    nlp, o = SR.nlp_for(Nr, N, T, False), {k: v.cpu().numpy() for k, v in out.items()}
    strict = np.array([SR.strict_active_set(nlp, dict(x=o["x"][b], lam_x=o["lam_x"][b], lam_g=o["lam_g"][b]), P[b], bounds)
                       for b in range(len(P))]) & (o["status"] == 0)
    assert strict.sum() >= 2
    tb = list(map(_t, bounds))
    jac, st = prob.solution_x0_jacobian(out, _t(P), *tb)
    jac, eps = jac.cpu().numpy(), 1e-4
    for j in range(prob.ns):
        e = _unit(len(P), prob.np_, j)
        xp = prob.solve(out["x"].clone(), _t(P + eps * e), *tb)["x"].cpu().numpy()
        xm = prob.solve(out["x"].clone(), _t(P - eps * e), *tb)["x"].cpu().numpy()
        for b in np.nonzero(strict)[0]:
            assert _rel((xp[b] - xm[b]) / (2 * eps), jac[b, j]) <= 1e-5, (b, j)


def _feedback_case(pkg, hexagon_p, B=16):
    P = _jitter(np.tile(hexagon_p, (B, 1)), 6, 0.03, seed=21)
    prob, bounds, out = _gpu_solutions(pkg, 6, 20, 0.3, P, 0.3, 0.22)
    tb = list(map(_t, bounds))
    jac, st = prob.solution_x0_jacobian(out, _t(P), *tb)
    return prob, P, bounds, tb, out, jac, st


@pytest.mark.gpu
def test_gpu_feedback_against_numpy(pkg, hexagon_p):
    torch = _torch()
    prob, P, bounds, tb, out, jac, st = _feedback_case(pkg, hexagon_p)
    ns, x, J = prob.ns, out["x"].cpu().numpy(), jac.cpu().numpy()
    assert bool((st == 0).all())
    rng = np.random.default_rng(22)
    for scale in (1e-3, 5e-2):        # 5e-2: large enough that corrected controls leave their bounds and get clamped
        meas = P[:, :ns] + scale * rng.normal(size=(len(P), ns))
        xc = prob.advanced_step(out, jac, st, _t(P), _t(meas), tb[0], tb[1]).cpu().numpy()
        ref = AR.advanced_step(x, J, np.zeros(len(P)), P, meas, bounds[0], bounds[1])
        assert np.array_equal(xc[:, :ns], meas)
        dlt = np.abs(meas - P[:, :ns])
        tol = 1e-15 * np.einsum("bjn,bj->bn", np.abs(J), dlt) + 2 * np.finfo(float).eps * np.abs(ref)
        assert np.all(np.abs(xc - ref) <= tol)
        free = x + np.einsum("bjn,bj->bn", J, meas - P[:, :ns])
        lo, hi = np.minimum(bounds[0], x), np.maximum(bounds[1], x)
        assert np.all(xc[:, ns:] >= lo[:, ns:]) and np.all(xc[:, ns:] <= hi[:, ns:])
        if scale > 1e-2:
            clamped = ((free < lo) | (free > hi))[:, ns:]
            assert clamped.sum() > 0                        # the clamp rule was exercised at saturated controls
            assert np.all((xc[:, ns:] == lo[:, ns:]) | (xc[:, ns:] == hi[:, ns:]) | ~clamped)
    xz = prob.advanced_step(out, jac, st, _t(P), _t(P[:, :ns]), tb[0], tb[1])
    assert torch.equal(xz[:, ns:], out["x"][:, ns:])       # zero correction: x bit for bit outside X_0


@pytest.mark.gpu
def test_gpu_status_1_instance_is_left_uncorrected(pkg):
    torch = _torch()
    Nr, N, T = 2, 10, 0.1
    P = np.stack([_swap(Nr), _swap(Nr)])
    prob, bounds, out = _gpu_solutions(pkg, Nr, N, T, P, 0.25, 0.22)
    bad = dict(out)
    bad["lam_g"] = out["lam_g"].clone()
    bad["lam_g"][1] *= -40.0                                 # the second instance gets the wrong inertia
    tb = list(map(_t, bounds))
    jac, st = prob.solution_x0_jacobian(bad, _t(P), *tb)
    assert st.tolist() == [0, 1] and bool(torch.isnan(jac[1]).all()) and bool(torch.isfinite(jac[0]).all())
    meas = _t(P[:, :3 * Nr] + 1e-3)
    xc = prob.advanced_step(out, jac, st, _t(P), meas, tb[0], tb[1])
    assert torch.equal(xc[1, 3 * Nr:], out["x"][1, 3 * Nr:]) and torch.equal(xc[:, :3 * Nr], meas)
    assert not torch.equal(xc[0, 3 * Nr:], out["x"][0, 3 * Nr:])


@pytest.mark.gpu
def test_gpu_reproducible_and_independent_of_bounds_batched(pkg, hexagon_p):
    torch = _torch()
    prob, P, bounds, tb, out, jac, st = _feedback_case(pkg, hexagon_p)
    tiled = [_t(np.tile(v, (len(P), 1))) for v in bounds]
    jac2, st2 = prob.solution_x0_jacobian(out, _t(P), *tb)
    jac3, st3 = prob.solution_x0_jacobian(out, _t(P), *tiled)
    assert torch.equal(jac, jac2) and torch.equal(jac, jac3) and torch.equal(st, st3)
    meas = _t(P[:, :prob.ns] + 1e-2 * np.random.default_rng(5).normal(size=(len(P), prob.ns)))
    a = prob.advanced_step(out, jac, st, _t(P), meas, tb[0], tb[1])
    b = prob.advanced_step(out, jac, st, _t(P), meas, tb[0], tb[1])
    c = prob.advanced_step(out, jac, st, _t(P), meas, tiled[0], tiled[1])
    assert torch.equal(a, b) and torch.equal(a, c)


def _loop_case(pkg, B, N=20, **opts):
    P = pkg.workload.synthetic_instances(B, 6, seed=20261022)
    prob = pkg.Problem(6, N, 0.3, **opts)
    return prob, P, list(map(_t, prob.bounds(0.3, 0.22, 2.84)))


LOOP_KEYS = ("traj", "u", "status", "iters", "active", "min_dist")


@pytest.mark.gpu
def test_gpu_zero_disturbance_loops_equal_todays_loop(pkg):
    torch = _torch()
    prob, P, tb = _loop_case(pkg, 512)
    steps = 40
    zero = torch.zeros((steps, 512, prob.ns), dtype=torch.float64, device="cuda:0")
    base = pkg.closed_loop(prob, _t(P), *tb, steps)
    ideal = pkg.closed_loop(prob, _t(P), *tb, steps, disturbance=zero)
    adv = pkg.closed_loop(prob, _t(P), *tb, steps, disturbance=zero, advanced_step=True)
    for k in LOOP_KEYS:
        assert torch.equal(base[k], ideal[k]) and torch.equal(base[k], adv[k]), k
    assert bool((adv["sens_status"][adv["active"] & (adv["status"] == 0)] == 0).all())
    assert torch.equal(adv["u_pred"], adv["u"])


@pytest.mark.gpu
def test_gpu_zero_disturbance_tracking_loop(pkg):
    torch = _torch()
    Nr, N, T, steps, B = 3, 10, 0.2, 20, 32
    rng = np.random.default_rng(13)
    refs = [rotation_reference(_circle(Nr, 1.0, phase=rng.uniform(0, 2 * np.pi)), N, T, steps) for _ in range(B)]
    ref = np.stack(refs, axis=1)                                    # [steps + N, B, 5 Nr]
    P = ref[0, :, :3 * Nr] + 0.03 * rng.normal(size=(B, 3 * Nr))
    prob = pkg.Problem(Nr, N, T, tracking=True)
    tb = list(map(_t, prob.bounds(0.3, 0.6, np.pi / 2)))
    zero = torch.zeros((steps, B, prob.ns), dtype=torch.float64, device="cuda:0")
    base = pkg.closed_loop(prob, _t(P), *tb, steps, reference=_t(ref))
    adv = pkg.closed_loop(prob, _t(P), *tb, steps, reference=_t(ref), disturbance=zero, advanced_step=True)
    for k in ("traj", "u", "status", "iters", "active", "track_err"):
        assert torch.equal(base[k], adv[k]), k


def _advanced_step_loop_with_ideal(prob, P, tb, w, tol=1e-1):
    """The advanced-step loop of closed_loop written out, with the ideal control at every step: U_0 of a solve at the true
    state, primal-started from the step's solution so that it stays in the same local optimum.  Returns the applied, predicted
    and ideal U_0 [steps, B, 2Nr] and the instance-steps where every solve and the Jacobian succeeded on an active instance."""
    torch = _torch()
    ns, nc, N = prob.ns, prob.nc, prob.N
    u0s = slice(ns * (N + 1), ns * (N + 1) + nc)
    p = _t(P)
    x_true = p[:, :ns].clone()
    x0 = _t(prob.cold_start(P[:, :ns]))
    u, u_pred, u_id, ok = [], [], [], []
    for t in range(w.shape[0]):
        active = (x_true - p[:, ns:2 * ns]).norm(dim=1) > tol
        out = prob.solve(x0, p, *tb)
        jac, st = prob.solution_x0_jacobian(out, p, *tb)
        xa = prob.advanced_step(out, jac, st, p, x_true, tb[0], tb[1])
        pt = p.clone()
        pt[:, :ns] = x_true
        ideal = prob.solve(out["x"].clone(), pt, *tb)
        u.append(xa[:, u0s]); u_pred.append(out["x"][:, u0s]); u_id.append(ideal["x"][:, u0s])
        ok.append(active & (out["status"] == 0) & (st == 0) & (ideal["status"] == 0))
        nxt = prob.plant(x_true, xa)
        p[:, :ns] = torch.where(active[:, None], nxt, x_true)
        x_true = torch.where(active[:, None], nxt + w[t], x_true)
        x0 = prob.shift(xa)
    return torch.stack(u), torch.stack(u_pred), torch.stack(u_id), torch.stack(ok)


@pytest.mark.gpu
def test_gpu_disturbed_loops_second_order_feedback_and_clearance(pkg):
    B, steps, dmin = 64, 20, 0.3
    prob, P, tb = _loop_case(pkg, B, tol=1e-10, acceptable_tol=1e-10)
    w = np.random.default_rng(23).normal(size=(steps, B, prob.ns))
    med = {}
    for sigma in (1e-3, 5e-4):
        dist = _t(sigma * w)
        ideal_loop = pkg.closed_loop(prob, _t(P), *tb, steps, disturbance=dist)
        adv = pkg.closed_loop(prob, _t(P), *tb, steps, disturbance=dist, advanced_step=True)
        for r in (ideal_loop, adv):
            assert float(r["min_dist"].min()) >= dmin - 10 * sigma
        u, u_pred, u_id, ok = _advanced_step_loop_with_ideal(prob, P, tb, dist)
        ok[0] = False                                       # step 0 solves at the true state: no correction to measure
        e_corr = (u - u_id).abs().amax(dim=2)[ok].cpu().numpy()
        e_pred = (u_pred - u_id).abs().amax(dim=2)[ok].cpu().numpy()
        assert e_corr.size >= B * steps // 2
        med[sigma] = (np.median(e_corr), np.median(e_pred))
        print("sigma %.1e: median |u - u_ideal| corrected %.3e, predicted %.3e (%d instance-steps)"
              % (sigma, med[sigma][0], med[sigma][1], e_corr.size))
        assert med[sigma][0] <= 0.1 * med[sigma][1]
    print("ratios sigma -> sigma/2: corrected %.2f, predicted %.2f" % (med[1e-3][0] / med[5e-4][0], med[1e-3][1] / med[5e-4][1]))
    assert med[1e-3][0] / med[5e-4][0] >= 3.0                    # second order
    assert 1.5 <= med[1e-3][1] / med[5e-4][1] <= 2.7              # first order


@pytest.mark.gpu
def test_gpu_error_paths(pkg):
    torch = _torch()
    cabi = pkg._cabi
    L = cabi.lib()
    unsupported = [pkg.Problem(1, 5, 0.1, obstacles=[[0.0, 0.0, 0.3]]), pkg.Problem(1, 5, 0.1, moving_obstacles=2),
                   pkg.Problem(1, 5, 0.1, tracking_obstacles=2), pkg.Problem(11, 3, 0.1), pkg.SmallOcp()]
    dummy = torch.zeros(64, dtype=torch.float64, device="cuda:0")
    d, st = dummy.data_ptr(), torch.zeros(4, dtype=torch.int32, device="cuda:0").data_ptr()
    for prob in unsupported:
        assert L.nmpc_solution_x0_jacobian(prob.h, 1, *[d] * 8, 0, d, None, d, 512, None) == -3, L.nmpc_last_error()
        assert L.nmpc_advanced_step(prob.h, 1, d, d, st, d, d, d, d, 0, d, None) == -3, L.nmpc_last_error()
    with pytest.raises(ValueError):
        pkg.closed_loop(unsupported[0], torch.zeros((1, 6), dtype=torch.float64, device="cuda:0"), dummy, dummy, dummy, dummy, 1,
                        advanced_step=True)
    Nr, N, T = 2, 10, 0.1
    P = _swap(Nr)[None]
    prob, bounds, out = _gpu_solutions(pkg, Nr, N, T, P, 0.25, 0.22)
    tb, tP = list(map(_t, bounds)), _t(P)
    need = L.nmpc_sensitivity_workspace_bytes(prob.h, 1, 0)
    ws = torch.empty(need, dtype=torch.uint8, device="cuda:0")
    jac = torch.empty((1, prob.ns, prob.n), dtype=torch.float64, device="cuda:0")
    sst = torch.empty(1, dtype=torch.int32, device="cuda:0")
    xc = torch.empty_like(out["x"])
    ptrs = [out["x"].data_ptr(), out["lam_x"].data_ptr(), out["lam_g"].data_ptr(), tP.data_ptr()] + [b.data_ptr() for b in tb]
    jbase = lambda: [prob.h, 1] + ptrs + [0, jac.data_ptr(), sst.data_ptr(), ws.data_ptr(), need, None]
    abase = lambda: [prob.h, 1, out["x"].data_ptr(), jac.data_ptr(), sst.data_ptr(), tP.data_ptr(), tP.data_ptr(), tb[0].data_ptr(),
                     tb[1].data_ptr(), 0, xc.data_ptr(), None]
    assert L.nmpc_solution_x0_jacobian(*jbase()) == 0
    assert L.nmpc_advanced_step(*abase()) == 0
    for base, fn in ((jbase, L.nmpc_solution_x0_jacobian), (abase, L.nmpc_advanced_step)):
        a = base(); a[2] = None                                  # NULL x
        assert fn(*a) == -1
        a = base(); a[1] = 0                                     # B = 0
        assert fn(*a) == -1
        if torch.cuda.device_count() > 1:                        # wrong device current
            with torch.cuda.device(1):
                assert fn(*base()) == -1
    a = jbase(); a[-2] = need - 8                                # small workspace
    assert L.nmpc_solution_x0_jacobian(*a) == -1
    a = abase(); a[4] = None                                     # NULL sens_status
    assert L.nmpc_advanced_step(*a) == -1
    torch.cuda.synchronize()
    assert torch.equal(xc[:, 3 * Nr:], out["x"][:, 3 * Nr:])    # measured = predicted: no correction

"""GPU parity tests: the CUDA path, called through the C-ABI, against the CPU oracle.

Tolerances are the ones BASELINE.json's north_star states:
    max |u - u_ref| <= 1e-4,  relative objective <= 1e-6,  constraint violation <= 1e-6.
The derivative-evaluation / shift / plant kernels are deterministic arithmetic: 1e-12 relative.
"""
import numpy as np
import pytest

from oracle.nlp_numpy import synthetic_instances
from oracle.oracle_lib import Oracle

pytestmark = pytest.mark.gpu
U_TOL, F_RTOL, C_TOL = 1e-4, 1e-6, 1e-6


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _t(torch, a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda")


@pytest.mark.parametrize("Nr,N,T", [(1, 25, 0.25), (2, 7, 0.1), (3, 5, 0.05), (6, 20, 0.3), (6, 35, 0.3), (8, 5, 0.02), (10, 20, 0.1),
                                    (16, 20, 0.3), (32, 6, 0.1)])   # the last two: records larger than shared memory (eval_kernel_big)
def test_eval_kernel_matches_oracle(pkg, torch_cuda, Nr, N, T):
    torch = torch_cuda
    rng = np.random.default_rng(Nr + N)
    prob, orc = pkg.Problem(Nr, N, T), Oracle(Nr, N, T)
    assert (prob.n, prob.mg, prob.nnz_jac, prob.nnz_hess) == (orc.n, orc.mg, orc.nnz_jac, orc.nnz_hess)
    for a, b in zip(prob.jac_pattern() + prob.hess_pattern(), orc.jac_pattern() + orc.hess_pattern()):
        np.testing.assert_array_equal(a, b)
    B = 37
    w, p, lam = rng.normal(size=(B, orc.n)), rng.normal(size=(B, 6 * Nr)), rng.normal(size=(B, orc.mg))
    out = prob.eval(_t(torch, w), _t(torch, p), _t(torch, lam))
    torch.cuda.synchronize()
    for b in range(B):
        e = orc.eval(w[b], p[b], lam[b])
        assert np.isclose(out["f"][b].item(), e["f"], rtol=1e-12)
        for k in ("grad", "g", "jac", "hess"):
            np.testing.assert_allclose(out[k][b].cpu().numpy(), e[k], rtol=1e-12, atol=1e-12, err_msg=k)


def test_shift_and_plant_kernels_exact(pkg, torch_cuda):
    torch = torch_cuda
    rng = np.random.default_rng(3)
    for Nr, N in ((1, 25), (6, 20), (4, 3), (3, 1)):
        prob, orc = pkg.Problem(Nr, N, 0.3), Oracle(Nr, N, 0.3)
        w = rng.normal(size=(65, orc.n))
        sh = prob.shift(_t(torch, w)).cpu().numpy()
        st = rng.normal(size=(65, 3 * Nr))
        pl = prob.plant(_t(torch, st), _t(torch, w)).cpu().numpy()
        for b in range(65):
            np.testing.assert_array_equal(sh[b], orc.shift(w[b]))
            np.testing.assert_allclose(pl[b], orc.plant(st[b], w[b][3 * Nr * (N + 1):3 * Nr * (N + 1) + 2 * Nr]), rtol=1e-14, atol=1e-15)


def _compare(out, ref, Nr, N, lbg, what):
    nX = 3 * Nr * (N + 1)
    x, f, g = out["x"].cpu().numpy(), out["f"].cpu().numpy(), out["g"].cpu().numpy()
    st, it = out["status"].cpu().numpy(), out["iters"].cpu().numpy()
    assert np.all(st == ref["status"]), (what, st, ref["status"])
    du = np.abs(x - ref["x"])[:, nX:].max(axis=1)
    df = np.abs(f - ref["f"]) / np.maximum(1.0, np.abs(ref["f"]))
    same = (du <= U_TOL) & (df <= F_RTOL)
    # constraint violation of OUR solution, independent of the oracle
    eq = np.isfinite(lbg) & (lbg == lbg)
    viol = np.maximum(lbg[None] - g, 0.0).max()
    assert viol <= C_TOL, (what, viol)
    return same, du, df, it


def test_solve_matches_oracle_small_cases(pkg, torch_cuda):
    torch = torch_cuda
    cases = [
        (1, 25, 0.25, 0.3, np.array([[0, 0, 0, 2.5, 2.0, 1.57]])),                       # C-1 casadi_test.py
        (2, 50, 0.1, 0.25, np.array([[-1, -1, 0.785, 1, 1, 2.356, 1, 1, 0.785, -1, -1, -2.356]])),   # C-2 second_scenario.py
        (3, 20, 0.05, 0.3, np.array([[-1, -1, 1.57, 0, -1, 1.57, 1, -1, 1.57, 2, 2, 0, 2, 1, 0, 2, 0, 0]])),  # C-3
    ]
    for Nr, N, T, dmin, P in cases:
        prob, orc = pkg.Problem(Nr, N, T), Oracle(Nr, N, T)
        lbx, ubx, lbg, ubg = prob.bounds(dmin, 0.22, 2.84)
        x0 = prob.cold_start(P[:, :3 * Nr])
        out = prob.solve(_t(torch, x0), _t(torch, P), _t(torch, lbx), _t(torch, ubx), _t(torch, lbg), _t(torch, ubg))
        torch.cuda.synchronize()
        ref = orc.solve_batch(x0, P, lbx, ubx, lbg, ubg)
        same, du, df, it = _compare(out, ref, Nr, N, lbg, (Nr, N))
        assert same.all(), (Nr, N, du, df, it, ref["iters"])
        assert np.abs(it - ref["iters"]).max() <= 3


def test_solve_six_robot_hexagon_and_synthetic_batch(pkg, torch_cuda, hexagon_p):
    torch = torch_cuda
    Nr, N, T = 6, 20, 0.3
    prob, orc = pkg.Problem(Nr, N, T), Oracle(Nr, N, T)
    lbx, ubx, lbg, ubg = prob.bounds(0.3, 0.22, 2.84)
    P = np.concatenate([hexagon_p[None], synthetic_instances(95)])
    x0 = prob.cold_start(P[:, :18])
    out = prob.solve(_t(torch, x0), _t(torch, P), _t(torch, lbx), _t(torch, ubx), _t(torch, lbg), _t(torch, ubg))
    torch.cuda.synchronize()
    ref = orc.solve_batch(x0, P, lbx, ubx, lbg, ubg)
    same, du, df, it = _compare(out, ref, Nr, N, lbg, "six")
    # the NLP is multi-modal (SURVEY.md 7): identical algorithms can still part ways through rounding;
    # require the same KKT point on >= 95 % of instances and a KKT point everywhere
    assert same.mean() >= 0.95, (same.mean(), du[~same], df[~same])
    assert out["stats"][:, 0].max().item() <= 1e-8
    d2 = out["g"].cpu().numpy().reshape(-1, N + 1, 18 + 15)[:, 1:, 18:]
    assert d2.min() >= 0.09 - C_TOL


def test_full_size_batch_properties(pkg, torch_cuda):
    """BASELINE size-independent properties at 4096 instances: all converge, KKT error, no collisions, bounds."""
    torch = torch_cuda
    Nr, N, T = 6, 20, 0.3
    prob = pkg.Problem(Nr, N, T)
    lbx, ubx, lbg, ubg = prob.bounds(0.3, 0.22, 2.84)
    P = synthetic_instances(4096)
    x0 = prob.cold_start(P[:, :18])
    out = prob.solve(_t(torch, x0), _t(torch, P), _t(torch, lbx), _t(torch, ubx), _t(torch, lbg), _t(torch, ubg))
    torch.cuda.synchronize()
    st = out["status"].cpu().numpy()
    assert (st == 0).mean() >= 0.995, np.bincount(st, minlength=5)
    ok = st == 0
    assert out["stats"][:, 0].cpu().numpy()[ok].max() <= 1e-8
    x, g = out["x"].cpu().numpy()[ok], out["g"].cpu().numpy()[ok]
    assert np.all(x >= lbx - 1e-6) and np.all(x <= ubx + 1e-6)
    assert np.abs(g.reshape(-1, 21, 33)[:, :, :18]).max() <= C_TOL
    assert g.reshape(-1, 21, 33)[:, 1:, 18:].min() >= 0.09 - C_TOL
    # warm start: apply u0 through the plant, shift, re-solve -> far fewer iterations, still solved
    xo = out["x"]
    state = prob.plant(_t(torch, P[:, :18]), xo)
    p2 = _t(torch, P).clone(); p2[:, :18] = state
    out2 = prob.solve(prob.shift(xo), p2, _t(torch, lbx), _t(torch, ubx), _t(torch, lbg), _t(torch, ubg))
    torch.cuda.synchronize()
    st2 = out2["status"].cpu().numpy()
    assert (st2 == 0).mean() >= 0.99
    assert out2["iters"].double().mean().item() < out["iters"].double().mean().item()


def test_host_api_equals_device_api_and_nlpsol_shim(pkg, torch_cuda):
    torch = torch_cuda
    Nr, N, T = 2, 10, 0.1
    prob = pkg.Problem(Nr, N, T)
    lbx, ubx, lbg, ubg = prob.bounds(0.25, 0.22, 2.84)
    P = np.array([[-1, -1, 0.785, 1, 1, 2.356, 1, 1, 0.785, -1, -1, -2.356]])
    x0 = prob.cold_start(P[:, :6])
    dev = prob.solve(_t(torch, x0), _t(torch, P), _t(torch, lbx), _t(torch, ubx), _t(torch, lbg), _t(torch, ubg))
    host = prob.solve_host(x0, P, lbx, ubx, lbg, ubg)
    for k in ("x", "f", "g", "lam_x", "lam_g"):
        np.testing.assert_array_equal(dev[k].cpu().numpy(), host[k])
    # the reference's call surface: keyword call, DM slicing, .full(), (1,mg) row bounds, (n,1) column bounds
    solver = pkg.nlpsol("solver", "ipopt", {"family": "unicycle_centralized", "Nr": Nr, "N": N, "T": T},
                        {"print_time": 0, "ipopt": {"max_iter": 2000, "print_level": 0, "acceptable_tol": 1e-8,
                                                    "acceptable_obj_change_tol": 1e-6}})
    sol = solver(x0=x0.reshape(-1, 1), p=P.reshape(-1, 1), lbx=lbx.reshape(-1, 1), ubx=ubx.reshape(-1, 1),
                 lbg=lbg.reshape(1, -1), ubg=ubg.reshape(1, -1))
    u = sol["x"][3 * Nr * (N + 1):].full()
    assert u.shape == (2 * Nr * N, 1)
    np.testing.assert_array_equal(u[:, 0], host["x"][0, 3 * Nr * (N + 1):])
    assert solver.stats()["success"]
    u_mat = np.transpose(pkg.reshape(np.transpose(u), 2 * Nr, N))          # the reference's unpack (:436-437)
    assert u_mat.shape == (N, 2 * Nr)
    # lam_p = dL/dp with L = f + lam_g'g (CasADi's convention), checked against central differences of the NumPy restatement
    from oracle.nlp_numpy import UnicycleNLP
    nlp = UnicycleNLP(Nr, N, T)
    w, lg = np.asarray(sol["x"].full()).ravel(), np.asarray(sol["lam_g"].full()).ravel()
    L = lambda pp: nlp.f(w, pp) + lg @ nlp.g(w, pp)
    eps = 1e-6
    fd = np.array([(L(P[0] + eps * e) - L(P[0] - eps * e)) / (2 * eps) for e in np.eye(6 * Nr)])
    np.testing.assert_allclose(np.asarray(sol["lam_p"].full()).ravel(), fd, rtol=1e-6, atol=1e-6)


def test_bound_errors_and_unsupported(pkg, torch_cuda):
    prob = pkg.Problem(2, 3, 0.1)
    lbx, ubx, lbg, ubg = prob.bounds(0.25, 0.22, 2.84)
    P = np.array([[0, 0, 0, 1, 0, 0, 1, 1, 0, 0, 1, 0.0]])
    x0 = prob.cold_start(P[:, :6])
    bad = lbx.copy(); bad[0] = 20.0
    with pytest.raises(pkg.NmpcError):
        prob.solve_host(x0, P, bad, ubx, lbg, ubg)
    bad = ubg.copy(); bad[0] = 1.0
    with pytest.raises(pkg.NmpcError):
        prob.solve_host(x0, P, lbx, ubx, lbg, bad)
    with pytest.raises(pkg.NmpcError):
        pkg.Problem(65, 5, 0.1)   # 11..64 robots run on the dense-block path (tests/test_gpu_block.py)


def test_infeasible_instance_reports_status_not_hang(pkg, torch_cuda):
    """Family A's first MPC step: all robots at the origin (centralized_six...py:361-362)."""
    prob = pkg.Problem(2, 10, 0.1, max_iter=300)
    orc = Oracle(2, 10, 0.1, max_iter=300)
    lbx, ubx, lbg, ubg = prob.bounds(0.25, 0.22, 2.84)
    P = np.array([[0, 0, 0, 0, 0, 0, 1, 1, 0.785, -1, -1, -2.356]], float)
    x0 = prob.cold_start(P[:, :6])
    out = prob.solve_host(x0, P, lbx, ubx, lbg, ubg)
    ref = orc.solve(x0[0], P[0], lbx, ubx, lbg, ubg)
    assert out["status"][0] in (2, 3, 4) and out["status"][0] == ref["status"]
    assert np.all(np.isfinite(out["x"]))


def _ring(Nr):
    a = np.arange(Nr) * 2 * np.pi / Nr
    st = np.stack([np.cos(a), np.sin(a), (a + 2 * np.pi) % (2 * np.pi) - np.pi], 1)
    g = -st.copy(); g[:, 2] = st[:, 2]
    return np.concatenate([st.ravel() + 0.01 * np.sin(np.arange(3 * Nr)), g.ravel()])


@pytest.mark.parametrize("Nr,N,T,dmin", [(8, 5, 0.02, 0.25), (8, 12, 0.3, 0.25), (10, 20, 0.1, 0.3), (7, 10, 0.3, 0.3), (9, 8, 0.2, 0.3)])
def test_two_warp_team_path_matches_oracle(pkg, torch_cuda, Nr, N, T, dmin):
    """7..10 robots (mpc_online_casadi_tb3_eight_...py:148-156, ..._ten_...py:169-177): one instance per 64-thread CTA."""
    torch = torch_cuda
    prob, orc = pkg.Problem(Nr, N, T), Oracle(Nr, N, T)
    lbx, ubx, lbg, ubg = prob.bounds(dmin, 0.22, 2.84)
    rng = np.random.default_rng(Nr)
    P = _ring(Nr)[None] + np.concatenate([0.03 * rng.normal(size=(12, 3 * Nr)), np.zeros((12, 3 * Nr))], axis=1)
    x0 = prob.cold_start(P[:, :3 * Nr])
    out = prob.solve(_t(torch, x0), _t(torch, P), _t(torch, lbx), _t(torch, ubx), _t(torch, lbg), _t(torch, ubg))
    torch.cuda.synchronize()
    ref = orc.solve_batch(x0, P, lbx, ubx, lbg, ubg)
    same, du, df, it = _compare(out, ref, Nr, N, lbg, (Nr, N))
    assert same.mean() >= 0.9, (du, df)
    assert out["stats"][:, 0].max().item() <= 1e-8


def test_parity_statistics_2048_synthetic_instances(pkg, torch_cuda):
    """Basin-agreement rate at scale: 2,048 cold six-robot instances, CUDA path vs oracle (SURVEY.md 7, hard part 1)."""
    torch = torch_cuda
    Nr, N, T = 6, 20, 0.3
    prob, orc = pkg.Problem(Nr, N, T), Oracle(Nr, N, T)
    lbx, ubx, lbg, ubg = prob.bounds(0.3, 0.22, 2.84)
    P = synthetic_instances(2048, seed=7)
    x0 = prob.cold_start(P[:, :18])
    out = prob.solve(_t(torch, x0), _t(torch, P), _t(torch, lbx), _t(torch, ubx), _t(torch, lbg), _t(torch, ubg))
    torch.cuda.synchronize()
    ref = orc.solve_batch(x0, P, lbx, ubx, lbg, ubg)
    x, f = out["x"].cpu().numpy(), out["f"].cpu().numpy()
    st, it = out["status"].cpu().numpy(), out["iters"].cpu().numpy()
    du = np.abs(x - ref["x"])[:, 18 * 21:].max(axis=1)
    df = np.abs(f - ref["f"]) / np.maximum(1.0, np.abs(ref["f"]))
    same = (du <= U_TOL) & (df <= F_RTOL) & (st == ref["status"])
    print("agreement %.4f  solved gpu %.4f oracle %.4f  iters gpu %.2f oracle %.2f  max|it diff| %d" %
          (same.mean(), (st == 0).mean(), (ref["status"] == 0).mean(), it.mean(), ref["iters"].mean(), np.abs(it - ref["iters"]).max()))
    assert (st == 0).mean() >= 0.999 and (ref["status"] == 0).mean() >= 0.999
    assert same.mean() >= 0.99, (same.mean(), du[~same][:10], df[~same][:10])
    # where they part ways both are KKT points (different local minima of a multi-modal NLP), never a failure
    assert out["stats"][:, 0].cpu().numpy().max() <= 1e-8
    assert np.median(np.abs(it - ref["iters"])) == 0


def test_scheduling_order_does_not_change_results(pkg, torch_cuda):
    """nmpc_set_order only changes which resident team picks which instance: outputs are bit-identical."""
    torch = torch_cuda
    Nr, N, T = 6, 20, 0.3
    prob = pkg.Problem(Nr, N, T)
    lbx, ubx, lbg, ubg = prob.bounds(0.3, 0.22, 2.84)
    P = synthetic_instances(300, Nr=Nr, seed=77)
    x0 = prob.cold_start(P[:, :3 * Nr])
    args = [_t(torch, a) for a in (x0, P, lbx, ubx, lbg, ubg)]
    a = prob.solve(*args)
    torch.cuda.synchronize()
    prob.set_order(prob.order_from_iters(a["iters"]))
    b = prob.solve(*args)
    torch.cuda.synchronize()
    prob.set_order(None)
    for k in ("x", "f", "g", "lam_g", "status", "iters"):
        assert torch.equal(a[k], b[k]), k


def test_benchmark_config_matches_independent_polish(pkg, torch_cuda):
    """The BENCHMARK configuration (6 robots, N = 20) against two solvers that share no code with the kernel or the oracle:
    tests/golden/polish6_scipy.npz (made by tests/golden/make_polish_golden.py) holds, for the de-symmetrised hexagon and the
    first 32 synthetic instances, where SciPy SLSQP and SciPy's trust-constr SQP on the active face end when started from the
    restated IPOPT's x*, plus the second-order certificate of that point.  The CUDA solver, from the reference's cold start,
    must stop within north_star's tolerances of those independently polished strict local minimisers."""
    import os
    torch = torch_cuda
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "polish6_scipy.npz"))
    Nr, N, T = 6, 20, 0.3
    P = gold["P"]
    np.testing.assert_array_equal(P[1:], synthetic_instances(len(P) - 1, Nr, 20261018))
    prob = pkg.Problem(Nr, N, T)
    lbx, ubx, lbg, ubg = prob.bounds(0.3, 0.22, 2.84)
    x0 = prob.cold_start(P[:, :18])
    out = prob.solve(_t(torch, x0), _t(torch, P), _t(torch, lbx), _t(torch, ubx), _t(torch, lbg), _t(torch, ubg))
    torch.cuda.synchronize()
    x, f, st = out["x"].cpu().numpy(), out["f"].cpu().numpy(), out["status"].cpu().numpy()
    assert (st == 0).all()
    nX = 18 * (N + 1)
    cert = gold["cert"]
    assert (cert[:, 0] > 0).all() and (cert[:, 1] > 0).all() and (cert[:, 2] > 0).all()      # multiplier signs, reduced Hessian > 0
    res = {}
    for name in ("slsqp", "face"):
        du = np.abs(x - gold["x_" + name])[:, nX:].max(axis=1)
        df = np.abs(f - gold["f_" + name]) / np.abs(gold["f_" + name])
        res[name] = (du, df)
        print("vs %s polish: max du %.2e  max df %.2e  within tolerance %d / %d" % (name, du.max(), df.max(), ((du <= U_TOL) & (df <= F_RTOL)).sum(), len(P)))
    # SLSQP stays within 5e-6 of the restated IPOPT's point on all 33 instances, so the CUDA solver must meet north_star's
    # tolerances against it everywhere -- except that a rounding-level fork into another basin of this multi-modal NLP is
    # possible (GPU and oracle agree on >= 99 % of 2,048 instances): allow one.
    du, df = res["slsqp"]
    assert ((du <= U_TOL) & (df <= F_RTOL)).sum() >= len(P) - 1, (du, df)
    # the face SQP confirms the objective everywhere; on three instances it stops 4e-3 .. 1.2e-2 away along flat control
    # directions (|f - f*| / f <= 1e-8 there), so its control tolerance is required on the other 30
    du, df = res["face"]
    assert (df <= F_RTOL).sum() >= len(P) - 1 and (du <= U_TOL).sum() >= len(P) - 4, (du, df)
    assert out["stats"][:, 10].max().item() == 0      # the fixed-size filter never evicted an entry


def test_set_order_length_is_checked_and_bad_entries_are_skipped(pkg, torch_cuda):
    """nmpc_set_order(h, order, len): a solve with another batch size is refused; a non-permutation never indexes outside
    the batch (ADVICE r1: the raw pointer used to be trusted)."""
    torch = torch_cuda
    prob = pkg.Problem(2, 6, 0.1)
    lbx, ubx, lbg, ubg = prob.bounds(0.25, 0.22, 2.84)
    P = synthetic_instances(8, Nr=2, seed=5)
    args = [_t(torch, a) for a in (prob.cold_start(P[:, :6]), P, lbx, ubx, lbg, ubg)]
    ref = prob.solve(*args)
    torch.cuda.synchronize()
    order = torch.arange(7, -1, -1, dtype=torch.int32, device="cuda")
    prob._order = None
    pkg._cabi.check(prob.L.nmpc_set_order(prob.h, order.data_ptr(), 5))
    with pytest.raises(pkg.NmpcError):
        prob.solve(*args)
    bad = order.clone(); bad[0] = 1000; bad[1] = -3          # instances 7 and 6 are never scheduled
    pkg._cabi.check(prob.L.nmpc_set_order(prob.h, bad.data_ptr(), 8))
    out = {"x": torch.full((8, prob.n), -7.0, dtype=torch.float64, device="cuda")}
    prob.solve(*args, out=out)
    torch.cuda.synchronize()
    assert torch.equal(out["x"][:6], ref["x"][:6]) and (out["x"][6:] == -7.0).all()
    prob.set_order(None)


def test_six_robots_all_at_origin_first_step(pkg, torch_cuda):
    """Family A's very first MPC step (centralized_six_robots_implementation.py:361-362): x0 = 0 for all six robots, so every
    stage-0 distance row is violated by the pinned X_0 and the NLP is infeasible.  The reference never reads the status
    (SURVEY.md 5): the call must return in bounded time with a finite iterate and a non-success status, as the oracle does."""
    Nr, N, T = 6, 35, 0.3
    prob = pkg.Problem(Nr, N, T, max_iter=300)
    orc = Oracle(Nr, N, T, max_iter=300)
    lbx, ubx, lbg, ubg = prob.bounds(0.4, 0.15, 1.5)          # the real-robot constants (:197-205)
    goal = np.array([[-0.7, -0.4, 0.0], [0.0, -0.8, 0.0], [0.7, -0.4, 0.0], [0.7, 0.4, 0.0], [0.0, 0.8, 0.0], [-0.7, 0.4, 0.0]])
    P = np.concatenate([np.zeros(18), goal.ravel()])[None]
    x0 = prob.cold_start(P[:, :18])
    out = prob.solve_host(x0, P, lbx, ubx, lbg, ubg)
    ref = orc.solve(x0[0], P[0], lbx, ubx, lbg, ubg)
    assert out["status"][0] in (2, 3, 4) and out["status"][0] == ref["status"], (out["status"], ref["status"])
    assert np.all(np.isfinite(out["x"])) and out["iters"][0] <= 300


def test_randomised_configurations_match_oracle(pkg, torch_cuda):
    """Fuzz over the descriptor space the reference's scripts span (1-10 robots, horizons 1-40, T 0.02-0.5, dmin 0.15-0.4, the
    TurtleBot and the real-robot control bounds, tight and wide position boxes): every configuration through the C-ABI against the
    oracle -- same status, north_star's tolerances where both land on the same point, a KKT point and no collision everywhere."""
    torch = torch_cuda
    rng = np.random.default_rng(20261018)
    n_same = n_tot = 0
    for case in range(36):
        Nr = int(rng.integers(1, 11))
        N = int(rng.choice([1, 2, 3, 5, 8, 13, 20, 27, 40]))
        T = float(rng.choice([0.02, 0.05, 0.1, 0.25, 0.3, 0.5]))
        dmin = float(rng.choice([0.15, 0.25, 0.3, 0.4]))
        vmax, wmax = [(0.22, 2.84), (0.15, 1.5)][int(rng.integers(0, 2))]
        box = float(rng.choice([3.0, 10.0]))
        B = 4
        P = synthetic_instances(B, Nr=Nr, seed=1000 + case, box=min(2.0 + 0.3 * Nr, box - 0.5), sep=dmin + 0.2)
        prob, orc = pkg.Problem(Nr, N, T), Oracle(Nr, N, T)
        lbx, ubx, lbg, ubg = prob.bounds(dmin, vmax, wmax, xy_box=box)
        x0 = prob.cold_start(P[:, :3 * Nr])
        out = prob.solve(_t(torch, x0), _t(torch, P), _t(torch, lbx), _t(torch, ubx), _t(torch, lbg), _t(torch, ubg))
        torch.cuda.synchronize()
        ref = orc.solve_batch(x0, P, lbx, ubx, lbg, ubg)
        st = out["status"].cpu().numpy()
        assert (st == ref["status"]).all(), (case, Nr, N, T, st, ref["status"])
        ok = st == 0
        if ok.any():
            assert out["stats"][:, 0].cpu().numpy()[ok].max() <= 1e-8, (case, Nr, N)
            g = out["g"].cpu().numpy()[ok]
            assert np.maximum(lbg[None] - g, 0.0).max() <= C_TOL, (case, Nr, N)
        nX = 3 * Nr * (N + 1)
        du = np.abs(out["x"].cpu().numpy() - ref["x"])[:, nX:].max(axis=1)
        df = np.abs(out["f"].cpu().numpy() - ref["f"]) / np.maximum(1.0, np.abs(ref["f"]))
        same = (du <= U_TOL) & (df <= F_RTOL)
        n_same += int(same[ok].sum()); n_tot += int(ok.sum())
        assert np.abs(out["iters"].cpu().numpy() - ref["iters"])[same & ok].max(initial=0) <= 5, (case, Nr, N, out["iters"].cpu().numpy(), ref["iters"])
        assert out["stats"][:, 10].max().item() == 0
    print("fuzz: %d / %d solved instances on the oracle's point" % (n_same, n_tot))
    assert n_tot >= 100 and n_same >= 0.97 * n_tot, (n_same, n_tot)


def test_per_instance_bounds_match_oracle(pkg, torch_cuda):
    """bounds_batched = 1: every instance carries its own lbx/ubx/lbg/ubg rows ([B, n] / [B, mg]) -- different safety distances,
    speed limits and position boxes inside one launch (the reference builds one `args` dict per script:
    sixth_scenario.py:127-135 dmin 0.3, second_scenario.py:118-120 dmin 0.25, decentralized_first_scenario.py:190-192 box +-2).
    The oracle is given the same per-instance rows; and the batched call must equal B shared-bounds calls."""
    torch = torch_cuda
    Nr, N, T, B = 4, 12, 0.2, 24
    rng = np.random.default_rng(77)
    prob, orc = pkg.Problem(Nr, N, T), Oracle(Nr, N, T)
    P = synthetic_instances(B, Nr, 4242)
    rows = [prob.bounds(dmin, vmax, wmax, xy_box=box) for dmin, vmax, wmax, box in
            zip(rng.uniform(0.15, 0.35, B), rng.uniform(0.15, 0.4, B), rng.uniform(1.0, 2.84, B), rng.choice([3.0, 10.0], B))]
    lbx, ubx, lbg, ubg = (np.stack([r[i] for r in rows]) for i in range(4))
    x0 = prob.cold_start(P[:, :3 * Nr])
    out = prob.solve(_t(torch, x0), _t(torch, P), _t(torch, lbx), _t(torch, ubx), _t(torch, lbg), _t(torch, ubg))
    torch.cuda.synchronize()
    ref = orc.solve_batch(x0, P, lbx, ubx, lbg, ubg)
    nX = 3 * Nr * (N + 1)
    x, f, g = out["x"].cpu().numpy(), out["f"].cpu().numpy(), out["g"].cpu().numpy()
    assert np.all(out["status"].cpu().numpy() == ref["status"])
    du = np.abs(x - ref["x"])[:, nX:].max(axis=1)
    df = np.abs(f - ref["f"]) / np.maximum(1.0, np.abs(ref["f"]))
    assert ((du <= U_TOL) & (df <= F_RTOL)).mean() >= 0.95, (du, df)
    ok = ref["status"] == 0
    assert ok.sum() >= B - 2
    assert np.maximum(lbg - g, 0.0)[ok].max() <= C_TOL
    relax = 1.01e-8 * np.maximum(1.0, np.abs(ubx))      # IPOPT's bound_relax_factor: bounds are relaxed by 1e-8 max(1, |b|) (restated in bounds_prep.cuh)
    assert np.all(np.maximum(lbx - x, 0.0)[ok] <= relax[ok]) and np.all(np.maximum(x - ubx, 0.0)[ok] <= relax[ok])
    # each instance's own speed limit is what binds: the largest |v| of instance b reaches vmax_b but never exceeds it
    v = np.abs(x[:, nX::2]).max(axis=1)
    assert np.all(v[ok] <= ubx[ok, nX] + 1.01e-8) and (v[ok] >= ubx[ok, nX] - 1e-6).mean() >= 0.8
    for b in (0, 7, 23):       # the same instance through the shared-bounds entry: identical arithmetic, identical result
        one = prob.solve(_t(torch, x0[b:b + 1]), _t(torch, P[b:b + 1]), _t(torch, lbx[b]), _t(torch, ubx[b]), _t(torch, lbg[b]), _t(torch, ubg[b]))
        np.testing.assert_array_equal(one["x"].cpu().numpy()[0], x[b])
        assert one["iters"].item() == out["iters"][b].item()


def test_single_robot_long_horizon_goal_sequence(pkg, torch_cuda):
    """Family E (decentralized_first_scenario.py:94-95,190-192,246-260): one robot, N = 200 stages of T = 0.05 s, positions boxed
    to +-2, v <= 0.22, |omega| <= 2.84, solved for each pose of the script's goal list from the previous goal -- a horizon ten
    times the benchmark's, so the stage records (not the robots) fill the scratch.  Each is checked against the oracle."""
    torch = torch_cuda
    Nr, N, T = 1, 200, 0.05
    prob, orc = pkg.Problem(Nr, N, T), Oracle(Nr, N, T)
    lbx, ubx, lbg, ubg = prob.bounds(0.15, 0.22, 2.84, xy_box=2.0)
    goals = np.array([[0, 0, 0], [1.0, 0.5, 0.0], [0.0, 0.75, -1.57], [-0.5, 0.5, 3.14], [-0.5, -0.75, 0.785], [0.75, -0.75, -0.785], [0, 0, 0]])
    P = np.concatenate([goals[:-1], goals[1:]], axis=1)
    x0 = prob.cold_start(P[:, :3])
    out = prob.solve(_t(torch, x0), _t(torch, P), _t(torch, lbx), _t(torch, ubx), _t(torch, lbg), _t(torch, ubg))
    torch.cuda.synchronize()
    ref = orc.solve_batch(x0, P, lbx, ubx, lbg, ubg)
    same, du, df, it = _compare(out, ref, Nr, N, lbg, "family E")
    assert np.all(ref["status"] == 0), ref["status"]
    assert same.all(), (du, df, it, ref["iters"])
    assert np.abs(it - ref["iters"]).max() <= 3
    x = out["x"].cpu().numpy()
    assert np.abs(x[:, :3 * (N + 1)].reshape(-1, N + 1, 3)[:, :, :2]).max() <= 2.0 + 2.1e-8

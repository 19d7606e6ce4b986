"""Distributed NMPC (nmpc_neighbour_obstacles, Problem.neighbour_obstacles, distributed_loop): every robot solves its own
one-robot problem against the predicted paths of its K nearest teammates, exchanged on the device.  CPU: the NumPy
restatement of the exchange (shift rule, key and tie rule, padding, untouched entries, min_dist over all robots) and the
reference loop on the C oracle.  GPU: the kernel against the restatement bit for bit (past one grid, both layouts, with and
without plans, guards, reproducibility), distributed_loop against the reference loop, a 64-robot swarm and the error paths."""
import numpy as np
import pytest

from tests.distributed_ref import (FAR, circle_swap, exchange, four_robot_crossing, hexagon_swap, passing,
                                   predictions, reference_loop)
from tests.obstacles_in_p import MovingOracle
from tests.test_moving_obstacles import _orc_bounds

NB_WARPS, CTAS_PER_SM = 8, 8       # neighbour_kernel: robots per CTA, CTAs per SM of its grid


def _np_of(N, K, tracking):
    return (3 + 5 * N if tracking else 6) + 3 * N * K


def _plan(rng, S, R, N, spread=2.0):
    """Random plans [S R, n] (X in a box, U random)."""
    n = 3 * (N + 1) + 2 * N
    w = rng.uniform(-spread, spread, size=(S * R, n))
    return w


# ---------------------------------------------------------------------------------------------- CPU
def test_predictions_follow_the_shift_rule():
    rng = np.random.default_rng(1)
    S, R, N = 2, 3, 5
    state = rng.normal(size=(S, R, 3))
    plan = _plan(rng, S, R, N)
    pr = predictions(state, plan, N)
    X = plan.reshape(S, R, -1)[:, :, :3 * (N + 1)].reshape(S, R, N + 1, 3)
    assert np.array_equal(pr[:, :, 0], state[..., :2])
    for k in range(1, N):
        assert np.array_equal(pr[:, :, k], X[:, :, min(k + 1, N), :2])
    assert np.array_equal(pr[:, :, N - 1], X[:, :, N, :2])          # the last stage: X_N
    hold = predictions(state, None, N)
    assert np.array_equal(hold, np.repeat(state[:, :, None, :2], N, axis=2))
    # and the exchange writes exactly those predictions (K = R - 1: every teammate)
    p, _ = exchange(state, plan, 0.4, R - 1, N, np.zeros((S * R, _np_of(N, R - 1, False))))
    O = p[:, 6:].reshape(S, R, N, R - 1, 3)
    for s in range(S):
        for a in range(R):
            got = {tuple(O[s, a, :, o, :2].ravel()) for o in range(R - 1)}
            assert got == {tuple(pr[s, j].ravel()) for j in range(R) if j != a}
    assert (O[..., 2] == 0.4).all()


def test_key_and_tie_rule_on_a_circle():
    """Eight robots at (+-3, +-4), (+-4, +-3) on the radius-5 circle: integer squared distances that tie exactly."""
    pts = np.array([[3, 4], [4, 3], [4, -3], [3, -4], [-3, -4], [-4, -3], [-4, 3], [-3, 4]], float)
    state = np.concatenate([pts, np.zeros((8, 1))], 1)[None]
    N, K = 3, 7
    p, md = exchange(state, None, 0.5, K, N, np.zeros((8, _np_of(N, K, False))))
    O = p[:, 6:].reshape(8, N, K, 3)
    for a in range(8):
        d2 = ((pts - pts[a]) ** 2).sum(1)
        want = sorted((d2[j], j) for j in range(8) if j != a)
        got = [int(np.flatnonzero((pts == O[a, 0, o, :2]).all(1))[0]) for o in range(K)]
        assert got == [j for _, j in want], (a, got, want)
    # robot 0 at (3, 4): (4, 3) at 2, then a tie at 50 between robots 2 (4, -3) and 6 (-4, 3): the lower index first
    got0 = [int(np.flatnonzero((pts == O[0, 0, o, :2]).all(1))[0]) for o in range(K)]
    assert got0[:2] == [1, 7] and got0.index(2) < got0.index(6)
    assert np.array_equal(md[0], np.sqrt(np.full(8, 2.0)))


def test_padding_when_the_team_is_smaller_than_k():
    rng = np.random.default_rng(2)
    S, R, N, K = 2, 3, 4, 5
    state = rng.normal(size=(S, R, 3))
    p, md = exchange(state, _plan(rng, S, R, N), 0.3, K, N, np.zeros((S * R, _np_of(N, K, False))))
    O = p[:, 6:].reshape(S, R, N, K, 3)
    pad = O[:, :, :, R - 1:]
    assert np.array_equal(pad[..., 0], np.broadcast_to(state[:, :, None, None, 0] + FAR, pad[..., 0].shape))
    assert np.array_equal(pad[..., 1], np.broadcast_to(state[:, :, None, None, 1], pad[..., 1].shape))
    assert (pad[..., 2] == 0.0).all() and (O[:, :, :, :R - 1, 2] == 0.3).all()
    one, md1 = exchange(state[:, :1], None, 0.3, K, N, np.zeros((S, _np_of(N, K, False))))
    assert np.isinf(md1).all() and (one[:, 6:].reshape(S, N, K, 3)[..., 2] == 0).all()


@pytest.mark.parametrize("tracking", [False, True])
def test_exchange_leaves_the_goal_and_reference_entries(tracking):
    rng = np.random.default_rng(3)
    S, R, N, K = 3, 5, 6, 2
    np_ = _np_of(N, K, tracking)
    p0 = rng.normal(size=(S * R, np_))
    p, _ = exchange(rng.normal(size=(S, R, 3)), _plan(rng, S, R, N), 0.3, K, N, p0)
    keep = np.ones(np_, bool)
    keep[:3] = False
    keep[np_ - 3 * N * K:] = False
    assert np.array_equal(p[:, keep], p0[:, keep])
    assert not np.array_equal(p[:, :3], p0[:, :3])


def test_min_dist_covers_every_robot_not_only_the_selected():
    """K = 1 selects the teammate whose plan comes closest later, while min_dist reports the nearest current pose."""
    N = 4
    state = np.array([[[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [3.0, 0.0, 0.0]]])
    plan = np.zeros((3, 3 * (N + 1) + 2 * N))
    for j in range(3):
        plan[j, :3 * (N + 1)] = np.tile(state[0, j], N + 1)
    plan[2, 3 * 2:3 * (N + 1):3] = 0.1          # robot 2's plan passes through (0.1, 0) from stage 1 on
    p, md = exchange(state, plan, 0.3, 1, N, np.zeros((3, _np_of(N, 1, False))))
    O = p[:, 6:].reshape(3, N, 1, 3)
    assert O[0, 1, 0, 0] == 0.1 and O[0, 0, 0, 0] == 3.0      # robot 0 selected robot 2
    assert md[0, 0] == 1.0 and md[0, 2] == 2.0
    d = np.linalg.norm(state[0, :, None, :2] - state[0, None, :, :2], axis=-1) + np.eye(3) * 1e9
    np.testing.assert_allclose(md[0], d.min(1), rtol=0, atol=1e-15)


def _ref_setup(case, N=20, T=0.3, margin=0.05):
    state0, goals = case()
    R = state0.shape[1]
    K = R - 1
    orc = MovingOracle(1, N, T, K)
    return state0, goals, K, _orc_bounds(orc, K, margin, dmin=0.0, v=0.2, w=np.pi / 4)


LOOP_CASES = {"crossing4": four_robot_crossing, "hexagon": hexagon_swap}
# feasible at every step of both loops (passing), or with a failed solve in the reference loop from step 1 on (see below)
GPU_LOOP_CASES = {"passing": (passing, 40), "crossing4": (four_robot_crossing, 2), "hexagon": (hexagon_swap, 2)}
DMIN = 0.3       # the centre distance the loops' rows keep, before the 0.05 lbg margin


@pytest.mark.parametrize("case", list(LOOP_CASES))
def test_reference_loop(case):
    N, T, steps = 20, 0.3, 40
    state0, goals, K, bnd = _ref_setup(LOOP_CASES[case], N, T)
    r = reference_loop(N, T, K, state0, goals, *bnd, steps, DMIN)
    assert r["traj"].shape == (steps + 1, 1, state0.shape[1], 3) and r["min_dist"].shape == (steps + 1, 1)
    # no pair ever closer than the clearance the rows keep
    assert r["min_dist"].min() >= DMIN, r["min_dist"].min()
    pos = r["traj"][..., :2]
    d = np.linalg.norm(pos[:, :, :, None] - pos[:, :, None], axis=-1) + np.eye(state0.shape[1]) * 1e9
    np.testing.assert_allclose(d.min(axis=(2, 3)), r["min_dist"], rtol=0, atol=1e-12)
    assert (r["status"] <= 1).mean() >= 0.8, np.bincount(r["status"].ravel())
    # everyone gets closer to the goal
    d0 = np.linalg.norm(state0[..., :2] - goals[..., :2], axis=-1)
    d1 = np.linalg.norm(r["traj"][-1, ..., :2] - goals[..., :2], axis=-1)
    assert (d1 < d0 - 0.5).all(), (d0, d1)


# ---------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _t(torch, a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda:0")


def _raw_exchange(torch, prob, state, plan, clearance, p_fill, guard=3):
    """nmpc_neighbour_obstacles on buffers with `guard` guard elements before and after p and min_dist.  Returns
    (rc, p, min_dist, guards intact)."""
    S, R = state.shape[:2]
    pbuf = _t(torch, np.concatenate([np.full(guard, -7.5), p_fill.ravel(), np.full(guard, -7.5)]))
    mbuf = _t(torch, np.full(S * R + 2 * guard, -7.5))
    st = _t(torch, state)
    pl = None if plan is None else _t(torch, plan)
    rc = prob.L.nmpc_neighbour_obstacles(prob.h, S, R, st.data_ptr(), None if pl is None else pl.data_ptr(), float(clearance),
                                         pbuf[guard:].data_ptr(), mbuf[guard:].data_ptr(), None)
    torch.cuda.synchronize()
    pb, mb = pbuf.cpu().numpy(), mbuf.cpu().numpy()
    ok = (pb[:guard] == -7.5).all() and (pb[-guard:] == -7.5).all() and (mb[:guard] == -7.5).all() and (mb[-guard:] == -7.5).all()
    return rc, pb[guard:-guard].reshape(p_fill.shape), mb[guard:-guard].reshape(S, R), ok


def _scenarios(R, sm_count):
    """Enough scenarios for the robot groups to pass one grid (CTAS_PER_SM x SMs CTAs) with an uneven last round; the largest
    teams are kept to a few scenarios."""
    groups = (R + NB_WARPS - 1) // NB_WARPS
    if R >= 1000:
        return 3
    return (CTAS_PER_SM * sm_count + 37) // groups + 1


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 6, 32])
@pytest.mark.parametrize("R", [1, 2, 7, 33, 64, 1000])
def test_gpu_exchange_matches_the_reference_bitwise(pkg, torch_cuda, R, K):
    torch = torch_cuda
    rng = np.random.default_rng(100 * R + K)
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    N, T = (6, 0.3) if R < 1000 else (10, 0.3)
    S = _scenarios(R, sm)
    state = np.concatenate([rng.uniform(-4, 4, size=(S, R, 2)), rng.uniform(-3, 3, size=(S, R, 1))], axis=2)
    if R == 33:     # exact ties: a lattice of integer positions
        state[..., :2] = rng.integers(-3, 4, size=(S, R, 2))
    for tracking in (False, True):
        prob = pkg.Problem(1, N, T, **({"tracking_obstacles": K} if tracking else {"moving_obstacles": K}))
        assert prob.np_ == _np_of(N, K, tracking)
        for with_plan in (False, True):
            plan = _plan(rng, S, R, N, 4.0) if with_plan else None
            fill = np.full((S * R, prob.np_), 0.25)
            before = prob.launch_count()
            rc, p, md, ok = _raw_exchange(torch, prob, state, plan, 0.35, fill)
            assert rc == 0 and ok
            assert prob.launch_count() == before + 1
            ref_p, ref_md = exchange(state, plan, 0.35, K, N, fill)
            assert np.array_equal(p, ref_p), (tracking, with_plan, np.argwhere(p != ref_p)[:5])
            assert np.array_equal(md, ref_md), (tracking, with_plan)
            # reproducible, and the Python entry gives the same
            rc2, p2, md2, _ = _raw_exchange(torch, prob, state, plan, 0.35, fill)
            assert np.array_equal(p2, p) and np.array_equal(md2, md)
            pt, mdt = prob.neighbour_obstacles(_t(torch, state), None if plan is None else _t(torch, plan), clearance=0.35,
                                               p=_t(torch, fill))
            assert np.array_equal(pt.cpu().numpy(), p) and np.array_equal(mdt.cpu().numpy(), md)


def _gpu_bounds(prob, margin=0.05):
    return prob.bounds_obstacles(margin, 0.2, np.pi / 4)


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(GPU_LOOP_CASES))
def test_gpu_loop_matches_the_reference_loop(pkg, torch_cuda, case):
    torch = torch_cuda
    N, T, steps = 20, 0.3, 40
    make, feasible_steps = GPU_LOOP_CASES[case]
    state0, goals, K, bnd = _ref_setup(make, N, T)
    prob = pkg.Problem(1, N, T, moving_obstacles=K)
    gb = _gpu_bounds(prob)
    assert all(np.array_equal(a, b) for a, b in zip(gb, bnd))
    res = pkg.distributed_loop(prob, _t(torch, state0), _t(torch, goals), *(_t(torch, a) for a in gb), steps, DMIN)
    ref = reference_loop(N, T, K, state0, goals, *bnd, steps, DMIN)
    # A solve that ends with status 3 returns its last iterate, which is the solver's path and not a property of the problem,
    # so the loops are compared up to and including the first step in which the reference loop has one.  In the crossing and
    # the hexagon that is step 1, with every pair more than 0.9 m apart: the shifted warm start runs through a teammate's new
    # predicted path and the solver exits locally infeasible (from the held pose the same instance solves).  The passing case
    # stays feasible for all 40 steps; its robot 0 holds its pose from the start and two more robots arrive and stop, so the
    # stop test, the held-pose plans, the order and the shift warm start are compared over the whole run.
    bad = np.flatnonzero((ref["status"] > 1).any(axis=(1, 2)))
    te = steps if bad.size == 0 else int(bad[0]) + 1
    assert te >= feasible_steps, te
    if case == "passing":
        act = ref["active"][:, 0]
        assert te == steps and not act[0, 0] and (act[0, 1:] & ~act[-1, 1:]).sum() >= 2, act[[0, -1]]
    u = res["u"].cpu().numpy()[:te]
    assert np.abs(u - ref["u"][:te]).max() <= 1e-4, np.abs(u - ref["u"][:te]).max()
    assert np.array_equal(res["status"].cpu().numpy()[:te], ref["status"][:te])
    assert np.array_equal(res["active"].cpu().numpy()[:te], ref["active"][:te])
    np.testing.assert_allclose(res["traj"].cpu().numpy()[:te + 1], ref["traj"][:te + 1], atol=1e-4)
    np.testing.assert_allclose(res["min_dist"].cpu().numpy()[:te + 1], ref["min_dist"][:te + 1], atol=1e-4)
    assert res["min_dist"].min().item() >= DMIN
    print("\n%s: loops compared over %d of %d steps" % (case, te, steps))


def _swarm(S, R=64, radius=7.5, seed=7):
    rng = np.random.default_rng(seed)
    return circle_swap(R, radius, S, rng, jitter=0.05)


def _pair_min(torch, traj):
    pos = traj[..., :2]
    S, R = pos.shape[1], pos.shape[2]
    out = []
    for t in range(pos.shape[0]):
        d = torch.cdist(pos[t], pos[t]) + torch.eye(R, dtype=pos.dtype, device=pos.device) * 1e9
        out.append(d.amin(dim=(1, 2)))
    return torch.stack(out)


@pytest.mark.gpu
def test_gpu_swarm_of_64_keeps_its_distance(pkg, torch_cuda):
    """The 64-robot circle swap (radius 7.5 m: 0.74 m between neighbours, 5 cm jitter), 32 seeded scenarios, K = 16.  The rows
    keep clearance = dmin + 0.2 = 0.5 m between centres, plus the 0.05 lbg margin: 0.25 m for the difference between a teammate's
    predicted and actual path; the plant must never bring a pair closer than dmin = 0.3 m."""
    torch = torch_cuda
    N, T, K, steps, dmin = 20, 0.3, 16, 150, 0.3
    clearance = dmin + 0.2
    state0, goals = _swarm(32)
    prob = pkg.Problem(1, N, T, moving_obstacles=K)
    bnd = [_t(torch, a) for a in _gpu_bounds(prob)]
    res = pkg.distributed_loop(prob, _t(torch, state0), _t(torch, goals), *bnd, steps, clearance)
    md = res["min_dist"]
    assert torch.allclose(md, _pair_min(torch, res["traj"]), rtol=0, atol=1e-12)
    assert md.min().item() >= dmin, md.min().item()
    st = res["status"]
    ok = (st <= 1).double().mean().item()
    # Not held to 99 % (about half end with status 3): as the 64 robots converge on the centre, many instances are infeasible
    # from any start (on the C oracle the four-robot crossing and the hexagon show it from the held pose too: a teammate inside
    # the stage-0 row's clearance + margin, or a predicted stage-1 position nearer than a unicycle can back away from in one
    # period), and others exit locally infeasible from the shifted warm start.  The 99 % criterion is asserted on the BASELINE
    # sampler below.
    dist = (res["traj"][-1, ..., :2] - _t(torch, goals)[..., :2]).norm(dim=-1)
    moving = res["active"][-1].double().mean().item()
    print("\nswarm 64 setpoint, %d steps: status 0/1 %.4f, min pair distance %.3f m, arrived (<= 0.1 m) %.3f, still active %.3f, "
          "median distance to goal %.2f m" % (steps, ok, md.min().item(), (dist <= 0.1).double().mean().item(), moving,
                                            dist.median().item()))


@pytest.mark.gpu
def test_gpu_swarm_of_64_on_the_baseline_sampler(pkg, torch_cuda):
    """32 scenarios of the 64-robot BASELINE workload (starts and goals 0.5 m apart in an 8 m box), K = 16, clearance dmin +
    0.05: at least 99 % of the solves end with status 0 or 1 and no pair comes closer than dmin."""
    torch = torch_cuda
    from oracle.nlp_numpy import synthetic_instances
    N, T, K, steps, dmin, S, R = 20, 0.3, 16, 30, 0.3, 32, 64
    P = synthetic_instances(S, Nr=R, seed=20261018, box=8.0)
    state0, goals = P[:, :3 * R].reshape(S, R, 3), P[:, 3 * R:].reshape(S, R, 3)
    prob = pkg.Problem(1, N, T, moving_obstacles=K)
    bnd = [_t(torch, a) for a in prob.bounds_obstacles(0.05, 0.22, 2.84)]
    res = pkg.distributed_loop(prob, _t(torch, state0), _t(torch, goals), *bnd, steps, dmin + 0.05)
    ok = (res["status"] <= 1).double().mean().item()
    assert ok >= 0.99, torch.bincount(res["status"].flatten().long())
    assert res["min_dist"].min().item() >= dmin, res["min_dist"].min().item()
    print("\nswarm 64 BASELINE sampler, %d steps: status 0/1 %.4f, min pair distance %.3f m" % (steps, ok, res["min_dist"].min().item()))


@pytest.mark.gpu
def test_gpu_swarm_of_64_on_a_rotating_formation(pkg, torch_cuda):
    """The same swarm tracking a reference that rotates the circle about its centre by pi at 0.03 rad/s (then holds), on the
    tracking-obstacle handle (the way DESIGN section 7 leaves the symmetric-swap standstill); arrival is reported."""
    torch = torch_cuda
    N, T, K, dmin, radius = 20, 0.3, 16, 0.3, 6.0
    om = 0.03
    steps = int(np.ceil(np.pi / om / T)) + 20
    state0, goals = _swarm(8, radius=radius)      # 6 m: 0.59 m between neighbours
    S, R = state0.shape[:2]
    tt = np.arange(steps + N) * T
    phi = np.minimum(om * tt, np.pi)
    w = np.where(om * tt < np.pi, om, 0.0)
    ang = np.arctan2(state0[..., 1], state0[..., 0])            # [S, R]
    a = ang[None] + phi[:, None, None]
    ref = np.zeros((steps + N, S, R, 5))
    ref[..., 0], ref[..., 1] = radius * np.cos(a), radius * np.sin(a)
    ref[..., 2] = a + np.pi / 2
    ref[..., 3], ref[..., 4] = radius * w[:, None, None], w[:, None, None]
    state0 = state0.copy()
    state0[..., 2] = ang + np.pi / 2
    prob = pkg.Problem(1, N, T, tracking_obstacles=K)
    bnd = [_t(torch, b) for b in prob.bounds_obstacles(0.05, 0.2, np.pi / 4, th_box=4 * np.pi)]
    res = pkg.distributed_loop(prob, _t(torch, state0), _t(torch, ref), *bnd, steps, dmin + 0.05)
    assert res["track_err"].shape == (steps + 1, S, R)
    # the sliding window: track_err is the distance to reference row t, so a wrongly laid out Z would not converge to it
    err = np.linalg.norm(res["traj"].cpu().numpy()[..., :2] - ref[:steps + 1, ..., :2], axis=-1)
    np.testing.assert_allclose(res["track_err"].cpu().numpy(), err, rtol=0, atol=1e-12)
    assert res["track_err"][-1].max().item() <= 0.05, res["track_err"][-1].max().item()
    assert res["min_dist"].min().item() >= dmin, res["min_dist"].min().item()
    ok = (res["status"] <= 1).double().mean().item()
    dist = (res["traj"][-1, ..., :2] - _t(torch, goals)[..., :2]).norm(dim=-1)
    assert ok >= 0.99 and (dist <= 0.1).double().mean().item() >= 0.95, (ok, (dist <= 0.1).double().mean().item())
    print("\nswarm 64 rotating formation, %d steps: status 0/1 %.4f, min pair distance %.3f m, arrived (<= 0.1 m of the "
          "antipode) %.3f, largest tracking error %.3f m, final %.3f m" % (steps, ok, res["min_dist"].min().item(),
                                                                          (dist <= 0.1).double().mean().item(),
                                                                          res["track_err"].max().item(),
                                                                          res["track_err"][-1].max().item()))


@pytest.mark.gpu
def test_gpu_errors(pkg, torch_cuda):
    torch = torch_cuda
    from nmpc_b200._cabi import NmpcError
    ENOTSUP, EINVAL = -3, -1
    state = _t(torch, np.zeros((2, 3, 3)))
    p = _t(torch, np.zeros((6, _np_of(5, 2, False))))
    L = pkg.lib()

    def call(prob, S=2, R=3, st=state.data_ptr(), pp=p.data_ptr(), c=0.3):
        return L.nmpc_neighbour_obstacles(prob.h, S, R, st, None, c, pp, None, None)
    for bad in (pkg.Problem(2, 5, 0.3), pkg.Problem(2, 5, 0.3, moving_obstacles=2), pkg.Problem(1, 5, 0.3, obstacles=[[1, 1, 0.3]]),
                pkg.SmallOcp("van_der_pol")):
        assert call(bad) == ENOTSUP
    prob = pkg.Problem(1, 5, 0.3, moving_obstacles=2)
    assert call(prob) == 0
    for kw in (dict(S=0), dict(R=0), dict(S=-1), dict(S=1 << 16, R=1 << 16), dict(st=None), dict(pp=None), dict(c=float("nan")),
               dict(c=-0.1), dict(c=float("inf"))):
        assert call(prob, **kw) == EINVAL, kw
    for bad in (pkg.Problem(2, 5, 0.3, moving_obstacles=2), pkg.Problem(1, 5, 0.3, tracking=True)):
        with pytest.raises(ValueError):
            bad.neighbour_obstacles(state, clearance=0.3)
    with pytest.raises(ValueError):
        prob.neighbour_obstacles(state[:, :, :2].contiguous(), clearance=0.3)
    with pytest.raises(ValueError):
        prob.neighbour_obstacles(state, p=p[:, 1:].contiguous(), clearance=0.3)
    with pytest.raises(ValueError):
        prob.neighbour_obstacles(state, plan=_t(torch, np.zeros((6, 7))), clearance=0.3)
    with pytest.raises(NmpcError):
        prob.neighbour_obstacles(state, clearance=-1.0)
    bnd = [_t(torch, a) for a in prob.bounds_obstacles(0.05, 0.2, np.pi / 4)]
    with pytest.raises(ValueError):      # goals of the wrong shape, a reference on the setpoint handle
        pkg.distributed_loop(prob, state, _t(torch, np.zeros((2, 3, 2))), *bnd, 3, 0.3)
    with pytest.raises(ValueError):
        pkg.distributed_loop(prob, state, _t(torch, np.zeros((8, 2, 3, 5))), *bnd, 3, 0.3)
    with pytest.raises(ValueError):
        pkg.distributed_loop(pkg.Problem(1, 5, 0.3, tracking_obstacles=2), state, _t(torch, np.zeros((2, 3, 3))), *bnd, 3, 0.3)

"""References for tests/test_distributed.py (distributed NMPC) -- TEST INFRASTRUCTURE ONLY.

  * exchange: a NumPy restatement of nmpc_neighbour_obstacles, bit for bit: the same predictions, the same rounded squares and
    sums (NumPy does not contract a * a + b * b into an FMA), the same lexicographic selection, the same padding;
  * reference_loop: distributed_loop with that exchange, every robot solved by the C oracle's moving-obstacle build
    (tests/obstacles_in_p.MovingOracle(1, N, T, K)) and the oracle's Euler plant and shift.
"""
import numpy as np

from tests.obstacles_in_p import MovingOracle

FAR = 1e6     # the padding obstacle sits at the robot's own pose + (FAR, 0), clearance 0


def predictions(state, plan, N):
    """[S, R, N, 2]: stage 0 the pose, stage k >= 1 X_{min(k+1, N)} of the plan [S R, n] (None: the pose)."""
    S, R, _ = state.shape
    pr = np.repeat(state[:, :, None, :2], N, axis=2).copy()
    if plan is not None:
        X = np.asarray(plan).reshape(S, R, -1)[:, :, :3 * (N + 1)].reshape(S, R, N + 1, 3)
        src = np.minimum(np.arange(1, N) + 1, N)
        pr[:, :, 1:] = X[:, :, src, :2]
    return pr


def exchange(state, plan, clearance, K, N, p):
    """nmpc_neighbour_obstacles on NumPy arrays: returns (p with x0bar and O written, min_dist [S, R]).  state [S, R, 3], plan
    [S R, n] or None, p [S R, np] (copied, the other entries kept)."""
    state = np.asarray(state, np.float64)
    S, R, _ = state.shape
    p = np.array(p, np.float64, copy=True)
    np_, kk = p.shape[1], min(K, R - 1)
    pr = predictions(state, plan, N)
    O = np.empty((S, R, N, K, 3))
    O[..., 0] = state[:, :, None, None, 0] + FAR      # padding, overwritten by the selected teammates
    O[..., 1] = state[:, :, None, None, 1]
    O[..., 2] = 0.0
    min_dist = np.empty((S, R))
    jj = np.arange(R)
    me = jj[:, None] == jj[None, :]
    chunk = max(1, int(2e7 // (R * R * N)))
    for s0 in range(0, S, chunk):
        q = pr[s0:s0 + chunk]                                       # [c, R, N, 2]
        c = q.shape[0]
        d = q[:, :, None] - q[:, None]                              # [c, a, j, N, 2]
        d2 = d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]          # rounded products, one rounded sum: no FMA, as on the device
        key = np.where(me, np.inf, np.fmin.reduce(d2, axis=3, initial=np.inf))     # [c, a, j]
        d0 = np.where(me, np.inf, d2[..., 0])
        min_dist[s0:s0 + c] = np.sqrt(np.fmin.reduce(d0, axis=2, initial=np.inf))
        # (key, j) in lexicographic order, the robot itself last
        order = np.lexsort((np.broadcast_to(jj, key.shape), np.broadcast_to(me, key.shape), key), axis=-1)[..., :kk]
        sel = q[np.arange(c)[:, None, None], order]                 # [c, a, kk, N, 2]
        O[s0:s0 + c, :, :, :kk, :2] = sel.transpose(0, 1, 3, 2, 4)
        O[s0:s0 + c, :, :, :kk, 2] = clearance
    p[:, :3] = state.reshape(S * R, 3)
    p[:, np_ - 3 * N * K:] = O.reshape(S * R, -1)
    return p, min_dist


def reference_loop(N, T, K, state0, goals, lbx, ubx, lbg, ubg, steps, clearance, tol=1e-1):
    """distributed_loop of a Problem(1, N, T, moving_obstacles=K) restated on the C oracle: state0, goals [S, R, 3].  Returns
    traj [steps+1, S, R, 3], u [steps, S, R, 2], status, iters, active [steps, S, R], min_dist [steps+1, S]."""
    orc = MovingOracle(1, N, T, K)
    S, R, _ = state0.shape
    B = S * R
    state, goals = np.array(state0, np.float64).reshape(B, 3), np.asarray(goals, np.float64).reshape(B, 3)
    p = np.zeros((B, orc.np_))
    p[:, 3:6] = goals
    x0 = np.stack([orc.cold_start(s) for s in state])
    plan = None
    traj = np.empty((steps + 1, B, 3)); traj[0] = state
    u = np.zeros((steps, B, 2)); st = np.zeros((steps, B), np.int32); its = np.zeros((steps, B), np.int32)
    act = np.zeros((steps, B), bool); md = np.empty((steps + 1, S))
    for t in range(steps):
        active = np.linalg.norm(state - goals, axis=1) > tol
        act[t] = active
        if plan is not None:
            plan = np.where(active[:, None], plan, np.stack([orc.cold_start(s) for s in state]))
        p, d = exchange(state.reshape(S, R, 3), plan, clearance, K, N, p)
        md[t] = d.min(axis=1)
        xs = np.empty((B, orc.n))
        for b in range(B):
            r = orc.solve(x0[b], p[b], lbx, ubx, lbg, ubg)
            xs[b], st[t, b], its[t, b] = r["x"], r["status"], r["iters"]
            u0 = r["x"][3 * (N + 1):3 * (N + 1) + 2]
            if active[b]:
                u[t, b] = u0
                state[b] = orc.plant(state[b], u0)
            x0[b] = orc.shift(r["x"])
        plan = xs
        traj[t + 1] = state
    md[steps] = exchange(state.reshape(S, R, 3), None, clearance, K, N, p)[1].min(axis=1)
    sh = lambda a: a.reshape((a.shape[0], S, R) + a.shape[2:])
    return dict(traj=sh(traj), u=sh(u), status=sh(st), iters=sh(its), active=sh(act), min_dist=md)


def circle_swap(R, radius, S=1, rng=None, jitter=0.0):
    """R robots on a circle facing the centre, each going to the antipodal point: state0, goals [S, R, 3] (optionally jittered
    per scenario)."""
    ang = 2 * np.pi * np.arange(R) / R
    head = np.angle(np.exp(1j * (ang + np.pi)))
    start = np.stack([radius * np.cos(ang), radius * np.sin(ang), head], 1)
    goal = np.stack([-radius * np.cos(ang), -radius * np.sin(ang), head], 1)
    st, gl = np.repeat(start[None], S, 0), np.repeat(goal[None], S, 0)
    if jitter and rng is not None:
        st[..., :2] += jitter * rng.uniform(-1, 1, size=(S, R, 2))
        gl[..., :2] += jitter * rng.uniform(-1, 1, size=(S, R, 2))
    return st, gl


def four_robot_crossing():
    """Four robots crossing to the far side of a 1.2 m circle through its centre region, at uneven angles (no exact
    symmetry for a solve to balance on): state0, goals [1, 4, 3]."""
    ang = np.array([0.1, 1.75, 3.3, 4.6])
    head = np.angle(np.exp(1j * (ang + np.pi)))
    start = np.stack([1.2 * np.cos(ang), 1.2 * np.sin(ang), head], 1)
    goal = np.stack([-1.2 * np.cos(ang), -1.2 * np.sin(ang), head], 1)
    return start[None], goal[None]


def passing():
    """Four robots whose solves stay feasible: robot 0 starts at its goal and stops, robot 1 drives past it 0.25 m off its line
    (the rows keep 0.4 m, so it must go round the held pose), robot 2 crosses the far lane the other way and robot 3 drives
    0.8 m, arrives and stops: state0, goals [1, 4, 3]."""
    start = np.array([[0.0, 0.0, 0.0], [-1.2, 0.25, 0.0], [1.0, -0.9, np.pi], [-0.6, 1.0, 0.0]])
    goal = np.array([[0.0, 0.0, 0.0], [1.0, 0.25, 0.0], [-1.0, -0.9, np.pi], [0.2, 1.0, 0.0]])
    return start[None], goal[None]


def hexagon_swap():
    """C-6: six robots on the unit hexagon swapping antipodally (tests/conftest.py hexagon_p): state0, goals [1, 6, 3]."""
    s3 = np.sqrt(3) / 2
    start = np.array([[s3, 0.5, -2.618], [0, 1, -1.571], [-s3, 0.5, -0.524],
                      [-s3, -0.5, 0.524], [0, -1, 1.571], [s3, -0.5, 2.618]])
    goal = -start.copy()
    goal[:, 2] = start[:, 2]
    return start[None], goal[None]

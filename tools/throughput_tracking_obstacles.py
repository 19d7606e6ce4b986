"""Batch throughput of trajectory tracking among obstacles (nmpc_create_tracking_obstacles) against the moving-obstacle handle.

One robot, N = 20, six obstacles moving at 0.05..0.15 m/s (the third scenario's layout at stage 0), B = 8192 cold starts,
warp-per-instance path.  Three cases, timed in alternation (reps rounds of a, b, c):
  (a) moving-obstacle handle (nmpc_create_moving_obstacles), p = [x0bar; xs; O];
  (b) the tracking-among-obstacles handle on the constant reference Z[k] = [xs; 0] with the same O -- must return (a)'s outputs
      bit for bit (asserted);
  (c) the tracking-among-obstacles handle on line references from the start to the goal at 0.15 m/s with feed-forward
      controls, crossed by the same moving obstacles.
Prints solves/s (median, min..max over the rounds), the launches per solve, the mean iterations, the card and its power limit,
and writes the numbers as JSON (default profiles/throughput_tracking_obstacles.json).

    python tools/throughput_tracking_obstacles.py [--B 8192] [--reps 5] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402
from tests.tracking_ref import line_reference  # noqa: E402
from tools.throughput_moving_obstacles import THIRD, card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "throughput_tracking_obstacles.json"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    pkg = ge.load_package()
    B, N, T = a.B, 20, 0.3
    obs = np.array([[x, y, r + 0.15] for x, y, r in THIRD])
    rng = np.random.default_rng(0)
    P = np.tile(np.array([[0.0, 0.6, 1.57, 0.1, 3.9, 1.57]]), (B, 1))
    P[:, :2] += 0.1 * rng.normal(size=(B, 2)); P[:, 3:5] += 0.2 * rng.normal(size=(B, 2))
    ang = rng.uniform(0, 2 * np.pi, size=(B, len(obs)))
    vel = rng.uniform(0.05, 0.15, size=(B, len(obs)))[..., None] * np.stack([np.cos(ang), np.sin(ang)], -1)   # [B, n_obs, 2]
    O = np.repeat(np.repeat(obs[None, None], B, axis=0), N, axis=1)                                            # [B, N, n_obs, 3]
    O[..., :2] += (np.arange(N) * T)[None, :, None, None] * vel[:, None]
    Z = np.stack([line_reference(P[b, :3], P[b, 3:], N, T, speed=0.15) for b in range(B)])                     # [B, N, 5]
    dev = torch.device("cuda:0")
    t = lambda x: torch.as_tensor(np.ascontiguousarray(x), dtype=torch.float64, device=dev)
    mv = pkg.Problem(1, N, T, moving_obstacles=len(obs))
    tr = pkg.Problem(1, N, T, tracking_obstacles=len(obs))
    lbx, ubx, lbg, ubg = (t(x) for x in mv.bounds_obstacles(0.1, 0.2, np.pi / 4))
    x0 = t(mv.cold_start(P[:, :3]))
    x0bar, xs, Ot = t(P[:, :3]), t(P[:, 3:]), t(O)
    pa = mv.params(x0bar, xs, Ot)
    pb = tr.params(x0bar, xs, obstacles=Ot)
    pc = tr.params(x0bar, t(Z[..., :3]), obstacles=Ot, uref=t(Z[..., 3:]))
    cases = {"a_moving_obstacles": (mv, pa), "b_tracking_constant_reference": (tr, pb), "c_tracking_line_references": (tr, pc)}
    outs, times, launches, solved, iters = {}, {k: [] for k in cases}, {}, {}, {}
    for k, (prob, p) in cases.items():     # warm-up (module load, workspace allocation)
        prob.solve(x0, p, lbx, ubx, lbg, ubg)
    torch.cuda.synchronize()
    for _ in range(a.reps):
        for k, (prob, p) in cases.items():
            l0 = prob.launch_count()
            torch.cuda.synchronize(); t0 = time.perf_counter()
            outs[k] = prob.solve(x0, p, lbx, ubx, lbg, ubg)
            torch.cuda.synchronize(); times[k].append(time.perf_counter() - t0)
            launches[k] = prob.launch_count() - l0
    for k in cases:
        solved[k] = (outs[k]["status"] == 0).double().mean().item()
        iters[k] = outs[k]["iters"].double().mean().item()
    for key in ("x", "f", "g", "lam_x", "lam_g", "status", "iters"):
        assert torch.equal(outs["a_moving_obstacles"][key], outs["b_tracking_constant_reference"][key]), "(a) and (b) differ in " + key
    name, plim = card()
    res = dict(card=name, power_limit=plim, B=B, Nr=1, N=N, n_obs=len(obs), reps=a.reps, bitwise_a_equals_b=True, cases={})
    print("%s, power limit %s; B=%d, Nr=1, N=%d, %d obstacles, cold starts, %d rounds" % (name, plim, B, N, len(obs), a.reps))
    for k in cases:
        r = np.array([B / s for s in times[k]])
        res["cases"][k] = dict(solves_per_s_median=float(np.median(r)), solves_per_s_min=float(r.min()), solves_per_s_max=float(r.max()),
                               launches_per_solve=launches[k], solved=solved[k], mean_iters=iters[k])
        print("  %-30s %8.0f solves/s (%.0f .. %.0f)  launches/solve %d  solved %.3f  mean iters %.1f"
              % (k, np.median(r), r.min(), r.max(), launches[k], solved[k], iters[k]))
    ra = res["cases"]["a_moving_obstacles"]["solves_per_s_median"]
    rb = res["cases"]["b_tracking_constant_reference"]["solves_per_s_median"]
    res["b_over_a"] = rb / ra
    print("  (b)/(a) = %.3f;  (a) == (b) bit for bit" % (rb / ra))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()

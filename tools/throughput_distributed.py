"""Distributed NMPC throughput (distributed_loop): control steps per second of S scenarios of R robots, each robot a one-robot
moving-obstacle instance against its K nearest teammates' predicted paths, the neighbour exchange's share of a step (CUDA
events around nmpc_neighbour_obstacles) and the kernel launches per step; beside it the centralized 64-robot swarm's step on the
dense-block path (the solve tools/time_swarm64.py times: 148 instances, the BASELINE workload), and the card's name and power
limit read in the same run.  The two loops solve different problems (K nearest predicted paths per robot against all 2,016
pairs at every stage), so the comparison is one of cost per control step, not a substitute for parity.

    python tools/throughput_distributed.py [--out profiles/throughput_distributed.json] [--steps 30]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402

pkg = ge.load_package()
from oracle.nlp_numpy import synthetic_instances  # noqa: E402

N, T, DMIN, MARGIN = 20, 0.3, 0.3, 0.05


def t64(a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda:0")


def swarm(S, R, seed):
    """S scenarios of R robots: the BASELINE start/goal sampler (8 m box, 0.5 m separation) for R = 64; for larger R (where
    rejection sampling of a whole team never succeeds) starts and goals on a jittered 1 m lattice, goals a random permutation of
    its points, so that the separation stays >= 0.5 m.  Returns state0, goals [S, R, 3] and the half-width of the area."""
    if R == 64:
        P = synthetic_instances(S, Nr=R, seed=seed, box=8.0)
        return P[:, :3 * R].reshape(S, R, 3), P[:, 3 * R:].reshape(S, R, 3), 8.0
    rng = np.random.default_rng(seed)
    side = int(np.ceil(np.sqrt(R)))
    lat = np.stack(np.meshgrid(np.arange(side), np.arange(side)), -1).reshape(-1, 2)[:R] - (side - 1) / 2.0

    def draw():
        xy = lat[rng.permutation(R)] + rng.uniform(-0.25, 0.25, size=(R, 2))
        return np.concatenate([xy, rng.uniform(-np.pi, np.pi, size=(R, 1))], 1)
    return (np.stack([draw() for _ in range(S)]), np.stack([draw() for _ in range(S)]), side / 2.0 + 0.5)


def run_distributed(S, R, K, steps, seed=20261018):
    state0, goals, box = swarm(S, R, seed)
    prob = pkg.Problem(1, N, T, moving_obstacles=K)
    bnd = [t64(a) for a in prob.bounds_obstacles(MARGIN, 0.22, 2.84, xy_box=box + 2.0)]
    st0, gl = t64(state0), t64(goals)
    pkg.distributed_loop(prob, st0, gl, *bnd, 3, DMIN + MARGIN)          # warm-up: modules, allocations
    torch.cuda.synchronize()
    l0 = prob.launch_count()
    t0 = time.perf_counter()
    res = pkg.distributed_loop(prob, st0, gl, *bnd, steps, DMIN + MARGIN)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    launches = (prob.launch_count() - l0) / steps
    # the exchange alone, on the loop's last state and plans, CUDA events over 50 launches
    state = res["traj"][-1].contiguous()
    plan = torch.zeros((S * R, prob.n), dtype=torch.float64, device="cuda:0")
    plan[:, :3 * (N + 1)] = state.reshape(S * R, 3).repeat(1, N + 1)
    p = torch.zeros((S * R, prob.np_), dtype=torch.float64, device="cuda:0")
    for _ in range(5):
        prob.neighbour_obstacles(state, plan, clearance=DMIN + MARGIN, p=p)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(50):
        prob.neighbour_obstacles(state, plan, clearance=DMIN + MARGIN, p=p)
    e1.record()
    torch.cuda.synchronize()
    ex_ms = e0.elapsed_time(e1) / 50
    step_ms = 1e3 * wall / steps
    st = res["status"]
    return dict(S=S, R=R, K=K, N=N, instances_per_step=S * R, steps=steps, steps_per_s=steps / wall, step_ms=step_ms,
                exchange_ms=ex_ms, exchange_share=ex_ms / step_ms, launches_per_step=launches,
                solves_per_s=S * R * steps / wall, status_0_1=(st <= 1).double().mean().item(),
                mean_iters=res["iters"].double().mean().item(), min_pair_distance=res["min_dist"].min().item())


def run_centralized(B=148, reps=2):
    """One control step of the centralized 64-robot swarm (tools/time_swarm64.py's solve, cold start, BASELINE instances)."""
    Nr = 64
    P = synthetic_instances(B, Nr=Nr, seed=20261018, box=8.0)
    prob = pkg.Problem(Nr, N, T)
    lbx, ubx, lbg, ubg = prob.bounds(DMIN, 0.22, 2.84)
    args = [t64(prob.cold_start(P[:, :3 * Nr])), t64(P), t64(lbx), t64(ubx), t64(lbg), t64(ubg)]
    times = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = prob.solve(*args)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    return dict(Nr=Nr, B=B, step_s=min(times), step_s_all=times, status_0_1=(out["status"] <= 1).double().mean().item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "throughput_distributed.json"))
    ap.add_argument("--steps", type=int, default=30)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    rows = []
    for S, R, K in ((148, 64, 8), (148, 64, 16), (148, 64, 8), (148, 64, 16), (16, 1024, 8), (16, 1024, 16)):   # R = 64 alternated
        r = run_distributed(S, R, K, a.steps)
        print(json.dumps(r), flush=True)
        rows.append(r)
    cen = run_centralized()
    print(json.dumps(cen), flush=True)
    res = dict(gpu=smi, torch=torch.__version__, T=T, dmin=DMIN, margin=MARGIN, distributed=rows, centralized_swarm64=cen,
               note="distributed: S scenarios x R robots, one one-robot moving-obstacle instance per robot against its K nearest "
                    "teammates' predicted paths; centralized: one 64-robot NLP per scenario with all 2,016 pair rows per stage. "
                    "Different problems: cost per control step only.")
    for r in rows:
        if r["R"] == 64:
            r["speedup_per_step_vs_centralized"] = cen["step_s"] / (r["step_ms"] / 1e3)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()

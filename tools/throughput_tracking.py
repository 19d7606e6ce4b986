"""Batch throughput of trajectory tracking (nmpc_create_tracking) against the setpoint handle (nmpc_create).

The benchmark workload: six robots, N = 20, T = 0.3, B = 8192 cold starts of the synthetic start/goal table, warp-per-instance
path.  Three cases, timed in alternation (reps rounds of a, b, c):
  (a) nmpc_create, p = [x0bar; xs];
  (b) the tracking handle with the constant reference Z[k] = [xs; 0] -- must return (a)'s outputs bit for bit (asserted);
  (c) the tracking handle with a time-varying, feasible reference: every robot on the straight line from its start to its goal
      at 0.15 m/s (v_max = 0.22) with the matching feed-forward control, holding at the goal.
Also runs, as characterisation, scenario C-6r (six robots swapping across a 0.8 m hexagon, dmin 0.4) in closed loop: once with
the setpoint handle (it ends in a collision-free deadlock), once tracking a reference that rotates the hexagon about its
centre by pi (0.15 rad/s, then holding), and reports how far each ends from the goal.
With --parent-tree DIR (a checkout of an earlier commit with its library built), also re-times the 64-robot swarm (148
instances, dense-block path) and the stand-alone evaluation K1 (B = 65,536 six-robot points) on that tree and on this one,
alternating, each timing in a fresh process.
Prints and writes (default profiles/throughput_tracking.json) solves/s (median, min..max over the rounds), mean iterations,
launches per solve, and the card and its power limit.

    python tools/throughput_tracking.py [--B 8192] [--reps 5] [--parent-tree DIR] [--out FILE]
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
from tests.tracking_ref import line_reference, rotation_reference  # noqa: E402

NR, N, T, DMIN, VMAX, WMAX = 6, 20, 0.3, 0.3, 0.22, 2.84      # the benchmark's problem (bench.py)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30).stdout.strip().splitlines()[0]
        name, plim = [s.strip() for s in q.split(",")]
        return name, plim
    except Exception:
        return torch.cuda.get_device_name(0), "unknown"


def dev(x):
    return torch.as_tensor(np.ascontiguousarray(x), dtype=torch.float64, device="cuda:0")


def throughput(pkg, B, reps):
    P = pkg.workload.synthetic_instances(B, Nr=NR)
    ns = 3 * NR
    reg = pkg.Problem(NR, N, T)
    trk = pkg.Problem(NR, N, T, tracking=True)
    bnd = [dev(a) for a in reg.bounds(DMIN, VMAX, WMAX)]
    x0 = dev(reg.cold_start(P[:, :ns]))
    pa = dev(P)
    pb = trk.params(dev(P[:, :ns]), dev(P[:, ns:]))
    Z = np.stack([line_reference(P[b, :ns], P[b, ns:], N, T) for b in range(B)])          # [B, N, 5 Nr]
    pc = trk.params(dev(P[:, :ns]), dev(Z[:, :, :ns]), uref=dev(Z[:, :, ns:]))
    cases = {"a_setpoint": (reg, pa), "b_tracking_constant": (trk, pb), "c_tracking_line": (trk, pc)}
    outs, times, launches = {}, {k: [] for k in cases}, {}
    for k, (prob, p) in cases.items():     # warm-up (module load, workspace allocation)
        prob.solve(x0, p, *bnd)
    torch.cuda.synchronize()
    for _ in range(reps):
        for k, (prob, p) in cases.items():
            l0 = prob.launch_count()
            torch.cuda.synchronize(); t0 = time.perf_counter()
            outs[k] = prob.solve(x0, p, *bnd)
            torch.cuda.synchronize(); times[k].append(time.perf_counter() - t0)
            launches[k] = prob.launch_count() - l0
    for key in ("x", "f", "g", "lam_x", "lam_g", "status", "iters", "stats"):
        assert torch.equal(outs["a_setpoint"][key], outs["b_tracking_constant"][key]), "(a) and (b) differ in " + key
    res = {}
    for k in cases:
        r = np.array([B / s for s in times[k]])
        res[k] = dict(solves_per_s_median=float(np.median(r)), solves_per_s_min=float(r.min()), solves_per_s_max=float(r.max()),
                      launches_per_solve=launches[k], solved=(outs[k]["status"] == 0).double().mean().item(),
                      mean_iters=outs[k]["iters"].double().mean().item())
    return res


def c6r(pkg, steps_setpoint=400, steps_tracking=120, omega=0.15):
    Nr, T6, N6, dmin, vmax, wmax, start, goal, _ = pkg.mpc_loop.SCENARIOS["C-6r"]
    ns = 3 * Nr
    start = np.asarray(start, float) + 0.02 * np.sin(1.0 + 2.0 * np.arange(ns))     # de-symmetrised as in tests/test_closed_loop.py
    goal = np.asarray(goal, float)
    out = {}
    reg = pkg.Problem(Nr, N6, T6)
    bnd = [dev(a) for a in reg.bounds(dmin, vmax, wmax)]
    r = pkg.closed_loop(reg, dev(np.concatenate([start, goal])[None]), *bnd, steps_setpoint, dmin=dmin)
    xy = r["traj"].cpu().numpy()[:, 0].reshape(-1, Nr, 3)[..., :2]
    out["setpoint"] = dict(steps=steps_setpoint, final_max_xy_dist_to_goal=float(np.linalg.norm(xy[-1] - goal.reshape(Nr, 3)[:, :2], axis=1).max()),
                           min_pair_dist=float(r["min_dist"].item()))
    trk = pkg.Problem(Nr, N6, T6, tracking=True)
    ref = rotation_reference(start, N6, T6, steps_tracking, omega=omega)[:, None, :]       # [steps + N, 1, 5 Nr]
    r = pkg.closed_loop(trk, dev(start[None]), *bnd, steps_tracking, reference=dev(ref))
    xy = r["traj"].cpu().numpy()[:, 0].reshape(-1, Nr, 3)[..., :2]
    out["tracking_rotation"] = dict(steps=steps_tracking, omega=omega,
                                    final_max_xy_dist_to_goal=float(np.linalg.norm(xy[-1] - goal.reshape(Nr, 3)[:, :2], axis=1).max()),
                                    min_pair_dist=float(r["min_dist"].item()),
                                    final_track_err=float(r["track_err"][-1].item()), max_track_err=float(r["track_err"].max().item()),
                                    all_solved=bool((r["status"] <= 1).all().item()))
    return out


def leg(kind, root):
    """One timing leg in this process on the package of the tree `root` (used with --parent-tree): prints a JSON line."""
    sys.path.insert(0, root)
    for m in [m for m in sys.modules if m == "__graft_entry__" or m.startswith("nmpc_b200")]:
        del sys.modules[m]
    import __graft_entry__ as ge_root
    pkg = ge_root.load_package()
    if kind == "swarm64":
        Nr, B = 64, 148
        P = pkg.workload.synthetic_instances(B, Nr=Nr, box=8.0)
        prob = pkg.Problem(Nr, N, T)
        args = [dev(prob.cold_start(P[:, :3 * Nr])), dev(P)] + [dev(a) for a in prob.bounds(DMIN, VMAX, WMAX)]
        prob.solve(*args)
        ts = []
        for _ in range(3):
            torch.cuda.synchronize(); t0 = time.perf_counter()
            out = prob.solve(*args)
            torch.cuda.synchronize(); ts.append(time.perf_counter() - t0)
        print(json.dumps(dict(leg=kind, solves_per_s=B / min(ts), iters=out["iters"].double().mean().item())))
    else:
        B = 65536
        P = pkg.workload.synthetic_instances(1024, Nr=NR)
        prob = pkg.Problem(NR, N, T)
        rng = np.random.default_rng(0)
        w = dev(np.tile(prob.cold_start(P[:, :3 * NR]), (B // 1024, 1)) + 0.01 * rng.normal(size=(B, prob.n)))
        p, lam = dev(np.tile(P, (B // 1024, 1))), dev(rng.normal(size=(B, prob.mg)))
        for _ in range(3):
            prob.eval(w, p, lam)
        ts = []
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); prob.eval(w, p, lam); e1.record()
            torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1) * 1e-3)
        print(json.dumps(dict(leg=kind, points_per_s=B / min(ts))))


def parent_compare(parent_tree, rounds=3):
    """swarm64 and K1 eval on the parent tree and on this one, alternating, each leg in a fresh process."""
    res = {}
    for kind in ("swarm64", "eval_k1"):
        runs = {"parent": [], "this": []}
        for _ in range(rounds):
            for who, root in (("parent", os.path.abspath(parent_tree)), ("this", ROOT)):
                o = subprocess.run([sys.executable, os.path.abspath(__file__), "--leg", kind, "--root", root], capture_output=True,
                                   text=True, check=True).stdout.strip().splitlines()[-1]
                d = json.loads(o)
                runs[who].append(d.get("solves_per_s", d.get("points_per_s")))
        res[kind] = {w: dict(median=float(np.median(v)), min=float(min(v)), max=float(max(v))) for w, v in runs.items()}
        res[kind]["this_over_parent"] = res[kind]["this"]["median"] / res[kind]["parent"]["median"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parent-tree", default=None)
    ap.add_argument("--leg", default=None, choices=["swarm64", "eval_k1"])
    ap.add_argument("--root", default=ROOT)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "throughput_tracking.json"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    if a.leg:
        return leg(a.leg, a.root)
    pkg = ge.load_package()
    name, plim = card()
    res = dict(card=name, power_limit=plim, B=a.B, Nr=NR, N=N, T=T, reps=a.reps, workload="synthetic_instances (bench.py), cold starts",
               bitwise_a_equals_b=True)
    res["cases"] = throughput(pkg, a.B, a.reps)
    ra, rb = res["cases"]["a_setpoint"]["solves_per_s_median"], res["cases"]["b_tracking_constant"]["solves_per_s_median"]
    res["b_over_a"] = rb / ra
    print("%s, power limit %s; B=%d, Nr=%d, N=%d, cold starts, %d rounds" % (name, plim, a.B, NR, N, a.reps))
    for k, c in res["cases"].items():
        print("  %-20s %8.0f solves/s (%.0f .. %.0f)  launches/solve %d  solved %.3f  mean iters %.2f"
              % (k, c["solves_per_s_median"], c["solves_per_s_min"], c["solves_per_s_max"], c["launches_per_solve"], c["solved"],
                 c["mean_iters"]))
    print("  (b)/(a) = %.3f;  (a) == (b) bit for bit" % res["b_over_a"])
    res["c6r"] = c6r(pkg)
    print("  C-6r:", json.dumps(res["c6r"]))
    if a.parent_tree:
        res["vs_parent"] = parent_compare(a.parent_tree)
        print("  vs parent:", json.dumps(res["vs_parent"]))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()

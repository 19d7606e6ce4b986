"""Throughput and latency of the parametric sensitivities (nmpc_solution_vjp / nmpc_solution_jvp) against the solve.

Six robots, N = 20, the synthetic workload of bench.py (synthetic_instances, reference bounds), B = 8192 returned solutions of
a cold solve.  Each round runs in a fresh process and times, on the same handle:
  vjp / jvp:     one call on the B solutions (random seeds), calls of B instances per second;
  cold / warm:   the cold solve of the batch, and the warm solve one MPC step later (plant step + shift of the cold solution);
  latency:       batch-1 wall time (host clock around the call and a synchronise) of one VJP and of one cold solve, median of
                 50 calls.
Prints medians (min..max over the rounds), the card and its power limit, and writes them as JSON
(default profiles/throughput_sensitivity.json).

    python tools/throughput_sensitivity.py [--B 8192] [--rounds 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def child(B):
    import torch
    import __graft_entry__ as ge
    from oracle.nlp_numpy import synthetic_instances
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    pkg = ge.load_package()
    Nr, N, T = 6, 20, 0.1
    dev = torch.device("cuda:0")
    t = lambda x: torch.as_tensor(np.ascontiguousarray(x), dtype=torch.float64, device=dev)
    prob = pkg.Problem(Nr, N, T)
    P = synthetic_instances(B, Nr)
    lbx, ubx, lbg, ubg = (t(x) for x in prob.bounds(0.4, 0.22, 2.84))
    p, x0 = t(P), t(prob.cold_start(P[:, :3 * Nr]))
    rng = np.random.default_rng(1)
    x_bar, p_dot = t(rng.normal(size=(B, prob.n))), t(rng.normal(size=(B, prob.np_)))

    def timed(fn, reps=1):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        return ts

    res = {}
    out = {}
    res["cold_s"] = timed(lambda: out.update(prob.solve(x0, p, lbx, ubx, lbg, ubg)))[0]
    state = prob.plant(p[:, :3 * Nr].contiguous(), out["x"])
    x0w = prob.shift(out["x"])
    pw = torch.cat([state, p[:, 3 * Nr:]], 1).contiguous()
    res["warm_s"] = timed(lambda: prob.solve(x0w, pw, lbx, ubx, lbg, ubg))[0]
    st = {}
    res["vjp_s"] = min(timed(lambda: st.update(vjp=prob.solution_vjp(out, p, lbx, ubx, lbg, ubg, x_bar)[1]), 3))
    res["jvp_s"] = min(timed(lambda: st.update(jvp=prob.solution_jvp(out, p, lbx, ubx, lbg, ubg, p_dot)[1]), 3))
    res["sens_status_ok"] = float(((st["vjp"] == 0) & (st["jvp"] == 0)).double().mean().item())
    res["solved"] = float((out["status"] == 0).double().mean().item())
    o1 = {k: v[:1].contiguous() for k, v in out.items()}
    res["lat_vjp_s"] = float(np.median(timed(lambda: prob.solution_vjp(o1, p[:1], lbx, ubx, lbg, ubg, x_bar[:1]), 50)))
    res["lat_solve_s"] = float(np.median(timed(lambda: prob.solve(x0[:1], p[:1], lbx, ubx, lbg, ubg), 50)))
    print(json.dumps(res))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=8192)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "throughput_sensitivity.json"))
    ap.add_argument("--child", action="store_true")
    a = ap.parse_args()
    if a.child:
        return child(a.B)
    rounds = []
    for _ in range(a.rounds):
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--B", str(a.B)], check=True, capture_output=True, text=True)
        rounds.append(json.loads(r.stdout.strip().splitlines()[-1]))
    from tools.throughput_moving_obstacles import card
    name, plim = card()
    B = a.B
    rate = lambda k: np.array([B / r[k] for r in rounds])
    res = dict(card=name, power_limit=plim, B=B, Nr=6, N=20, rounds=a.rounds, per_round=rounds, summary={})
    print("%s, power limit %s; B=%d, Nr=6, N=20, %d rounds in fresh processes" % (name, plim, B, a.rounds))
    for k, label in (("vjp_s", "VJP"), ("jvp_s", "JVP"), ("cold_s", "cold solve"), ("warm_s", "warm solve")):
        r = rate(k)
        res["summary"][label] = dict(instances_per_s_median=float(np.median(r)), min=float(r.min()), max=float(r.max()))
        print("  %-11s %12.0f instances/s (%.0f .. %.0f)" % (label, np.median(r), r.min(), r.max()))
    for k, label in (("lat_vjp_s", "batch-1 VJP"), ("lat_solve_s", "batch-1 solve")):
        v = np.array([r[k] for r in rounds]) * 1e3
        res["summary"][label] = dict(ms_median=float(np.median(v)), min=float(v.min()), max=float(v.max()))
        print("  %-13s %8.3f ms (%.3f .. %.3f)" % (label, np.median(v), v.min(), v.max()))
    res["summary"]["vjp_over_cold"] = float(np.median(rate("vjp_s")) / np.median(rate("cold_s")))
    res["summary"]["jvp_over_cold"] = float(np.median(rate("jvp_s")) / np.median(rate("cold_s")))
    print("  VJP / cold solve = %.0f x, JVP / cold solve = %.0f x;  solved %.4f, sens status 0 on %.4f"
          % (res["summary"]["vjp_over_cold"], res["summary"]["jvp_over_cold"], rounds[-1]["solved"], rounds[-1]["sens_status_ok"]))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()

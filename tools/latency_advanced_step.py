"""Latency and throughput of advanced-step NMPC (nmpc_solution_x0_jacobian / nmpc_advanced_step) against the solve.

The six-robot N = 20 configuration of bench.py (T = 0.3, dmin = 0.3, reference bounds, synthetic_instances).  One process, one
handle, the card's name and power limit read in the same call:
  batch 1 (host clock around the call and a synchronise, 20 warm-up calls, p50 / p90 of 200): the warm solve (one MPC step
  after a cold solve: plant step + shift), the VJP (for comparison), nmpc_solution_x0_jacobian (preparation) and
  nmpc_advanced_step (feedback);
  B = 8192: one Jacobian pass against one nmpc_solution_jvp call on the same solutions (CUDA events, best of 5), instances/s;
  closed loops of 512 instances x 40 steps with x, y, theta noise of sigma = 1e-3: wall time of the ideal loop
  (closed_loop(disturbance=)) and of the advanced-step loop (advanced_step=True), each after one warm-up loop.

    python tools/latency_advanced_step.py [--out profiles/latency_advanced_step.json]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "latency_advanced_step.json"))
    a = ap.parse_args()
    import torch
    import __graft_entry__ as ge
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    pkg = ge.load_package()
    Nr, N, T, dmin, vmax, wmax = 6, 20, 0.3, 0.3, 0.22, 2.84
    dev = torch.device("cuda:0")
    t = lambda x: torch.as_tensor(np.ascontiguousarray(x), dtype=torch.float64, device=dev)
    prob = pkg.Problem(Nr, N, T)
    ns = prob.ns
    bounds = [t(x) for x in prob.bounds(dmin, vmax, wmax)]
    lbx, ubx, lbg, ubg = bounds
    res = {}
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    res["gpu"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"
    res["device_name"] = torch.cuda.get_device_name(dev)
    res["config"] = dict(Nr=Nr, N=N, T=T, dmin=dmin, vmax=vmax, wmax=wmax)

    def host_clock(fn, reps=200, warm=20):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
        return dict(p50_ms=float(np.percentile(ts, 50)), p90_ms=float(np.percentile(ts, 90)))

    # ---- batch 1
    P1 = pkg.workload.synthetic_instances(1, Nr)
    p1 = t(P1)
    cold = prob.solve(t(prob.cold_start(P1[:, :ns])), p1, *bounds)
    p1w = p1.clone()
    p1w[:, :ns] = prob.plant(p1[:, :ns].contiguous(), cold["x"])
    x0w = prob.shift(cold["x"])
    warm = prob.solve(x0w, p1w, *bounds)
    jac1, st1 = prob.solution_x0_jacobian(warm, p1w, *bounds)
    meas = (p1w[:, :ns] + 1e-3).contiguous()
    xb = torch.ones_like(warm["x"])
    lat = {}
    lat["warm_solve"] = host_clock(lambda: prob.solve(x0w, p1w, *bounds))
    lat["vjp"] = host_clock(lambda: prob.solution_vjp(warm, p1w, *bounds, xb))
    lat["x0_jacobian"] = host_clock(lambda: prob.solution_x0_jacobian(warm, p1w, *bounds))
    lat["advanced_step"] = host_clock(lambda: prob.advanced_step(warm, jac1, st1, p1w, meas, lbx, ubx))
    res["batch1"] = lat
    res["batch1_sens_status"] = int(st1.item())

    # ---- B = 8192: Jacobian pass against one JVP call
    B = 8192
    P = pkg.workload.synthetic_instances(B, Nr)
    p = t(P)
    out = prob.solve(t(prob.cold_start(P[:, :ns])), p, *bounds)
    p_dot = t(np.random.default_rng(1).normal(size=(B, prob.np_)))

    def events(fn, reps=5):
        fn()
        torch.cuda.synchronize()
        best = float("inf")
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1) / 1e3)
        return best

    st = {}
    tj = events(lambda: st.update(jac=prob.solution_x0_jacobian(out, p, *bounds)[1]))
    tv = events(lambda: st.update(jvp=prob.solution_jvp(out, p, *bounds, p_dot)[1]))
    res["B8192"] = dict(x0_jacobian_s=tj, jvp_s=tv, x0_jacobian_inst_per_s=B / tj, jvp_inst_per_s=B / tv,
                        jacobian_over_jvp_time=tj / tv, columns=ns,
                        sens_status_ok=float(((st["jac"] == 0) & (st["jvp"] == 0)).double().mean().item()),
                        solved=float((out["status"] == 0).double().mean().item()))

    # ---- closed loops
    Bl, steps, sigma = 512, 40, 1e-3
    Pl = t(pkg.workload.synthetic_instances(Bl, Nr, seed=20261022))
    w = t(sigma * np.random.default_rng(2).normal(size=(steps, Bl, ns)))
    loops = {}
    for name, kw in (("ideal", {}), ("advanced_step", dict(advanced_step=True))):
        pkg.closed_loop(prob, Pl, *bounds, steps, disturbance=w, **kw)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = pkg.closed_loop(prob, Pl, *bounds, steps, disturbance=w, **kw)
        torch.cuda.synchronize()
        loops[name] = dict(wall_s=time.perf_counter() - t0, min_dist=float(r["min_dist"].min()),
                           solved=float((r["status"][r["active"]] == 0).double().mean().item()))
    res["closed_loop_512x40"] = loops
    print(json.dumps(res, indent=1))
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()

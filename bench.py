#!/usr/bin/env python
"""bench.py -- 6-robot, N=20 NMPC solves/sec on B200 (BASELINE.json metric), one JSON line.

  python bench.py --gpus 1 --steps K --warmup W          (N>1: launched by torch.distributed.run)
  python bench.py --impl reference ...                    CPU arm: the restated IPOPT path on host cores
  python bench.py ... --dump-outputs DIR                  also write the last timed step's outputs as DIR/<name>.npy

A step = one cold-start solve (X_k = start, U = 0; centralized_six_robots_implementation.py:398-400)
of a batch of synthetic start/goal instances (SURVEY.md 8d recipe).  Instances are independent, so
ranks shard them with no collective on the data path ("weak": 8192 instances per GPU = 65536 / 8).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NR, NH, T, DMIN, VMAX, WMAX = 6, 20, 0.3, 0.3, 0.22, 2.84      # sixth_scenario.py:127-135, N overridden to 20
PER_GPU = 8192
ALG_BYTES_PER_SOLVE = 15728       # SURVEY.md 8d: p + w0 in, x + f + g out
F_FACT, F_SOLVE, F_EVAL = 1100160, 92160, 14700   # SURVEY.md 8d dense-stage FP64 flop counts @ Nr=6, N=20
F_ITER = F_FACT + F_SOLVE + F_EVAL                # 1.207 MFLOP per interior-point iteration (SURVEY.md 8d's unit of work)
DUMP_BYTES = 64_000_000           # --dump-outputs: bytes written, all files together


def dump_outputs(out, path):
    """Write the arrays one solve returned to its caller (x, f, g, stats, status, iters) as float64 DIR/<name>.npy, row b
    of every file being the same instance.  When the whole batch would exceed DUMP_BYTES, a default_rng(0) sample of
    instances is written instead (the same one for every run at a given batch size); instance.npy holds their indices."""
    arrs = {k: v.cpu().numpy().astype(np.float64) for k, v in out.items()}
    B = len(arrs["x"])
    row_bytes = 8 * (1 + sum(a[0].size for a in arrs.values()))      # 1: the instance index
    keep = min(B, (DUMP_BYTES - 4096) // row_bytes)                    # 4096: room for the .npy headers
    idx = np.arange(B) if keep == B else np.sort(np.random.default_rng(0).choice(B, keep, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "instance.npy"), idx.astype(np.float64))
    for k, a in arrs.items():
        np.save(os.path.join(path, k + ".npy"), a[idx])


def measured_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of solve_kernel<6> per solve, from the latest committed ncu --set full
    capture (profiles/solve_kernel_traffic.json names the capture); None when the file is missing."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "solve_kernel_traffic.json")))
        return (t["dram_bytes_read"] + t["dram_bytes_write"]) / t["instances"], t["source"]
    except (OSError, KeyError, ValueError):
        return None, None


def load_pkg():
    import __graft_entry__ as ge
    return ge.load_package()


def shard(rank, world, per_gpu):
    """This rank's slice of ONE default_rng(20261018) table of world * per_gpu instances (65,536 at 8 x 8,192; BASELINE.md 2),
    split by sharding.shard_range.  Host-only code of the package (workload.py): no CUDA needed."""
    return load_pkg().workload.bench_shard(rank, world, per_gpu, NR)


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.sm_max = index, False, [], set(), None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                     nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
            while not self.stop_flag:
                self.sm.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.05)
        except Exception as e:      # no NVML: report what we have
            self.reasons.add("nvml_unavailable:%s" % type(e).__name__)

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons)}


def cpu_arm(P, nthreads, budget_s=20.0):
    """Restated IPOPT path (oracle/, 'port') on the host cores, bounded sample of the same workload."""
    from oracle.oracle_lib import Oracle
    o = Oracle(NR, NH, T)
    lbx, ubx, lbg, ubg = o.bounds(DMIN, VMAX, WMAX)
    n = 0
    t0 = time.perf_counter()
    chunk = max(2 * nthreads, 16)
    iters = []
    while n < len(P) and time.perf_counter() - t0 < budget_s:
        Pi = P[n:n + chunk]
        x0 = np.stack([o.cold_start(q[:3 * NR]) for q in Pi])
        r = o.solve_batch(x0, Pi, lbx, ubx, lbg, ubg, nthreads=nthreads)
        iters.append(r["iters"])
        n += len(Pi)
    dt = time.perf_counter() - t0
    return n / dt, n, dt, float(np.concatenate(iters).mean())


def cpu_one_core(steps=60):
    """BASELINE.md 2: the CPU path on ONE core -- cold solves/s over the first instances of the workload and p50 / p95
    single-solve latency over the closed-loop hexagon swap (the loop timed at centralized_six...py:482), restated IPOPT."""
    from oracle.oracle_lib import Oracle
    wl = load_pkg().workload
    o = Oracle(NR, NH, T)
    lbx, ubx, lbg, ubg = o.bounds(DMIN, VMAX, WMAX)
    P = wl.synthetic_instances(48, NR)
    t0 = time.perf_counter()
    n = 0
    for q in P:
        o.solve(o.cold_start(q[:3 * NR]), q, lbx, ubx, lbg, ubg)
        n += 1
        if time.perf_counter() - t0 > 6.0:
            break
    cold = n / (time.perf_counter() - t0)
    p1 = wl.hexagon_swap(True)
    w = o.cold_start(p1[:18])
    times = []
    for _ in range(steps):
        t1 = time.perf_counter()
        r = o.solve(w, p1, lbx, ubx, lbg, ubg)
        times.append(time.perf_counter() - t1)
        x = r["x"]
        p1[:18] = o.plant(p1[:18], x[18 * (NH + 1):18 * (NH + 1) + 12])
        w = o.shift(x)
    return {"cold_solves_per_s": cold, "cold_sample": n, "p50_ms": 1e3 * float(np.median(times[1:])), "p95_ms": 1e3 * float(np.percentile(times[1:], 95)),
            "first_cold_ms": 1e3 * times[0], "loop_steps": steps,
            "note": "one host core, restated IPOPT (oracle/): cold solves of the first instances; p50/p95 over the %d-step closed-loop hexagon swap" % steps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--per-gpu", type=int, default=PER_GPU)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--swarm", type=int, default=148, help="N=1 only: also time this many 64-robot swarm instances (BASELINE.json configs[4]) on the dense-block path; 0 = skip")
    ap.add_argument("--clone", type=int, default=-1, help="diagnostic: replicate one instance B times (all warps run in lockstep)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned (rank 0's shard) as DIR/<name>.npy, "
                                                          "at most 64 MB (a fixed sample of instances when the batch is larger)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs records the CUDA path; the reference arm solves a time-bounded, run-dependent sample")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    ncores = os.cpu_count() or 1
    config = {"workload": "6-robot N=20 cold-start NMPC (sixth_scenario.py constants), %d synthetic start/goal instances per GPU: rank r's "
                          "slice of one default_rng(20261018) table of n_gpus x %d instances (65536 at 8 GPUs)" % (a.per_gpu, a.per_gpu),
              "Nr": NR, "N": NH, "T": T, "dmin": DMIN, "batch_per_gpu": a.per_gpu, "l2": "flushed between timed steps (512 MiB write)"}

    if a.impl == "reference":
        if rank != 0:
            return
        P, _ = shard(0, 1, a.per_gpu)
        per_step = []
        tot_n = tot_t = 0
        mean_it = 0.0
        for s in range(a.warmup + a.steps):
            v, n, dt, mean_it = cpu_arm(P, ncores, budget_s=8.0 if s >= a.warmup else 2.0)
            if s >= a.warmup:
                per_step.append(dt); tot_n += n; tot_t += dt
        val = tot_n / tot_t
        line = {"impl": "reference", "metric": "6-robot N=20 NMPC solves/sec", "value": val, "unit": "solves/s", "n_gpus": a.gpus,
                "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * float(np.mean(per_step)), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": val, "unit": "solves/s", "cores": ncores, "kind": "port",
                                 "sample": "first %d cold-start instances of the same workload per step (~8 s), restated IPOPT "
                                           "(oracle/nmpc_oracle.c, OpenMP); CasADi/IPOPT are not installable here" % (tot_n // max(1, a.steps)),
                                 "mean_iters": mean_it, "one_core": cpu_one_core()},
                "e2e": {"value": val, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import torch
    pkg = load_pkg()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    B = a.per_gpu
    P, (shard_lo, shard_hi) = shard(rank, world, B)
    if a.clone >= 0:
        P = np.repeat(P[a.clone:a.clone + 1], B, axis=0)
    prob = pkg.Problem(NR, NH, T)
    lbx, ubx, lbg, ubg = prob.bounds(DMIN, VMAX, WMAX)
    x0 = prob.cold_start(P[:, :3 * NR])
    t = lambda v: torch.as_tensor(np.ascontiguousarray(v), dtype=torch.float64, device=dev)
    d_x0, d_p, d_lbx, d_ubx, d_lbg, d_ubg = t(x0), t(P), t(lbx), t(ubx), t(lbg), t(ubg)
    out = {}
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)

    def step():
        prob.solve(d_x0, d_p, d_lbx, d_ubx, d_lbg, d_ubg, want=("f", "g", "stats"), out=out)

    for _ in range(a.warmup):
        step()
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = prob.launch_count()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    evs = []
    for _ in range(a.steps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); step(); e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize()
    if a.dump_outputs and rank == 0:
        dump_outputs(out, a.dump_outputs)
    if world > 1:
        dist.barrier()
    ms = [e0.elapsed_time(e1) for e0, e1 in evs]
    launches = prob.launch_count() - launches0
    sampler.stop_flag = True
    sampler.join(timeout=2)
    st = out["status"].cpu().numpy()
    stats = out["stats"].cpu().numpy()
    iters = out["iters"].cpu().numpy()
    solved = float((st == 0).mean())
    # per-rank record: its own device time and the iteration statistics of its shard (the makespan of a rank is decided by
    # the tail of its 4.6 waves, so the MAX over ranks grows with the number of different shards)
    mine = torch.tensor([sum(ms) / a.steps, float(iters.mean()), float(iters.max()), float(stats[:, 8].mean()), float(stats[:, 8].max()),
                         float(shard_lo)], dtype=torch.float64, device=dev)
    allr = [torch.zeros_like(mine) for _ in range(world)]
    if world > 1:
        dist.all_gather(allr, mine)
    else:
        allr = [mine]
    per_rank = [{"rank": r, "ms_per_step": v[0].item(), "mean_ip_iters": v[1].item(), "max_ip_iters": int(v[2].item()),
                 "mean_factorisations": v[3].item(), "max_factorisations": int(v[4].item()), "first_instance": int(v[5].item())}
                for r, v in enumerate(allr)]
    tot_ms = torch.tensor([sum(ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot_ms, op=dist.ReduceOp.MAX)
    tot_ms = tot_ms.item()

    # ---- end to end through the host-buffer C-ABI call (pinned inputs, H2D + solve + D2H of x, status, iters) ----
    pin = lambda v: torch.as_tensor(np.ascontiguousarray(v), dtype=torch.float64).pin_memory().numpy()
    h_x0, h_p = pin(x0), pin(P)
    h_out = {"x": torch.empty((B, prob.n), dtype=torch.float64).pin_memory().numpy(),
             "status": torch.empty(B, dtype=torch.int32).pin_memory().numpy(),
             "iters": torch.empty(B, dtype=torch.int32).pin_memory().numpy()}
    prob.solve_host(h_x0, h_p, lbx, ubx, lbg, ubg, want=(), out=h_out)      # warm-up (allocates the staging buffers)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(a.e2e_steps):
        prob.solve_host(h_x0, h_p, lbx, ubx, lbg, ubg, want=(), out=h_out)
    e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    h2d = 8 * (h_x0.size + h_p.size + 2 * lbx.size + 2 * lbg.size)
    d2h = 8 * h_out["x"].size + 4 * 2 * B
    e2e_val = world * B * a.e2e_steps / e2e_s.item()

    # ---- second timed mode (SURVEY.md 8d): warm start = apply u0 through the Euler plant, shift, re-solve ----
    xo = out["x"].clone()
    d_p2 = d_p.clone()
    d_p2[:, :3 * NR] = prob.plant(d_p[:, :3 * NR].contiguous(), xo)
    d_x0w = prob.shift(xo)
    outw = {}
    prob.solve(d_x0w, d_p2, d_lbx, d_ubx, d_lbg, d_ubg, want=("stats",), out=outw)
    torch.cuda.synchronize()
    # longest-first scheduling from the PREVIOUS solve's iteration counts (what a closed loop has at hand: nmpc_set_order)
    prob.set_order(prob.order_from_iters(out["iters"]))
    prob.solve(d_x0w, d_p2, d_lbx, d_ubx, d_lbg, d_ubg, want=("stats",), out=outw)      # untimed warm-up in the new order
    torch.cuda.synchronize()
    wev = []
    for _ in range(a.steps):
        flush.fill_(1)
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record()
        prob.solve(d_x0w, d_p2, d_lbx, d_ubx, d_lbg, d_ubg, want=("stats",), out=outw)
        w1.record()
        wev.append((w0, w1))
    torch.cuda.synchronize()
    prob.set_order(None)
    warm_ms = torch.tensor([sum(e0.elapsed_time(e1) for e0, e1 in wev) / a.steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(warm_ms, op=dist.ReduceOp.MAX)
    warm = {"value": world * B / (warm_ms.item() * 1e-3), "unit": "solves/s", "ms_steps": [round(e0.elapsed_time(e1), 2) for e0, e1 in wev], "mean_ip_iters": float(outw["iters"].double().mean().item()),
            "solved_frac": float((outw["status"] == 0).double().mean().item()), "max_ip_iters": int(outw["iters"].max().item()),
            "note": "one MPC step later: Euler plant + reference shift as initial guess (the closed-loop regime); instances "
                    "scheduled longest-first by the previous step's iteration counts (nmpc_set_order)"}

    # ---- the same cold steps issued back to back on two streams (two handles, two workspaces): the next batch's CTAs take the SMs that the
    #      tail of the previous batch leaves idle.  An EXTRA: `value` above stays one step at a time (each step drains before the next starts) ----
    piped = None
    if rank == 0 and world == 1:
        prob2 = pkg.Problem(NR, NH, T)
        streams = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)]
        pouts = [{}, {}]
        pp = [prob, prob2]
        for i in range(2):
            with torch.cuda.stream(streams[i]):
                pp[i].solve(d_x0, d_p, d_lbx, d_ubx, d_lbg, d_ubg, want=("stats",), out=pouts[i])
        torch.cuda.synchronize()
        k2 = a.steps
        flush.fill_(1)
        p0 = torch.cuda.Event(enable_timing=True)
        p0.record()
        ends = []
        for sidx in range(k2):
            st_ = streams[sidx % 2]
            st_.wait_event(p0)
            with torch.cuda.stream(st_):
                pp[sidx % 2].solve(d_x0, d_p, d_lbx, d_ubx, d_lbg, d_ubg, want=("stats",), out=pouts[sidx % 2])
                e_ = torch.cuda.Event(enable_timing=True)
                e_.record()
                ends.append(e_)
        torch.cuda.synchronize()
        p_ms = max(p0.elapsed_time(e_) for e_ in ends)
        piped = {"value": k2 * B / (p_ms * 1e-3), "unit": "solves/s", "steps": k2, "ms_total": p_ms,
                 "solved_frac": float((pouts[0]["status"] == 0).double().mean().item()),
                 "note": "extra, not the headline: the same cold batches launched alternately on two streams with two workspaces, so that "
                         "batch s+1 back-fills the SMs idled by the tail of batch s (the per-step figure pays that tail every step); "
                         "the working set of a step (667 MB) is larger than L2, no flush between the overlapped steps"}
        del prob2

    # ---- p50 single-solve latency: hexagon swap (C-6 constants, N=20), closed loop, batch = 1, host buffers ----
    lat = None
    if rank == 0:
        p1 = pkg.workload.hexagon_swap(True)[None]        # de-symmetrised (see tests/test_closed_loop.py)
        w1_ = prob.cold_start(p1[:, :18])
        times, o1 = [], {}
        for step in range(60):
            t0 = time.perf_counter()
            prob.solve_host(w1_, p1, lbx, ubx, lbg, ubg, want=(), out=o1)
            times.append(time.perf_counter() - t0)
            u0 = o1["x"][0, 18 * (NH + 1):18 * (NH + 1) + 12]
            for i in range(6):
                th = p1[0, 3 * i + 2]
                p1[0, 3 * i] += T * u0[2 * i] * np.cos(th); p1[0, 3 * i + 1] += T * u0[2 * i] * np.sin(th); p1[0, 3 * i + 2] += T * u0[2 * i + 1]
            X = o1["x"][0, :18 * (NH + 1)].reshape(NH + 1, 18); U = o1["x"][0, 18 * (NH + 1):].reshape(NH, 12)
            w1_ = np.concatenate([np.concatenate([X[1:], X[NH - 1:NH]]).ravel(), np.concatenate([U[1:], U[-1:]]).ravel()])[None]
        lat = {"p50_ms": 1e3 * float(np.median(times[1:])), "p95_ms": 1e3 * float(np.percentile(times[1:], 95)), "first_cold_ms": 1e3 * times[0],
               "steps": 60, "note": "batch=1 closed loop through nmpc_solve_host (H2D of p and guess, solve, D2H of x), wall clock"}

    # ---- BASELINE.json configs[4]: 64-robot swarm on the CTA-per-instance dense-block path (one timed launch) ----
    swarm = None
    if rank == 0 and world == 1 and a.swarm > 0:
        Bs, Ns = a.swarm, 64
        Ps = pkg.workload.synthetic_instances(min(Bs, 8), Nr=Ns, seed=20261018, box=8.0)
        Ps = np.tile(Ps, ((Bs + len(Ps) - 1) // len(Ps), 1))[:Bs]      # 8 distinct instances, repeated (rejection sampling 64 robots is slow)
        sp = pkg.Problem(Ns, NH, T)
        sb = sp.bounds(DMIN, VMAX, WMAX)
        sargs = [t(sp.cold_start(Ps[:, :3 * Ns])), t(Ps)] + [t(v) for v in sb]
        so = {}
        sp.solve(sargs[0][:1], sargs[1][:1], *sargs[2:], want=("stats",), out={})      # warm-up launch: one instance
        torch.cuda.synchronize()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(); sp.solve(*sargs, want=("stats",), out=so); s1.record()
        torch.cuda.synchronize()
        s_ms = s0.elapsed_time(s1)
        nf = so["stats"][:, 8].double().mean().item()
        nx, nu = 3 * Ns, 2 * Ns
        dense = NH * (4 * nx ** 3 + 6 * nx * nx * nu + 3 * nx * nu * nu + nu ** 3 / 3.0)       # SURVEY.md 8d dense-stage count
        executed = NH * (nu ** 3 / 3.0 + nu * nu * (nx + 1) + nx * nx * nu)                    # Cholesky + triangular solve + symmetric rank-k update
        swarm = {"workload": "64-robot N=20 cold-start swarm (2016 pair rows per stage), %d instances, one CTA per instance" % Bs,
                 "value": Bs / (s_ms * 1e-3), "unit": "solves/s", "ms": s_ms, "solved_frac": float((so["status"] == 0).double().mean().item()),
                 "mean_ip_iters": float(so["iters"].double().mean().item()), "mean_factorisations": nf,
                 "fp64_tflops_dense_stage_count": Bs / (s_ms * 1e-3) * nf * dense / 1e12,
                 "fp64_tflops_executed_upper_bound": Bs / (s_ms * 1e-3) * nf * executed / 1e12}
        del sp, sargs, so

    # ---- BASELINE.json configs[0]: the Van der Pol multiple-shooting demo (mpc_pose_control_casadi.py), thread per instance ----
    vdp = None
    if rank == 0 and world == 1 and a.swarm > 0:
        ocp = pkg.SmallOcp("van_der_pol", N=20, T=10.0, rk_steps=4)
        w0, lbw, ubw, lbg0, ubg0 = ocp.demo_arrays()
        o1 = ocp.solve_host(w0, lbw, ubw, lbg0, ubg0)                       # warm-up (module load, staging buffers)
        t0 = time.perf_counter(); o1 = ocp.solve_host(w0, lbw, ubw, lbg0, ubg0); t_one = time.perf_counter() - t0
        Bv = 16384
        rngv = np.random.default_rng(1)
        W0 = np.tile(w0, (Bv, 1)); W0[:, 2:] += 0.1 * rngv.normal(size=(Bv, ocp.n - 2))
        ob = ocp.solve_host(W0, lbw, ubw, lbg0, ubg0, want=())
        t0 = time.perf_counter(); ob = ocp.solve_host(W0, lbw, ubw, lbg0, ubg0, want=()); t_b = time.perf_counter() - t0
        vdp = {"workload": "Van der Pol demo, N=20, T=10, 4 RK4 steps per interval (62 variables, 40 shooting rows)",
               "single_solve_ms": 1e3 * t_one, "iters": int(o1["iters"][0]), "status": int(o1["status"][0]), "f": float(o1["f"][0]),
               "batch": Bv, "batch_solves_per_s": Bv / t_b, "batch_solved_frac": float((ob["status"] == 0).mean()),
               "note": "host buffers, wall clock; batch = the demo's problem from 16384 perturbed initial guesses"}

    if rank != 0:
        return
    value = world * B * a.steps / (tot_ms * 1e-3)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    per_gpu_solves = B * a.steps / (tot_ms * 1e-3)
    import ctypes
    tf, tdm = ctypes.c_double(0.0), ctypes.c_double(0.0)
    pkg.lib().nmpc_probe_fp64(ctypes.byref(tf))
    pkg.lib().nmpc_probe_dmma(ctypes.byref(tdm))
    # SURVEY.md 8d: achieved = solves/s x mean interior-point iterations x 1.207 MFLOP (dense-stage count of ONE factorisation,
    # back-solve and evaluation per iteration; failed inertia attempts are not useful work and are not counted)
    ach_tf = per_gpu_solves * float(iters.mean()) * F_ITER / 1e12
    flops_refact = float((stats[:, 8] * F_FACT + iters * (F_SOLVE + F_EVAL)).mean())
    traffic_per_solve, traffic_src = measured_traffic()
    cpu_val, cpu_n, cpu_dt, cpu_it = cpu_arm(P, ncores, budget_s=15.0)     # same instances as the GPU arm, bounded to ~15 s
    line = {
        "metric": "6-robot N=20 NMPC solves/sec", "value": value, "unit": "solves/s", "n_gpus": world, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": tot_ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": config,
        "solved_frac": solved, "mean_ip_iters": float(iters.mean()), "max_ip_iters": int(iters.max()),
        "mean_factorisations": float(stats[:, 8].mean()),
        "roofline": {"bound": "fp64", "achieved": ach_tf, "peak": tf.value, "unit": "TFLOP/s", "frac": ach_tf / tf.value if tf.value else None,
                     "traffic": traffic_per_solve * B if traffic_per_solve else None, "traffic_source": traffic_src,
                     "flops_per_unit": F_ITER, "units_per_launch": float(iters.sum()),
                     "peak_source": "nmpc_probe_fp64: register-only DFMA kernel timed in this run (MEASURED_PEAKS.json has no FP64 figure)",
                     "note": "solve_kernel<6>: the binding resource is the FP64 pipe / dependent-issue latency / instruction fetch, not HBM "
                             "and not tensor cores (tcgen05 has no f64 kind; DMMA probe below); see roofline_hbm for the memory view"},
        "roofline_hbm": {"achieved": per_gpu_solves * traffic_per_solve / 1e9 if traffic_per_solve else None, "peak": hbm_peak, "unit": "GB/s",
                         "frac": per_gpu_solves * traffic_per_solve / 1e9 / hbm_peak if traffic_per_solve else None,
                         "algorithmic_gbs": per_gpu_solves * ALG_BYTES_PER_SOLVE / 1e9, "algorithmic_bytes_per_solve": ALG_BYTES_PER_SOLVE,
                         "measured_bytes_per_solve": traffic_per_solve, "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md)",
                         "note": "measured DRAM traffic of the committed ncu capture x this run's solves/s: the scratch rows of the resident "
                                 "instances stream through HBM (they do not fit L2)"},
        "fp64_extras": {"refactorisation_inclusive_tflops": per_gpu_solves * flops_refact / 1e12,
                        "refactorisation_inclusive_frac": per_gpu_solves * flops_refact / 1e12 / tf.value if tf.value else None,
                        "dmma_probe_tflops": tdm.value, "dfma_probe_tflops": tf.value,
                        "note": "refactorisation-inclusive = every factorisation attempt (also those that fail the inertia test) at the dense-stage "
                                "count; dmma_probe = mma.sync.m8n8k4.f64 micro-probe (nmpc_probe_dmma)"},
        "per_rank": per_rank,
        "cpu_baseline": {"value": cpu_val, "unit": "solves/s", "cores": ncores, "kind": "port",
                         "sample": "%d cold-start instances of the same workload in %.1f s, restated IPOPT (oracle/), OpenMP" % (cpu_n, cpu_dt),
                         "mean_iters": cpu_it, "one_core": cpu_one_core()},
        "e2e": {"value": e2e_val, "unit": "solves/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "warm_start": warm, "pipelined": piped, "latency": lat, "swarm64": swarm, "van_der_pol": vdp,
        "gpu_launches": launches, "clocks": sampler.summary(),
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

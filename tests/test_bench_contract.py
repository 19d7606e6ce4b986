"""bench.py's output: the JSON line (one line, the keys of the measurement contract) of the reference arm (`--impl reference`,
the CPU restatement of the path timed on the host cores, no GPU needed), and the arrays `--dump-outputs DIR` writes."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip().startswith("{")]
    assert len(lines) == 1, p.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["n_gpus"] == 1
    assert d["unit"] == "solves/s" and d["value"] > 0 and d["steps"] == 1
    assert "6-robot" in d["metric"] and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    oc = cb["one_core"]      # BASELINE.md 2: one-core solves/s and the closed-loop p50 / p95
    assert oc["cold_solves_per_s"] > 0 and 0 < oc["p50_ms"] <= oc["p95_ms"]


def _read_dump(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_outputs_fits_the_cap_and_samples_the_same_instances_every_run(tmp_path):
    """A full 8,192-instance step (6 robots, N = 20) is larger than the cap: a fixed sample of whole instances is written,
    the same in every run, and the files together stay within 64 MB.  A small batch is written whole."""
    import torch
    from bench import DUMP_BYTES, dump_outputs
    rng = np.random.default_rng(3)
    for B, sampled in ((8192, True), (40, False)):
        out = {"x": torch.from_numpy(rng.normal(size=(B, 618))), "f": torch.from_numpy(rng.normal(size=B)),
               "g": torch.from_numpy(rng.normal(size=(B, 693))), "stats": torch.from_numpy(rng.normal(size=(B, 11))),
               "status": torch.from_numpy(rng.integers(0, 5, B).astype(np.int32)),
               "iters": torch.from_numpy(rng.integers(5, 60, B).astype(np.int32))}
        runs = []
        for rep in range(2):
            d = str(tmp_path / ("B%d_%d" % (B, rep)))
            dump_outputs(out, d)
            assert sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)) <= DUMP_BYTES <= 64 * 10 ** 6
            runs.append(_read_dump(d))
        got = runs[0]
        assert sorted(got) == ["f", "g", "instance", "iters", "stats", "status", "x"]
        idx = got["instance"].astype(np.int64)
        assert np.array_equal(idx, got["instance"]) and np.all(np.diff(idx) > 0)
        assert (len(idx) < B) == sampled and len(idx) > 0.5 * B
        for k, v in out.items():
            assert got[k].dtype == np.float64 and np.array_equal(got[k], v.numpy()[idx].astype(np.float64)), k
        for k in got:
            assert np.array_equal(got[k], runs[1][k]), k


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step_and_honours_steps(tmp_path, pkg):
    """--dump-outputs writes what the timed cold solve returned: bit for bit what a direct solve of the same instances gives.
    --steps sets the number of timed steps of every leg that repeats the step."""
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    B = 256
    d = str(tmp_path / "dump")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                        "--per-gpu", str(B), "--swarm", "0", "--e2e-steps", "1", "--dump-outputs", d],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip().startswith("{")]
    assert len(lines) == 1, p.stdout[-2000:]
    res = json.loads(lines[0])
    assert res["steps"] == 2 and res["pipelined"]["steps"] == 2 and len(res["warm_start"]["ms_steps"]) == 2
    got = _read_dump(d)
    assert np.array_equal(got["instance"], np.arange(B))
    P, _ = pkg.workload.bench_shard(0, 1, B, 6)
    prob = pkg.Problem(6, 20, 0.3)
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda")
    ref = prob.solve(t(prob.cold_start(P[:, :18])), t(P), *[t(a) for a in prob.bounds(0.3, 0.22, 2.84)], want=("f", "g", "stats"))
    torch.cuda.synchronize()
    for k, v in ref.items():
        assert np.array_equal(got[k], v.cpu().numpy().astype(np.float64)), k

#!/usr/bin/env python
"""The pruned arg-max (ombo_score, fast mode, exact 2-D EHVI) against OMBO_NO_PRUNE=1 on the C5 headline of bench.py.

Runs `bench.py --gpus 1` RUNS times each way, alternating, on one card; then the depth-2 bound (OMBO_PRUNE_DEPTH=2)
and 8 instead of 16 generator warps in the bound pass (OMBO_FAST_GEN_WARPS=8), one profiled step per variant
(torch.profiler: bound-pass kernel time, i.e. the BOUND instantiations of k_posterior_fast8, against the full launches
of the threshold and the survivors), and one complete default `bench.py` line (value, roofline, accuracy record).
Survivor counts come from OMBO_PRUNE_LOG.  Card name and power limit are read in the same call.
Writes profiles/r04_prune.{json,md} (or --out DIR)."""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--no-e2e", "--no-fit", "--no-refresh-timing",
         "--no-extras", "--no-cpu-baseline"]


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    name, power, clk = [c.strip() for c in q.split(",")]
    return {"name": name, "power_limit": power, "sm_max_clock": clk}


def bench(env_extra, steps, warmup, dump=None):
    env = dict(os.environ, OMBO_PRUNE_LOG="1", **env_extra)
    cmd = BENCH + ["--steps", str(steps), "--warmup", str(warmup)] + (["--dump-outputs", dump] if dump else [])
    out = subprocess.run(cmd, env=env, capture_output=True, text=True, cwd=ROOT)
    if out.returncode:
        raise SystemExit(out.stderr[-3000:])
    line = json.loads(out.stdout.strip().splitlines()[-1])
    surv = [int(m.group(1)) for m in re.finditer(r"\[prune\] m \d+ survivors (\d+)", out.stderr)]
    return {"value": line["value"], "ms_per_step": (1 << 24) / line["value"] * 1e3, "survivors": surv[-steps:],
            "clocks": line.get("clocks")}


PROFILE = r"""
import json, sys, numpy as np, torch
sys.path.insert(0, {root!r})
import bench as B, optimobo_b200 as ob
X, Y, ells, sf2 = B.workload()
models = [ob.GPModel(X, Y[:, i], ells[i], sf2[i], device="cuda:0") for i in range(2)]
PF, r = ob.host_prep.calc_pf(Y), Y.max(0)
spec = ob.spec_ehvi(r, PF, ob.host_prep.cached_samples(2, 5, seed=0), "exact")
pool = ob.CandidatePool.counter(1 << 24, np.zeros(10), np.ones(10), seed=1)
for _ in range(2):
    ob.score(models, spec, pool, precision="fast")
torch.cuda.synchronize()
from torch.profiler import profile, ProfilerActivity
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    ob.score(models, spec, pool, precision="fast")
    torch.cuda.synchronize()
k = {{}}
for e in prof.events():
    if e.device_type.name == "CUDA":
        k[e.name] = k.get(e.name, 0.0) + e.device_time / 1e3
print(json.dumps(k))
"""


def profile_step(env_extra):
    env = dict(os.environ, **env_extra)
    out = subprocess.run([sys.executable, "-c", PROFILE.format(root=ROOT)], env=env, capture_output=True, text=True)
    if out.returncode:
        return {"error": out.stderr[-2000:]}
    k = json.loads(out.stdout.strip().splitlines()[-1])
    f8 = {n: t for n, t in k.items() if "k_posterior_fast8" in n}
    bound = sum(t for n, t in f8.items() if _is_bound(n))
    full = sum(f8.values()) - bound
    return {"bound_pass_ms": bound, "full_launches_ms": full, "other_ms": sum(k.values()) - sum(f8.values()),
            "kernels": k}


def _is_bound(name):
    # k_posterior_fast8<DP, R, GW, MATERN, BOUND>: the last template argument
    m = re.search(r"k_posterior_fast8<([^>]*)>", name)
    return bool(m) and m.group(1).split(",")[-1].strip() == "true"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=4)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    a = ap.parse_args()
    rec = {"card": card(), "workload": "bench.py C5 headline: 2^24 candidates, n = 1024, d = 10, 2 GPs, exact 2-D EHVI",
           "pruned": [], "unpruned": []}
    dumps = os.path.join(a.out, "r04_dumps")
    for i in range(a.runs):
        rec["unpruned"].append(bench({"OMBO_NO_PRUNE": "1"}, a.steps, a.warmup,
                                     os.path.join(dumps, "A") if i == 0 else None))
        rec["pruned"].append(bench({}, a.steps, a.warmup, os.path.join(dumps, "B") if i == 0 else None))
    # the default bound pass: chunk 0 (depth 1), 16 generator warps; the other three corners
    rec["depth2"] = bench({"OMBO_PRUNE_DEPTH": "2"}, a.steps, a.warmup)
    rec["gen8"] = bench({"OMBO_FAST_GEN_WARPS": "8"}, a.steps, a.warmup)
    rec["depth2_gen8"] = bench({"OMBO_PRUNE_DEPTH": "2", "OMBO_FAST_GEN_WARPS": "8"}, a.steps, a.warmup)
    import numpy as np
    same = all(np.array_equal(np.load(os.path.join(dumps, "A", f)), np.load(os.path.join(dumps, "B", f)))
               for f in ("best_value.npy", "best_index.npy"))
    rec["outputs_identical"] = same
    rec["profile"] = {"depth1": profile_step({}), "depth2": profile_step({"OMBO_PRUNE_DEPTH": "2"}),
                      "unpruned": profile_step({"OMBO_NO_PRUNE": "1"})}
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "5", "--warmup", "2"],
                         capture_output=True, text=True, cwd=ROOT)
    if out.returncode:
        raise SystemExit(out.stderr[-3000:])
    line = json.loads(out.stdout.strip().splitlines()[-1])
    rec["full_bench_line"] = {k: line.get(k) for k in ("value", "ms_per_step", "roofline", "clocks", "accuracy", "best")}
    rec["card_after"] = card()
    ms = {k: [r["ms_per_step"] for r in rec[k]] for k in ("pruned", "unpruned")}
    rec["summary"] = {k: {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v)} for k, v in ms.items()}
    rec["summary"]["speedup_median"] = statistics.median(ms["unpruned"]) / statistics.median(ms["pruned"])
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "r04_prune.json"), "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({"summary": rec["summary"], "card": rec["card"], "outputs_identical": same,
                      "depth2_ms": rec["depth2"]["ms_per_step"], "gen8_ms": rec["gen8"]["ms_per_step"],
                      "depth2_gen8_ms": rec["depth2_gen8"]["ms_per_step"],
                      "survivors": rec["pruned"][0]["survivors"],
                      "full_bench_line": {k: rec["full_bench_line"][k] for k in ("value", "ms_per_step")},
                      "same_argmax": (rec["full_bench_line"]["accuracy"] or {}).get("same_argmax"),
                      "profile": {k: {kk: vv for kk, vv in v.items() if kk != "kernels"} for k, v in rec["profile"].items()}},
                     indent=1))


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""The two-stage pruned arg-max (mean-only stage 1 in front of the chunk-0 bound) against the depth-1 path alone
(OMBO_PRUNE_STAGE1=0) on the C5 headline of bench.py.

Runs `bench.py --gpus 1` RUNS times each way, alternating, on one card, and compares the --dump-outputs of the two
arms; then one profiled step per arm (torch.profiler, a run of its own): stage 1 (k_posterior_mean8), the BOUND
launches of k_posterior_fast8 (the depth-1 pass over the whole pool, or over the stage-1 survivors) and the rest.
Survivor counts per stage come from OMBO_PRUNE_LOG.  Card name, power limit and NVML clocks are read in the same call.
Writes profiles/r08_cascade.json (or --out DIR)."""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--no-e2e", "--no-fit", "--no-refresh-timing",
         "--no-extras", "--no-cpu-baseline"]


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    name, power, clk_max, clk = [c.strip() for c in q.split(",")]
    return {"name": name, "power_limit": power, "sm_max_clock": clk_max, "sm_clock_now": clk}


def bench(env_extra, steps, warmup, dump=None):
    env = dict(os.environ, OMBO_PRUNE_LOG="1", **env_extra)
    cmd = BENCH + ["--steps", str(steps), "--warmup", str(warmup)] + (["--dump-outputs", dump] if dump else [])
    out = subprocess.run(cmd, env=env, capture_output=True, text=True, cwd=ROOT)
    if out.returncode:
        raise SystemExit(out.stderr[-3000:])
    line = json.loads(out.stdout.strip().splitlines()[-1])
    s1 = [int(m.group(1)) for m in re.finditer(r"\[prune1\] m \d+ survivors (\d+)", out.stderr)]
    s2 = [int(m.group(1)) for m in re.finditer(r"\[prune\] m \d+ survivors (\d+)", out.stderr)]
    return {"value": line["value"], "ms_per_step": (1 << 24) / line["value"] * 1e3, "stage1_survivors": s1[-steps:],
            "stage2_survivors": s2[-steps:], "clocks": line.get("clocks")}


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


THRESHOLD = r"""
import ctypes as C, json, sys, numpy as np, torch
sys.path.insert(0, {root!r})
import bench as B, optimobo_b200 as ob
from optimobo_b200 import _cabi
X, Y, ells, sf2 = B.workload()
models = [ob.GPModel(X, Y[:, i], ells[i], sf2[i], device="cuda:0") for i in range(2)]
PF, r = ob.host_prep.calc_pf(Y), Y.max(0)
spec = ob.spec_ehvi(r, PF, ob.host_prep.cached_samples(2, 5, seed=0), "exact")
m = 1 << 24
pool = ob.CandidatePool.counter(m, np.zeros(10), np.ones(10), seed=1)
val = ob.score(models, spec, pool, precision="fast", want_acq=True).acq        # full values (unpruned)
fn = _cabi.lib().ombo_debug_mean8
fn.argtypes = [C.c_void_p, C.POINTER(_cabi.Gp), C.POINTER(_cabi.Pool), C.POINTER(_cabi.Acq)] + [C.c_void_p] * 4
mu = torch.empty((2, m), dtype=torch.float64, device="cuda:0")
ub = torch.empty(m, dtype=torch.float64, device="cuda:0")
best = torch.empty(2, dtype=torch.int64, device="cuda:0")
gps = (_cabi.Gp * 2)(*[md.c_struct(1e-15) for md in models])
p, a = pool.c_struct(), spec.c_struct(torch.device("cuda:0"))
_cabi.check(fn(_cabi.Context.get(0).handle, gps, C.byref(p), C.byref(a), C.c_void_p(mu.data_ptr()),
               C.c_void_p(ub.data_ptr()), C.c_void_p(best.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
torch.cuda.synchronize()
ubn = torch.where(torch.isnan(ub), torch.full_like(ub, -np.inf), ub)
ub_max = float(ubn.max())
vn = torch.where(torch.isnan(val), torch.full_like(val, -np.inf), val)
n_sms = torch.cuda.get_device_properties(0).multi_processor_count
def survivors(cand):
    v0 = float(vn[cand].max())
    return int((torch.isnan(ub) | (ub >= v0 - 2e-3 * ub_max)).sum()), v0
out = {{"pool_best": float(vn.max())}}
# CTA c of the launch walks the 256-candidate tiles c, c + grid, ...: its maximum is the shipped threshold row
cta = (torch.arange(m, device="cuda:0") // 256) % n_sms
per_cta = torch.stack([torch.argmax(torch.where(cta == c, ubn, torch.full_like(ubn, -np.inf))) for c in range(n_sms)])
for name, cand in (("T=1 (bound arg-max)", torch.argmax(ubn)[None]), ("T=32 (top 32 bounds)", torch.topk(ubn, 32).indices),
                   ("T=%d (per-CTA maxima, shipped)" % n_sms, per_cta), ("T=1024 (top 1024 bounds)", torch.topk(ubn, 1024).indices)):
    n, v0 = survivors(cand)
    out[name] = {{"stage1_survivors": n, "v0": v0}}
print(json.dumps(out))
"""


def threshold_study():
    """stage-1 survivors on the 2^24 pool for several choices of the threshold candidates"""
    out = subprocess.run([sys.executable, "-c", THRESHOLD.format(root=ROOT)], capture_output=True, text=True)
    if out.returncode:
        return {"error": out.stderr[-2000:]}
    return json.loads(out.stdout.strip().splitlines()[-1])


def profile_step(env_extra):
    env = dict(os.environ, **env_extra)
    out = subprocess.run([sys.executable, "-c", PROFILE.format(root=ROOT)], env=env, capture_output=True, text=True)
    if out.returncode:
        return {"error": out.stderr[-2000:]}
    k = json.loads(out.stdout.strip().splitlines()[-1])
    stage1 = sum(t for n, t in k.items() if "k_posterior_mean8" in n)
    bound = sum(t for n, t in k.items() if _is_bound(n))
    return {"stage1_ms": stage1, "bound_pass_ms": bound, "rest_ms": sum(k.values()) - stage1 - bound, "kernels": k}


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
           "cascade": [], "depth1": []}
    tmp = tempfile.TemporaryDirectory()
    dumps = tmp.name
    for i in range(a.runs):
        rec["depth1"].append(bench({"OMBO_PRUNE_STAGE1": "0"}, a.steps, a.warmup,
                                   os.path.join(dumps, "A") if i == 0 else None))
        rec["cascade"].append(bench({}, a.steps, a.warmup, os.path.join(dumps, "B") if i == 0 else None))
    import numpy as np
    same = all(np.array_equal(np.load(os.path.join(dumps, "A", f)), np.load(os.path.join(dumps, "B", f)))
               for f in ("best_value.npy", "best_index.npy"))
    rec["outputs_identical"] = same
    tmp.cleanup()
    rec["threshold_study"] = threshold_study()
    rec["profile"] = {"cascade": profile_step({}), "depth1": profile_step({"OMBO_PRUNE_STAGE1": "0"})}
    rec["card_after"] = card()
    ms = {k: [r["ms_per_step"] for r in rec[k]] for k in ("cascade", "depth1")}
    rec["summary"] = {k: {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v), "all_ms": v}
                      for k, v in ms.items()}
    rec["summary"]["speedup_median"] = statistics.median(ms["depth1"]) / statistics.median(ms["cascade"])
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "r08_cascade.json"), "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({"summary": rec["summary"], "card": rec["card"], "card_after": rec["card_after"],
                      "outputs_identical": same,
                      "stage1_survivors": rec["cascade"][0]["stage1_survivors"],
                      "stage2_survivors": rec["cascade"][0]["stage2_survivors"],
                      "depth1_survivors": rec["depth1"][0]["stage2_survivors"],
                      "threshold_study": rec["threshold_study"],
                      "profile": {k: {kk: vv for kk, vv in v.items() if kk != "kernels"} for k, v in rec["profile"].items()}},
                     indent=1))


if __name__ == "__main__":
    main()

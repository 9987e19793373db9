#!/usr/bin/env python
"""Stage 1 of the pruned arg-max on the tensor core (posterior_stage1_tc.cu, the default) against the exact-mean stage 1
(OMBO_STAGE1_KERNEL=mean8) on the C5 headline of bench.py.

Runs `bench.py --gpus 1` RUNS times each way, alternating, on one card, compares the --dump-outputs of the two arms and
records the stage-1 / stage-2 survivor counts (OMBO_PRUNE_LOG); then one profiled step per arm (torch.profiler, a run
of its own): stage-1 kernel time and its cycles per 128-candidate x 64-column block at the SM clock read in the same
call.  Card name, power limit and NVML clocks are read in the same call.  Writes profiles/r10_stage1_tc.json (or
--out DIR)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from cascade_bench import PROFILE, ROOT, bench, card  # noqa: E402

ARMS = {"tc": {}, "mean8": {"OMBO_STAGE1_KERNEL": "mean8"}}
STAGE1 = ("k_stage1_tc", "k_posterior_mean8")


def profile_step(env_extra, clock_mhz):
    env = dict(os.environ, **env_extra)
    out = subprocess.run([sys.executable, "-c", PROFILE.format(root=ROOT)], env=env, capture_output=True, text=True)
    if out.returncode:
        return {"error": out.stderr[-2000:]}
    k = json.loads(out.stdout.strip().splitlines()[-1])
    stage1 = sum(t for n, t in k.items() if any(s in n for s in STAGE1))
    # 2 GPs x 2^24 candidates / 148 SMs, in 128-row tiles of 16 K-blocks of 64 training points (n = 1024)
    blocks_per_sm = 2 * (1 << 24) / 148 / 128 * 16
    return {"stage1_ms": stage1, "rest_ms": sum(k.values()) - stage1,
            "stage1_cycles_per_block": stage1 * 1e-3 * clock_mhz * 1e6 / blocks_per_sm, "kernels": k}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=4)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    a = ap.parse_args()
    rec = {"card": card(), "workload": "bench.py C5 headline: 2^24 candidates, n = 1024, d = 10, 2 GPs, exact 2-D EHVI",
           "tc": [], "mean8": []}
    tmp = tempfile.TemporaryDirectory()
    for i in range(a.runs):
        for arm in ("mean8", "tc"):
            rec[arm].append(bench(ARMS[arm], a.steps, a.warmup, os.path.join(tmp.name, arm) if i == 0 else None))
    import numpy as np
    rec["outputs_identical"] = all(
        np.array_equal(np.load(os.path.join(tmp.name, "mean8", f)), np.load(os.path.join(tmp.name, "tc", f)))
        for f in ("best_value.npy", "best_index.npy"))
    tmp.cleanup()
    clock = float(rec["card"]["sm_max_clock"].split()[0])
    if not a.no_profile:
        rec["profile"] = {arm: profile_step(env, clock) for arm, env in ARMS.items()}
    rec["card_after"] = card()
    ms = {arm: [r["ms_per_step"] for r in rec[arm]] for arm in ARMS}
    rec["summary"] = {arm: {"median_ms": statistics.median(v), "spread_ms": max(v) - min(v), "all_ms": v}
                      for arm, v in ms.items()}
    rec["summary"]["speedup_median"] = statistics.median(ms["mean8"]) / statistics.median(ms["tc"])
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "r10_stage1_tc.json"), "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({"summary": rec["summary"], "card": rec["card"], "card_after": rec["card_after"],
                      "outputs_identical": rec["outputs_identical"],
                      "survivors": {arm: [rec[arm][0]["stage1_survivors"][:1], rec[arm][0]["stage2_survivors"][:1]]
                                    for arm in ARMS},
                      "clocks": {arm: [r["clocks"] for r in rec[arm]] for arm in ARMS},
                      "profile": {k: {kk: vv for kk, vv in v.items() if kk != "kernels"}
                                  for k, v in rec.get("profile", {}).items()}}, indent=1))


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Batch proposals on one card: what the exact device top-k (ombo_score_topk) costs next to ombo_score, and what the
Kriging-believer batch (propose_batch) costs with its shortlist certificate against a brute-force believer.

1. C5 step (n = 1024, d = 10, exact 2-D EHVI, fast mode, 2^24 counter candidates): ombo_score_topk at
   k in {1, 256, 4096, 65536} against ombo_score unpruned (the same spec without OMBO_ACQ_FRONT_VALID, so the call
   takes the passes the top-k takes) and pruned.  CUDA events around each call; variants alternate inside every
   repetition after a warm-up of each.
2. Time per batch, q in {2, 4, 8}: propose_batch (default shortlist) against a brute-force believer that runs one
   ombo_score per step (pruned where eligible) with the same fantasy models, on C5 EHVI exact (2^24), C4-shaped box
   EHVI (n = 512, d = 12, k = 3, 2^22) and EI on one GP of the C2 shape (ZDT1, n = 256, d = 10, 2^24).
3. Certification rate (steps 1..7 of q = 8 decided by the shortlist) against shortlist in {256, 1024, 4096, 16384}
   on the same workloads, over three pool seeds.
Card name and power limit are read in the same call.  Writes profiles/r05_batch.{json,md} (or --out DIR)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import optimobo_b200 as ob  # noqa: E402
from optimobo_b200 import _cabi  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    name, power, clk = [c.strip() for c in q.split(",")]
    return {"name": name, "power_limit": power, "sm_max_clock": clk}


def zdt(n, d, k=2, seed=0):
    rng = np.random.default_rng(seed)
    X = rng.random((n, d))
    f1 = X[:, 0]
    g = 1 + 9.0 / (d - 1) * X[:, 1:].sum(1)
    return X, np.column_stack([f1, g * (1 - np.sqrt(f1 / g)), g * (1 - X[:, 1]) + 0.5 * f1][:k])


def front_spec_for(build, PF, r):
    def spec_for(Yb):
        inside = Yb[np.all(Yb <= r, axis=1)] if len(Yb) else Yb
        return build(ob.host_prep.calc_pf(np.vstack([PF, inside])) if len(inside) else PF)
    return spec_for


def workloads():
    out = {}
    X, Y = zdt(1024, 10)
    models = [ob.GPModel(X, Y[:, i], [0.7, 0.8][i] * np.ones(10), [1.0, 2.0][i]) for i in range(2)]
    PF, r = ob.host_prep.calc_pf(Y), Y.max(0)
    cache = ob.host_prep.cached_samples(2, 5, seed=0)
    out["C5 EHVI exact"] = (models, front_spec_for(lambda F: ob.spec_ehvi(r, F, cache, "exact"), PF, r), 10, 24,
                            "fast")
    X, Y = zdt(512, 12, k=3)
    models = [ob.GPModel(X, Y[:, i], [0.7, 0.8, 0.9][i] * np.ones(12), [1.0, 2.0, 1.5][i]) for i in range(3)]
    PF, r = ob.host_prep.calc_pf(Y), Y.max(0)
    out["C4 box"] = (models, front_spec_for(lambda F: ob.spec_ehvi_box(r, F), PF, r), 12, 22, "fast")
    X, Y = zdt(256, 10)
    model = ob.GPModel(X, Y[:, 1], 0.8 * np.ones(10), 2.0)
    best = float(Y[:, 1].min())
    out["C2 EI"] = ([model], lambda Yb: ob.spec_ei(min(best, float(Yb.min())) if len(Yb) else best), 10, 24, "fast")
    return out


def timed(fn):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e)


def brute_batch(models, spec_for, pool, q, precision):
    Yb = np.empty((0, len(models)))
    picked = []
    for j in range(q):
        if j > 0:
            x = pool.rows(picked[-1], 1)
            mu, _ = ob.posterior(models, x, precision="fp64")
            y = mu[:, 0].cpu().numpy()
            Yb = np.vstack([Yb, y[None, :]])
            models = [m.with_observations(x, y[g:g + 1]) for g, m in enumerate(models)]
        res = ob.score(models, spec_for(Yb), pool, precision=precision)
        picked.append(res.best_index)
    return picked


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    info = dict(card=card(), reps=args.reps)
    wl = workloads()
    # 1. top-k selection overhead at C5
    models, spec_for, d, log2m, prec = wl["C5 EHVI exact"]
    spec = spec_for(np.empty((0, 2)))
    unpruned = ob.acquisition.AcquisitionSpec(**{**spec.__dict__, "reserved": 0, "_dev": {}})
    pool = ob.CandidatePool.counter(1 << log2m, np.zeros(d), np.ones(d), seed=1)
    variants = {"score unpruned": lambda: ob.score(models, unpruned, pool, precision=prec, sync=False),
                "score pruned": lambda: ob.score(models, spec, pool, precision=prec, sync=False)}
    for k in (1, 256, 4096, 65536):
        variants[f"topk k={k}"] = (lambda k=k: ob.score_topk(models, spec, pool, k, precision=prec))
    for fn in variants.values():
        fn(), fn()
    times = {name: [] for name in variants}
    for _ in range(args.reps):
        for name, fn in variants.items():
            times[name].append(timed(fn))
    info["c5_step_ms"] = {name: statistics.median(t) for name, t in times.items()}
    info["c5_step_ms_spread"] = {name: [min(t), max(t)] for name, t in times.items()}
    print(json.dumps(info["c5_step_ms"]), flush=True)
    # 2. + 3. batches
    info["batch_ms"], info["cert_rate"] = {}, {}
    for wname, (models, spec_for, d, log2m, prec) in wl.items():
        pool = ob.CandidatePool.counter(1 << log2m, np.zeros(d), np.ones(d), seed=5)
        ob.propose_batch(models, spec_for, pool, 2, precision=prec)                   # warm-up
        brute_batch(models, spec_for, pool, 2, prec)
        rows = {}
        for q in (2, 4, 8):
            t = {"shortlist": [], "brute": []}
            agree = True
            for _ in range(max(1, args.reps // 2)):
                t0 = time.perf_counter()
                _, _, idx, _ = ob.propose_batch(models, spec_for, pool, q, precision=prec)
                torch.cuda.synchronize()
                t["shortlist"].append(1e3 * (time.perf_counter() - t0))
                t0 = time.perf_counter()
                want = brute_batch(models, spec_for, pool, q, prec)
                torch.cuda.synchronize()
                t["brute"].append(1e3 * (time.perf_counter() - t0))
                agree &= list(idx) == want
            rows[q] = {k: statistics.median(v) for k, v in t.items()}
            rows[q]["same_picks"] = bool(agree)
        info["batch_ms"][wname] = rows
        rates = {}
        for K in (256, 1024, 4096, 16384):
            c = n = 0
            for seed in (5, 6, 7):
                pool = ob.CandidatePool.counter(1 << log2m, np.zeros(d), np.ones(d), seed=seed)
                _, _, _, cert = ob.propose_batch(models, spec_for, pool, 8, precision=prec, shortlist=K)
                c += int(cert[1:].sum())
                n += 7
            rates[K] = c / n
        info["cert_rate"][wname] = rates
        print(wname, json.dumps(rows), json.dumps(rates), flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r05_batch.json"), "w") as f:
        json.dump(info, f, indent=1)
    c = info["card"]
    lines = [f"# Batch proposals: top-k overhead and Kriging-believer batches ({c['name']}, power limit "
             f"{c['power_limit']}, max SM clock {c['sm_max_clock']})", "",
             "Written by scripts/batch_bench.py; medians of the repetitions, CUDA events (section 1) or a host clock "
             "around work that ends in a device synchronise (section 2).", "",
             "## C5 step, 2^24 candidates, exact 2-D EHVI, fast mode", "", "| call | ms | min..max |", "|---|---|---|"]
    for name, v in info["c5_step_ms"].items():
        lo, hi = info["c5_step_ms_spread"][name]
        lines.append(f"| {name} | {v:.2f} | {lo:.2f}..{hi:.2f} |")
    base = info["c5_step_ms"]["score unpruned"]
    lines += ["", "Selection overhead over the unpruned step: " + ", ".join(
        f"k={k}: {100 * (info['c5_step_ms'][f'topk k={k}'] / base - 1):+.1f} %" for k in (1, 256, 4096, 65536)), "",
              f"## Time per batch (default shortlist {ob.acquisition.BATCH_SHORTLIST}) against a brute-force believer",
              "", "| workload | q | shortlist KB ms | brute-force KB ms | same picks |", "|---|---|---|---|---|"]
    for wname, rows in info["batch_ms"].items():
        for q, r in rows.items():
            lines.append(f"| {wname} | {q} | {r['shortlist']:.1f} | {r['brute']:.1f} | {r['same_picks']} |")
    lines += ["", "## Certification rate (steps 1..7 of q = 8, three pools)", "",
              "| workload | K=256 | K=1024 | K=4096 | K=16384 |", "|---|---|---|---|---|"]
    for wname, rates in info["cert_rate"].items():
        lines.append(f"| {wname} | " + " | ".join(f"{rates[K]:.2f}" for K in (256, 1024, 4096, 16384)) + " |")
    with open(os.path.join(args.out, "r05_batch.md"), "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()

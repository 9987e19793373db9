"""The box decomposition behind the exact box EHVI built on the device (device_prep.ehvi_boxes, ombo_ehvi_boxes)
against the host (host_prep.ehvi_boxes), on one GPU:

  1. One decomposition, host clock from the numpy front to the device tensors after a device synchronise, for sphere
     fronts at k = 3 (66 / 256 / 512 points) and k = 4 (150 / 256 / 400 points), and at small fronts (4 to 32 points)
     for the crossover behind prep_on_device="auto".  Warm-up first; host and device calls alternate.  Every device
     result is checked equal to the host's.
  2. One q = 8 Kriging-believer batch (propose_batch) with box EHVI at a 3-objective front of 256 points over 2^22
     candidates, each step's spec built from scratch on the host and on the device (the optimiser's spec_for), host
     clock with a device synchronise.  Both pick the same rows.

Card name and power limit are read in the same run.  Writes profiles/r07_ehvi_boxes_device.{json,md} (or --out DIR).
Run from the repository root."""
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
import optimobo_b200 as ob  # noqa: E402
from optimobo_b200 import device_prep, host_prep  # noqa: E402

DEV = "cuda:0"


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    name, power, clk = [c.strip() for c in q.split(",")]
    return {"name": name, "power_limit": power, "sm_max_clock": clk}


def sphere(P, k, seed):
    X = np.abs(np.random.default_rng(seed).normal(size=(P, k)))
    return X / np.linalg.norm(X, axis=1, keepdims=True)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t0) * 1e3


def decomposition(k, P, reps):
    F, r = sphere(P, k, 100 * k + P), np.full(k, 1.1)
    table, boxes = host_prep.ehvi_boxes(F, r)
    t_dev, b_dev = device_prep.ehvi_boxes(F, r, DEV)                       # warm-up (and the buffer size)
    assert np.array_equal(t_dev.cpu().numpy(), table) and np.array_equal(b_dev.cpu().numpy(), boxes)
    host_ms, dev_ms = [], []
    for _ in range(reps):
        host_ms.append(timed(lambda: host_prep.ehvi_boxes(F, r))[1])
        dev_ms.append(timed(lambda: device_prep.ehvi_boxes(F, r, DEV))[1])
    return {"k": k, "points": P, "boxes": len(boxes), "B": table.shape[1], "reps": reps,
            "host_ms": float(np.median(host_ms)), "device_ms": float(np.median(dev_ms)),
            "device_ms_min": float(np.min(dev_ms)), "device_ms_max": float(np.max(dev_ms))}


def batch(device, models, pf, pool, q):
    max_point = np.full(3, 1.1)

    def spec_for(Y_bel):                    # MultiSurrogateOptimiser._batch_spec_for with ehvi="box"
        inside = np.asarray(Y_bel, dtype=float).reshape(-1, 3)
        inside = inside[np.all(inside <= max_point, axis=1)]
        front = host_prep.calc_pf(np.vstack([pf, inside])) if len(inside) else pf
        return ob.spec_ehvi_box(max_point, front, device=device)

    (X, _, idx, cert), ms = timed(lambda: ob.propose_batch(models, spec_for, pool, q, precision="fast"))
    return idx, cert, ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--batch-reps", type=int, default=2)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs the GPU"
    info = {"card": card(), "decomposition": [], "crossover": []}
    print(info["card"], flush=True)
    for k, Ps in ((3, (66, 256, 512)), (4, (150, 256, 400))):
        for P in Ps:
            row = decomposition(k, P, args.reps if P < 400 else max(2, args.reps // 2))
            info["decomposition"].append(row)
            print(json.dumps(row), flush=True)
    for k in (3, 4):
        for P in (4, 8, 12, 16, 24, 32):
            row = decomposition(k, P, 4 * args.reps)
            info["crossover"].append(row)
            print(json.dumps(row), flush=True)

    # q = 8 Kriging-believer batch, k = 3, front of 256 points, 2^22 candidates
    rng = np.random.default_rng(7)
    n, d, m, q = 300, 6, 1 << 22, 8
    X = rng.random((n, d))
    W = rng.normal(size=(d, 3))
    Y = 0.5 + 0.3 * np.sin(3 * X @ W)
    models = [ob.GPModel(X, Y[:, i], 0.5 * np.ones(d), 0.1, device=DEV) for i in range(3)]
    pf = sphere(256, 3, 9)
    pool = ob.CandidatePool.counter(m, np.zeros(d), np.ones(d), seed=5)
    batch(DEV, models, pf, pool, q)                                            # warm-up
    rows = {"host": [], "device": []}
    picks = {}
    for _ in range(args.batch_reps):
        for name, device in (("host", None), ("device", DEV)):
            idx, cert, ms = batch(device, models, pf, pool, q)
            rows[name].append(ms)
            picks[name] = idx.tolist()
    assert picks["host"] == picks["device"], picks
    info["batch"] = {"k": 3, "front": 256, "boxes": len(host_prep.ehvi_boxes(pf, np.full(3, 1.1))[1]), "q": q,
                     "candidates": m, "precision": "fast", "reps": args.batch_reps,
                     "host_ms": float(np.median(rows["host"])), "device_ms": float(np.median(rows["device"])),
                     "same_rows": True}
    print(json.dumps(info["batch"]), flush=True)

    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r07_ehvi_boxes_device.json"), "w") as f:
        json.dump(info, f, indent=1)
    c = info["card"]
    lines = [f"# Box decomposition on the device against the host ({c['name']}, power limit {c['power_limit']}, "
             f"max SM clock {c['sm_max_clock']})", "",
             "`scripts/ehvi_boxes_device_bench.py`.  Host clock from the numpy front to the result after a device "
             "synchronise, median over the repetitions after a warm-up; host (`host_prep.ehvi_boxes`, one CPU thread "
             "of the GPU host) and device (`device_prep.ehvi_boxes`) calls alternate.  Sphere fronts, r = 1.1.  Every "
             "device result equals the host's element for element.", "",
             "| k | front points | boxes | B | host ms | device ms (min-max) | host / device |", "|---|---|---|---|---|---|---|"]
    for row in info["decomposition"] + info["crossover"]:
        lines.append(f"| {row['k']} | {row['points']} | {row['boxes']} | {row['B']} | {row['host_ms']:.3f} | "
                     f"{row['device_ms']:.3f} ({row['device_ms_min']:.3f}-{row['device_ms_max']:.3f}) | "
                     f"{row['host_ms'] / row['device_ms']:.1f} |")
    b = info["batch"]
    lines += ["", f"One q = {b['q']} Kriging-believer batch (`propose_batch`, fast precision) with box EHVI at a 3-objective "
              f"front of {b['front']} points ({b['boxes']} boxes) over 2^22 candidates, every step's spec rebuilt "
              f"from scratch: host decomposition {b['host_ms']:.1f} ms, device decomposition {b['device_ms']:.1f} ms "
              f"(median of {b['reps']}); both pick the same rows.", ""]
    with open(os.path.join(args.out, "r07_ehvi_boxes_device.md"), "w") as f:
        f.write("\n".join(lines))
    print("\n".join(lines))


if __name__ == "__main__":
    main()

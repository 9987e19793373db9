"""Cost of the box HV-PoI (OMBO_ACQ_HV_POI_BOX, spec_hv_poi_box) against the box EHVI (OMBO_ACQ_EHVI_BOX) on one GPU:

  1. K4 alone, 2^22 candidates, the same boxes for both kinds (the HV-PoI table is the EHVI table clamped at the
     ideal point), FP32 and FP64: device time of the k_acquire_box kernels inside score() from torch.profiler, kind 8
     and kind 10 alternating in one session, on
     a. the C4 front (DTLZ2, n = 512, d = 12, k = 3) and the C4 models;
     b. a 4-objective front of 256 points on the unit sphere, with four models on the C4 inputs (the fourth
        objective a further DTLZ2 coordinate).
  2. The whole score() step at C4, CUDA events, kinds 8 and 10 alternating after a warm-up, a 256 MB L2 flush before
     each call, fast and FP64.

Prints markdown and writes JSON (--out) and markdown (--md), with the card's name and power limit read in the same
run.  Run from the repository root."""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import optimobo_b200 as ob  # noqa: E402
from optimobo_b200 import _cabi  # noqa: E402
from ehvi_box_bench import c4_problem, card  # noqa: E402
from ehvi_feas_bench import alternate, profiled_box_ms  # noqa: E402

DEV = torch.device("cuda:0")


def sphere4(P, seed):
    F = np.abs(np.random.default_rng(seed).normal(size=(P, 4)))
    return F / np.linalg.norm(F, axis=1, keepdims=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2m", type=int, default=22)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--md", default=None)
    args = ap.parse_args()
    m = 1 << args.log2m
    info = dict(card=card(), candidates=m, fast_path=_cabi.fast_path_available(), reps=args.reps, warmup=args.warmup)
    precisions = ("fp64", "fast") if info["fast_path"] else ("fp64",)
    lines = [f"card: {info['card']['name']}, power limit {info['card']['power_limit']}, "
             f"max SM clock {info['card']['max_sm_clock']}; 2^{args.log2m} candidates", ""]

    X, Y = c4_problem()
    d = X.shape[1]
    # a fourth DTLZ2-like objective on the same inputs for the 4-model case
    Y4 = np.column_stack([Y, (1 + ((X[:, 3:] - 0.5) ** 2).sum(1)) * np.sin(0.5 * np.pi * X[:, 2])])
    models = [ob.GPModel(X, Y4[:, i], np.ones(d), 1.0, device=DEV) for i in range(4)]
    pool = ob.CandidatePool.counter(m, np.zeros(d), np.ones(d), seed=1)
    PF3 = ob.host_prep.calc_pf(Y)
    PF4 = sphere4(256, 7)
    fronts = [("C4 front, k = 3", PF3, Y.min(0), Y.max(0), 3),
              ("4-objective sphere front, 256 points", PF4, PF4.min(0), PF4.max(0) + 0.1, 4)]

    # ---- 1. K4 alone ----
    k4 = []
    lines += ["## K4 alone (k_acquire_box inside score(), torch.profiler device time)", "",
              "| front | boxes | breakpoints | precision | EHVI_BOX ms | HV_POI_BOX ms | ratio |",
              "|---|---|---|---|---|---|---|"]
    for name, PF, ideal, maxp, k in fronts:
        hv = ob.spec_hv_poi_box(ideal, maxp, PF, device=DEV)
        eh = ob.spec_ehvi_box(np.asarray(hv.ref), PF, device=DEV)
        assert torch.equal(hv.cells, eh.cells)
        n_boxes, B = hv.cells.shape[0], hv.stripes.shape[1]
        for prec in precisions:
            t = profiled_box_ms({"8": lambda: ob.score(models[:k], eh, pool, precision=prec, sync=False),
                                 "10": lambda: ob.score(models[:k], hv, pool, precision=prec, sync=False)},
                                max(3, args.reps // 2))
            k4.append(dict(front=name, boxes=int(n_boxes), breakpoints=int(B), precision=prec, ehvi_box_ms=t["8"],
                           hv_poi_box_ms=t["10"], ratio=t["10"][0] / t["8"][0]))
            x = k4[-1]
            lines.append(f"| {name} | {n_boxes} | {B} | {prec} | {x['ehvi_box_ms'][0]:.3f} ± {x['ehvi_box_ms'][1]:.3f} "
                         f"| {x['hv_poi_box_ms'][0]:.3f} ± {x['hv_poi_box_ms'][1]:.3f} | {x['ratio']:.3f} |")

    # ---- 2. the whole step at C4 ----
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)
    hv = ob.spec_hv_poi_box(Y.min(0), Y.max(0), PF3)
    eh = ob.spec_ehvi_box(np.asarray(hv.ref), PF3)
    steps = []
    lines += ["", "## Whole score() step at C4 (n = 512, d = 12, k = 3; L2 flushed before each call)", "",
              "| precision | EHVI_BOX ms | HV_POI_BOX ms | difference ms |", "|---|---|---|---|"]
    for prec in precisions:
        t = alternate({"8": lambda: ob.score(models[:3], eh, pool, precision=prec, sync=False),
                       "10": lambda: ob.score(models[:3], hv, pool, precision=prec, sync=False)},
                      args.warmup, args.reps, flush)
        steps.append(dict(precision=prec, ehvi_box_ms=t["8"], hv_poi_box_ms=t["10"], difference_ms=t["10"][0] - t["8"][0]))
        x = steps[-1]
        lines.append(f"| {prec} | {x['ehvi_box_ms'][0]:.2f} ± {x['ehvi_box_ms'][1]:.2f} | "
                     f"{x['hv_poi_box_ms'][0]:.2f} ± {x['hv_poi_box_ms'][1]:.2f} | {x['difference_ms']:.2f} |")
    info.update(k4=k4, steps=steps)
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(info, f, indent=1)
    if args.md:
        os.makedirs(os.path.dirname(os.path.abspath(args.md)), exist_ok=True)
        with open(args.md, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()

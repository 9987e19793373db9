"""Cost of the constrained box EHVI (OMBO_ACQ_EHVI_BOX_FEAS, spec_ehvi_box_feasible) against the plain box EHVI
(OMBO_ACQ_EHVI_BOX) on one GPU:

  1. K4 alone at the box bench's C4 shape (k = 3, the C4 front, 2^22 candidates), c = 1 and 2 constraint models:
     a. FP64 through acquire_from_posterior's C entry on device-resident synthetic posteriors, CUDA events around
        each call, kind 8 and kind 9 alternating after a warm-up;
     b. FP32 and FP64 inside score() on the C4 models' posteriors: device time of the k_acquire_box kernels read from
        torch.profiler (the only way to isolate K4 inside score), kind 8 and kind 9 alternating in one session.
  2. The whole score() step, CUDA events, kind 8 and kind 9 alternating after a warm-up, a 256 MB L2 flush before each
     call:
     a. BNH shape: n = 100, d = 2, k = 2, c = 2, 2^22 candidates, precision "auto";
     b. C4 shape: n = 512, d = 12, k = 3, c = 2, 2^22 candidates, fast and FP64.
     Next to each, the posterior of the c constraint models alone (ACQ_NONE, mean and variance), the work kind 9 adds
     besides the c feasibility factors per candidate.

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
from ehvi_box_bench import acquire_direct, c4_problem, card  # noqa: E402

DEV = torch.device("cuda:0")


def bnh_problem(n=100):
    rng = np.random.default_rng(3)
    X = ob.host_prep.latin_hypercube(n, [(0.0, 5.0), (0.0, 3.0)], rng)
    Y = np.column_stack([4 * X[:, 0] ** 2 + 4 * X[:, 1] ** 2, (X[:, 0] - 5) ** 2 + (X[:, 1] - 5) ** 2])
    G = np.column_stack([((X[:, 0] - 5) ** 2 + X[:, 1] ** 2 - 25) / 25,
                         -((X[:, 0] - 8) ** 2 + (X[:, 1] + 3) ** 2 - 7.7) / 7.7])
    return X, Y, G


def c4_constraints(X):
    return np.column_stack([X[:, :3].sum(1) - 1.2, 0.4 - X[:, 3] - 0.5 * X[:, 4]]) * 4.0


def alternate(fns, warmup, reps, flush=None):
    """Mean / std ms per call of each fn, CUDA events, the fns interleaved call by call after `warmup` rounds."""
    for _ in range(warmup):
        for fn in fns.values():
            fn()
    ts = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            if flush is not None:
                flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts[k].append(e0.elapsed_time(e1))
    return {k: (float(np.mean(v)), float(np.std(v))) for k, v in ts.items()}


def profiled_box_ms(fns, reps):
    """Device ms per call of each fn's k_acquire_box launches: one profiler session per fn pair member, alternating."""
    from torch.profiler import ProfilerActivity, profile
    for fn in fns.values():
        fn()
    torch.cuda.synchronize()
    out = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                fn()
                torch.cuda.synchronize()
            tot = 0.0
            for e in prof.key_averages():
                if "k_acquire_box" in e.key:
                    tot += getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
            out[k].append(tot / 1e3)
    return {k: (float(np.mean(v)), float(np.std(v))) for k, v in out.items()}


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
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)
    lines = [f"card: {info['card']['name']}, power limit {info['card']['power_limit']}, "
             f"max SM clock {info['card']['max_sm_clock']}; 2^{args.log2m} candidates", ""]

    # ---- 1. K4 alone at the C4 shape ----
    X, Y = c4_problem()
    d = X.shape[1]
    G = c4_constraints(X)
    PF, r = ob.host_prep.calc_pf(Y), Y.max(0) + 0.1
    plain = ob.spec_ehvi_box(r, PF)
    n_boxes = plain.cells.shape[0]
    info["c4_boxes"], info["c4_breakpoints"] = n_boxes, plain.stripes.shape[1]
    rng = np.random.default_rng(0)
    mu = np.vstack([(PF[rng.integers(0, len(PF), m)] + rng.normal(0, 0.05, size=(m, 3))).T,
                    rng.normal(0.0, 1.0, size=(2, m))])
    mu_t = torch.as_tensor(np.ascontiguousarray(mu)).to(DEV)
    var_t = torch.full((5, m), 0.05 ** 2, dtype=torch.float64, device=DEV)
    k4 = []
    lines += [f"## K4 alone, C4 front ({n_boxes} boxes, k = 3)", "",
              "| source | precision | c | kind 8 ms | kind 9 ms | ratio |", "|---|---|---|---|---|---|"]
    for c in (1, 2):
        feas = ob.spec_ehvi_box_feasible(r, PF, c)
        t = alternate({"8": acquire_direct(plain, mu_t[:3], var_t[:3]),
                       "9": acquire_direct(feas, mu_t[:3 + c].contiguous(), var_t[:3 + c].contiguous())},
                      args.warmup, args.reps)
        k4.append(dict(source="acquire_from_posterior, CUDA events (incl. box packing + arg-max merge)",
                       precision="fp64", c=c, kind8_ms=t["8"], kind9_ms=t["9"], ratio=t["9"][0] / t["8"][0]))
    del mu_t, var_t
    models = [ob.GPModel(X, Y[:, i], np.ones(d), 1.0, device=DEV) for i in range(3)]
    cons = [ob.GPModel(X, G[:, j], np.ones(d), 1.0, device=DEV) for j in range(2)]
    pool = ob.CandidatePool.counter(m, np.zeros(d), np.ones(d), seed=1)
    for prec in precisions:
        for c in (1, 2):
            feas = ob.spec_ehvi_box_feasible(r, PF, c)
            t = profiled_box_ms({"8": lambda: ob.score(models, plain, pool, precision=prec, sync=False),
                                 "9": lambda: ob.score(models + cons[:c], feas, pool, precision=prec, sync=False)},
                                max(3, args.reps // 2))
            k4.append(dict(source="k_acquire_box inside score(), torch.profiler device time", precision=prec, c=c,
                           kind8_ms=t["8"], kind9_ms=t["9"], ratio=t["9"][0] / t["8"][0]))
    for x in k4:
        lines.append(f"| {x['source']} | {x['precision']} | {x['c']} | {x['kind8_ms'][0]:.3f} ± {x['kind8_ms'][1]:.3f} "
                     f"| {x['kind9_ms'][0]:.3f} ± {x['kind9_ms'][1]:.3f} | {x['ratio']:.4f} |")

    # ---- 2. whole steps ----
    steps = []
    Xb, Yb, Gb = bnh_problem()
    bm = [ob.GPModel(Xb, Yb[:, i], np.array([1.5, 1.0]), float(np.var(Yb[:, i])), device=DEV) for i in range(2)]
    bc = [ob.GPModel(Xb, Gb[:, j], np.array([1.5, 1.0]), float(np.var(Gb[:, j])), device=DEV) for j in range(2)]
    feasible = np.all(Gb <= 0, axis=1)
    bpf, br = ob.host_prep.calc_pf(Yb[feasible]), Yb.max(0)
    bpool = ob.CandidatePool.counter(m, [0.0, 0.0], [5.0, 3.0], seed=2)
    cases = [("BNH n=100 d=2 k=2 c=2", bm, bc, ob.spec_ehvi_box(br, bpf), ob.spec_ehvi_box_feasible(br, bpf, 2),
              bpool, "auto")]
    feas2 = ob.spec_ehvi_box_feasible(r, PF, 2)
    for prec in precisions:
        cases.append(("C4 n=512 d=12 k=3 c=2", models, cons, plain, feas2, pool, prec))
    lines += ["", "## Whole score() step (L2 flushed before each call)", "",
              "| shape | precision | kind 8 ms | kind 9 ms | difference ms | c constraint posteriors alone ms |",
              "|---|---|---|---|---|---|"]
    for name, mo, co, s8, s9, pl, prec in cases:
        resolved = ob.resolve_precision(mo + co, prec)
        post = {}

        def cons_post():
            post["r"] = ob.score(co, None, pl, precision=resolved, want_posterior=True, sync=False)

        t = alternate({"8": lambda: ob.score(mo, s8, pl, precision=resolved, sync=False),
                       "9": lambda: ob.score(mo + co, s9, pl, precision=resolved, sync=False),
                       "post": cons_post}, args.warmup, args.reps, flush)
        post.clear()
        steps.append(dict(shape=name, precision=prec, resolved=resolved, kind8_ms=t["8"], kind9_ms=t["9"],
                          constraint_posteriors_ms=t["post"], difference_ms=t["9"][0] - t["8"][0]))
        x = steps[-1]
        lines.append(f"| {name} | {prec} ({resolved}) | {x['kind8_ms'][0]:.2f} ± {x['kind8_ms'][1]:.2f} | "
                     f"{x['kind9_ms'][0]:.2f} ± {x['kind9_ms'][1]:.2f} | {x['difference_ms']:.2f} | "
                     f"{x['constraint_posteriors_ms'][0]:.2f} ± {x['constraint_posteriors_ms'][1]:.2f} |")
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

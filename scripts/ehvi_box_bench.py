"""Cost of the exact box EHVI (spec_ehvi_box, k_acquire_box) against the crude 3-D EHVI (spec_ehvi3d, k_acquire) on
one GPU:

  1. K4 alone: kernel time of the acquisition (+ the box packing) read from torch.profiler inside score() over 2^22
     candidates of the C4 models, in FP64 and in the fast mode (FP32 K4), for the C4 front and sphere fronts of
     P = 100 / 200 points; plus the FP64 K4 through acquire_from_posterior's C entry on 2^22 synthetic posteriors
     (CUDA events, device-resident inputs).  Reports ms and boxes per candidate-second.
  2. The whole score() step at the C4 shape (n = 512, d = 12, k = 3, 2^22 candidates, fast and FP64): CUDA events,
     3 warm-up + 5 timed passes, a 256 MB L2 flush before each.

Prints a markdown table and writes everything, with the card's name and power limit read in the same run, as JSON
to --out (default: stdout only).  Run from the repository root."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import optimobo_b200 as ob  # noqa: E402
from optimobo_b200 import _cabi  # noqa: E402
from optimobo_b200.gp import current_stream_ptr  # noqa: E402

DEV = torch.device("cuda:0")


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")] if q.returncode == 0 else ("?", "?", "?")
    return dict(name=name or torch.cuda.get_device_name(0), power_limit=power, max_sm_clock=clock,
                torch_name=torch.cuda.get_device_name(0))


def c4_problem(n=512, d=12):
    X = np.random.default_rng(4).random((n, d))
    g = ((X[:, 2:] - 0.5) ** 2).sum(1)
    a, b = 0.5 * np.pi * X[:, 0], 0.5 * np.pi * X[:, 1]
    Y = np.column_stack([(1 + g) * np.cos(a) * np.cos(b), (1 + g) * np.cos(a) * np.sin(b), (1 + g) * np.sin(a)])
    return X, Y


def sphere_front(P, seed):
    F = np.abs(np.random.default_rng(seed).normal(size=(P, 3)))
    return F / np.linalg.norm(F, axis=1, keepdims=True)


def kernel_ms(fn, names, reps):
    """Device time per call of the kernels whose name contains one of `names` (torch.profiler, its own run)."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    total = 0.0
    for e in prof.key_averages():
        if any(n in e.key for n in names):
            total += getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
    return total / 1e3 / reps


def step_ms(fn, flush, warmup=3, reps=5):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.mean(ts)), float(np.std(ts))


def acquire_direct(spec, mu_t, var_t):
    """acquire_from_posterior's C entry on device-resident posteriors (no host copies in the timed region)."""
    a = spec.c_struct(DEV)
    G, m = mu_t.shape
    acq = torch.empty((m,), dtype=torch.float64, device=DEV)
    best = torch.empty((2,), dtype=torch.int64, device=DEV)
    ctx = _cabi.Context.get(0)

    def run():
        _cabi.check(_cabi.lib().ombo_acquire_posterior(
            ctx.handle, C.byref(a), G, C.c_void_p(mu_t.data_ptr()), C.c_void_p(var_t.data_ptr()), m, m, 0,
            C.c_void_p(acq.data_ptr()), C.c_void_p(best.data_ptr()), current_stream_ptr(DEV)))
    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2m", type=int, default=22)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    m = 1 << args.log2m
    info = dict(card=card(), candidates=m, fast_path=_cabi.fast_path_available())
    X, Y = c4_problem()
    d = X.shape[1]
    models = [ob.GPModel(X, Y[:, i], np.ones(d), 1.0, device=DEV) for i in range(3)]
    cache = ob.host_prep.cached_samples(3, 5, seed=4)
    pool = ob.CandidatePool.counter(m, np.zeros(d), np.ones(d), seed=1)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)
    c4_pf, c4_r = ob.host_prep.calc_pf(Y), Y.max(0) + 0.1
    fronts = {"C4": (c4_pf, c4_r)}
    for P in (100, 200):
        F = sphere_front(P, P)
        fronts[f"sphere P={P}"] = (F, np.full(3, 1.1))
    precisions = ("fp64", "fast") if info["fast_path"] else ("fp64",)
    rows = []
    # 1. K4 alone
    rng = np.random.default_rng(0)
    for fname, (PF, r) in fronts.items():
        box = ob.spec_ehvi_box(r, PF)
        crude = ob.spec_ehvi3d(r, PF, cache)
        n_boxes, B = box.cells.shape[0], box.stripes.shape[1]
        mu = PF[rng.integers(0, len(PF), m)] + rng.normal(0, 0.05, size=(m, 3))
        mu_t = torch.as_tensor(np.ascontiguousarray(mu.T)).to(DEV)
        var_t = torch.full((3, m), 0.05 ** 2, dtype=torch.float64, device=DEV)
        for kind, spec in (("EHVI_3D", crude), ("EHVI_BOX", box)):
            run = acquire_direct(spec, mu_t, var_t)
            ms = kernel_ms(run, ("k_acquire", "k_pack_boxes"), args.reps)
            rows.append(dict(part="K4 alone, acquire_from_posterior (synthetic posteriors)", front=fname, P=len(PF),
                             B=B, n_boxes=n_boxes, kind=kind, precision="fp64", k4_ms=ms,
                             boxes_per_cand_s=(n_boxes * m / (ms * 1e-3)) if kind == "EHVI_BOX" else None))
            for prec in precisions:
                ms = kernel_ms(lambda: ob.score(models, spec, pool, precision=prec, sync=False),
                               ("k_acquire", "k_pack_boxes"), args.reps)
                rows.append(dict(part="K4 inside score() (C4 models' posteriors)", front=fname, P=len(PF), B=B,
                                 n_boxes=n_boxes, kind=kind, precision=prec, k4_ms=ms,
                                 boxes_per_cand_s=(n_boxes * m / (ms * 1e-3)) if kind == "EHVI_BOX" else None))
        del mu_t, var_t
    # 2. the whole score() step at the C4 shape
    box = ob.spec_ehvi_box(c4_r, c4_pf)
    crude = ob.spec_ehvi3d(c4_r, c4_pf, cache)
    crude_x = ob.spec_ehvi3d(c4_r, c4_pf, cache, semantics="exact")     # reads all three variances, as the box kind
    steps = []
    for prec in precisions:
        for kind, spec in (("EHVI_3D", crude), ("EHVI_3D exact semantics", crude_x), ("EHVI_BOX", box)):
            mean, sd = step_ms(lambda: ob.score(models, spec, pool, precision=prec, sync=False), flush)
            steps.append(dict(kind=kind, precision=prec, step_ms=mean, step_ms_std=sd))
    for prec in precisions:
        s = {x["kind"]: x["step_ms"] for x in steps if x["precision"] == prec}
        steps.append(dict(kind="ratio EHVI_BOX / EHVI_3D", precision=prec, step_ms=s["EHVI_BOX"] / s["EHVI_3D"]))
    info.update(k4=rows, c4_step=steps)
    print(f"card: {info['card']}")
    print("| part | front | B | boxes | kind | precision | K4 ms | boxes per candidate-s |\n|---|---|---|---|---|---|---|---|")
    for x in rows:
        bps = f"{x['boxes_per_cand_s']:.3e}" if x["boxes_per_cand_s"] else "-"
        print(f"| {x['part']} | {x['front']} | {x['B']} | {x['n_boxes']} | {x['kind']} | {x['precision']} | "
              f"{x['k4_ms']:.3f} | {bps} |")
    print("| C4 step, 2^%d candidates | kind | precision | ms |\n|---|---|---|---|" % args.log2m)
    for x in steps:
        print(f"| | {x['kind']} | {x['precision']} | {x['step_ms']:.3f} |")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(info, f, indent=1)


if __name__ == "__main__":
    main()

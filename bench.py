#!/usr/bin/env python
"""bench.py -- candidates scored per second on the acquisition hot path.

Workload (BASELINE.json configs[4], SURVEY.md section 8d "C5"): n_train = 1024, d = 10,
2 objectives (ZDT1 values), injected hyper-parameters (sigma_f2 = (1, 2), ell = 0.7 / 0.8),
full GP posterior (mean + std for BOTH objectives) + 2-objective EHVI + arg-max, over a
counter-generated uniform candidate pool of m candidates per GPU per step (weak scaling).

  value  : candidates/s, whole job, inputs resident on the device (the pool is generated
           on-chip from a counter RNG: 0 input bytes), CUDA-event time per step, max over ranks.
  e2e    : same metric through the host entry of the C ABI (ombo_score_host): the candidate
           pool lives in PINNED HOST memory, is copied host->device inside the timed region
           (chunked, overlapped with scoring) and the 16-byte result is read back.
  roofline: the dominant kernel (posterior: K1+K2) timed with CUDA events on its stream
           inside the timed region (C-ABI profile hooks), algorithmic FLOPs/candidate from
           SURVEY section 8d (G_var follows --semantics).
  cpu_baseline: the numpy/LAPACK oracle port (oracle/oracle.py) on the host cores on a
           bounded sample of the same workload, plus `reference_call_pattern`: the REFERENCE'S OWN
           util_functions.EHVI, one candidate per call (the pattern differential_evolution drives),
           timed on 256 candidates when the reference package is present (baseline/_ref).
  sweep / strong / fp64 / reference_semantics / accuracy / parity_nranks: sub-records that tell the
           rest of the C5 story in the same line (pool sizes 2^20..2^26 per GPU, fixed-pool strong
           scaling at this N, the FP64 tolerance mode with its own DGEMM roofline, the reference's
           model-0-variance semantics, the measured fast-mode error, and the N-rank result parity).
  --impl reference : the same oracle port as the measured arm (the reference is pure Python and
           scores one candidate per call; the batched port is its best case).  Rank 0 only.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_TRAIN, DIM, N_OBJ = 1024, 10, 2


def zdt1(X):
    f1 = X[:, 0]
    g = 1 + 9.0 / (X.shape[1] - 1) * X[:, 1:].sum(1)
    return np.column_stack([f1, g * (1 - np.sqrt(f1 / g))])


def workload(n=N_TRAIN, d=DIM):
    rng = np.random.default_rng(0)
    X = rng.random((n, d))
    Y = zdt1(X)
    ells = [0.7 * np.ones(d), 0.8 * np.ones(d)]
    sf2 = [1.0, 2.0]
    return X, Y, ells, sf2


def algorithmic_flops_per_candidate(n, d, G, G_var, P):
    """SURVEY.md section 8d: F = G_var n^2 + G (2n + n(3d+10)) + A, A(EHVI-2D) ~ 30 P."""
    return G_var * n * n + G * (2 * n + n * (3 * d + 10)) + 30 * P


def issued_units_per_mac(fmt):
    """Tensor-core products per algorithmic MAC, in units of one 16-bit product: the 16-bit x3 split issues 3, the
    f8c format 1 (fp16) + 2 x 1/2 (e4m3 at twice the rate)."""
    return 2.0 if fmt == "f8c" else 3.0


class ClockSampler(threading.Thread):
    """Samples SM clock, power and clock-event (throttle) reasons during the timed region: NVML every 20 ms when
    pynvml is importable (the same counters nvidia-smi prints), else the nvidia-smi query of the profiling recipe
    (one subprocess per sample, ~5 per second).  Also reads NVML's total-energy counter at both ends."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.rows, self._stop_ev = gpu_index, [], threading.Event()
        self.nv, self.h, self.e0, self.energy_j = None, None, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices: honour CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = int(vis.split(",")[gpu_index]) if vis and all(t.strip().isdigit() for t in vis.split(",")) else gpu_index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nv = pynvml
            self.e0 = pynvml.nvmlDeviceGetTotalEnergyConsumption(self.h)
        except Exception:
            self.nv = None

    def _nvml_row(self):
        nv, h = self.nv, self.h
        try:
            reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        flag = lambda bit: "Active" if reasons & bit else "Not Active"
        return [str(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), str(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)),
                str(nv.nvmlDeviceGetPowerUsage(h) / 1e3), hex(reasons),
                flag(0x8), flag(0x40), flag(0x20), flag(0x4)]      # hw_slowdown, hw_thermal, sw_thermal, sw_power_cap

    def run(self):
        while not self._stop_ev.is_set():
            try:
                if self.nv is not None:
                    self.rows.append(self._nvml_row())
                else:
                    out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits"], capture_output=True, text=True,
                                         timeout=5).stdout.strip()
                    if out:
                        self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop_ev.wait(0.02 if self.nv is not None else 0.2)
        if self.nv is not None and self.e0 is not None:
            try:
                self.energy_j = (self.nv.nvmlDeviceGetTotalEnergyConsumption(self.h) - self.e0) / 1e3
            except Exception:
                pass

    def summary(self):
        self._stop_ev.set()
        self.join(timeout=6)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            for name, col in (("hw_slowdown", 4), ("hw_thermal_slowdown", 5), ("sw_thermal_slowdown", 6),
                              ("sw_power_cap", 7)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]),
                "power_w_max": max(float(r[2]) for r in self.rows), "samples": len(self.rows),
                "reasons": sorted(reasons), "source": "nvml" if self.nv is not None else "nvidia-smi",
                "energy_j": self.energy_j}


def cpu_oracle_rate(budget_s, chunk=4096, semantics="exact"):
    """Batched FP64 posterior + vectorised EHVI of the oracle port on the host cores."""
    from oracle import oracle as O
    X, Y, ells, sf2 = workload()
    st = [O.gp_fit_state(X, Y[:, i], ells[i], sf2[i]) for i in range(N_OBJ)]
    PF, r = O.calc_pf(Y), Y.max(0)
    from scipy.stats import norm, qmc
    cache = norm.ppf(qmc.Sobol(d=2, scramble=True, seed=0).random_base2(m=5))
    lo, hi = np.zeros(DIM), np.ones(DIM)
    done, t0 = 0, time.perf_counter()
    best = (-np.inf, -1)
    while True:
        Xc = O.candidates_from_counter(1, done, chunk, lo, hi)
        post = [O.gp_posterior(s, Xc) for s in st]
        a = O.ehvi_batched(post[0][0], post[1][0], post[0][1], post[1][1], PF, r, cache, semantics)
        i = O.argmax_lowest_index(a)
        if a[i] > best[0]:
            best = (float(a[i]), done + i)
        done += chunk
        el = time.perf_counter() - t0
        if el >= budget_s and done >= 2 * chunk:
            break
    return done / el, done, el


def reference_call_pattern(n_cand=256):
    """SURVEY section 8d (i): the reference's own `util_functions.EHVI` (util_functions.py:136-167, EHVI_2D_aux
    :81-133) called with ONE x per call -- what scipy's differential_evolution does at optimisers.py:118 -- on the
    C5 workload, with sklearn's GaussianProcessRegressor behind a GPy-shaped predict (GPy is not installable).
    Needs the reference package (baseline/_ref, /root/reference or $OPTIMOBO_REF); otherwise the figure measured in
    the build container is reported as such."""
    from oracle import ref_loader as R
    from oracle import oracle as O
    if not R.reference_available():
        return {"value": 97.8, "unit": "candidates/s", "cores": 8, "measured": "build container (SURVEY probe), "
                "reference package not present on this box", "candidates": 256}
    uf = R.load_reference().util_functions
    from sklearn.gaussian_process import GaussianProcessRegressor
    from sklearn.gaussian_process.kernels import ConstantKernel, Matern
    from scipy.stats import norm, qmc
    X, Y, ells, sf2 = workload()
    models = []
    for i in range(N_OBJ):
        g = GaussianProcessRegressor(kernel=ConstantKernel(sf2[i]) * Matern(length_scale=ells[i], nu=2.5), alpha=1e-8,
                                     optimizer=None, normalize_y=False).fit(X, Y[:, i])

        def post(Xq, g=g):
            mu, sd = g.predict(Xq, return_std=True)
            return mu, sd * sd
        models.append(R.ShimGP(post))
    PF, r = uf.calc_pf(Y), Y.max(0)
    cache = norm.ppf(qmc.Sobol(d=2, scramble=True, seed=0).random_base2(m=5))
    Xc = O.candidates_from_counter(1, 0, n_cand, np.zeros(DIM), np.ones(DIM))
    uf.EHVI(Xc[0], models, r, PF, cache)
    t0 = time.perf_counter()
    vals = [float(np.asarray(uf.EHVI(x, models, r, PF, cache)).reshape(-1)[0]) for x in Xc]
    el = time.perf_counter() - t0
    return {"value": n_cand / el, "unit": "candidates/s", "cores": os.cpu_count(), "candidates": n_cand,
            "seconds": el, "measured": "this box: unmodified optimobo.util_functions.EHVI from " + R.reference_root() +
            ", one x per call, sklearn GPR behind a GPy-shaped predict", "best_value": max(vals)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count()
    t_budget = 6.0
    times, total = [], 0
    for it in range(args.warmup + args.steps):
        rate, done, el = cpu_oracle_rate(t_budget if it >= args.warmup else 2.0)
        if it >= args.warmup:
            times.append(el)
            total += done
    value = total / sum(times)
    line = {
        "impl": "reference", "metric": "candidates scored/sec (GP mean+std+EHVI)", "value": value,
        "unit": "candidates/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "C5: n_train=1024 d=10 k=2 EHVI-2D (exact semantics), counter-generated pool",
                   "sample_per_step": total // max(1, len(times))},
        "cpu_baseline": {"value": value, "unit": "candidates/s", "cores": cores, "kind": "port",
                         "sample": f"{total} candidates in {len(times)} steps, batched numpy/LAPACK oracle "
                                   "(4096-row chunks), all BLAS threads"},
        "e2e": {"value": value, "unit": "candidates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    try:
        line["cpu_baseline"]["reference_call_pattern"] = reference_call_pattern()
    except Exception as e:          # the batched port above is the measured arm; this is the extra baseline
        line["cpu_baseline"]["reference_call_pattern"] = {"error": repr(e)}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--precision", default=os.environ.get("OMBO_BENCH_PRECISION", "auto"))
    ap.add_argument("--log2m", type=int, default=0, help="candidates per GPU per step = 2**log2m")
    ap.add_argument("--semantics", default="exact")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-fit", action="store_true", help="skip the (untimed, separately reported) device hyper-parameter fit")
    ap.add_argument("--no-refresh-timing", action="store_true", help="skip the GP refresh timing loops (short profiler runs)")
    ap.add_argument("--no-extras", action="store_true", help="skip the sweep / strong / fp64 / reference-semantics / accuracy sub-records")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's result (best_value.npy, best_index.npy, float64) to DIR")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference" and args.dump_outputs:
        # the CPU arm scores as many candidates as fit its time budget, so its result is not reproducible
        ap.error("--dump-outputs applies to the GPU path only, not to --impl reference")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import optimobo_b200 as ob
    from optimobo_b200 import _cabi
    from optimobo_b200.distributed import score_sharded

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    precision = args.precision
    if precision == "auto":
        precision = "fast" if _cabi.fast_path_available() else "fp64"
    log2m = args.log2m or (24 if precision == "fast" else 20)
    m_per_gpu = 1 << log2m
    m_total = m_per_gpu * world

    X, Y, ells, sf2 = workload()
    t0 = time.perf_counter()
    models = [ob.GPModel(X, Y[:, i], ells[i], sf2[i], device=dev) for i in range(N_OBJ)]
    torch.cuda.synchronize()
    refresh_first_ms = 1e3 * (time.perf_counter() - t0)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ob.refresh_models(models)                  # warm-up of the side streams and host threads
    torch.cuda.synchronize()

    def median_ms(fn, reps=7):
        ts = []
        for _ in range(reps):
            ev0.record(); fn(); ev1.record(); torch.cuda.synchronize()
            ts.append(ev0.elapsed_time(ev1))
        return sorted(ts)[len(ts) // 2]

    refresh_ms = refresh_serial_ms = None
    if not args.no_refresh_timing:
        refresh_ms = median_ms(lambda: ob.refresh_models(models))          # both GPs' K3 chains overlapped on two streams
        refresh_serial_ms = median_ms(lambda: [mdl.refresh() for mdl in models])

    # hyper-parameter fit on the device (section 8f-1): reported separately, not part of the metric
    fit_ms, fit_info = None, {}
    if rank == 0 and not args.no_fit:
        from optimobo_b200.fit import fit_hyperparameters_device
        fit_hyperparameters_device(X, Y[:, 0], max_f_eval=3, device=dev)      # warm-up: lazy module load, pool growth
        torch.cuda.synchronize()
        fit_info = {}
        t0 = time.perf_counter()
        fit_hyperparameters_device(X, Y[:, 0], max_f_eval=40, device=dev, info=fit_info)
        fit_ms = 1e3 * (time.perf_counter() - t0)

    # first front + hypervolume of the evaluated sample (section 8f-2), device vs host; reported, not in the metric
    prep_ms = None
    if rank == 0:
        ob.device_prep.calc_pf(Y, dev)                                   # warm-up
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(10):
            pf_d = ob.device_prep.calc_pf(Y, dev)
            hv_d = ob.device_prep.hypervolume(Y, Y.max(0), dev)
        t1 = time.perf_counter()
        pf_h, hv_h = ob.host_prep.calc_pf(Y), ob.host_prep.hypervolume(Y, Y.max(0))
        t2 = time.perf_counter()
        assert np.array_equal(pf_d, pf_h) and hv_d == hv_h
        prep_ms = {"device": 1e2 * (t1 - t0), "host": 1e3 * (t2 - t1)}

    cache = ob.host_prep.cached_samples(2, 5, seed=0)
    PF, r = ob.host_prep.calc_pf(Y), Y.max(0)
    spec = ob.spec_ehvi(r, PF, cache, args.semantics)
    ctx = _cabi.Context.get(local)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step, steps, warmup, profile=False):
        """W untimed + K timed steps of `step` (L2 flushed between steps, outside the events), barrier +
        synchronize on both sides, CUDA events per step, MAX over ranks.  -> (total ms, last result, n_prof, prof_ms)"""
        for _ in range(warmup):
            flush.zero_()
            step()
        barrier()
        if profile:
            ctx.profile(True)
        starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        result = None
        for i in range(steps):
            flush.zero_()
            starts[i].record()
            result = step()
            ends[i].record()
        barrier()
        n_prof, prof_ms = ctx.profile_read() if profile else (0, 0.0)
        if profile:
            ctx.profile(False)
        t = torch.tensor([sum(s.elapsed_time(e) for s, e in zip(starts, ends))], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), result, n_prof, prof_ms

    # ---- headline: C5, 2^log2m candidates per GPU per step --------------------------------------
    pool = ob.CandidatePool.counter(m_total, np.zeros(DIM), np.ones(DIM), seed=1)

    def step():
        return score_sharded(models, spec, pool, precision=precision)

    for _ in range(args.warmup):
        flush.zero_()
        step()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ctx.launch_count(reset=True)
    wall0 = time.perf_counter()
    total_ms, result, n_prof, prof_ms = timed(step, args.steps, 0, profile=True)
    wall = time.perf_counter() - wall0
    launches = ctx.launch_count(reset=True)
    clocks = sampler.summary() if sampler else None
    if clocks and clocks.get("energy_j") is not None:
        # NVML total-energy counter over the timed region (the kernel runs at the power cap: time follows energy);
        # includes the 256 MB L2 flush between steps
        # (the counter advances in coarse ticks: below about a second of timed region the figure is noise)
        e_j = clocks.pop("energy_j")
        clocks["energy_j_per_step"] = e_j / args.steps if wall >= 1.0 else None
    value = m_total * args.steps / (total_ms / 1e3)
    if args.dump_outputs and rank == 0:
        # what score_sharded returns, identical on every rank; the index is exact in float64 (m_total < 2^53)
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "best_value.npy"), np.array([result[0]], dtype=np.float64))
        np.save(os.path.join(args.dump_outputs, "best_index.npy"), np.array([result[1]], dtype=np.float64))

    # ---- end-to-end: host candidates through the C-ABI host entry ------------------------------
    e2e = None
    if not args.no_e2e:
        host_dtype = torch.float32 if precision == "fast" else torch.float64
        gen = torch.Generator().manual_seed(1234 + rank)
        Xh = torch.rand((m_per_gpu, DIM), dtype=host_dtype, generator=gen).pin_memory()
        for _ in range(2):
            ob.propose_host(models, spec, Xh, precision=precision, index_base=rank * m_per_gpu)
        barrier()
        k_e2e = max(2, min(args.steps, 5))
        w0 = time.perf_counter()
        es = torch.cuda.Event(enable_timing=True); ee = torch.cuda.Event(enable_timing=True)
        es.record()
        for _ in range(k_e2e):
            bv, bi = ob.propose_host(models, spec, Xh, precision=precision, index_base=rank * m_per_gpu)
        ee.record()
        barrier()
        te = torch.tensor([es.elapsed_time(ee)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e = {"value": m_total * k_e2e / (float(te.item()) / 1e3), "unit": "candidates/s",
               "h2d_bytes_per_step": int(Xh.numel() * Xh.element_size()), "d2h_bytes_per_step": 16,
               "steps": k_e2e, "host_dtype": str(host_dtype).replace("torch.", ""),
               "wall_s": time.perf_counter() - w0}
        del Xh

    # ---- N-rank result parity (outside the timed region): the sharded winner == the single-GPU winner ----------
    parity_nranks = None
    if world > 1:
        ppool = ob.CandidatePool.counter(1 << 22, np.zeros(DIM), np.ones(DIM), seed=7)
        v_sh, i_sh = score_sharded(models, spec, ppool, precision=precision)
        whole = ob.score(models, spec, ppool, precision=precision)           # every rank: the whole pool on one GPU
        ok = (i_sh == whole.best_index) and (v_sh == whole.best_value)
        flag = torch.tensor([1 if ok else 0], dtype=torch.int64, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        parity_nranks = "ok" if int(flag.item()) == 1 else f"MISMATCH sharded=({v_sh}, {i_sh}) single=({whole.best_value}, {whole.best_index})"
        if parity_nranks != "ok":
            raise SystemExit("N-rank parity failed: " + parity_nranks)

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    n, d, P = N_TRAIN, DIM, len(PF)
    bf16_peak = peaks.get("bf16_tflops_sustained", 1400.0)
    bf16_src = ("MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)"
                if peaks else "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)")
    dgemm = {}

    def dgemm_peak():
        """no FP64 peak in MEASURED_PEAKS.json: cuBLAS DGEMM measured in this run (SURVEY section 5)"""
        if "v" not in dgemm:
            a = torch.randn(4096, 4096, dtype=torch.float64, device=dev)
            b = torch.randn(4096, 4096, dtype=torch.float64, device=dev)
            best = 1e9
            for _ in range(6):
                s_, e_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s_.record(); torch.matmul(a, b); e_.record(); torch.cuda.synchronize()
                best = min(best, s_.elapsed_time(e_))
            dgemm["v"] = 2 * 4096 ** 3 / (best / 1e3) / 1e12
        return dgemm["v"]

    def roofline_of(prec, semantics, m_gpu, steps, n_prof_, prof_ms_, tot_ms):
        """Roofline of the posterior kernel (K1 + K2): algorithmic FLOPs from SURVEY section 8d with G_var taken from
        the semantics (reference semantics reads only model 0's variance), over the CUDA-event time of its launches."""
        G_var = N_OBJ if semantics == "exact" else 1
        fl_cand = algorithmic_flops_per_candidate(n, d, N_OBJ, G_var, P)
        if prec == "fast":
            peak, src = bf16_peak, bf16_src
        else:
            peak, src = dgemm_peak(), "cuBLAS DGEMM 4096^3 measured in this run (best of 6)"
        launch_ms = prof_ms_ / max(1, n_prof_)
        # the profiled launches are the posterior kernels of all GPs; their algorithmic work per candidate is F - A
        fl_total = (fl_cand - 30 * P) * m_gpu * steps
        achieved = fl_total / (prof_ms_ / 1e3) / 1e12 if n_prof_ else None
        return {"bound": "tensor", "kernel": "k_posterior_" + ("fast" if prec == "fast" else "fp64"),
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": (achieved / peak) if achieved else None,
                "peak_source": src, "launches": n_prof_, "avg_launch_ms": launch_ms,
                "candidates_per_launch": m_gpu * steps * N_OBJ / max(1, n_prof_),
                "kernel_share_of_step": prof_ms_ / tot_ms if tot_ms else None, "flops_per_candidate": fl_cand,
                "g_var": G_var}

    # ---- sub-records: pool-size sweep, strong scaling, FP64 mode, reference semantics, accuracy ---------------
    extras = {}
    if not args.no_extras:
        def run_pool(m_tot, prec, sem, steps, warmup, profile=False):
            p_ = ob.CandidatePool.counter(m_tot, np.zeros(DIM), np.ones(DIM), seed=1)
            sp_ = spec if sem == args.semantics else ob.spec_ehvi(r, PF, cache, sem)
            tot, res, npf, pms = timed(lambda: score_sharded(models, sp_, p_, precision=prec), steps, warmup, profile)
            return {"candidates_total": m_tot, "candidates_per_gpu": m_tot // world, "steps": steps,
                    "ms_per_step": tot / steps, "value": m_tot * steps / (tot / 1e3), "best": list(res)}, npf, pms, tot

        if precision == "fast":
            sweep = []
            for lg in (20, 22, 24, 26):
                st_ = 2 if lg == 26 else 3
                rec, _, _, _ = run_pool((1 << lg) * world, "fast", args.semantics, st_, 1)
                rec["log2m_per_gpu"] = lg
                sweep.append(rec)
            extras["sweep"] = {"scaling": "weak", "unit": "candidates/s", "precision": "fast", "semantics": args.semantics,
                               "points": sweep}
            strong = []
            for lg in (24, 26):
                st_ = 2 if lg == 26 else 3
                rec, _, _, _ = run_pool(1 << lg, "fast", args.semantics, st_, 1)
                rec["log2m_total"] = lg
                strong.append(rec)
            extras["strong"] = {"scaling": "strong", "unit": "candidates/s", "n_gpus": world, "precision": "fast",
                                "note": "fixed total pool sharded over the run's N GPUs (includes refresh-free scoring, the "
                                        "16-byte all-gather and the readback)", "points": strong}
            rec, npf, pms, tot = run_pool((1 << 24) * world, "fast", "reference" if args.semantics == "exact" else "exact", 3, 1, True)
            other = "reference" if args.semantics == "exact" else "exact"
            rec["roofline"] = roofline_of("fast", other, 1 << 24, 3, npf, pms, tot)
            rec["note"] = ("reference semantics: EHVI scales both objectives by MODEL 0's variance (util_functions.py:233), so only "
                           "model 0 runs K2; model 1 runs the mean-only kernel" if other == "reference" else "exact semantics")
            extras[other + "_semantics"] = rec
        if precision == "fast":
            rec, npf, pms, tot = run_pool((1 << 20) * world, "fp64", args.semantics, 3, 1, True)
            rec["roofline"] = roofline_of("fp64", args.semantics, 1 << 20, 3, npf, pms, tot)
            extras["fp64"] = rec
        if precision == "fast" and rank == 0:
            # measured error of the fast mode against the FP64 CUDA path on the head of the same pool (2^16 candidates)
            hp = ob.CandidatePool.counter(1 << 16, np.zeros(DIM), np.ones(DIM), seed=1)
            f_ = ob.score(models, spec, hp, precision="fast", want_posterior=True, want_acq=True)
            q_ = ob.score(models, spec, hp, precision="fp64", want_posterior=True, want_acq=True)
            sf, sq = f_.var.sqrt(), q_.var.sqrt()
            af, aq = f_.acq, q_.acq
            amax = float(aq.abs().max())
            sel = aq.abs() > 1e-3 * amax
            extras["accuracy"] = {
                "sample": "first 2^16 candidates of the pool, fast vs FP64 CUDA path (FP64 path vs sklearn / oracle: tests)",
                "sigma_max_rel_err": float(((sf - sq).abs() / sq).max()),
                "sigma_max_abs_err_over_sigma_f": float(((sf - sq).abs() / torch.tensor(sf2, device=dev).sqrt()[:, None]).max()),
                "mu_max_abs_err_over_sigma": float(((f_.mu - q_.mu).abs() / sq).max()),
                "ehvi_max_rel_err_where_above_1e-3_of_max": float(((af - aq).abs()[sel] / aq.abs()[sel]).max()),
                "ehvi_max_abs_err_over_max": float((af - aq).abs().max() / amax),
                "same_argmax": bool(f_.best_index == q_.best_index),
                "plane_format": [g.plane_format for g in models], "conditioning": [g.conditioning for g in models]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel ---------------------------------------------------
    roofline = roofline_of(precision, args.semantics, m_per_gpu, args.steps, n_prof, prof_ms, total_ms)
    traffic = None
    try:   # dram__bytes_read.sum + dram__bytes_write.sum of one launch of the same size (ncu --set full capture)
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[precision]
    except Exception:
        pass
    roofline["traffic"] = traffic
    if precision == "fast" and roofline["achieved"]:
        # what the tensor cores actually execute: products per algorithmic MAC of the operand format in use, and the
        # diagonal blocks of the triangular factor rounded up to 64 columns (68 of 64 ideal units at n = 1024)
        fmt = models[0].plane_format
        nch = N_TRAIN // 128
        units = sum(2 * c + 2 for c in range(nch)) - 0.5 * nch
        issued = issued_units_per_mac(fmt) * units * (128 * 64) * 2      # FLOP-equivalents per candidate per GP
        G_var = roofline["g_var"]
        issued_tflops = issued * G_var * m_per_gpu * args.steps / (prof_ms / 1e3) / 1e12
        roofline["issued"] = {"tflops_bf16_equivalent": issued_tflops, "frac": issued_tflops / roofline["peak"],
                              "units_per_mac": issued_units_per_mac(fmt), "plane_format": fmt,
                              "note": "tensor-pipe work the kernel sustains, in units of one 16-bit product per MAC (an e4m3 "
                                      "product counts 1/2: twice the rate); includes the mean-only launches' time when G_var < G"}

    cpu = None
    if not args.no_cpu_baseline:
        rate, done, el = cpu_oracle_rate(args.cpu_seconds, semantics=args.semantics)
        cpu = {"value": rate, "unit": "candidates/s", "cores": os.cpu_count(), "kind": "port",
               "sample": f"{done} candidates of the same pool in {el:.1f} s: batched numpy/LAPACK oracle "
                         "(FP64 posterior x2 + vectorised EHVI, 4096-row chunks), all BLAS threads"}
        try:
            cpu["reference_call_pattern"] = reference_call_pattern()
        except Exception as e:
            cpu["reference_call_pattern"] = {"error": repr(e)}

    fmt0 = models[0].plane_format
    line = {
        "metric": "candidates scored/sec (GP mean+std+EHVI)", "value": value, "unit": "candidates/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": ("fp16+2xe4m3" if fmt0 == "f8c" else fmt0) if precision == "fast" else "f64", "data": "synthetic",
        "config": {"workload": f"C5: n_train={n} d={d} k=2, full posterior + EHVI-2D ({args.semantics} semantics) + arg-max",
                   "candidates_per_gpu_per_step": m_per_gpu, "precision": precision,
                   "l2": "256 MB flush between timed iterations",
                   "pool": "counter-generated on device (value) / pinned host buffer (e2e)",
                   "parallelism": f"dp{world} (pool sharded, GP state replicated, one 16-byte all-gather)"},
        "ms_per_bo_iter": {"gp_refresh_x2": refresh_ms, "gp_refresh_x2_one_stream": refresh_serial_ms,
                           "score_and_reduce": total_ms / args.steps,
                           "first_refresh_incl_init": refresh_first_ms,
                           "hyperparameter_fit_40_evals_one_gp": fit_ms,
                           "fit_likelihood_evaluations": fit_info.get("nfev"),
                           "fit_ms_per_evaluation": (fit_ms / fit_info["nfev"]) if fit_ms and fit_info.get("nfev") else None,
                           "first_front_and_hypervolume_n1024": prep_ms},
        "e2e": e2e, "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
        "best": {"value": result[0], "index": result[1]}, "wall_s_timed_region": wall,
    }
    if parity_nranks is not None:
        line["parity_nranks"] = parity_nranks
    line.update(extras)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py -- headline benchmark of the Kalman hot path (BASELINE.json config 2).

Workload: second-order (linear trend) DLM, polynomial(2), n = 2, p = 1; 1e6 independent
synthetic series x T = 1000 per GPU; fused Kalman filter + RTS smoother in fp64 writing the
full KfState (m, C, a, R, f, Q) and SmoothingState (s, S) of every step.
Metric: filter+smoother series-steps/s (whole job, all ranks).

A "step" = one pass over the rank's 1e6 series, issued as `--chunks` launches over resident
inputs; outputs go to one reused device buffer set (1e9 steps x 160 B does not fit next to
anything else in 180 GB).  Every launch reads/writes >> 126 MB (L2), so no explicit flush.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--series S] [--T T]
                  [--dump-outputs DIR]
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

N_STATE, N_OBS = 2, 1
ALGO_BYTES_PER_STEP = 8 * (N_OBS + (2 * N_STATE + 2 * N_STATE ** 2 + N_OBS + N_OBS ** 2)
                           + (N_STATE + N_STATE ** 2) + (N_STATE + N_STATE ** 2))  # 216 (SURVEY 8d)
# --dump-outputs sample: 256 series at T = 1000 are 41 MB; fewer when one series' outputs are larger
DUMP_SERIES, DUMP_BYTES, DUMP_SEED = 256, 60_000_000, 20260109


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--series", type=int, default=1_000_000, help="series per GPU")
    ap.add_argument("--T", type=int, default=1000)
    ap.add_argument("--chunks", type=int, default=0,
                    help="launches per step; 0 = launches of --waves full waves each")
    ap.add_argument("--waves", type=int, default=5, help="full GPU waves per launch")
    ap.add_argument("--e2e-series", type=int, default=0,
                    help="series per e2e step (0 = same as --series)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-ffbs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed for a fixed "
                         "sample of series as DIR/<field>.npy (float64, rank 0's series; f and Q "
                         "without the initial row, which holds no forecast)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    return args


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md): NVML in-process
    every 10 ms (the timed region of a few steps is only a fraction of a second), nvidia-smi as
    the fallback."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    BITS = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
            "sw_power_cap": 0x4}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_ev = index, [], threading.Event()
        self.reasons, self.smax, self.how = set(), None, "nvidia-smi"
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self._h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            self._nvml, self.how = pynvml, "nvml"
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        nv = self._nvml
        self.rows.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
        try:
            mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
        except Exception:
            mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        for name, bit in self.BITS.items():
            if mask & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        r = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                            "-i", str(self.index)], capture_output=True, text=True, timeout=5)
        if r.returncode == 0 and r.stdout.strip():
            c = [x.strip() for x in r.stdout.strip().split(",")]
            self.rows.append(float(c[0]))
            self.smax = float(c[1])
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), c[3:7]):
                if v.lower().startswith("active"):
                    self.reasons.add(name)

    def run(self):
        while not self._stop_ev.is_set():
            try:
                if self._nvml:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._stop_ev.wait(0.01 if self._nvml else 0.2)

    def stop(self):
        self._stop_ev.set()
        self.join(timeout=6)
        return {"sm_mhz": float(np.median(self.rows)) if self.rows else None,
                "sm_max_mhz": self.smax, "reasons": sorted(self.reasons),
                "samples": len(self.rows), "how": self.how}


def synth_params(B, seed, xp):
    """Per-series parameters: base x logU(0.5, 2) so nothing constant-folds (SURVEY 8d)."""
    rng = np.random.default_rng(seed + 1)
    sc = np.exp(rng.uniform(np.log(0.5), np.log(2.0), size=(2, B)))
    Vs = (3.0 * sc[0])[None, :]                                   # [1][B]
    Ws = np.array([2.0, 0.0, 0.0, 1.0])[:, None] * sc[1][None, :]  # [4][B] column-major diag(2,1)
    return np.ascontiguousarray(Vs), np.ascontiguousarray(Ws)


def timed_cpu(run, min_seconds=2.0, max_reps=100000):
    """BASELINE.md section 3: every CPU baseline is timed for >= 2 s of wall time AFTER one warm
    pass (page faults, OpenMP team start-up, first-touch of the outputs).  `run()` does one pass
    over the sample; returns (passes, seconds)."""
    run()
    reps, t0 = 0, time.perf_counter()
    while True:
        run()
        reps += 1
        dt = time.perf_counter() - t0
        if dt >= min_seconds or reps >= max_reps:
            return reps, dt


def cpu_reference_leg(series, T, seconds_target=15.0, threads=None, warm_passes=1, passes=None):
    """Time the CPU restatement of the reference (oracle, all host cores) on a bounded sample of
    the same workload.  The JVM reference itself cannot run here (no JDK): kind = "port".
    `passes` fixes the number of timed passes; without it they fill ~seconds_target."""
    import oracle
    from bayesian_dlms_b200 import dlm
    oracle.build()
    threads = threads or os.cpu_count()
    mod = dlm.polynomial(2)
    times = np.arange(1, T + 1.0)
    F, _, G, _, n, p = dlm.materialise(mod, times)
    rng = np.random.default_rng(20260101)

    # bounded sample: Bs series (<= 16384: 160 KB of outputs each), repeated into the same
    # output arrays until ~seconds_target of CPU work has been timed
    Bs = int(min(series, 16384))
    y = rng.standard_normal((Bs, T, 1)).cumsum(axis=1)
    Vs, Ws = synth_params(Bs, 20260101, np)
    Vt, Wt = np.ascontiguousarray(Vs.T), np.ascontiguousarray(Ws.T)
    m0, C0 = np.zeros(n), dlm.cm(100 * np.eye(n))

    def run(out=None):
        t0 = time.perf_counter()
        out = oracle.batch_filter_smooth(Bs, n, p, T, F, G, Vt, Wt, m0, C0, times, y,
                                         keep_init=True, nthreads=threads, out=out)
        return time.perf_counter() - t0, out

    _, out = run()          # warm: page-faults the output arrays, spins up the OpenMP team
    for _ in range(max(0, warm_passes - 1)):
        run(out)
    reps = passes
    if reps is None:
        dt1, out = run(out)
        reps = int(max(1, min(200, round(seconds_target / max(dt1, 1e-6)))))
    t0 = time.perf_counter()
    for _ in range(reps):
        run(out)
    dt = time.perf_counter() - t0
    return {"value": reps * Bs * T / dt, "unit": "series-steps/s", "cores": threads, "kind": "port",
            "sample": f"{Bs} series x T={T} x {reps} passes (config-2 model, full "
                      f"KfState+SmoothingState outputs into reused arrays), {dt:.2f} s wall, "
                      f"oracle/bdlm_oracle.c gcc -O2 OpenMP"}, reps * Bs, dt


def ffbs_leg(eng, dev, with_cpu=True, B=4096, T=2000):
    """Secondary metric (BASELINE.json config 3): FFBS draws/s for the seasonal DLM
    (polynomial(1) |+| seasonal(24, 6), n = 13, p = 1), 4096 chains x T = 2000 with 10 %
    missing observations, injected normals, Gibbs sufficient statistics fused.  FP64-bound:
    the roofline is the measured DFMA peak (halved: the parity contract forbids FMA)."""
    import torch
    from bayesian_dlms_b200 import Model, SERIES_MAJOR, dlm
    mod = dlm.polynomial(1) + dlm.seasonal(24, 6)
    n = 13
    W = np.diag([0.01] + [0.2, 0.4, 0.5, 0.2, 0.1, 0.4] * 2)
    params = dict(V=np.array([[1.0]]), W=W, m0=np.zeros(n), C0=np.eye(n))
    g = torch.Generator(device=dev).manual_seed(20260103)
    y = torch.randn((B, T, 1), generator=g, device=dev, dtype=torch.float64) * 2.0
    y[torch.rand((B, T, 1), generator=g, device=dev) < 0.1] = float("nan")
    z = torch.randn((B, T + 1, n), generator=g, device=dev, dtype=torch.float64)
    model = Model.build(mod, T=T)
    eng.ffbs(model, params, y, z, layout=SERIES_MAJOR, stats=True)  # warm-up
    torch.cuda.synchronize()
    ms = []
    for _ in range(2):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = eng.ffbs(model, params, y, z, layout=SERIES_MAJOR, stats=True)
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    t = min(ms) * 1e-3
    # dense algorithmic flops per step: filter 8n^3 + sampler 15n^3 + Jacobi eig ~ 60 n^3
    flops_step = 83.0 * n ** 3
    peak = eng.ctx.fp64_peak_tflops()
    res = {"config": "config3: seasonal n=13 p=1, %d chains x T=%d, 10%% missing, FFBS + Gibbs stats" % (B, T),
           "draws_per_s": B / t, "steps_per_s": B * (T + 1) / t, "ms_per_sweep": t * 1e3,
           "status_max": int(out["status"].max()),
           "roofline": {"bound": "fp64", "achieved": B * (T + 1) * flops_step / t / 1e12,
                        "peak": peak / 2.0, "unit": "TFLOP/s",
                        "frac": B * (T + 1) * flops_step / t / 1e12 / (peak / 2.0),
                        "flops_per_step": flops_step,
                        "peak_source": "bdlm_fp64_peak_tflops (DFMA microbenchmark) / 2: "
                                       "mul and add issue separately under the no-FMA parity contract"}}
    if with_cpu:
        import oracle
        F, _, G, _, _, p = dlm.materialise(mod, np.arange(1, T + 1.0))
        threads = os.cpu_count()
        Bs = threads
        rng = np.random.default_rng(3)
        yc = rng.standard_normal((Bs, T, 1)) * 2.0
        yc[rng.random(yc.shape) < 0.1] = np.nan
        zc = rng.standard_normal((Bs, T + 1, n))
        reps, dt = timed_cpu(lambda: oracle.batch_ffbs(
            Bs, n, p, T, F, G, [1.0], dlm.cm(W), np.zeros(n), dlm.cm(np.eye(n)),
            np.arange(1, T + 1.0), yc, zc, nthreads=threads))
        res["cpu_baseline"] = {"value": reps * Bs / dt, "unit": "draws/s", "cores": threads, "kind": "port",
                               "sample": f"{Bs} chains x T={T} x {reps} passes after one warm pass, "
                                         f"{dt:.2f} s wall, oracle port OpenMP"}
    return res


def svd_leg(eng, dev, with_cpu=True, B=65536, T=1000):
    """Secondary metric (BASELINE.json config 4): SVD-stabilised filter + sampler
    (SvdSampler.ffbs as GibbsSampling.stepSvd calls it) for the correlated model, 8-fold outer
    sum of polynomial(1), n = p = 8, full W; all 65 536 series of the config in one call."""
    import torch
    from bayesian_dlms_b200 import Model, SERIES_MAJOR, dlm
    mod = dlm.polynomial(1)
    for _ in range(7):
        mod = mod * dlm.polynomial(1)
    n = 8
    V = np.diag([1.0, 4.0] * 4)
    W = np.diag([0.75, 1.25] * 4) + 0.5 * (np.eye(8, k=1) + np.eye(8, k=-1))
    params = dict(V=V, W=W, m0=np.zeros(n), C0=np.eye(n))
    g = torch.Generator(device=dev).manual_seed(20260104)
    y = torch.randn((B, T, n), generator=g, device=dev, dtype=torch.float64) * 2.0
    z = torch.randn((B, T + 1, n), generator=g, device=dev, dtype=torch.float64)
    model = Model.build(mod, T=T)
    eng.ffbs(model, params, y, z, layout=SERIES_MAJOR, svd=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = eng.ffbs(model, params, y, z, layout=SERIES_MAJOR, svd=True)
    e1.record()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) * 1e-3
    # three thin Jacobi SVDs of 2n x n per step (~8 sweeps x n(n-1)/2 pairs x 6*3n flops) + products
    flops_step = 3 * 8 * (n * (n - 1) / 2) * 18 * n + 20.0 * n ** 3
    peak = eng.ctx.fp64_peak_tflops()
    res = {"config": "config4: correlated n=p=8, %d series x T=%d, SVD filter + SVD sampler" % (B, T),
           "draws_per_s": B / t, "steps_per_s": B * (T + 1) / t, "ms_per_sweep": t * 1e3,
           "status_max": int(out["status"].max()),
           "roofline": {"bound": "fp64", "achieved": B * (T + 1) * flops_step / t / 1e12,
                        "peak": peak / 2.0, "unit": "TFLOP/s",
                        "frac": B * (T + 1) * flops_step / t / 1e12 / (peak / 2.0),
                        "flops_per_step": flops_step}}
    if with_cpu:
        import oracle
        F, _, G, _, _, p = dlm.materialise(mod, np.arange(1, T + 1.0))
        threads = os.cpu_count()
        Bs = 4 * threads
        rng = np.random.default_rng(4)
        yc = rng.standard_normal((Bs, T, n)) * 2.0
        zc = rng.standard_normal((Bs, T + 1, n))
        reps, dt = timed_cpu(lambda: oracle.batch_ffbs(
            Bs, n, p, T, F, G, dlm.cm(V), dlm.cm(W), np.zeros(n), dlm.cm(np.eye(n)),
            np.arange(1, T + 1.0), yc, zc, svd=True, nthreads=threads))
        res["cpu_baseline"] = {"value": reps * Bs / dt, "unit": "draws/s", "cores": threads, "kind": "port",
                               "sample": f"{Bs} series x T={T} x {reps} passes after one warm pass, "
                                         f"{dt:.2f} s wall, oracle port OpenMP"}
    return res


def gibbs_leg(eng, dev, B=4096, T=2000, sweeps=3):
    """BASELINE.json config 3 as the reference runs it: FFBS INSIDE the d-inverse-gamma Gibbs
    sampler (GibbsSampling.sample, Gibbs.scala:153-180).  One sweep = normals for the sweep,
    FFBS with fused sufficient statistics, on-device conjugate draws of diag(V), diag(W); the
    drawn parameters feed the next sweep as per-chain arrays without leaving the GPU."""
    import torch
    from bayesian_dlms_b200 import Model, SERIES_MAJOR, dlm, gibbs
    mod = dlm.polynomial(1) + dlm.seasonal(24, 6)
    n = 13
    W = np.diag([0.01] + [0.2, 0.4, 0.5, 0.2, 0.1, 0.4] * 2)
    init = dict(V=np.array([[1.0]]), W=W, m0=np.zeros(n), C0=np.eye(n))
    prior = dict(v_shape=5.0, v_scale=4.0, w_shape=17.0, w_scale=4.0)  # SeasonalModel.scala:127
    g = torch.Generator(device=dev).manual_seed(20260103)
    y = torch.randn((B, T, 1), generator=g, device=dev, dtype=torch.float64) * 2.0
    y[torch.rand((B, T, 1), generator=g, device=dev) < 0.1] = float("nan")
    model = Model.build(mod, T=T)
    gibbs.sample(eng, model, y, prior, init, 1, seed=1, layout=SERIES_MAJOR)  # warm-up
    torch.cuda.synchronize()
    l0 = eng.ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    res = gibbs.sample(eng, model, y, prior, init, sweeps, seed=2, layout=SERIES_MAJOR)
    e1.record()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) * 1e-3
    return {"config": "config3: %d chains x T=%d, %d Gibbs sweeps (normals + FFBS + stats + "
                      "inverse-gamma draws of V, W), device-resident" % (B, T, sweeps),
            "chain_sweeps_per_s": B * sweeps / t, "ms_per_sweep": t * 1e3 / sweeps,
            "launches_per_sweep": (eng.ctx.launch_count() - l0) / sweeps,
            "status_max": int(res["status"].max()),
            "posterior_mean_V_last": float(res["V"][-1].mean())}


def gibbs_wishart_leg(eng, dev, B=65536, T=1000, sweeps=2):
    """BASELINE.json config 4 as a sampler: correlated model n = p = 8, SVD filter + SVD sampler
    (GibbsSampling.stepSvd's FFBS, Gibbs.scala:182-198) with an inverse-Wishart draw of the full W
    (GibbsWishart.sampleSystemMatrix, GibbsWishart.scala:16-35) and inverse-gamma draws of diag(V),
    65 536 series, every sweep device-resident."""
    import torch
    from bayesian_dlms_b200 import Model, SERIES_MAJOR, dlm, gibbs
    mod = dlm.polynomial(1)
    for _ in range(7):
        mod = mod * dlm.polynomial(1)
    n = 8
    V = np.diag([1.0, 4.0] * 4)
    W = np.diag([0.75, 1.25] * 4) + 0.5 * (np.eye(8, k=1) + np.eye(8, k=-1))
    init = dict(V=V, W=W, m0=np.zeros(n), C0=np.eye(n))
    prior = dict(v_shape=6.0, v_scale=5.0, w_nu=10.0, w_psi=np.eye(n))  # CorrelatedModel.scala:85-86
    g = torch.Generator(device=dev).manual_seed(20260104)
    y = torch.randn((B, T, n), generator=g, device=dev, dtype=torch.float64) * 2.0
    model = Model.build(mod, T=T)
    gibbs.sample(eng, model, y, prior, init, 1, seed=1, layout=SERIES_MAJOR, svd=True, record=False)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    res = gibbs.sample(eng, model, y, prior, init, sweeps, seed=2, layout=SERIES_MAJOR, svd=True,
                       record=False)
    e1.record()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) * 1e-3
    return {"config": "config4: %d series x T=%d, %d Gibbs sweeps (normals + SVD-FFBS + stats + "
                      "inverse-Wishart W, inverse-gamma V), device-resident" % (B, T, sweeps),
            "series_sweeps_per_s": B * sweeps / t, "ms_per_sweep": t * 1e3 / sweeps,
            "status_max": int(res["status"].max())}


def ar_leg(eng, dev, with_cpu=True, B=1_000_000, T=1000):
    """Next row f3: scalar AR(1) FFBS (FilterAr.ffbs, FilterAr.scala:77-83), the inner loop of the
    stochastic-volatility samplers, 1e6 series x T = 1000, per-series parameters and per-step
    per-series observation variances.  HBM-bound: y, v in; (m, C) spilled and re-read; z in;
    theta out = 8 * 8 B per series-step."""
    import torch
    from bayesian_dlms_b200 import TIME_MAJOR
    g = torch.Generator(device=dev).manual_seed(20260106)
    r = lambda *s: torch.rand(s, generator=g, device=dev, dtype=torch.float64)  # noqa: E731
    sv = dict(phi=0.5 + 0.45 * r(B), mu=r(B) - 0.5, sigma_eta=0.1 + r(B))
    y = torch.randn((T, B), generator=g, device=dev, dtype=torch.float64)
    v = 0.5 + r(T, B)
    z = torch.randn((T + 1, B), generator=g, device=dev, dtype=torch.float64)
    eng.ar_ffbs(sv, y, v, z, layout=TIME_MAJOR)
    torch.cuda.synchronize()
    ms = []
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = eng.ar_ffbs(sv, y, v, z, layout=TIME_MAJOR)
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    t = float(np.median(ms)) * 1e-3
    byt = 8 * 8
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    res = {"config": "f3: scalar AR(1) FFBS, %d series x T=%d, per-series phi/mu/sigma and v_t" % (B, T),
           "steps_per_s": B * T / t, "draws_per_s": B / t, "ms": t * 1e3,
           "finite": bool(torch.isfinite(out["theta"][:, :1000]).all()),
           "roofline": {"bound": "hbm", "achieved": B * T * byt / t / 1e9, "peak": peak,
                        "unit": "GB/s", "frac": B * T * byt / t / 1e9 / peak, "bytes_per_step": byt}}
    if with_cpu:
        import oracle
        Tc, per = T, 500
        yc, vc, zc = np.random.default_rng(6).standard_normal((3, Tc + 1))
        tt, vv = np.arange(1.0, Tc + 1), np.abs(vc[:Tc]) + 0.5

        def run_ar():
            for _ in range(per):
                f = oracle.ar_filter(0.8, 0.1, 0.3, tt, vv, yc[:Tc])
                oracle.ar_backward_sample(0.8, f, zc)

        reps, dt = timed_cpu(run_ar)
        res["cpu_baseline"] = {"value": reps * per * Tc / dt, "unit": "series-steps/s", "cores": 1,
                               "kind": "port",
                               "sample": f"{reps * per} series x T={Tc} after a warm pass of {per}, one "
                                         f"core, {dt:.2f} s wall"}
    return res


def scan_leg(eng, dev, with_cpu=True, logT=24):
    """Secondary metric (BASELINE.json config 5): ONE series, T = 2^24, polynomial(2),
    parallel-in-time filter + smoother on one GPU (the 8-GPU run shards the time axis and
    exchanges one aggregate per rank)."""
    import torch
    from bayesian_dlms_b200 import Model, dlm
    from bayesian_dlms_b200.scan import scan_filter_smooth
    n, T = 2, 1 << logT
    params = dict(V=[[3.0]], W=np.diag([2.0, 1.0]), m0=np.zeros(2), C0=100.0 * np.eye(2))
    g = torch.Generator(device=dev).manual_seed(20260105)
    y = torch.randn(T, generator=g, device=dev, dtype=torch.float64).cumsum(0) * 0.1
    model = Model.build(dlm.polynomial(2), T=T)
    for _ in range(2):
        scan_filter_smooth(eng, model, params, y)
    torch.cuda.synchronize()

    def timed(queue_ahead):
        ms = []
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            if queue_ahead:  # ~0.5 ms of spinning in front of e0: the call's launches are queued
                torch.cuda._sleep(1_000_000)  # before e0 fires, so the events see device time only
            e0.record()
            out = scan_filter_smooth(eng, model, params, y)
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        return float(np.median(ms)), out

    # One call is 9 dependent launches of 1.2-1.4 ms in total: events around the Python call also
    # count the ~0.1 ms the host needs before its first launch (GPU idle).  Both are reported; the
    # roofline uses the device time, like the headline (whose 12 ms launches hide the host).
    ms_host, out = timed(False)
    try:
        ms_dev, out = timed(True)
    except Exception:
        ms_dev = ms_host
    t = min(ms_dev, ms_host) * 1e-3
    byt = 8 * (1 + 14 + 6 + 6)  # SURVEY 8(d): y, KfState, (m, C) re-read, (s, S) = 216 B/step
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    res = {"config": "config5: one series, T=2^%d, polynomial(2), associative-scan filter+smoother" % logT,
           "steps_per_s": T / t, "ms": t * 1e3, "ms_incl_host_prep": ms_host,
           "timing": "CUDA events on the launching stream, median of 5 calls after 2 warm calls; ms = with the "
                     "call's launches queued behind a 0.5 ms spin kernel (device time), "
                     "ms_incl_host_prep = events around the bare Python call",
           "status": int(out["status"][0]),
           "roofline": {"bound": "hbm", "achieved": T * byt / t / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": T * byt / t / 1e9 / peak, "bytes_per_step": byt}}
    if with_cpu:
        import oracle
        Tc = 1 << 20  # the reference recursion is sequential: one core, bounded sample
        F, _, G, _, _, p = dlm.materialise(dlm.polynomial(2), np.arange(1, 9.0))
        yc = y[:Tc].cpu().numpy()
        tc = np.arange(1, Tc + 1.0)

        def run_seq():
            o = oracle.kf_filter(2, 1, F, G, [3.0], dlm.cm(np.diag([2.0, 1.0])), np.zeros(2),
                                 dlm.cm(100.0 * np.eye(2)), tc, yc)
            oracle.rts_smooth(2, G, o)

        reps, dt = timed_cpu(run_seq)
        res["cpu_baseline"] = {"value": reps * Tc / dt, "unit": "series-steps/s", "cores": 1, "kind": "port",
                               "sample": f"first 2^20 steps x {reps} passes after one warm pass, "
                                         f"sequential (the reference has no parallel-in-time path), "
                                         f"{dt:.2f} s wall"}
    return res


def ffbs_small_leg(eng, dev, with_cpu=True, B=1_000_000, T=1000):
    """FFBS for the config-2 model itself (polynomial(2), the reference's SecondOrder Gibbs example,
    SecondOrder.scala:53-97): 1e6 chains x T = 1000, one thread per chain, on-device normals,
    sufficient statistics fused."""
    import torch
    from bayesian_dlms_b200 import Model, TIME_MAJOR, dlm
    g = torch.Generator(device=dev).manual_seed(20260108)
    y = torch.randn((T, 1, B), generator=g, device=dev, dtype=torch.float64).cumsum(0)
    params = dict(V=[[3.0]], W=np.diag([2.0, 1.0]), m0=np.zeros(2), C0=100.0 * np.eye(2))
    model = Model.build(dlm.polynomial(2), T=T)
    eng.ctx.set_rng(20260108, 0)
    eng.ffbs(model, params, y, None, layout=TIME_MAJOR, stats=True)
    torch.cuda.synchronize()
    ms = []
    for it in range(3):
        eng.ctx.set_rng(20260108, it + 1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = eng.ffbs(model, params, y, None, layout=TIME_MAJOR, stats=True)
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    t = float(np.median(ms)) * 1e-3
    res = {"config": "FFBS of the config-2 model: polynomial(2), %d chains x T=%d, Philox normals, "
                     "Gibbs statistics fused" % (B, T),
           "draws_per_s": B / t, "steps_per_s": B * (T + 1) / t, "ms_per_sweep": t * 1e3,
           "status_max": int(out["status"].max())}
    if with_cpu:
        import oracle
        F, _, G, _, n, p = dlm.materialise(dlm.polynomial(2), np.arange(1, T + 1.0))
        threads = os.cpu_count()
        Bs = 64 * threads
        rng = np.random.default_rng(8)
        yc = rng.standard_normal((Bs, T, 1)).cumsum(axis=1)
        zc = rng.standard_normal((Bs, T + 1, 2))
        reps, dt = timed_cpu(lambda: oracle.batch_ffbs(
            Bs, n, p, T, F, G, [3.0], dlm.cm(np.diag([2.0, 1.0])), np.zeros(2),
            dlm.cm(100.0 * np.eye(2)), np.arange(1, T + 1.0), yc, zc, nthreads=threads))
        res["cpu_baseline"] = {"value": reps * Bs / dt, "unit": "draws/s", "cores": threads, "kind": "port",
                               "sample": f"{Bs} chains x T={T} x {reps} passes after one warm pass, "
                                         f"{dt:.2f} s wall, oracle port OpenMP"}
    return res


def loglik_leg(eng, dev, with_cpu=True, B=1_000_000, T=1000):
    """Row a9 of the scope table: KalmanFilter.likelihood (what Metropolis-Hastings evaluates per
    proposal, MetropolisHastings.scala:126-137) for the config-2 model, 1e6 series with their own
    V, W: both log-likelihoods per series, nothing stored per step (FP64-issue bound)."""
    import torch
    from bayesian_dlms_b200 import Model, TIME_MAJOR, dlm
    g = torch.Generator(device=dev).manual_seed(20260107)
    y = torch.randn((T, 1, B), generator=g, device=dev, dtype=torch.float64).cumsum(0)
    Vs_all, Ws_all = synth_params(B, 20260107, np)
    params = dict(V=torch.from_numpy(Vs_all).to(dev), W=torch.from_numpy(Ws_all).to(dev),
                  m0=np.zeros(2), C0=100.0 * np.eye(2), per_series=("V", "W"))
    model = Model.build(dlm.polynomial(2), T=T)
    eng.loglik(model, params, y, layout=TIME_MAJOR)
    torch.cuda.synchronize()
    ms = []
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = eng.loglik(model, params, y, layout=TIME_MAJOR)
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    t = float(np.median(ms)) * 1e-3
    res = {"config": "a9: KalmanFilter.likelihood, polynomial(2), %d series x T=%d, per-series V, W" % (B, T),
           "series_steps_per_s": B * T / t, "likelihoods_per_s": B / t, "ms": t * 1e3,
           "status_max": int(out["status"].max())}
    if with_cpu:
        import oracle
        F, _, G, _, n, p = dlm.materialise(dlm.polynomial(2), np.arange(1, T + 1.0))
        yc = y[:, 0, :64].cpu().numpy().T.copy()
        tt = np.arange(1, T + 1.0)

        def run_ll():
            for b in range(64):
                oracle.loglik(n, p, F, G, [float(Vs_all[0, b])], Ws_all[:, b].copy(), np.zeros(2),
                              dlm.cm(100.0 * np.eye(2)), tt, yc[b])

        reps, dt = timed_cpu(run_ll)
        res["cpu_baseline"] = {"value": reps * 64 * T / dt, "unit": "series-steps/s", "cores": 1, "kind": "port",
                               "sample": f"64 series x T={T} x {reps} passes after one warm pass, one "
                                         f"core, {dt:.2f} s wall"}
    return res


def jmh_leg(eng, with_cpu=True):
    """The reference's own JMH shapes (benchmark/src/main/scala/bench/KalmanFilter.scala:10-33,
    SvdFilter.scala:28-36, ffbs.scala:27-35): ONE series, polynomial(1), V = 3, W = 1, m0 = 0,
    C0 = 1, T = 10 -- KalmanFilter.filterDlm, SvdFilter.filterDlm, Smoothing.ffbsDlm,
    SvdSampler.ffbsDlm -- plus one series of T = 1000 (filterDlm + backwardsSmoother, the
    FirstOrderDlm example).  Microseconds per call through (a) the drop-in mirror of the Scala API
    (reference_api, host objects in and out), (b) the bare C ABI with host buffers, next to (c) the
    CPU port on one core.  A single short series cannot fill a GPU: this leg exists to state the
    per-call latency of the drop-in honestly, not to win."""
    from bayesian_dlms_b200 import (Data, DlmParameters, KalmanFilter, Model, SERIES_MAJOR, Smoothing,
                                    SvdFilter, SvdSampler, dlm, polynomial)
    mod = polynomial(1)
    p = DlmParameters(v=[[3.0]], w=[[1.0]], m0=[0.0], c0=[[1.0]])
    rng = np.random.default_rng(10)

    def series(T):
        x = np.cumsum(rng.standard_normal(T))
        return [Data(float(t + 1), np.array([x[t] + 1.7 * rng.standard_normal()])) for t in range(T)]

    def us(fn, min_s=0.5):
        fn(); fn()
        n, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < min_s:
            fn(); n += 1
        return (time.perf_counter() - t0) / n * 1e6

    res = {"model": "polynomial(1), V=3, W=1, m0=0, C0=1, one series (the JMH ModelState)", "unit": "us/call"}
    for T in (10, 1000):
        ys = series(T)
        z = rng.standard_normal((T + 1, 1))
        yarr = np.ascontiguousarray(np.array([d.observation for d in ys]).reshape(1, T, 1))
        model = Model.build(mod, T=T)
        par = dict(V=p.v, W=p.w, m0=p.m0, C0=p.c0)
        zz = z.reshape(1, T + 1, 1).copy()
        row = {}
        row["kalmanFilter"] = {
            "mirror": us(lambda: KalmanFilter.filterDlm(mod, ys, p)),
            "c_abi": us(lambda: eng.filter(model, par, yarr, layout=SERIES_MAJOR, keep_init=False))}
        row["svdFilter"] = {
            "mirror": us(lambda: SvdFilter.filterDlm(mod, ys, p)),
            "c_abi": us(lambda: eng.svd_filter(model, par, yarr, layout=SERIES_MAJOR, keep_init=False))}
        row["naiveFfbs"] = {
            "mirror": us(lambda: Smoothing.ffbsDlm(mod, ys, p, z=z)),
            "c_abi": us(lambda: eng.ffbs(model, par, yarr, zz, layout=SERIES_MAJOR))}
        row["svdFfbs"] = {
            "mirror": us(lambda: SvdSampler.ffbsDlm(mod, ys, p, z=z)),
            "c_abi": us(lambda: eng.ffbs(model, par, yarr, zz, layout=SERIES_MAJOR, svd=True))}
        row["filterSmooth"] = {
            "mirror": us(lambda: Smoothing.backwardsSmoother(mod)(KalmanFilter.filter(mod, ys, p))),
            "c_abi": us(lambda: eng.filter_smooth(model, par, yarr, layout=SERIES_MAJOR))}
        if with_cpu:
            import oracle
            F, _, G, _, n_, p_ = dlm.materialise(mod, np.arange(1, T + 1.0))
            tt, y1 = np.arange(1, T + 1.0), yarr[0]
            V, W, m0, C0 = [3.0], [1.0], [0.0], [1.0]
            row["kalmanFilter"]["cpu_port"] = us(lambda: oracle.kf_filter(1, 1, F, G, V, W, m0, C0, tt, y1, keep_init=False))
            row["svdFilter"]["cpu_port"] = us(lambda: oracle.svd_filter(1, 1, F, G, V, W, m0, C0, tt, y1, keep_init=False))
            row["naiveFfbs"]["cpu_port"] = us(lambda: oracle.ffbs(1, 1, F, G, V, W, m0, C0, tt, y1, z))
            row["svdFfbs"]["cpu_port"] = us(lambda: oracle.svd_ffbs(1, 1, F, G, V, W, m0, C0, tt, y1, z))
            row["filterSmooth"]["cpu_port"] = us(
                lambda: oracle.rts_smooth(1, G, oracle.kf_filter(1, 1, F, G, V, W, m0, C0, tt, y1)))
        res["T=%d" % T] = row
    res["note"] = ("c_abi = one bdlm_* call with numpy host buffers incl. ctypes marshalling; mirror adds "
                   "Data/KfState object (un)packing; cpu_port = oracle C via ctypes, one core. The "
                   "reference's JVM numbers for these harnesses are unpublished and no JVM exists here.")
    return res


def scan_dist_leg(comm, eng, dev, rank, world, logT=24, reps=5):
    """BASELINE.json config 5 on N GPUs: ONE series, T = 2^24, time-sharded across the ranks through
    the library's communicator (bdlm_comm_scan_filter_smooth: per pass one exchange of a <= 16-double
    chunk aggregate per rank, no host synchronisation).  Strong scaling: total work is fixed.
    Time = max over ranks.  Two variants: one process per GPU (this torchrun job; NCCL all-gathers
    issued by libbdlm.so) and, on rank 0 alone, ONE process driving all N GPUs with the aggregates
    stored straight into the peers' mailboxes over NVLink (no NCCL call on the path)."""
    import torch
    import torch.distributed as dist
    from bayesian_dlms_b200 import Model, dlm
    from bayesian_dlms_b200.comm import Comm
    from bayesian_dlms_b200.scan import scan_filter_smooth
    from bayesian_dlms_b200.sharding import shard_range
    T = 1 << logT
    params = dict(V=[[3.0]], W=np.diag([2.0, 1.0]), m0=np.zeros(2), C0=100.0 * np.eye(2))
    lo, hi = shard_range(T, rank, world)
    # every rank draws the SAME full series (134 MB) and keeps its own time chunk; the full copy
    # is only used for the parity check below
    g = torch.Generator(device=dev).manual_seed(20260105)
    yfull = torch.randn(T, generator=g, device=dev, dtype=torch.float64).cumsum(0) * 0.1
    yc = yfull[lo:hi].contiguous()
    h = comm.scan_setup([Model.build(dlm.polynomial(2), T=hi - lo)], params, [yc])
    comm.scan_run(h); comm.scan_run(h)
    ms = []
    for _ in range(reps):
        dist.barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); comm.scan_run(h); e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms.append(float(t.item()))
    st = h["status"][0].clone()
    dist.all_reduce(st, op=dist.ReduceOp.MAX)
    # parity on REAL ranks: this rank's rows of the exchanged run against the same rows of the
    # single-GPU scan of the whole series (itself checked against the CPU oracle at this size by
    # tests/test_gpu_scan.py::test_scan_full_config5_size_vs_cpu_oracle)
    one = scan_filter_smooth(eng, Model.build(dlm.polynomial(2), T=T), params, yfull)
    torch.cuda.synchronize()

    def worst_vs_one(out, r):
        lo_r, hi_r = shard_range(T, r, world)
        r0 = 0 if r == 0 else lo_r + 1      # global row of the chunk's first output row
        w = torch.zeros(1, device=dev, dtype=torch.float64)
        for k in ("m", "C", "a", "R", "s", "S"):
            a = out[k].to(dev)
            b = one[k][r0:r0 + a.shape[0]]
            den = torch.maximum(b.abs(), 1e-6 * one[k].abs().max())
            w = torch.maximum(w, ((a - b).abs() / den).max().reshape(1))
        return w

    worst = worst_vs_one(h["outs"][0], rank)
    dist.all_reduce(worst, op=dist.ReduceOp.MAX)
    t = float(np.median(ms)) * 1e-3
    res = {"config": "config5: one series, T=2^%d, polynomial(2), time-sharded over %d GPUs" % (logT, world),
           "scaling": "strong", "steps_per_s": T / t, "ms": t * 1e3, "status": int(st.item()),
           "max_rel_err": float(worst.item()),
           "max_rel_err_of": "every rank's (m, C, a, R, s, S) rows vs the single-GPU scan of the "
                             "whole series, max over ranks; bar 1e-9",
           "exchange": "bdlm_comm_scan_filter_smooth, one process per GPU: 2 ncclAllGather of <= 16 "
                       "doubles per rank per call, issued by libbdlm.so"}
    # ---- the same job from ONE process driving all N GPUs (a JVM host): peer-mailbox exchange.
    # The other ranks wait on the CPU (c10d store), not in an NCCL barrier whose spinning kernel
    # would share their GPU with this leg.
    store = dist.distributed_c10d._get_default_store()
    torch.cuda.synchronize()
    if rank == 0:
        try:
            res["single_process"] = scan_single_process(T, world, params, yfull, worst_vs_one, reps)
        except Exception as ex:
            res["single_process"] = {"error": repr(ex)}
        store.set("bdlm_single_process_scan_done", "1")
    else:
        store.wait(["bdlm_single_process_scan_done"])
    dist.barrier()
    return res


def scan_single_process(T, world, params, yfull, worst_vs_one, reps):
    import torch
    from bayesian_dlms_b200 import Model, dlm
    from bayesian_dlms_b200.comm import Comm
    from bayesian_dlms_b200.sharding import shard_range
    out = {}
    for peer in (True, False):
        if peer:
            os.environ.pop("BDLM_COMM_NO_PEER", None)
        else:
            os.environ["BDLM_COMM_NO_PEER"] = "1"
        pc = Comm.single_process(list(range(world)))
        os.environ.pop("BDLM_COMM_NO_PEER", None)
        streams = []
        for r, e in enumerate(pc.engines):   # contexts on torch streams so that torch events time them
            st = torch.cuda.Stream(device=r)
            streams.append(st)
            e.ctx.set_stream(st.cuda_stream)
        models, chunks = [], []
        for r in range(world):
            lo_r, hi_r = shard_range(T, r, world)
            models.append(Model.build(dlm.polynomial(2), T=hi_r - lo_r))
            chunks.append(yfull[lo_r:hi_r].to(torch.device("cuda", r)).contiguous())
        for r in range(world):
            torch.cuda.synchronize(r)
        guards = [torch.cuda.stream(st) for st in streams]
        for gd in guards:
            gd.__enter__()
        try:
            hp = pc.scan_setup(models, params, chunks)
            for _ in range(3):
                pc.scan_run(hp)
            pc.sync()
            dev_ms, host_ms = [], []
            for _ in range(reps):
                pc.sync()
                evs = []
                for st in streams:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(st)
                    evs.append((e0, e1))
                w0 = time.perf_counter()
                pc.scan_run(hp)
                for (e0, e1), st in zip(evs, streams):
                    e1.record(st)
                pc.sync()
                host_ms.append((time.perf_counter() - w0) * 1e3)
                dev_ms.append(max(e0.elapsed_time(e1) for e0, e1 in evs))
        finally:
            for gd in reversed(guards):
                gd.__exit__(None, None, None)
        worst_p = max(float(worst_vs_one(hp["outs"][r], r).item()) for r in range(world))
        out["peer_mailboxes" if pc.uses_peer_exchange else "nccl_allgather"] = {
            "ms": float(np.median(dev_ms)), "host_enqueue_plus_sync_ms": float(np.median(host_ms)),
            "status": max(int(s_.item()) for s_ in hp["status"]), "max_rel_err": worst_p}
        pc.close()
    out["timing"] = "CUDA events on every device's stream, max over devices, median of %d" % reps
    out["what"] = ("ONE process drives all %d GPUs through bdlm_comm_scan_filter_smooth; peer_mailboxes = "
                   "aggregates stored into the peers' memory over NVLink + flag, no NCCL call" % world)
    return out


def loglik_dist_leg(comm, eng, dev, rank, world, B=1_000_000, T=1000):
    """The reduction north_star names: KalmanFilter.likelihood of every series of every rank and
    ONE ncclAllReduce of the two sums inside the library (bdlm_comm_loglik) -- the pooled
    log-likelihood a Metropolis step over shared parameters needs (MetropolisHastings.scala:126-137)."""
    import torch
    import torch.distributed as dist
    from bayesian_dlms_b200 import Model, TIME_MAJOR, dlm
    g = torch.Generator(device=dev).manual_seed(20260107 + rank)
    y = torch.randn((T, 1, B), generator=g, device=dev, dtype=torch.float64).cumsum(0)
    params = dict(V=[[3.0]], W=np.diag([2.0, 1.0]), m0=np.zeros(2), C0=100.0 * np.eye(2))
    model = Model.build(dlm.polynomial(2), T=T)
    out = comm.loglik(model, params, y, layout=TIME_MAJOR)
    ms = []
    for _ in range(3):
        dist.barrier(); torch.cuda.synchronize()
        w0 = time.perf_counter()
        out = comm.loglik(model, params, y, layout=TIME_MAJOR)   # returns after the all-reduce
        w = torch.tensor([time.perf_counter() - w0], device=dev, dtype=torch.float64)
        dist.all_reduce(w, op=dist.ReduceOp.MAX)
        ms.append(float(w.item()) * 1e3)
    local = torch.stack([out["transition"].sum(), out["innovations"].sum()])
    dist.all_reduce(local)   # torch's own reduce as the cross-check of the library's
    t = float(np.median(ms)) * 1e-3
    return {"config": "a9 on %d GPUs: %d series/GPU x T=%d, sums reduced by ncclAllReduce inside "
                      "libbdlm.so" % (world, B, T),
            "series_steps_per_s": world * B * T / t, "ms": t * 1e3,
            "sum_innovations": out["sum_innovations"], "sum_transition": out["sum_transition"],
            "rel_diff_vs_torch_allreduce": float(max(
                abs(out["sum_transition"] - local[0].item()) / abs(local[0].item()),
                abs(out["sum_innovations"] - local[1].item()) / abs(local[1].item())))}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    T, B = args.T, args.series
    # identical in both arms (the driver compares the dicts); run-derived launch geometry goes to
    # its own key
    config = {"workload": "config2: polynomial(2) n=2 p=1, %d series/GPU x T=%d, fused Kalman filter + "
                          "RTS smoother, full KfState+SmoothingState outputs" % (B, T),
              "series_per_gpu": B, "T": T, "global_series": world * B,
              "device_layout": "time-major SoA [rows][k][B]",
              "l2": "inputs+outputs per launch >> 126 MB L2 (no flush needed)"}
    geometry = {}

    if args.impl == "reference":
        if rank != 0:
            return
        # K timed steps, each one pass over the bounded sample (W untimed passes first)
        base, nser, dt = cpu_reference_leg(B, T, passes=args.steps, warm_passes=max(1, args.warmup))
        v = base["value"]
        print(json.dumps({
            "impl": "reference", "metric": "filter+smoother series-steps/s", "value": v,
            "unit": "series-steps/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / max(1, args.steps), "higher_is_better": True,
            "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "cpu_baseline": base,
            "e2e": {"value": v, "unit": "series-steps/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0},
            "note": "JVM/Scala toolchain absent: CPU restatement of the reference (oracle port), "
                    "all host cores, bounded sample"}))
        return

    import torch
    import torch.distributed as dist
    from bayesian_dlms_b200 import Engine, Model, TIME_MAJOR, dlm

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    comm = None
    if world > 1:
        # torch.distributed is plumbing (rendezvous, barriers, max-over-ranks of the timings); the
        # data-path collectives go through the library's own communicator (bdlm_comm_*)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        from bayesian_dlms_b200.comm import Comm
        comm = Comm.from_torch_distributed(local)
        eng = comm.engines[0]
    else:
        eng = Engine(local)
    eng.use_torch_stream()

    # ---- synthetic inputs, resident in HBM (Dlm.simStep generative model, Dlm.scala:245-282)
    if args.chunks > 0:
        nch = args.chunks
        bounds = [(i * B) // nch for i in range(nch + 1)]
    else:
        # every series of a launch takes the same time: launches that are whole waves
        # (resident blocks x SMs x 128 series) leave no partially filled last wave
        from bayesian_dlms_b200.sharding import shard_range, wave_aligned_slabs
        glo, ghi = shard_range(world * B, rank, world)  # this rank's block of the global batch
        assert ghi - glo == B
        slabs = wave_aligned_slabs(0, B, eng.ctx.wave_series(N_STATE, N_OBS), args.waves)
        bounds = [s[0] for s in slabs] + [B]
        nch = len(bounds) - 1
    geometry["launches_per_step"] = nch
    geometry["series_per_launch"] = bounds[1] - bounds[0]
    Bc_max = max(bounds[i + 1] - bounds[i] for i in range(nch))
    rows = T + 1
    # The rank's whole batch is drawn first and then cut into launches, so that a series gets the
    # same data whatever the launch geometry (which follows the kernel's occupancy): two builds of
    # the library then see identical inputs and their outputs compare series for series.
    g = torch.Generator(device=dev).manual_seed(20260101 + rank)
    Vs_all, Ws_all = synth_params(B, 20260101 + 1000 * rank, np)
    Vd, Wd = torch.from_numpy(Vs_all).to(dev), torch.from_numpy(Ws_all).to(dev)
    x0 = 10.0 * torch.randn((B,), generator=g, device=dev, dtype=torch.float64)
    x1 = 10.0 * torch.randn((B,), generator=g, device=dev, dtype=torch.float64)
    yall = torch.empty((T, 1, B), device=dev, dtype=torch.float64)
    sw0, sw1, sv = Wd[0].sqrt(), Wd[3].sqrt(), Vd[0].sqrt()
    for t in range(T):
        x0 = x0 + x1 + sw0 * torch.randn((B,), generator=g, device=dev, dtype=torch.float64)
        x1 = x1 + sw1 * torch.randn((B,), generator=g, device=dev, dtype=torch.float64)
        yall[t, 0] = x0 + sv * torch.randn((B,), generator=g, device=dev, dtype=torch.float64)
    ys, pars = [], []
    for i in range(nch):
        b0, b1 = bounds[i], bounds[i + 1]
        ys.append(yall[:, :, b0:b1].contiguous())
        pars.append(dict(V=Vd[:, b0:b1].contiguous(), W=Wd[:, b0:b1].contiguous(), m0=np.zeros(2),
                         C0=100.0 * np.eye(2), per_series=("V", "W")))
    del yall, x0, x1
    model = Model.build(dlm.polynomial(2), T=T)
    dims = dict(m=2, C=4, a=2, R=4, f=1, Q=1, s=2, S=4)
    outbuf = {k: torch.empty((rows, d, Bc_max), device=dev, dtype=torch.float64)
              for k, d in dims.items()}
    outbuf["status"] = torch.empty((Bc_max,), device=dev, dtype=torch.int32)

    def views(Bc):
        if Bc == Bc_max:
            return outbuf
        o = {k: outbuf[k].view(-1)[: rows * dims[k] * Bc].view(rows, dims[k], Bc) for k in dims}
        o["status"] = outbuf["status"][:Bc]
        return o

    chk = torch.zeros(4, device=dev, dtype=torch.float64)

    # --dump-outputs: the full outputs of a step (160 B per series-step) never coexist -- every
    # launch overwrites the buffers -- so the last timed step keeps a fixed, seeded sample of series
    # right after each launch (a gather of at most DUMP_BYTES, small next to a launch's traffic)
    picks = kept = None
    if args.dump_outputs and rank == 0:
        per_series = 8 * (rows * sum(dims.values()) + 1)
        ns = min(B, DUMP_SERIES, DUMP_BYTES // per_series)
        if ns < 1:
            sys.exit("--dump-outputs: the outputs of one series exceed %d bytes" % DUMP_BYTES)
        pick = np.sort(np.random.default_rng(DUMP_SEED).choice(B, size=ns, replace=False))
        picks = [torch.from_numpy(pick[(pick >= b0) & (pick < b1)] - b0).to(dev)
                 for b0, b1 in zip(bounds[:-1], bounds[1:])]
        kept = [{k: v.new_empty(v.shape[:-1] + (len(p),)) for k, v in views(b1 - b0).items()}
                for p, b0, b1 in zip(picks, bounds[:-1], bounds[1:])]

    def keep_sample(i, o):
        for k, v in o.items():
            torch.index_select(v, -1, picks[i], out=kept[i][k])

    def step(timers=None, keep=False):
        for i in range(nch):
            Bc = bounds[i + 1] - bounds[i]
            if timers is not None:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            o = eng.filter_smooth(model, pars[i], ys[i], out=views(Bc))
            if timers is not None:
                e1.record()
                timers.append((e0, e1, Bc))
            if keep:
                keep_sample(i, o)
        chk[0] = o["s"][0, 0, 0]; chk[1] = o["S"][0, 0, 0]; chk[2] = o["m"][-1, 0, 0]
        chk[3] = o["status"].max().double()
        if world > 1:
            # the only inter-GPU traffic of a step: ncclAllReduce of 4 doubles, issued by libbdlm.so
            # on the stream the kernels run on
            comm.allreduce_sum_device(chk)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    if picks is not None:  # untimed first gather: a kernel's first launch loads its module
        for i in range(nch):
            keep_sample(i, views(bounds[i + 1] - bounds[i]))
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    timers = []
    launches0 = eng.ctx.launch_count()
    barrier()
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    for it in range(args.steps):
        step(timers, keep=picks is not None and it == args.steps - 1)
    t1.record()
    barrier()
    ms = t0.elapsed_time(t1)
    if kept:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for k in kept[0]:   # [rows][k][sampled series] as the launches return them; status [series]
            a = torch.cat([c[k] for c in kept], dim=-1).cpu().numpy().astype(np.float64)
            if k in ("f", "Q"):  # row 0 is the initial state's placeholder (NaN: no forecast yet)
                a = a[1:]        # so only the T one-step forecasts are written
            np.save(os.path.join(args.dump_outputs, k + ".npy"), a)
        kept.clear()
    launches = eng.ctx.launch_count() - launches0
    clocks = sampler.stop() if sampler else None
    tt = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms = float(tt.item())
    status_max = float(chk[3].item())
    kern_ms = [a.elapsed_time(b) for a, b, _ in timers]
    kern_steps = [bc * T for _, _, bc in timers]
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = sum(kern_steps) * ALGO_BYTES_PER_STEP / (sum(kern_ms) * 1e-3) / 1e9
    value = world * B * T * args.steps / (ms * 1e-3)

    # ---- e2e: same metric through the C ABI with pinned HOST buffers (H2D + D2H timed)
    e2e = None
    if not args.no_e2e:
        Be = args.e2e_series or B
        slab = min(Be, 50_000)
        hy = torch.empty((slab, T, 1), dtype=torch.float64).pin_memory()
        hy.copy_(torch.randn((slab, T, 1), dtype=torch.float64).cumsum(1))
        hV = torch.from_numpy(np.ascontiguousarray(Vs_all[:, :slab].T.copy())).pin_memory()
        hW = torch.from_numpy(np.ascontiguousarray(Ws_all[:, :slab].T.copy())).pin_memory()
        hout = {k: torch.empty((slab, rows, d), dtype=torch.float64).pin_memory() for k, d in dims.items()}
        hout["status"] = torch.empty((slab,), dtype=torch.int32).pin_memory()
        hp = dict(V=hV, W=hW, m0=np.zeros(2), C0=100.0 * np.eye(2), per_series=("V", "W"))
        from bayesian_dlms_b200 import SERIES_MAJOR
        ncall = (Be + slab - 1) // slab

        def e2e_step():
            for _ in range(ncall):
                eng.filter_smooth(model, hp, hy, layout=SERIES_MAJOR, out=hout)

        e2e_step()  # warm-up (arena allocation, page faults)
        barrier()
        w0 = time.perf_counter()
        ksteps = max(1, min(args.steps, 3))
        for _ in range(ksteps):
            e2e_step()
        barrier()
        wall = time.perf_counter() - w0
        wt = torch.tensor([wall], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(wt, op=dist.ReduceOp.MAX)
        wall = float(wt.item())
        h2d = ncall * slab * (T * 8 + 5 * 8)
        d2h = ncall * slab * (rows * sum(dims.values()) * 8 + 4)
        e2e = {"value": world * ncall * slab * T * ksteps / wall, "unit": "series-steps/s",
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": ksteps,
               "host_layout": "series-major [B][T+1][k], pinned", "series_per_call": slab,
               "calls_per_step": ncall,
               "outputs": "full KfState (m,C,a,R,f,Q) + SmoothingState (s,S): 160 B/series-step over PCIe"}
        # PCIe roofline of this leg, measured on the SAME buffers at this N: bare pinned-host
        # copies (torch non_blocking copy_ = one cudaMemcpyAsync each), all ranks at once
        dout = {k: torch.empty((slab, rows, d), device=dev, dtype=torch.float64) for k, d in dims.items()}
        dy = torch.empty((slab, T, 1), device=dev, dtype=torch.float64)

        def bare(direction):
            barrier()
            w0 = time.perf_counter()
            for _ in range(2):
                if direction in ("d2h", "both"):
                    for k in dims:
                        hout[k].copy_(dout[k], non_blocking=True)
                if direction in ("h2d", "both"):
                    dy.copy_(hy, non_blocking=True)
            barrier()
            w = torch.tensor([time.perf_counter() - w0], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(w, op=dist.ReduceOp.MAX)
            nbytes = 0
            if direction in ("d2h", "both"):
                nbytes += slab * rows * sum(dims.values()) * 8
            if direction in ("h2d", "both"):
                nbytes += slab * T * 8
            return 2 * nbytes / float(w.item()) / 1e9    # GB/s per rank, slowest rank

        bare("d2h")
        d2h_peak, h2d_peak = bare("d2h"), bare("h2d")
        del dout, dy
        per_rank_gbs = (h2d + d2h) * ksteps / wall / 1e9
        e2e["roofline"] = {
            "bound": "pcie", "achieved": per_rank_gbs, "peak": d2h_peak, "unit": "GB/s per GPU",
            "frac": per_rank_gbs / d2h_peak,
            "h2d_peak": h2d_peak,
            "peak_source": "bare cudaMemcpyAsync D2H of the same pinned output buffers (8 fields x "
                           "%d series), all %d ranks concurrently, slowest rank" % (slab, world),
            "bytes_per_series_step": (h2d + d2h) / (ncall * slab * T)}
        # the same call asking only for what the reference's SmoothDlm app writes out
        # (smoothed mean and covariance, FirstOrderDlm.scala:248-254): 48 B/series-step D2H
        lean = {k: hout[k] for k in ("s", "S", "status")}
        eng.filter_smooth(model, hp, hy, layout=SERIES_MAJOR, out=lean)
        barrier()
        w0 = time.perf_counter()
        for _ in range(ncall):
            eng.filter_smooth(model, hp, hy, layout=SERIES_MAJOR, out=lean)
        barrier()
        wl = torch.tensor([time.perf_counter() - w0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(wl, op=dist.ReduceOp.MAX)
        e2e["lean_outputs_value"] = world * ncall * slab * T / float(wl.item())
        e2e["lean_outputs"] = "s, S only (what SmoothDlm writes): 48 B/series-step over PCIe"

    scan_dist = loglik_dist = None
    if world > 1 and not args.no_ffbs:  # collective: every rank takes part
        outbuf.clear(); ys.clear(); pars.clear()
        torch.cuda.empty_cache()
        try:
            scan_dist = scan_dist_leg(comm, eng, dev, rank, world)
        except Exception as ex:
            scan_dist = {"error": repr(ex)}
        torch.cuda.empty_cache()
        try:
            loglik_dist = loglik_dist_leg(comm, eng, dev, rank, world)
        except Exception as ex:
            loglik_dist = {"error": repr(ex)}
        torch.cuda.empty_cache()

    if rank == 0:
        line = {
            "metric": "filter+smoother series-steps/s", "value": value, "unit": "series-steps/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "launch_geometry": geometry,
            "gpu_launches": int(launches), "clocks": clocks, "status_max": status_max,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak,
                         # ncu --set full capture of this kernel (profiles/r1_kf_small_full.txt):
                         # dram read + write = 61.298 GB for a 284 160-series launch whose
                         # algorithmic bytes are 61.379 GB -> 0.9987 x algorithmic, scaled here
                         # to this run's average launch
                         "traffic": 0.9987 * ALGO_BYTES_PER_STEP * float(np.mean(kern_steps)) / 1e9,
                         "traffic_unit": "GB per launch",
                         "traffic_source": "NOT measured by this run: ratio from the ncu --set full "
                                           "capture profiles/r1_kf_small_full.txt (kernel as of commit 48f6a5e; "
                                           "61.298 GB measured / 61.379 GB algorithmic for its "
                                           "284160-series launch); kf_small.cu unchanged since",
                         "kernel": "kf_small_kernel<2,true> (fused filter+smoother)",
                         "algorithmic_bytes_per_series_step": ALGO_BYTES_PER_STEP,
                         "launch_ms_avg": float(np.mean(kern_ms)),
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650"},
        }
        if e2e:
            line["e2e"] = e2e
        if not args.no_ffbs and world == 1:
            outbuf.clear(); ys.clear(); pars.clear()  # release the headline buffers (84 GB)
            torch.cuda.empty_cache()
            try:
                line["ffbs"] = ffbs_leg(eng, dev, with_cpu=not args.no_cpu)
            except Exception as ex:  # secondary metric: never take the headline down
                line["ffbs"] = {"error": repr(ex)}
            for key, fn in (("svd_ffbs", svd_leg), ("scan", scan_leg), ("ar_ffbs", ar_leg),
                            ("loglik", loglik_leg), ("ffbs_small", ffbs_small_leg)):
                try:
                    line[key] = fn(eng, dev, with_cpu=not args.no_cpu)
                except Exception as ex:
                    line[key] = {"error": repr(ex)}
                torch.cuda.empty_cache()
            try:
                line["jmh"] = jmh_leg(eng, with_cpu=not args.no_cpu)
            except Exception as ex:
                line["jmh"] = {"error": repr(ex)}
            for key, fn in (("gibbs", gibbs_leg), ("gibbs_wishart", gibbs_wishart_leg)):
                try:
                    line[key] = fn(eng, dev)
                except Exception as ex:
                    line[key] = {"error": repr(ex)}
                torch.cuda.empty_cache()
        if scan_dist is not None:
            line["scan"] = scan_dist
        if loglik_dist is not None:
            line["loglik"] = loglik_dist
        if not args.no_cpu and world >= 1:
            try:
                base, _, _ = cpu_reference_leg(B, T)
                line["cpu_baseline"] = base
            except Exception as ex:  # the baseline leg must never take the bench line down
                line["cpu_baseline"] = {"error": repr(ex)}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

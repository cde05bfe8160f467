"""Device time of the parallel-in-time scan on a dynamic regression (per-step F, f_tv) next to the
time-invariant scan of the same length, and the sequential kernel on the regression series.

    python tools/scan_regression_time.py [--log2T 24] [--reps 5] [--json out.json]

Calls timed (filter + textbook smoother, bdlm_scan_filter_smooth unless named otherwise), n = 2:
  regression, host F     F_t = (1, x_t) as a host [T][n] array, copied to the device by every call
  regression, device F   the same F as a device array (BDLM_PS_F), read in place
  polynomial(2)          the time-invariant scan (level 1 from the model table)
  log-likelihoods        bdlm_scan_loglik of the regression (device F) and of polynomial(2)
  sequential             bdlm_kf_filter_smooth without BDLM_PARALLEL_IN_TIME on the regression
CUDA events around each call on torch's current stream, median of --reps calls after two warm-up
calls (one call for the sequential kernel).  y, F and the workspace exceed L2 at T = 2^24.  Then one
call of each scan under torch.profiler gives its device time per kernel.  The card's name, power
limit and maximum SM clock are read in the same run (nvidia-smi, read-only query)."""
import argparse
import json
import os
import re
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        return out.splitlines()[1] if len(out.splitlines()) > 1 else out
    except (OSError, subprocess.SubprocessError) as e:
        return "nvidia-smi unavailable (%s)" % e


def median_ms(fn, reps, warm=2):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def kernel_ms(fn):
    """Device time per kernel (template arguments dropped) of one call."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        name = re.sub(r"<.*", "", ev.name.replace("(anonymous namespace)::", "")).split("(")[0].split("::")[-1]
        out[name] = out.get(name, 0.0) + ev.device_time / 1e3  # us -> ms
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2T", type=int, default=24)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    import torch
    from bayesian_dlms_b200 import Engine, Model, TIME_MAJOR, dlm
    from bayesian_dlms_b200.scan import scan_filter_smooth, scan_loglik
    T = 1 << args.log2T
    eng = Engine(0)
    eng.use_torch_stream()
    rng = np.random.default_rng(1)
    # regression with one covariate: beta_t a random walk (G = I), y_t = beta_t . (1, x_t) + v_t
    x = rng.standard_normal(T)
    F = np.ascontiguousarray(np.column_stack([np.ones(T), x]))
    W = np.diag([0.05, 0.01])
    beta = np.cumsum(rng.standard_normal((T, 2)) * np.sqrt(np.diag(W)), axis=0)
    y = np.einsum("ti,ti->t", F, beta) + rng.standard_normal(T)
    y[rng.random(T) < 0.01] = np.nan
    params = dict(V=np.array([[1.0]]), W=W, m0=np.zeros(2), C0=10.0 * np.eye(2))
    yd = torch.from_numpy(y).cuda()
    reg_host = Model(F.ravel(), dlm.cm(np.eye(2)), True, False, 2, 1, T, None)
    reg_dev = Model(torch.from_numpy(F).cuda(), dlm.cm(np.eye(2)), True, False, 2, 1, T, None, None, ("F",))
    poly = Model.build(dlm.polynomial(2), T=16)
    poly = Model(poly.F, poly.G, False, False, 2, 1, T, None)
    calls = {
        "scan filter+smoother, regression, host F": lambda: scan_filter_smooth(eng, reg_host, params, yd),
        "scan filter+smoother, regression, device F": lambda: scan_filter_smooth(eng, reg_dev, params, yd),
        "scan filter+smoother, polynomial(2)": lambda: scan_filter_smooth(eng, poly, params, yd),
        "scan log-likelihoods, regression, device F": lambda: scan_loglik(eng, reg_dev, params, yd),
        "scan log-likelihoods, polynomial(2)": lambda: scan_loglik(eng, poly, params, yd),
    }
    res = dict(card=card(), T=T, n=2, missing=0.01, reps=args.reps, ms={}, kernels_ms={})
    print("card:", res["card"])
    for name, fn in calls.items():
        res["ms"][name] = median_ms(fn, args.reps)
        print("%-48s %10.3f ms" % (name, res["ms"][name]))
    y3 = yd.reshape(T, 1, 1)
    seq = lambda: eng.filter_smooth(reg_host, params, y3, layout=TIME_MAJOR, textbook=True)  # noqa: E731
    res["ms"]["sequential filter+smoother, regression"] = median_ms(seq, 1, warm=0)
    print("%-48s %10.3f ms" % ("sequential filter+smoother, regression", res["ms"]["sequential filter+smoother, regression"]))
    for name in ("scan filter+smoother, regression, device F", "scan filter+smoother, polynomial(2)"):
        res["kernels_ms"][name] = kernel_ms(calls[name])
        print(name + ":")
        for k, v in res["kernels_ms"][name].items():
            print("    %-36s %9.3f ms" % (k, v))
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()

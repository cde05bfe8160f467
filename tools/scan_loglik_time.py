"""Device time of the parallel-in-time log-likelihood (bdlm_scan_loglik) for one long series, next to
the scan's filter + smoother (bdlm_scan_filter_smooth) at the same shape and the sequential
thread-per-series bdlm_loglik at B = 1.

    python tools/scan_loglik_time.py [--reps 7] [--seq-max-log2 20] [--json out.json]

CUDA events around each call on torch's current stream, median of --reps calls after two warm-up
calls per shape.  y (8 B per step) and the scan's workspace exceed L2 from T = 2^22 on.  The card's
name, power limit and maximum SM clock are read in the same run (nvidia-smi, read-only query)."""
import argparse
import json
import os
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


def model(n):
    from bayesian_dlms_b200 import dlm
    mod = {1: dlm.polynomial(1), 2: dlm.polynomial(2), 4: dlm.polynomial(2) + dlm.seasonal(7, 1)}[n]
    W = np.diag(np.linspace(0.5, 1.0, n))
    return mod, dict(V=np.array([[2.0]]), W=W, m0=np.ones(n), C0=10.0 * np.eye(n))


def median_ms(fn, reps):
    import torch
    for _ in range(2):
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--seq-max-log2", type=int, default=20)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    import torch
    from bayesian_dlms_b200 import Engine, Model, TIME_MAJOR
    from bayesian_dlms_b200.scan import scan_filter_smooth, scan_loglik
    assert torch.cuda.is_available(), "needs a GPU"
    print("card (name, power limit, max SM clock):", card())
    eng = Engine(0)
    rows = []
    print("%3s %6s %12s %16s %14s %10s %10s" % ("n", "log2T", "loglik ms", "filt+smooth ms", "sequential ms",
                                                "ll/fs", "seq/ll"))
    for n in (1, 2, 4):
        mod, params = model(n)
        for lg in (20, 22, 24):
            T = 1 << lg
            rng = np.random.default_rng(lg + n)
            y = np.cumsum(rng.standard_normal(T)) + rng.standard_normal(T)
            y[rng.random(T) < 0.01] = np.nan
            yd = torch.from_numpy(y).cuda()
            md = Model.build(mod, T=T)
            ll = median_ms(lambda: scan_loglik(eng, md, params, yd, last=True), args.reps)
            fs = median_ms(lambda: scan_filter_smooth(eng, md, params, yd), args.reps)
            seq = None
            if lg <= args.seq_max_log2:
                y3 = yd.reshape(T, 1, 1)
                seq = median_ms(lambda: eng.loglik(md, params, y3, layout=TIME_MAJOR), max(5, args.reps // 2))
            rows.append(dict(n=n, log2T=lg, loglik_ms=ll, filter_smooth_ms=fs, sequential_ms=seq))
            print("%3d %6d %12.3f %16.3f %14s %10.3f %10s" % (n, lg, ll, fs, "%.1f" % seq if seq else "-", ll / fs,
                                                           "%.0f" % (seq / ll) if seq else "-"))
            del yd
            torch.cuda.empty_cache()
    if args.json:
        with open(args.json, "w") as f:
            json.dump(dict(card=card(), rows=rows), f, indent=1)


if __name__ == "__main__":
    main()

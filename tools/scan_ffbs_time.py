"""Device time of the parallel-in-time FFBS (bdlm_scan_ffbs) for one long series -- with and without
the Gibbs statistics, with injected normals and with Philox normals -- next to the scan's filter +
smoother (bdlm_scan_filter_smooth) at the same shape, the opt-in bdlm_ffbs (BDLM_PARALLEL_IN_TIME)
and the sequential thread-per-chain bdlm_ffbs at B = 1 (2^20 only by default: it walks T dependent
steps forward and back on one thread).

    python tools/scan_ffbs_time.py [--reps 7] [--seq-max-log2 20] [--json out.json]

CUDA events around each call on torch's current stream, median of --reps calls after two warm-up
calls per shape.  y, z, theta and the (m, C) spill exceed L2 from T = 2^22 on.  The card's name,
power limit and maximum SM clock are read in the same run (nvidia-smi, read-only query)."""
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
    from bayesian_dlms_b200.scan import scan_ffbs, scan_filter_smooth
    assert torch.cuda.is_available(), "needs a GPU"
    print("card (name, power limit, max SM clock):", card())
    eng = Engine(0)
    eng.ctx.set_rng(11, 0, 0)
    rows = []
    cols = ("ffbs+stats z", "ffbs+stats philox", "ffbs z", "filt+smooth", "opt-in ffbs", "sequential")
    print("%3s %6s" % ("n", "log2T") + "".join("%19s" % c for c in cols) + "%10s %10s" % ("ffbs/fs", "seq/opt"))
    for n in (1, 2, 4):
        mod, params = model(n)
        for lg in (20, 22, 24):
            T = 1 << lg
            rng = np.random.default_rng(lg + n)
            y = np.cumsum(rng.standard_normal(T)) + rng.standard_normal(T)
            y[rng.random(T) < 0.01] = np.nan
            yd = torch.from_numpy(y).cuda()
            zd = torch.from_numpy(rng.standard_normal((T + 1, n))).cuda()
            md = Model.build(mod, T=T)
            r = dict(n=n, log2T=lg)
            r["ffbs_stats_z_ms"] = median_ms(lambda: scan_ffbs(eng, md, params, yd, zd), args.reps)
            r["ffbs_stats_philox_ms"] = median_ms(lambda: scan_ffbs(eng, md, params, yd), args.reps)
            r["ffbs_z_ms"] = median_ms(lambda: scan_ffbs(eng, md, params, yd, zd, stats=False), args.reps)
            r["filter_smooth_ms"] = median_ms(lambda: scan_filter_smooth(eng, md, params, yd), args.reps)
            r["opt_in_ms"] = r["sequential_ms"] = None
            if lg <= args.seq_max_log2:
                y3, z3 = yd.reshape(T, 1, 1), zd.reshape(T + 1, n, 1)
                r["opt_in_ms"] = median_ms(lambda: eng.ffbs(md, params, y3, z3, layout=TIME_MAJOR, stats=True,
                                                            parallel_in_time=True), args.reps)
                r["sequential_ms"] = median_ms(lambda: eng.ffbs(md, params, y3, z3, layout=TIME_MAJOR, stats=True),
                                               max(3, args.reps // 2))
            rows.append(r)
            v = [r["ffbs_stats_z_ms"], r["ffbs_stats_philox_ms"], r["ffbs_z_ms"], r["filter_smooth_ms"],
                 r["opt_in_ms"], r["sequential_ms"]]
            print("%3d %6d" % (n, lg) + "".join("%19s" % ("%.3f" % x if x is not None else "-") for x in v) +
                  "%10.2f %10s" % (v[0] / v[3], "%.0f" % (v[5] / v[4]) if v[5] else "-"))
            del yd, zd
            torch.cuda.empty_cache()
    if args.json:
        with open(args.json, "w") as f:
            json.dump(dict(card=card(), rows=rows), f, indent=1)


if __name__ == "__main__":
    main()

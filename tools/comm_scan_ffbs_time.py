"""Device time of the time-sharded log-likelihoods and FFBS of one long series, in three forms:

* the single-GPU calls (bdlm_scan_loglik, bdlm_scan_ffbs with statistics) of the whole series;
* the communicator calls (bdlm_comm_scan_loglik / _ffbs) on a world-1 communicator: the same work
  plus the phases' extra launches and the NCCL all-gathers on one rank;
* emulated ranks: --emulate contexts on ONE GPU run the bdlm_scan_dist_* phases of their chunks,
  the all-gathers done by device concatenations.  That is the sum of the ranks' work on one device,
  not an N-GPU time.

    python tools/comm_scan_ffbs_time.py [--reps 7] [--emulate 8] [--json out.json]

CUDA events around each call on torch's current stream (every context is put on it), median of
--reps calls after two warm-up calls, n = 1, 2, 4 at T = 2^20 and 2^24.  With several GPUs the
communicator form runs over all of them and the time is the largest over the devices.  The card's
name, power limit and maximum SM clock are read in the same run (nvidia-smi, read-only query)."""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from scan_ffbs_time import card, median_ms, model  # noqa: E402


def comm_ms(comm, fn, reps):
    """Median over reps of the largest per-device event time of one communicator call."""
    import torch
    devs = comm.devices
    for _ in range(2):
        fn()
    comm.sync()
    ts = []
    for _ in range(reps):
        ev = []
        for d in devs:
            with torch.cuda.device(d):
                a = torch.cuda.Event(enable_timing=True)
                a.record()
                ev.append(a)
        fn()
        t = 0.0
        for d, a in zip(devs, ev):
            with torch.cuda.device(d):
                b = torch.cuda.Event(enable_timing=True)
                b.record()
                b.synchronize()
                t = max(t, a.elapsed_time(b))
        ts.append(t)
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--emulate", type=int, default=8)
    ap.add_argument("--log2", type=int, nargs="*", default=[20, 24])
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    import torch
    from bayesian_dlms_b200 import Engine, Model
    from bayesian_dlms_b200.comm import Comm
    from bayesian_dlms_b200.scan import DistFfbs, DistLoglik, scan_ffbs, scan_loglik
    from bayesian_dlms_b200.sharding import time_chunk
    assert torch.cuda.is_available(), "needs a GPU"
    info = card()
    print("card (name, power limit, max SM clock):", info)
    ngpu = torch.cuda.device_count()
    eng = Engine(0)
    eng.use_torch_stream()
    eng.ctx.set_rng(11, 0, 0)
    comm = Comm.single_process(list(range(ngpu)))
    for e in comm.engines:
        with torch.cuda.device(e.device):
            e.use_torch_stream()
        e.ctx.set_rng(11, 0, 0)
    rows = []
    cols = ("loglik 1 GPU", "loglik comm", "loglik emul", "ffbs 1 GPU", "ffbs comm", "ffbs emul")
    print("%3s %6s" % ("n", "log2T") + "".join("%15s" % c for c in cols))
    for n in (1, 2, 4):
        mod, params = model(n)
        for lg in args.log2:
            T = 1 << lg
            rng = np.random.default_rng(lg + n)
            y = np.cumsum(rng.standard_normal(T)) + rng.standard_normal(T)
            y[rng.random(T) < 0.01] = np.nan
            yd = torch.from_numpy(y).cuda()
            md = Model.build(mod, T=T)
            r = dict(n=n, log2T=T.bit_length() - 1, gpus=ngpu, emulated_ranks=args.emulate)
            r["loglik_one_ms"] = median_ms(lambda: scan_loglik(eng, md, params, yd, last=True), args.reps)
            r["ffbs_one_ms"] = median_ms(lambda: scan_ffbs(eng, md, params, yd), args.reps)
            # communicator over every GPU of the box, one chunk per device
            models, chunks, firsts = [], [], []
            for i, d in enumerate(comm.devices):
                lo, hi, first = time_chunk(T, i, comm.world)
                models.append(Model.build(mod, T=hi - lo))
                chunks.append(yd[lo:hi].to(f"cuda:{d}").contiguous())
                firsts.append(first)
            h = comm.scan_setup(models, params, chunks)
            r["loglik_comm_ms"] = comm_ms(comm, lambda: comm.scan_loglik(h), args.reps)
            r["ffbs_comm_ms"] = comm_ms(comm, lambda: comm.scan_ffbs(h, firsts, T), args.reps)
            del h, chunks
            # emulated ranks on device 0
            W = args.emulate
            ll, fb = [], []
            for k in range(W):
                lo, hi, first = time_chunk(T, k, W)
                e = Engine(0)
                e.use_torch_stream()
                e.ctx.set_rng(11, 0, 0)
                mk = Model.build(mod, T=hi - lo)
                yk = yd[lo:hi].contiguous()
                ll.append(DistLoglik(e, mk, params, yk, k, W))
                fb.append(DistFfbs(e, mk, params, yk, k, W, first, T))

            def gather(ranks, src, dst):
                g = torch.cat([getattr(d, src) for d in ranks])
                for d in ranks:
                    getattr(d, dst).copy_(g)

            def run_ll():
                for d in ll:
                    d.forward_local()
                gather(ll, "agg_f", "aggs_f")
                for d in ll:
                    d.partial()
                gather(ll, "part", "parts")
                for d in ll:
                    d.finish()

            def run_fb():
                for d in fb:
                    d.forward_local()
                gather(fb, "agg_f", "aggs_f")
                for d in fb:
                    d.local()
                gather(fb, "agg_s", "aggs_s")
                for d in fb:
                    d.finish()
                gather(fb, "part", "parts")
                for d in fb:
                    d.stats_finish()
            r["loglik_emulated_ms"] = median_ms(run_ll, args.reps)
            r["ffbs_emulated_ms"] = median_ms(run_fb, args.reps)
            del ll, fb
            rows.append(r)
            v = [r["loglik_one_ms"], r["loglik_comm_ms"], r["loglik_emulated_ms"], r["ffbs_one_ms"],
                 r["ffbs_comm_ms"], r["ffbs_emulated_ms"]]
            print("%3d %6d" % (n, lg) + "".join("%15.3f" % x for x in v))
            del yd
            torch.cuda.empty_cache()
    comm.close()
    if args.json:
        with open(args.json, "w") as f:
            json.dump(dict(card=info, rows=rows), f, indent=1)


if __name__ == "__main__":
    main()

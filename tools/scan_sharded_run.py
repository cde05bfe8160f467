"""Config 5 on N GPUs: ONE series, time-sharded across ranks (run under torchrun).

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port 29517 tools/scan_sharded_run.py --logT 24

Each rank owns a contiguous time chunk and runs the device-side phases (DistScan); the only
inter-GPU traffic is the all-gather of one scan aggregate per rank and pass (3n^2+2n / 2n^2+n
doubles).  Checks the sharded result against the single-GPU scan and prints one JSON line
(time = max over ranks, device events).
"""
import argparse, json, os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bayesian_dlms_b200 import Engine, Model, dlm
from bayesian_dlms_b200.scan import DistScan, scan_filter_smooth
from bayesian_dlms_b200.sharding import shard_range

ap = argparse.ArgumentParser(); ap.add_argument("--logT", type=int, default=24); ap.add_argument("--reps", type=int, default=5)
a = ap.parse_args()
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
dev = torch.device("cuda", local)
eng = Engine(local); eng.use_torch_stream()
T, n = 1 << a.logT, 2
mod = dlm.polynomial(2)
params = dict(V=[[3.0]], W=np.diag([2.0, 1.0]), m0=np.zeros(2), C0=100.0 * np.eye(2))
g = torch.Generator(device=dev).manual_seed(20260105)      # same series on every rank
y = torch.randn(T, generator=g, device=dev, dtype=torch.float64).cumsum(0) * 0.1
lo, hi = shard_range(T, rank, world)
yc = y[lo:hi].contiguous()
cmodel = Model.build(mod, T=hi - lo)     # flattened once, outside the timed region
run = DistScan(eng, cmodel, params, yc, rank, world).run
out = run()   # warm-up (NCCL communicator, arena, table)
out = run()
torch.cuda.synchronize(); dist.barrier()
ms = []
for _ in range(a.reps):
    dist.barrier(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); out = run(); e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms.append(float(t.item()))
# parity against the single-GPU scan of the whole series (each rank checks its own chunk)
full = scan_filter_smooth(eng, Model.build(mod, T=T), params, y)
torch.cuda.synchronize()
r0 = lo + (0 if rank == 0 else 1)         # row offset of this chunk inside the T + 1 rows
err = 0.0
for k in ("m", "C", "s", "S", "a", "R"):
    ref = full[k][r0:r0 + out[k].shape[0]]
    den = ref.abs().clamp_min(1e-6 * float(ref.abs().max()))
    err = max(err, float(((out[k] - ref).abs() / den).max()))
e = torch.tensor([err], device=dev, dtype=torch.float64); dist.all_reduce(e, op=dist.ReduceOp.MAX)
if rank == 0:
    med = float(np.median(ms))
    print(json.dumps({"config": "config5 sharded: one series T=2^%d over %d GPUs (time chunks)" % (a.logT, world),
                      "n_gpus": world, "ms": med, "steps_per_s": T / med * 1e3,
                      "max_rel_err_vs_single_gpu": float(e.item())}))
dist.barrier(); dist.destroy_process_group()

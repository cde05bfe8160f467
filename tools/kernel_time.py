"""Time the fused filter+smoother register kernel alone at an exact number of waves.

    [BDLM_LIB_PATH=variants/libbdlm_x.so] python tools/kernel_time.py [--waves 3] [--n 2] [--T 1000]
        [--seg 4] [--per-series-g]

--seg K: the library's kSeg (kf_small.cu), for the byte count only: with K > 0 the fused kernel
for n <= 2 reads back one (m, C) row in K and y again for the others; --seg 0 counts the full
(m, C) re-read of a library without the recompute (and of n > 2).
--per-series-g (n = 2): every series on its own irregular grid with G(dt) = [[1, dt], [0, 1]], so
the kernel loads dt and G per series and step (the non-REG path); those loads are not counted.
"""
import argparse
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bayesian_dlms_b200 import Engine, Model, dlm  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--waves", type=float, default=3)
ap.add_argument("--n", type=int, default=2)
ap.add_argument("--T", type=int, default=1000)
ap.add_argument("--iters", type=int, default=5)
ap.add_argument("--lean", action="store_true")
ap.add_argument("--seg", type=int, default=4)
ap.add_argument("--per-series-g", action="store_true")
a = ap.parse_args()
eng = Engine(0)
n, T = a.n, a.T
wave = eng.ctx.wave_series(n, 1)
B = int(a.waves * wave)
dev = torch.device("cuda", 0)
y = torch.randn((T, 1, B), device=dev, dtype=torch.float64).cumsum(0)
Vs = (3.0 * torch.exp(torch.rand((1, B), device=dev, dtype=torch.float64) - 0.5)).contiguous()
W0 = np.diag(np.linspace(2.0, 1.0, n)) if n > 1 else np.array([[3.0]])
Ws = (torch.from_numpy(dlm.cm(W0)).to(dev)[:, None] *
      torch.exp(torch.rand((1, B), device=dev, dtype=torch.float64) - 0.5)).contiguous()
params = dict(V=Vs, W=Ws, m0=np.zeros(n), C0=100.0 * np.eye(n), per_series=("V", "W"))
model = Model.build(dlm.polynomial(n), T=T)
if a.per_series_g:
    assert n == 2, "--per-series-g builds a 2-state trend"
    g = torch.Generator(device=dev).manual_seed(1)
    dts = torch.randint(0, 4, (T, 1, B), generator=g, device=dev).double() * 0.5  # dt = 0 included
    dts[0] = 1.0                                    # first dt = 1 (times start at min - 1)
    times = dts.cumsum(0)
    G = torch.zeros((T, 4, B), device=dev, dtype=torch.float64)
    G[:, 0], G[:, 2], G[:, 3] = 1.0, dts[:, 0], 1.0  # column-major [[1, dt], [0, 1]]
    model = Model(np.array([1.0, 0.0]), G, False, True, 2, 1, T, times, None, ("times", "G"))
dims = dict(m=n, C=n * n, a=n, R=n * n, f=1, Q=1, s=n, S=n * n)
if a.lean:
    dims = dict(m=n, C=n * n, s=n, S=n * n)
out = {k: torch.empty((T + 1, d, B), device=dev, dtype=torch.float64) for k, d in dims.items()}
out["status"] = torch.empty((B,), device=dev, dtype=torch.int32)
for _ in range(2):
    eng.filter_smooth(model, params, y, out=out)
torch.cuda.synchronize()
ms = []
for _ in range(a.iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    eng.filter_smooth(model, params, y, out=out)
    e1.record()
    torch.cuda.synchronize()
    ms.append(e0.elapsed_time(e1))
# y + outputs, then what the backward pass reads back (see --seg)
back = (n + n * n + a.seg - 1) / a.seg if n <= 2 and a.seg > 0 else n + n * n
byt = 8 * (1 + sum(dims.values()) + back)
best, med = min(ms), float(np.median(ms))
print(f"lib={os.environ.get('BDLM_LIB_PATH', 'default')} n={n} wave={wave} B={B} T={T} "
      f"{'per-series G ' if a.per_series_g else ''}"
      f"bytes/step={byt:g} median={med:.3f} ms best={best:.3f} ms  "
      f"{B * T / med / 1e6:.2f} G steps/s  {B * T * byt / med / 1e6:.0f} GB/s (median) "
      f"{B * T * byt / best / 1e6:.0f} GB/s (best) status_max={int(out['status'].max())}")

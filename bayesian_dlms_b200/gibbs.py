"""Device-resident Gibbs sampling for batches of independent chains / series.

Mirrors ``GibbsSampling.sample`` / ``sampleSvd`` (Gibbs.scala:134-217: FFBS, then the conjugate
inverse-gamma draws of diag(V) and diag(W)) and ``GibbsWishart.sample`` (GibbsWishart.scala:40-80:
FFBS, inverse-Wishart draw of W, inverse-gamma draw of diag(V)).  One sweep is three launches
on one stream -- FFBS kernel with fused sufficient statistics, the draw kernel(s) -- and nothing
returns to the host between sweeps: the drawn V, W are written as per-series parameter arrays
that the next sweep's FFBS reads directly.
"""
from __future__ import annotations

from typing import Dict, Optional

from . import _capi as capi
from .batch import Engine, Model, TIME_MAJOR


def sample(eng: Engine, model: Model, y, prior: Dict, init: Dict, n_iters: int, *, seed: int = 0,
           layout=TIME_MAJOR, svd: bool = False, record: bool = True,
           z: Optional[object] = None, first_series: int = 0, parallel_in_time: bool = False) -> Dict:
    """Run ``n_iters`` Gibbs sweeps for every chain of the batch.

    y       CUDA tensor, (T, p, B) time-major or (B, T, p) series-major; NaN = missing
    prior   dict(v_shape, v_scale, and w_shape, w_scale  or  w_nu, w_psi)
    init    dict(V, W, m0, C0): initial DlmParameters shared by all chains (numpy)
    z       optional pre-drawn normals (n_iters, *theta-shape) for bit-exact comparisons;
            default: the FFBS kernels draw their own (Philox keyed by (seed, sweep)), so no
            normals are materialised in HBM at all
    parallel_in_time
            ONE long series (B = 1) may draw its path with the scan's sampler (include/bdlm.h
            BDLM_PARALLEL_IN_TIME; ignored where the problem is not eligible).  The scan builds
            its model table on the host from shared parameters, so each sweep hands the drawn
            V and W to the next FFBS as host arrays: p*p + n*n doubles copied back and one host
            synchronisation per sweep, instead of the device-resident per-series parameters
    Returns dict(V=(iters, p, B) diagonals, W=(iters, n or n*n, B), theta=last path, status=...)
    in time-major orientation regardless of ``layout`` for the recorded chains.
    """
    import torch
    n, p, T = model.n, model.p, model.T
    B = y.shape[2] if layout == TIME_MAJOR else y.shape[0]
    wishart = prior.get("w_psi") is not None
    params = dict(init)
    chain_v = torch.empty((n_iters, p, B), dtype=torch.float64, device=y.device) if record else None
    wk = n * n if wishart else n
    chain_w = torch.empty((n_iters, wk, B), dtype=torch.float64, device=y.device) if record else None
    bad = torch.zeros((B,), dtype=torch.int32, device=y.device)
    draw_out = None
    out = None
    pit = parallel_in_time and B == 1 and not svd
    vdiag = torch.arange(p, device=y.device) * (p + 1)
    wdiag = torch.arange(n, device=y.device) * (n + 1)
    for it in range(n_iters):
        zi = z[it] if z is not None else None
        eng.ctx.set_rng(seed, it, first_series)  # ranks sharding the chains pass their offset
        out = eng.ffbs(model, params, y, zi, layout=layout, stats=True, status=True, svd=svd,
                       parallel_in_time=pit)
        draw_out = eng.gibbs_draw(n, p, T, out, prior, layout=layout, seed=seed, sweep=it,
                                  out=draw_out)
        bad |= out["status"] | draw_out["status"]
        if pit:  # shared host parameters: the scan's model table is built from them
            params = dict(V=draw_out["V"].reshape(p, p).T.cpu().numpy(),
                          W=draw_out["W"].reshape(n, n).T.cpu().numpy(), m0=init["m0"], C0=init["C0"])
        else:
            params = dict(V=draw_out["V"], W=draw_out["W"], m0=init["m0"], C0=init["C0"],
                          per_series=("V", "W"))
        if record:
            V = draw_out["V"] if layout == TIME_MAJOR else draw_out["V"].t()
            W = draw_out["W"] if layout == TIME_MAJOR else draw_out["W"].t()
            chain_v[it] = V[vdiag]
            chain_w[it] = W if wishart else W[wdiag]
    return dict(V=chain_v, W=chain_w, theta=out["theta"] if out else None, status=bad,
                last_params=params)

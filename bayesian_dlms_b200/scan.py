"""Parallel-in-time Kalman filter + smoother for ONE long series (BASELINE config 5).

Not in the reference (strictly sequential recursion, Filter.scala:41-62); temporal
parallelisation by associative scan (Sarkka & Garcia-Fernandez 2021), kernels in csrc/scan.cu.
``scan_filter_smooth`` is the single-GPU call, ``scan_loglik`` the log-likelihoods and last
filtered state by the forward pass alone, ``scan_ffbs`` a backward-sampled path with its Gibbs
statistics; ``DistScan`` runs one rank's time chunk of a
sharded series with the device-side phases (one all-gather of a 3n^2+2n-double aggregate per rank
for the filter, 2n^2+n for the smoother), ``DistLoglik`` and ``DistFfbs`` the log-likelihoods and
FFBS of such a chunk (``sharding.time_chunk`` gives each rank its observations and first row).

A model with a per-step F (``f_tv``: dynamic regression, F_t = (1, x_t)) runs on every one of these
calls: ``model.F`` (T, n) on the host is copied to the device with each call, or, with
``model.per_series = ("F",)``, a CUDA tensor of T * n doubles is read in place.  A chunk's model
holds the F rows of its own observations.
"""
from __future__ import annotations

from typing import Dict

import numpy as np

from . import _capi as capi
from . import dlm as _dlm
from .batch import Engine, Model, SERIES_MAJOR, _mem_and_ptr, bound_engine


def _problem(model: Model, params: Dict, y, keep_init: bool):
    assert model.p == 1 and model.n <= 4 and model.times is None and not model.g_tv
    assert tuple(model.per_series) in ((), ("F",)) and (model.f_tv or not model.per_series)
    keep = [_dlm.cm(np.atleast_2d(np.asarray(params["V"], float))),
            _dlm.cm(np.atleast_2d(np.asarray(params["W"], float))),
            np.ascontiguousarray(np.asarray(params["m0"], float).ravel()),
            _dlm.cm(np.atleast_2d(np.asarray(params["C0"], float)))]
    mem, yptr = _mem_and_ptr(y)
    assert mem == capi.DEVICE, "scan path takes device-resident y"
    F, per = model.F, 0
    if model.per_series:  # device F [T][n], read in place
        assert model.F.numel() == model.T * model.n, tuple(model.F.shape)
        fmem, F = _mem_and_ptr(model.F)
        assert fmem == capi.DEVICE, "per-series F lives with y on the device"
        per = capi.PS_F
    elif model.f_tv:  # host F [T][n]
        F = np.ascontiguousarray(np.asarray(model.F, float).reshape(model.T, model.n))
        keep.append(F)
    pr = capi.make_problem(B=1, T=model.T, n=model.n, p=1, layout=SERIES_MAJOR, mem=capi.DEVICE,
                           keep_init=keep_init, F=F, G=model.G, times=None, V=keep[0],
                           W=keep[1], m0=keep[2], C0=keep[3], y=yptr, per_series=per, f_tv=model.f_tv)
    return pr, keep


_FIELDS = ("m", "C", "a", "R", "f", "Q", "s", "S")


def _outputs(like, rows: int, n: int, want=_FIELDS):
    """[rows, k] float64 tensors on ``like``'s device for the fields in ``want``, and the
    ``KfOut`` / ``SmoothOut`` structs that point at them (NULL for the fields left out)."""
    import torch
    dims = dict(m=n, C=n * n, a=n, R=n * n, f=1, Q=1, s=n, S=n * n)
    out = {k: torch.empty((rows, dims[k]), dtype=torch.float64, device=like.device) for k in want}
    ko, so = capi.KfOut(), capi.SmoothOut()
    for k in ("m", "C", "a", "R", "f", "Q"):
        setattr(ko, k, out[k].data_ptr() if k in out else None)
    for k in ("s", "S"):
        setattr(so, k, out[k].data_ptr() if k in out else None)
    return out, ko, so


def scan_filter_smooth(eng: Engine, model: Model, params: Dict, y, *, keep_init=True, want=_FIELDS):
    """y: CUDA tensor [T] (or [T, 1]).  Returns [rows, k] tensors (+ int status)."""
    import torch
    with bound_engine(eng):
        pr, keep = _problem(model, params, y, keep_init)
    out, ko, so = _outputs(y, model.T + int(keep_init), model.n, want)
    st = torch.zeros((1,), dtype=torch.int32, device=y.device)
    eng.ctx.check(capi.load().bdlm_scan_filter_smooth(eng.ctx.handle, pr, ko, so, st.data_ptr()))
    out["status"] = st
    return out


def scan_loglik(eng: Engine, model: Model, params: Dict, y, *, transition=True, innovations=True,
                last=False):
    """Both log-likelihoods (as ``Engine.loglik``) and, with ``last``, the final filtered state
    (as ``Engine.filter_last``) of ONE long series by the scan's forward pass (bdlm_scan_loglik).
    y: CUDA tensor [T] (or [T, 1]).  Returns [1] / [n] / [n*n] device tensors + int32 status [1]."""
    import torch
    with bound_engine(eng):
        pr, keep = _problem(model, params, y, True)
    n = model.n
    z = lambda k: torch.empty((k,), dtype=torch.float64, device=y.device)  # noqa: E731
    out = {}
    if transition:
        out["transition"] = z(1)
    if innovations:
        out["innovations"] = z(1)
    if last:
        out["m"], out["C"] = z(n), z(n * n)
    ptr = lambda k: out[k].data_ptr() if k in out else None  # noqa: E731
    st = torch.zeros((1,), dtype=torch.int32, device=y.device)
    eng.ctx.check(capi.load().bdlm_scan_loglik(eng.ctx.handle, pr, ptr("m"), ptr("C"), ptr("transition"),
                                               ptr("innovations"), st.data_ptr()))
    out["status"] = st
    return out


def scan_ffbs(eng: Engine, model: Model, params: Dict, y, z=None, *, stats=True, want_kf=()):
    """Smoothing.ffbsDlm of ONE long series by the scan (bdlm_scan_ffbs): the path theta [T+1, n],
    with ``stats`` the Gibbs statistics ssy [1], ny [1], ssw [n], scatter [n*n] of it, and the
    filter fields named in ``want_kf`` [T+1, k].  y: CUDA tensor [T] (or [T, 1]); z: CUDA tensor
    [T+1, n] of injected normals, or None for the Philox normals of ``eng.ctx.set_rng`` (the values
    the sequential ``Engine.ffbs`` consumes).  Adds the int32 status [1]."""
    import torch
    with bound_engine(eng):
        pr, keep = _problem(model, params, y, True)
    n, rows = model.n, model.T + 1
    assert z is None or (tuple(z.shape) == (rows, n) and _mem_and_ptr(z)[0] == capi.DEVICE), z.shape
    out, ko, _ = _outputs(y, rows, n, want_kf)
    out["theta"] = torch.empty((rows, n), dtype=torch.float64, device=y.device)
    gs = capi.GibbsStats()
    if stats:
        for k, d in (("ssy", 1), ("ny", 1), ("ssw", n), ("scatter", n * n)):
            out[k] = torch.empty((d,), dtype=torch.float64, device=y.device)
            setattr(gs, k, out[k].data_ptr())
    st = torch.zeros((1,), dtype=torch.int32, device=y.device)
    eng.ctx.check(capi.load().bdlm_scan_ffbs(eng.ctx.handle, pr, None if z is None else z.data_ptr(),
                                             out["theta"].data_ptr(), ko, gs if stats else None, st.data_ptr()))
    out["status"] = st
    return out


def elem_doubles(n: int, backward: bool) -> int:
    return int(capi.load().bdlm_scan_elem_doubles(n, int(backward)))


def dist_doubles(n: int, what: int) -> int:
    """Sizes of the time-sharded loglik / FFBS exchanges (capi.SCAN_DIST_*)."""
    return int(capi.load().bdlm_scan_dist_doubles(n, what))


class _DistChunk:
    """One rank's chunk of a time-sharded series: the problem struct, the forward local phase and
    the exchange buffers [size] -> [world * size] of the phases that follow it."""

    def __init__(self, eng: Engine, model: Model, params: Dict, y_chunk, rank: int, world: int):
        self.eng, self.rank, self.world, self.n = eng, rank, world, model.n
        self.model, self.y = model, y_chunk   # the problem struct points into model.F / model.G
        self.keep_init = rank == 0
        self.rows = model.T + int(self.keep_init)
        with bound_engine(eng):
            self.pr, self._keep = _problem(model, params, y_chunk, self.keep_init)
        self.agg_f, self.aggs_f = self._xch(elem_doubles(self.n, False))

    def _xch(self, size):
        import torch
        z = lambda k: torch.zeros(k, dtype=torch.float64, device=self.y.device)  # noqa: E731
        return z(size), z(self.world * size)

    def _ck(self, rc):
        self.eng.ctx.check(rc)

    def forward_local(self):
        self._ck(capi.load().bdlm_scan_dist_forward_local(self.eng.ctx.handle, self.pr, self.rank,
                                                          self.world, self.agg_f.data_ptr()))

    @staticmethod
    def _gather(all_gather_into):
        if all_gather_into is None:
            import torch.distributed as dist
            all_gather_into = dist.all_gather_into_tensor
        return all_gather_into


class DistScan(_DistChunk):
    """Time-sharded scan of ONE series over ``world`` GPUs with no host round trip
    (``bdlm_scan_dist_*``): per pass one all-gather of a 3n^2+2n (filter) / 2n^2+n (smoother)
    double aggregate per rank, issued on the engine's stream between the local and the finish
    kernels.  ``all_gather_into(out, x)`` defaults to ``torch.distributed.all_gather_into_tensor``
    (NCCL); tests pass their own to emulate several ranks on one GPU."""

    def __init__(self, eng: Engine, model: Model, params: Dict, y_chunk, rank: int, world: int):
        import torch
        super().__init__(eng, model, params, y_chunk, rank, world)
        self.out, self.ko, self.so = _outputs(y_chunk, self.rows, self.n)
        self.agg_b, self.aggs_b = self._xch(elem_doubles(self.n, True))
        self.status = torch.zeros(1, dtype=torch.int32, device=y_chunk.device)

    def forward_finish(self):
        self._ck(capi.load().bdlm_scan_dist_forward_finish(
            self.eng.ctx.handle, self.pr, self.rank, self.world, self.aggs_f.data_ptr(), self.ko,
            self.status.data_ptr()))

    def backward_local(self):
        self._ck(capi.load().bdlm_scan_dist_backward_local(
            self.eng.ctx.handle, self.pr, self.rank, self.world, self.ko, self.so,
            self.agg_b.data_ptr()))

    def backward_finish(self):
        self._ck(capi.load().bdlm_scan_dist_backward_finish(
            self.eng.ctx.handle, self.pr, self.rank, self.world, self.aggs_b.data_ptr(), self.ko,
            self.so, self.status.data_ptr()))

    def run(self, all_gather_into=None):
        gather = self._gather(all_gather_into)
        self.forward_local()
        gather(self.aggs_f, self.agg_f)
        self.forward_finish()
        self.backward_local()
        gather(self.aggs_b, self.agg_b)
        self.backward_finish()
        return self.out


class DistLoglik(_DistChunk):
    """Log-likelihoods of a time-sharded series (``bdlm_scan_dist_loglik_*``): every rank ends with
    the sums and status of ``scan_loglik`` on the whole series, bit-identical across ranks; the rank
    holding the series' last observation also has its final filtered state (m, C).  ``run`` takes
    the same injectable all-gather as ``DistScan``."""

    def __init__(self, eng: Engine, model: Model, params: Dict, y_chunk, rank: int, world: int):
        import torch
        super().__init__(eng, model, params, y_chunk, rank, world)
        self.part, self.parts = self._xch(dist_doubles(self.n, capi.SCAN_DIST_LOGLIK_PART))
        z = lambda k: torch.zeros(k, dtype=torch.float64, device=y_chunk.device)  # noqa: E731
        self.out = dict(transition=z(1), innovations=z(1), m=z(self.n), C=z(self.n * self.n),
                        status=torch.zeros(1, dtype=torch.int32, device=y_chunk.device))

    def partial(self):
        self._ck(capi.load().bdlm_scan_dist_loglik_partial(
            self.eng.ctx.handle, self.pr, self.rank, self.world, self.aggs_f.data_ptr(),
            self.out["m"].data_ptr(), self.out["C"].data_ptr(), self.part.data_ptr()))

    def finish(self):
        o = self.out
        self._ck(capi.load().bdlm_scan_dist_loglik_finish(
            self.eng.ctx.handle, self.world, self.parts.data_ptr(), o["transition"].data_ptr(),
            o["innovations"].data_ptr(), o["status"].data_ptr()))

    def run(self, all_gather_into=None):
        gather = self._gather(all_gather_into)
        self.forward_local()
        gather(self.aggs_f, self.agg_f)
        self.partial()
        gather(self.parts, self.part)
        self.finish()
        return self.out


class DistFfbs(_DistChunk):
    """FFBS + Gibbs statistics of a time-sharded series (``bdlm_scan_dist_ffbs_*``): theta of the
    chunk's rows (concatenated over ranks: ``scan_ffbs``'s path of the whole series), the filter
    fields in ``want_kf`` (m and C are always kept: the sampler reads them), and the statistics and
    status of the whole series, bit-identical on every rank.  ``first_row`` / ``total_T`` place the
    chunk in the series (``sharding.time_chunk``); z: CUDA tensor [rows, n] of the chunk's injected
    normals, or None for the Philox normals of ``eng.ctx.set_rng`` at the global rows."""

    def __init__(self, eng: Engine, model: Model, params: Dict, y_chunk, rank: int, world: int,
                 first_row: int, total_T: int, z=None, want_kf=()):
        import torch
        super().__init__(eng, model, params, y_chunk, rank, world)
        n = self.n
        assert z is None or (tuple(z.shape) == (self.rows, n) and _mem_and_ptr(z)[0] == capi.DEVICE)
        self.first_row, self.total_T, self.z = int(first_row), int(total_T), z
        self.out, self.ko, _ = _outputs(y_chunk, self.rows, n, tuple(dict.fromkeys(("m", "C") + tuple(want_kf))))
        dev = y_chunk.device
        self.out["theta"] = torch.empty((self.rows, n), dtype=torch.float64, device=dev)
        self.gs = capi.GibbsStats()
        for k, d in (("ssy", 1), ("ny", 1), ("ssw", n), ("scatter", n * n)):
            self.out[k] = torch.zeros((d,), dtype=torch.float64, device=dev)
            setattr(self.gs, k, self.out[k].data_ptr())
        self.out["status"] = torch.zeros(1, dtype=torch.int32, device=dev)
        self.agg_s, self.aggs_s = self._xch(dist_doubles(n, capi.SCAN_DIST_SAMPLER_ELEM))
        self.part, self.parts = self._xch(dist_doubles(n, capi.SCAN_DIST_FFBS_PART))

    def local(self):
        self._ck(capi.load().bdlm_scan_dist_ffbs_local(
            self.eng.ctx.handle, self.pr, self.rank, self.world, self.first_row, self.total_T,
            self.aggs_f.data_ptr(), None if self.z is None else self.z.data_ptr(),
            self.out["theta"].data_ptr(), self.ko, self.agg_s.data_ptr(), self.out["status"].data_ptr()))

    def finish(self):
        self._ck(capi.load().bdlm_scan_dist_ffbs_finish(
            self.eng.ctx.handle, self.pr, self.rank, self.world, self.aggs_s.data_ptr(),
            self.out["theta"].data_ptr(), self.ko, self.part.data_ptr(), self.out["status"].data_ptr()))

    def stats_finish(self):
        self._ck(capi.load().bdlm_scan_dist_ffbs_stats_finish(
            self.eng.ctx.handle, self.n, self.world, self.parts.data_ptr(), self.gs,
            self.out["status"].data_ptr()))

    def run(self, all_gather_into=None):
        gather = self._gather(all_gather_into)
        self.forward_local()
        gather(self.aggs_f, self.agg_f)
        self.local()
        gather(self.aggs_s, self.agg_s)
        self.finish()
        gather(self.parts, self.part)
        self.stats_finish()
        return self.out

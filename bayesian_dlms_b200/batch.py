"""Batched entry points over libbdlm.so: many independent series / chains per call.

This is the host-side shim a Scala facade would sit on (INTEGRATION.md): it flattens the
model closures (``dlm.materialise``), picks the memory space from the arrays it is given
(torch CUDA tensors -> device pointers, numpy arrays -> host pointers) and calls the C
ABI.  PyTorch is used only to own device memory and streams.

Array shapes (k = components per row, rows = T + keep_init):
  layout TIME_MAJOR   : y (T, p, B)   outputs (rows, k, B)   per-series params (k, B)
  layout SERIES_MAJOR : y (B, T, p)   outputs (B, rows, k)   per-series params (B, k)
Matrices are column-major inside a row (Breeze ``DenseMatrix.data`` order).
"""
from __future__ import annotations

import functools
import threading
from dataclasses import dataclass
from typing import Dict, Optional, Sequence

import numpy as np

from . import _capi as capi
from . import dlm as _dlm

TIME_MAJOR, SERIES_MAJOR = capi.TIME_MAJOR, capi.SERIES_MAJOR

KF_FIELDS = ("m", "C", "a", "R", "f", "Q")
SVD_FIELDS = ("m", "dc", "uc", "a", "dr", "ur", "f")


@dataclass
class Model:
    """Materialised ``Dlm`` for one time grid (see ``dlm.materialise``)."""

    F: np.ndarray
    G: np.ndarray
    f_tv: bool
    g_tv: bool
    n: int
    p: int
    T: int
    times: Optional[np.ndarray]  # None = regular grid 1..T
    t_init: Optional[np.ndarray] = None  # 1-element array: time of the saved state to resume from
    # names among ("times", "F", "G") that are given PER SERIES: arrays laid out like y with
    # k = 1 / n*p / n*n, living in the same memory space as y (numpy or torch)
    per_series: tuple = ()

    @staticmethod
    def build(mod: _dlm.Dlm, times: Optional[Sequence[float]] = None, T: Optional[int] = None,
              t_init: Optional[float] = None):
        if times is None:
            assert T is not None and T > 0, "give times or T"
            tgrid = np.arange(1, T + 1, dtype=np.float64)
        else:
            tgrid = np.ascontiguousarray(times, dtype=np.float64)
        if tgrid.size == 0:
            raise ValueError("empty observation vector (NoSuchElementException in the reference)")
        F, f_tv, G, g_tv, n, p = _dlm.materialise(mod, tgrid, t_init)
        regular = t_init is None and (times is None or
                                      np.array_equal(tgrid, np.arange(1, tgrid.size + 1)))
        return Model(np.ascontiguousarray(F.ravel()), np.ascontiguousarray(G.ravel()),
                     bool(f_tv), bool(g_tv), n, p, int(tgrid.size),
                     None if regular else tgrid,
                     None if t_init is None else np.array([float(t_init)]))


def build_batch_model(mod: _dlm.Dlm, times, layout=capi.SERIES_MAJOR) -> Model:
    """Model for a batch whose series sit on DIFFERENT time grids (``Data(time, observation)`` is
    per series in the reference, Dlm.scala:94; AqMeshExample.scala:86-127 has per-sensor irregular
    times): ``times`` is (B, T).  The closures are evaluated per series on the host; F / G are
    passed per series only where they really differ (polynomial G does not depend on dt,
    regression F depends on time).  Ragged batches: pad a short series at the end with its last
    time (dt = 0 passes the state through) and NaN observations."""
    times = np.ascontiguousarray(times, dtype=np.float64)
    assert times.ndim == 2 and times.shape[1] > 0
    B, T = times.shape
    mods = list(mod) if isinstance(mod, (list, tuple)) else [mod] * B   # one Dlm per series, e.g.
    assert len(mods) == B                                              # regression covariates
    Fs, Gs, f_any, g_any = [], [], False, False
    n = p = None
    for b in range(B):
        F, f_tv, G, g_tv, n, p = _dlm.materialise(mods[b], times[b])
        Fs.append(np.broadcast_to(F.reshape(-1, n * p), (T, n * p)))
        Gs.append(np.broadcast_to(G.reshape(-1, n * n), (T, n * n)))
        f_any, g_any = f_any or bool(f_tv), g_any or bool(g_tv)
    Fs, Gs = np.stack(Fs), np.stack(Gs)          # (B, T, k)
    f_ps = f_any or not np.array_equal(Fs, np.broadcast_to(Fs[:1, :1], Fs.shape))
    g_ps = g_any or not np.array_equal(Gs, np.broadcast_to(Gs[:1, :1], Gs.shape))
    lay = (lambda a: np.ascontiguousarray(a.transpose(1, 2, 0))) if layout == capi.TIME_MAJOR \
        else np.ascontiguousarray
    per = ["times"] + (["F"] if f_ps else []) + (["G"] if g_ps else [])
    return Model(lay(Fs) if f_ps else np.ascontiguousarray(Fs[0, 0]),
                 lay(Gs) if g_ps else np.ascontiguousarray(Gs[0, 0]),
                 bool(f_ps), bool(g_ps), n, p, T, lay(times[:, :, None]), None, tuple(per))


def model_to_device(model: Model, device) -> Model:
    """Copy of ``model`` whose per-series arrays are CUDA tensors (for device-resident calls)."""
    import torch
    kw = {k: getattr(model, k) for k in ("F", "G", "f_tv", "g_tv", "n", "p", "T", "times", "t_init",
                                         "per_series")}
    for name in model.per_series:
        kw[name] = torch.from_numpy(np.ascontiguousarray(kw[name])).to(device)
    return Model(**kw)


_engines_by_device = {}
_tls = threading.local()   # .engine: the Engine whose method is running on this thread


class bound_engine:
    """``with bound_engine(eng): ...`` -- device tensors marshalled inside the block make ``eng``
    (and no other engine of that device) adopt torch's current stream."""

    def __init__(self, eng):
        self.eng = eng

    def __enter__(self):
        self.prev = getattr(_tls, "engine", None)
        _tls.engine = self.eng
        return self.eng

    def __exit__(self, *exc):
        _tls.engine = self.prev
        return False


def _on_engine_stream(fn):
    @functools.wraps(fn)
    def wrap(self, *args, **kwargs):
        with bound_engine(self):
            return fn(self, *args, **kwargs)
    return wrap


def _adopt_torch_stream(x):
    """Device-mode calls are enqueued on torch's CURRENT stream of the tensor's device, so they
    are ordered with the torch ops that produced the inputs and consume the outputs.  The engine
    is the one whose method is running (thread-local); the per-device registry is only the
    fallback for helpers called outside an Engine method."""
    import torch
    eng = getattr(_tls, "engine", None) or _engines_by_device.get(x.device.index)
    if eng is not None:
        eng.ctx.set_stream(torch.cuda.current_stream(x.device).cuda_stream)


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _mem_and_ptr(x):
    if x is None:
        return None, None
    if _is_torch(x):
        if x.is_cuda:
            _adopt_torch_stream(x)
        assert x.is_contiguous() and str(x.dtype) in ("torch.float64", "torch.int32"), \
            "contiguous fp64 tensors only"
        return (capi.DEVICE if x.is_cuda else capi.HOST), x.data_ptr()
    assert isinstance(x, np.ndarray) and x.flags.c_contiguous
    return capi.HOST, x.ctypes.data


def _shared_param(x, rows, cols):
    """Shared (host) parameter -> flat column-major numpy array."""
    a = np.asarray(x, dtype=np.float64)
    if a.ndim == 2 and a.shape == (rows, cols):
        return _dlm.cm(a)
    a = np.ascontiguousarray(a.ravel())
    assert a.size == rows * cols, (a.shape, rows, cols)
    return a


class Engine:
    """One GPU context.  All methods return dicts of arrays in the caller's memory space."""

    def __init__(self, device: int = 0):
        self.ctx = capi.Context(device)
        self.device = device
        _engines_by_device[device] = self  # latest engine of a device adopts torch's stream

    # ------------------------------------------------------------------ helpers
    def use_torch_stream(self):
        import torch
        self.ctx.set_stream(torch.cuda.current_stream(self.device).cuda_stream)

    def _alloc(self, like, shape, dtype="float64", pinned=False):
        if _is_torch(like):
            import torch
            dt = torch.float64 if dtype == "float64" else torch.int32
            if like.is_cuda:
                return torch.empty(shape, dtype=dt, device=like.device)
            return torch.empty(shape, dtype=dt, pin_memory=pinned)
        return np.empty(shape, dtype=np.float64 if dtype == "float64" else np.int32)

    def _shape(self, layout, B, rows, k):
        return (rows, k, B) if layout == TIME_MAJOR else (B, rows, k)

    def _problem(self, model: Model, params: Dict, y, layout, keep_init, compat, B, mem):
        n, p = model.n, model.p
        per = 0
        ptrs = {}
        keep = []
        # params["v_tv"] = True: V varies with t (StudentTGibbs.filter): shared V is (T, p*p)
        # column-major per row [or (T, p, p)]; per-series V is laid out like y with k = p*p
        v_tv = bool(params.get("v_tv", False))
        w_tv = bool(params.get("w_tv", False))  # same for W (DlmFsvSystem.ffbs), k = n*n
        for name, bit, r, c in (("V", capi.PS_V, p, p), ("W", capi.PS_W, n, n),
                                ("m0", capi.PS_M0, n, 1), ("C0", capi.PS_C0, n, n)):
            x = params.get(name)
            if x is None:
                ptrs[name] = None
                continue
            # per-series parameters are named explicitly: params["per_series"] = ("V", "W")
            if name in params.get("per_series", ()):
                expect = (r * c, B) if layout == TIME_MAJOR else (B, r * c)
                if (name == "V" and v_tv) or (name == "W" and w_tv):
                    expect = self._shape(layout, B, model.T, r * c)
                assert tuple(x.shape) == expect, (name, tuple(x.shape), expect)
                m_, ptr = _mem_and_ptr(x)
                assert m_ == mem, f"{name} lives in a different memory space than y"
                per |= bit
                ptrs[name] = ptr
            elif (name == "V" and v_tv) or (name == "W" and w_tv):
                a = np.asarray(x, dtype=np.float64)
                if a.ndim == 3:  # (T, p, p) -> column-major rows
                    a = a.transpose(0, 2, 1)
                a = np.ascontiguousarray(a.reshape(model.T, r * c))
                keep.append(a)
                ptrs[name] = a
            else:
                a = _shared_param(x, r, c)
                keep.append(a)
                ptrs[name] = a
        _, yptr = _mem_and_ptr(y)
        grid = {"F": model.F, "G": model.G, "times": model.times}
        for name, bit, k in (("times", capi.PS_TIMES, 1), ("F", capi.PS_F, n * p),
                             ("G", capi.PS_G, n * n)):
            if name in model.per_series:
                x = grid[name]
                expect = self._shape(layout, B, model.T, k)
                assert tuple(x.shape) == expect, (name, tuple(x.shape), expect)
                m_, ptr = _mem_and_ptr(x)
                assert m_ == mem, f"per-series {name} lives in a different memory space than the data"
                per |= bit
                grid[name] = ptr
        pr = capi.make_problem(B=B, T=model.T, n=n, p=p, layout=layout, mem=mem,
                               keep_init=keep_init, F=grid["F"], G=grid["G"], times=grid["times"],
                               V=ptrs["V"], W=ptrs["W"], m0=ptrs["m0"], C0=ptrs["C0"], y=yptr,
                               per_series=per, compat=compat, f_tv=model.f_tv, g_tv=model.g_tv,
                               v_tv=v_tv, w_tv=w_tv, t_init=model.t_init)
        return pr, keep

    def _batch_of(self, model, y, layout):
        shp = tuple(y.shape)
        if layout == TIME_MAJOR:
            assert shp[0] == model.T and shp[1] == model.p, (shp, model.T, model.p)
            return shp[2]
        assert shp[1] == model.T and shp[2] == model.p, (shp, model.T, model.p)
        return shp[0]

    def _outs(self, cls, fields, want, like, layout, B, rows, dims, pinned):
        out, struct = {}, cls()
        for name in fields:
            if name in want:
                out[name] = self._alloc(like, self._shape(layout, B, rows, dims[name]),
                                        pinned=pinned)
                setattr(struct, name, _mem_and_ptr(out[name])[1])
            else:
                setattr(struct, name, None)
        return out, struct

    def _kf_dims(self, model):
        n, p = model.n, model.p
        return dict(m=n, C=n * n, a=n, R=n * n, f=p, Q=p * p, s=n, S=n * n)

    def _svd_dims(self, model):
        n, p = model.n, model.p
        return dict(m=n, dc=n, uc=n * n, a=n, dr=n, ur=n * n, f=p)

    def _status(self, like, B, want):
        if not want:
            return None, None
        st = self._alloc(like, (B,), dtype="int32")
        return st, _mem_and_ptr(st)[1]

    # ------------------------------------------------------------------ filter / smoother
    @_on_engine_stream
    def filter(self, model: Model, params: Dict, y, *, layout=TIME_MAJOR, keep_init=True,
               want=KF_FIELDS, status=True, pinned=False):
        """KalmanFilter.filterDlm / .filter batched (KalmanFilter.scala:291-294, Filter.scala:41-45)."""
        mem, _ = _mem_and_ptr(y)
        B = self._batch_of(model, y, layout)
        rows = model.T + int(keep_init)
        pr, keep = self._problem(model, params, y, layout, keep_init, 0, B, mem)
        out, ko = self._outs(capi.KfOut, KF_FIELDS, want, y, layout, B, rows,
                             self._kf_dims(model), pinned)
        st, stp = self._status(y, B, status)
        self.ctx.check(capi.load().bdlm_kf_filter(self.ctx.handle, pr, ko, stp))
        if st is not None:
            out["status"] = st
        return out

    @_on_engine_stream
    def smooth(self, model: Model, params: Dict, filt: Dict, *, layout=TIME_MAJOR,
               keep_init=True, textbook=False, status=True, pinned=False):
        """Smoothing.backwardsSmoother batched (Smoothing.scala:57-64)."""
        m = filt["m"]
        mem, _ = _mem_and_ptr(m)
        B = m.shape[2] if layout == TIME_MAJOR else m.shape[0]
        rows = model.T + int(keep_init)
        pr, keep = self._problem(model, params, None, layout, keep_init,
                                 capi.TEXTBOOK_SMOOTHER if textbook else 0, B, mem)
        ko = capi.KfOut()
        for name in KF_FIELDS:
            setattr(ko, name, _mem_and_ptr(filt[name])[1] if name in ("m", "C", "a", "R")
                    and filt.get(name) is not None else None)
        out, so = self._outs(capi.SmoothOut, ("s", "S"), ("s", "S"), m, layout, B, rows,
                             self._kf_dims(model), pinned)
        st, stp = self._status(m, B, status)
        self.ctx.check(capi.load().bdlm_rts_smooth(self.ctx.handle, pr, ko, so, stp))
        if st is not None:
            out["status"] = st
        return out

    @_on_engine_stream
    def filter_smooth(self, model: Model, params: Dict, y, *, layout=TIME_MAJOR, keep_init=True,
                      want=KF_FIELDS + ("s", "S"), textbook=False, status=True, pinned=False,
                      out: Optional[Dict] = None, parallel_in_time=False):
        """Fused KalmanFilter(adv).filter + Smoothing.backwardsSmoother.  ``parallel_in_time``: ONE
        long eligible series may run through the associative-scan kernels (1e-9 instead of
        bit-for-bit; include/bdlm.h BDLM_PARALLEL_IN_TIME)."""
        mem, _ = _mem_and_ptr(y)
        B = self._batch_of(model, y, layout)
        rows = model.T + int(keep_init)
        pr, keep = self._problem(model, params, y, layout, keep_init,
                                 (capi.TEXTBOOK_SMOOTHER if textbook else 0) |
                                 (capi.PARALLEL_IN_TIME if parallel_in_time else 0), B, mem)
        dims = self._kf_dims(model)
        if out is None:
            res, ko = self._outs(capi.KfOut, KF_FIELDS, want, y, layout, B, rows, dims, pinned)
            res2, so = self._outs(capi.SmoothOut, ("s", "S"), want, y, layout, B, rows, dims, pinned)
            res.update(res2)
            st, stp = self._status(y, B, status)
            if st is not None:
                res["status"] = st
        else:  # caller-provided output buffers (benchmarks reuse them across steps)
            res, ko, so = out, capi.KfOut(), capi.SmoothOut()
            for name in KF_FIELDS:
                setattr(ko, name, _mem_and_ptr(out[name])[1] if name in out else None)
            for name in ("s", "S"):
                setattr(so, name, _mem_and_ptr(out[name])[1] if name in out else None)
            stp = _mem_and_ptr(out["status"])[1] if "status" in out else None
        self.ctx.check(capi.load().bdlm_kf_filter_smooth(self.ctx.handle, pr, ko, so, stp))
        return res

    @_on_engine_stream
    def loglik(self, model: Model, params: Dict, y, *, layout=TIME_MAJOR, status=True,
               parallel_in_time=False):
        """KalmanFilter.likelihood (transition form, KalmanFilter.scala:299-306) and the
        innovations form (conditionalLikelihood, :138-153) per series.  ``parallel_in_time``: ONE
        long eligible series may run through the scan's forward pass (1e-9 instead of bit-for-bit;
        include/bdlm.h BDLM_PARALLEL_IN_TIME)."""
        mem, _ = _mem_and_ptr(y)
        B = self._batch_of(model, y, layout)
        pr, keep = self._problem(model, params, y, layout, True,
                                 capi.PARALLEL_IN_TIME if parallel_in_time else 0, B, mem)
        tr, inn = self._alloc(y, (B,)), self._alloc(y, (B,))
        st, stp = self._status(y, B, status)
        self.ctx.check(capi.load().bdlm_loglik(self.ctx.handle, pr, _mem_and_ptr(tr)[1],
                                               _mem_and_ptr(inn)[1], stp))
        out = dict(transition=tr, innovations=inn)
        if st is not None:
            out["status"] = st
        return out

    @_on_engine_stream
    def filter_last(self, model: Model, params: Dict, y, *, layout=TIME_MAJOR, loglik=False,
                    status=True, parallel_in_time=False):
        """``ys.foldLeft(init)(kf.step(mod, p))`` batched (NoModel.scala:153-155): only the state
        after the last observation, nothing stored per step.  Returns m (n, B) / (B, n) and
        C (n*n, B) / (B, n*n) [+ both log-likelihoods].  ``parallel_in_time`` as in ``loglik``."""
        mem, _ = _mem_and_ptr(y)
        B = self._batch_of(model, y, layout)
        pr, keep = self._problem(model, params, y, layout, True,
                                 capi.PARALLEL_IN_TIME if parallel_in_time else 0, B, mem)
        n = model.n
        row = (lambda k: (k, B)) if layout == TIME_MAJOR else (lambda k: (B, k))
        out = dict(m=self._alloc(y, row(n)), C=self._alloc(y, row(n * n)))
        if loglik:
            out["transition"], out["innovations"] = self._alloc(y, (B,)), self._alloc(y, (B,))
        st, stp = self._status(y, B, status)
        ptr = lambda k: _mem_and_ptr(out[k])[1] if k in out else None  # noqa: E731
        self.ctx.check(capi.load().bdlm_kf_filter_last(self.ctx.handle, pr, ptr("m"), ptr("C"),
                                                       ptr("transition"), ptr("innovations"), stp))
        if st is not None:
            out["status"] = st
        return out

    # ------------------------------------------------------------------ samplers
    def _stats(self, like, layout, B, model, want):
        if not want:
            return {}, None
        n, p = model.n, model.p
        dims = dict(ssy=p, ny=p, ssw=n, scatter=n * n)
        out, gs = {}, capi.GibbsStats()
        for k, d in dims.items():
            out[k] = self._alloc(like, (d, B) if layout == TIME_MAJOR else (B, d))
            setattr(gs, k, _mem_and_ptr(out[k])[1])
        return out, gs

    @_on_engine_stream
    def ffbs(self, model: Model, params: Dict, y, z, *, layout=TIME_MAJOR, want_kf=(),
             stats=False, status=True, svd=False, consistent_w=False, pinned=False,
             parallel_in_time=False):
        """Smoothing.ffbsDlm (Smoothing.scala:173-180) or, with svd=True, SvdSampler.ffbsDlm
        (SvdSampler.scala:79-82), batched over chains, with injected normals z.
        ``parallel_in_time``: ONE long eligible series may run through the scan's sampler (same
        normals, path within 1e-9 instead of bit-for-bit; include/bdlm.h BDLM_PARALLEL_IN_TIME)."""
        mem, _ = _mem_and_ptr(y)
        B = self._batch_of(model, y, layout)
        rows = model.T + 1
        # z=None: the kernels draw their own normals (Philox, Context.set_rng(seed, sweep))
        assert z is None or tuple(z.shape) == self._shape(layout, B, rows, model.n), \
            (z.shape, rows, model.n)
        zptr = None if z is None else _mem_and_ptr(z)[1]
        compat = capi.SVD_CONSISTENT_W if (svd and consistent_w) else 0
        if parallel_in_time and not svd:
            compat |= capi.PARALLEL_IN_TIME
        pr, keep = self._problem(model, params, y, layout, True, compat, B, mem)
        theta = self._alloc(y, self._shape(layout, B, rows, model.n), pinned=pinned)
        out = dict(theta=theta)
        sout, gs = self._stats(y, layout, B, model, stats)
        out.update(sout)
        st, stp = self._status(y, B, status)
        lib = capi.load()
        if svd:
            fo, so = self._outs(capi.SvdOut, SVD_FIELDS, want_kf, y, layout, B, rows,
                                self._svd_dims(model), pinned)
            out.update({"svd_" + k: v for k, v in fo.items()})
            self.ctx.check(lib.bdlm_svd_ffbs(self.ctx.handle, pr, zptr,
                                             _mem_and_ptr(theta)[1], so, gs, stp))
        else:
            fo, ko = self._outs(capi.KfOut, KF_FIELDS, want_kf, y, layout, B, rows,
                                self._kf_dims(model), pinned)
            out.update(fo)
            self.ctx.check(lib.bdlm_ffbs(self.ctx.handle, pr, zptr,
                                         _mem_and_ptr(theta)[1], ko, gs, stp))
        if st is not None:
            out["status"] = st
        return out

    @_on_engine_stream
    def svd_filter(self, model: Model, params: Dict, y, *, layout=TIME_MAJOR, keep_init=True,
                   want=SVD_FIELDS, consistent_w=False, status=True, pinned=False):
        """SvdFilter.filterDlm / .filter batched (SvdFilter.scala:100-119,158-161)."""
        mem, _ = _mem_and_ptr(y)
        B = self._batch_of(model, y, layout)
        rows = model.T + int(keep_init)
        pr, keep = self._problem(model, params, y, layout, keep_init,
                                 capi.SVD_CONSISTENT_W if consistent_w else 0, B, mem)
        out, so = self._outs(capi.SvdOut, SVD_FIELDS, want, y, layout, B, rows,
                             self._svd_dims(model), pinned)
        st, stp = self._status(y, B, status)
        self.ctx.check(capi.load().bdlm_svd_filter(self.ctx.handle, pr, so, stp))
        if st is not None:
            out["status"] = st
        return out

    @_on_engine_stream
    def gibbs_stats(self, model: Model, y, theta, *, layout=TIME_MAJOR):
        """Sufficient statistics of a given path (Gibbs.scala:29-43,63-73; GibbsWishart.scala:22-29)."""
        mem, _ = _mem_and_ptr(y)
        B = self._batch_of(model, y, layout)
        pr, keep = self._problem(model, {}, y, layout, True, 0, B, mem)
        out, gs = self._stats(y, layout, B, model, True)
        self.ctx.check(capi.load().bdlm_gibbs_suffstats(self.ctx.handle, pr,
                                                        _mem_and_ptr(theta)[1], gs))
        return out

    # ------------------------------------------------------------------ "next" rows (8f)
    def _ar_problem(self, sv: Dict, y, v, times, layout, ou):
        """sv: dict(phi, mu, sigma_eta) -- python floats (shared) or [B] arrays living with y."""
        mem, yptr = _mem_and_ptr(y)
        if layout == TIME_MAJOR:
            T, B = int(y.shape[0]), int(y.shape[1])
        else:
            B, T = int(y.shape[0]), int(y.shape[1])
        keep = []
        pr = capi.ArProblem()
        pr.B, pr.T, pr.layout, pr.mem = B, T, int(layout), int(mem)
        pr.process = capi.OU if ou else capi.AR1
        per = not np.isscalar(sv["phi"])
        pr.per_series = int(per)
        for name in ("phi", "mu", "sigma_eta"):
            x = sv[name]
            if per:
                m_, ptr = _mem_and_ptr(x)
                assert m_ == mem and tuple(x.shape) == (B,), name
                setattr(pr, name, ptr)
            else:
                a = np.array([float(x)])
                keep.append(a)
                setattr(pr, name, a.ctypes.data)
        if np.isscalar(v):
            a = np.array([float(v)]); keep.append(a)
            pr.v_mode, pr.v = capi.V_SCALAR, a.ctypes.data
        elif isinstance(v, np.ndarray) and v.ndim == 1:  # y is always 2-D, so 1-D = per step
            a = np.ascontiguousarray(v, dtype=np.float64); keep.append(a)
            assert a.size == T
            pr.v_mode, pr.v = capi.V_PER_STEP, a.ctypes.data
        else:
            m_, ptr = _mem_and_ptr(v)
            assert m_ == mem and tuple(v.shape) == tuple(y.shape)
            pr.v_mode, pr.v = capi.V_PER_SERIES_STEP, ptr
        if times is not None:
            a = np.ascontiguousarray(times, dtype=np.float64); keep.append(a)
            assert a.size == T
            pr.times = a.ctypes.data
        pr.y = yptr
        return pr, keep, B, T

    @_on_engine_stream
    def ar_filter(self, sv: Dict, y, v, *, times=None, ou=False, layout=TIME_MAJOR,
                  want=("m", "C", "a", "R")):
        """FilterAr / FilterOu.filterUnivariate batched (FilterAr.scala:37-47, FilterOu.scala:30-45).
        y: (T, B) time-major or (B, T) series-major, NaN = missing.  Outputs have T + 1 rows."""
        pr, keep, B, T = self._ar_problem(sv, y, v, times, layout, ou)
        shape = (T + 1, B) if layout == TIME_MAJOR else (B, T + 1)
        out, ao = {}, capi.ArOut()
        for k in ("m", "C", "a", "R"):
            if k in want:
                out[k] = self._alloc(y, shape)
                setattr(ao, k, _mem_and_ptr(out[k])[1])
        self.ctx.check(capi.load().bdlm_ar_filter(self.ctx.handle, pr, ao))
        return out

    @_on_engine_stream
    def ar_ffbs(self, sv: Dict, y, v, z, *, times=None, ou=False, layout=TIME_MAJOR, want=()):
        """FilterAr / FilterOu.ffbs batched (FilterAr.scala:77-83, FilterOu.scala:73-79) with
        injected normals z (T + 1 rows)."""
        pr, keep, B, T = self._ar_problem(sv, y, v, times, layout, ou)
        shape = (T + 1, B) if layout == TIME_MAJOR else (B, T + 1)
        assert tuple(z.shape) == shape, (tuple(z.shape), shape)
        out, ao = dict(theta=self._alloc(y, shape)), capi.ArOut()
        for k in ("m", "C", "a", "R"):
            if k in want:
                out[k] = self._alloc(y, shape)
                setattr(ao, k, _mem_and_ptr(out[k])[1])
        self.ctx.check(capi.load().bdlm_ar_ffbs(self.ctx.handle, pr, _mem_and_ptr(z)[1],
                                                _mem_and_ptr(out["theta"])[1], ao))
        return out

    @_on_engine_stream
    def conjugate_filter(self, model: Model, params: Dict, prior_shape: float, prior_scale: float,
                         y, *, layout=TIME_MAJOR, want=("m", "C"), status=True):
        """ConjugateFilter(prior, advanceState).filter batched (ConjugateFilter.scala:17-112)."""
        mem, _ = _mem_and_ptr(y)
        B = self._batch_of(model, y, layout)
        rows = model.T + 1
        pr, keep = self._problem(model, params, y, layout, True, 0, B, mem)
        out, ko = self._outs(capi.KfOut, KF_FIELDS, want, y, layout, B, rows, self._kf_dims(model), False)
        out["shape"] = self._alloc(y, self._shape(layout, B, rows, 1))
        out["scale"] = self._alloc(y, self._shape(layout, B, rows, 1))
        st, stp = self._status(y, B, status)
        self.ctx.check(capi.load().bdlm_conjugate_filter(
            self.ctx.handle, pr, float(prior_shape), float(prior_scale), ko,
            _mem_and_ptr(out["shape"])[1], _mem_and_ptr(out["scale"])[1], stp))
        if st is not None:
            out["status"] = st
        return out

    @_on_engine_stream
    def gibbs_draw(self, n: int, p: int, T: int, stats: Dict, prior: Dict, *, layout=TIME_MAJOR,
                   seed=0, sweep=0, inject: Optional[Dict] = None, want_shape_rate=False,
                   out: Optional[Dict] = None):
        """Conjugate draws of V (diagonal inverse gamma) and W (diagonal inverse gamma, or inverse
        Wishart when prior has ``w_psi``) from Gibbs sufficient statistics, on the device
        (Gibbs.scala:41-49,72-77; GibbsWishart.scala:16-35).  Returns per-chain ``V`` (p*p) and
        ``W`` (n*n) arrays usable as per-series parameters of the next sweep."""
        like = stats["ssy"]
        mem, _ = _mem_and_ptr(like)
        B = like.shape[1] if layout == TIME_MAJOR else like.shape[0]
        pr = capi.Problem()
        pr.B, pr.T, pr.n, pr.p, pr.layout, pr.mem, pr.keep_init = B, T, n, p, int(layout), int(mem), 1
        gs = capi.GibbsStats()
        for k in ("ssy", "ny", "ssw", "scatter"):
            setattr(gs, k, _mem_and_ptr(stats[k])[1] if stats.get(k) is not None else None)
        gp = capi.GibbsPrior()
        gp.v_shape, gp.v_scale = prior["v_shape"], prior["v_scale"]
        gp.w_shape, gp.w_scale = prior.get("w_shape", 0.0), prior.get("w_scale", 0.0)
        keep = []
        if prior.get("w_psi") is not None:
            psi = _shared_param(prior["w_psi"], n, n); keep.append(psi)
            gp.w_nu, gp.w_psi = float(prior["w_nu"]), psi.ctypes.data
        rng = capi.GibbsRng()
        rng.seed, rng.sweep = int(seed), int(sweep)
        for k in ("gamma_v", "gamma_w", "bartlett"):
            setattr(rng, k, _mem_and_ptr(inject[k])[1] if inject and inject.get(k) is not None else None)
        row = (lambda k: (k, B)) if layout == TIME_MAJOR else (lambda k: (B, k))
        res = out if out is not None else dict(V=self._alloc(like, row(p * p)), W=self._alloc(like, row(n * n)))
        if want_shape_rate:
            res["v_shape_rate"] = self._alloc(like, row(2 * p))
            res["w_shape_rate"] = self._alloc(like, row(2 * n))
        if "status" not in res:
            res["status"] = self._alloc(like, (B,), dtype="int32")
        ptr = lambda k: _mem_and_ptr(res[k])[1] if k in res else None  # noqa: E731
        self.ctx.check(capi.load().bdlm_gibbs_draw(self.ctx.handle, pr, gs, gp, rng, ptr("V"), ptr("W"),
                                                   ptr("v_shape_rate"), ptr("w_shape_rate"),
                                                   ptr("status")))
        return res

    def sync(self):
        self.ctx.sync()


_default: Dict[int, Engine] = {}


def default_engine(device: int = 0) -> Engine:
    """Process-wide engine per device; raises if libbdlm.so or a CUDA device is missing."""
    if device not in _default:
        _default[device] = Engine(device)
    return _default[device]

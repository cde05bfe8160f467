"""Multi-GPU communicator (``bdlm_comm_*``, include/bdlm.h): NCCL and the per-device contexts
behind one object, in the library -- the host only passes plain pointers.

* ``Comm.single_process(devices)``: one process drives all GPUs (what a JVM host does); sharded
  calls take HOST arrays for the whole batch and cut them over the devices.
* ``Comm.from_torch_distributed(device)``: one process per GPU under ``torchrun``; the 128-byte
  rendezvous id is broadcast with ``torch.distributed`` (plumbing), the collectives themselves are
  issued by libbdlm.so on its own NCCL communicator.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence

import numpy as np

from . import _capi as capi
from .batch import (Engine, KF_FIELDS, Model, SERIES_MAJOR, SVD_FIELDS, TIME_MAJOR, _mem_and_ptr,
                    bound_engine)


class Comm:
    def __init__(self, devices: Sequence[int], first_rank: int = 0, world: Optional[int] = None,
                 uid: Optional[bytes] = None):
        lib = capi.load()
        devs = (C.c_int32 * len(devices))(*[int(d) for d in devices])
        world = len(devices) if world is None else int(world)
        h = C.c_void_p()
        idbuf = None if uid is None else C.create_string_buffer(bytes(uid), capi.COMM_ID_BYTES)
        rc = lib.bdlm_comm_create(devs, len(devices), int(first_rank), world, idbuf, C.byref(h))
        if rc != 0:
            raise capi.BdlmError(rc, lib.bdlm_comm_last_error(None).decode())
        self._h = h
        self.devices, self.first_rank, self.world = list(devices), int(first_rank), world
        # Engines over the communicator's own contexts (borrowed handles)
        self.engines: List[Engine] = []
        for i, d in enumerate(devices):
            e = Engine.__new__(Engine)
            e.ctx = capi.Context(d, borrowed_handle=lib.bdlm_comm_ctx(h, i))
            e.device = d
            self.engines.append(e)

    # ------------------------------------------------------------------ construction
    @staticmethod
    def unique_id() -> bytes:
        buf = C.create_string_buffer(capi.COMM_ID_BYTES)
        rc = capi.load().bdlm_comm_unique_id(buf)
        if rc != 0:
            raise capi.BdlmError(rc, capi.load().bdlm_comm_last_error(None).decode())
        return buf.raw

    @classmethod
    def single_process(cls, devices: Sequence[int]) -> "Comm":
        return cls(devices)

    @classmethod
    def from_torch_distributed(cls, device: int) -> "Comm":
        import torch
        import torch.distributed as dist
        rank, world = dist.get_rank(), dist.get_world_size()
        t = torch.zeros(capi.COMM_ID_BYTES, dtype=torch.uint8)
        if rank == 0:
            t = torch.frombuffer(bytearray(cls.unique_id()), dtype=torch.uint8).clone()
        if dist.get_backend() == "nccl":
            t = t.cuda(device)
        dist.broadcast(t, 0)
        return cls([device], first_rank=rank, world=world, uid=bytes(t.cpu().numpy().tobytes()))

    def close(self):
        if getattr(self, "_h", None):
            capi.load().bdlm_comm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc < 0:
            raise capi.BdlmError(rc, capi.load().bdlm_comm_last_error(self._h).decode())
        return rc

    @property
    def uses_peer_exchange(self) -> bool:
        return bool(capi.load().bdlm_comm_uses_peer_exchange(self._h))

    def sync(self):
        self._ck(capi.load().bdlm_comm_sync(self._h))

    # ------------------------------------------------------------------ collectives
    def allreduce_sum(self, values: np.ndarray) -> np.ndarray:
        """Sum over all PROCESSES of a small host vector (ncclAllReduce inside the library)."""
        v = np.ascontiguousarray(values, dtype=np.float64).copy()
        self._ck(capi.load().bdlm_comm_allreduce_sum(self._h, v.ctypes.data, v.size))
        return v

    def allreduce_sum_device(self, t):
        """In place on a CUDA fp64 tensor (one device per process); enqueue-only."""
        with bound_engine(self.engines[0]):
            _, ptr = _mem_and_ptr(t)
        self._ck(capi.load().bdlm_comm_allreduce_sum_device(self._h, ptr, t.numel()))
        return t

    # ------------------------------------------------------------------ sharded batched calls
    def _eng0(self) -> Engine:
        return self.engines[0]

    def filter_smooth(self, model: Model, params: Dict, y, *, layout=SERIES_MAJOR, keep_init=True,
                      want=KF_FIELDS + ("s", "S"), textbook=False):
        e = self._eng0()
        with bound_engine(e):
            mem, _ = _mem_and_ptr(y)
            B = e._batch_of(model, y, layout)
            rows = model.T + int(keep_init)
            pr, keep = e._problem(model, params, y, layout, keep_init,
                                  capi.TEXTBOOK_SMOOTHER if textbook else 0, B, mem)
            dims = e._kf_dims(model)
            res, ko = e._outs(capi.KfOut, KF_FIELDS, want, y, layout, B, rows, dims, False)
            res2, so = e._outs(capi.SmoothOut, ("s", "S"), want, y, layout, B, rows, dims, False)
            res.update(res2)
            st, stp = e._status(y, B, True)
        self._ck(capi.load().bdlm_comm_kf_filter_smooth(self._h, pr, ko, so, stp))
        res["status"] = st
        return res

    def filter(self, model: Model, params: Dict, y, *, layout=SERIES_MAJOR, keep_init=True,
               want=KF_FIELDS):
        """``bdlm_comm_kf_filter``: KalmanFilter.filterDlm / .filter over the devices."""
        e = self._eng0()
        with bound_engine(e):
            mem, _ = _mem_and_ptr(y)
            B = e._batch_of(model, y, layout)
            rows = model.T + int(keep_init)
            pr, keep = e._problem(model, params, y, layout, keep_init, 0, B, mem)
            res, ko = e._outs(capi.KfOut, KF_FIELDS, want, y, layout, B, rows, e._kf_dims(model), False)
            st, stp = e._status(y, B, True)
        self._ck(capi.load().bdlm_comm_kf_filter(self._h, pr, ko, stp))
        res["status"] = st
        return res

    def svd_filter(self, model: Model, params: Dict, y, *, layout=SERIES_MAJOR, keep_init=True,
                   want=SVD_FIELDS, consistent_w=False):
        """``bdlm_comm_svd_filter``: SvdFilter.filterDlm / .filter over the devices."""
        e = self._eng0()
        with bound_engine(e):
            mem, _ = _mem_and_ptr(y)
            B = e._batch_of(model, y, layout)
            rows = model.T + int(keep_init)
            pr, keep = e._problem(model, params, y, layout, keep_init,
                                  capi.SVD_CONSISTENT_W if consistent_w else 0, B, mem)
            res, so = e._outs(capi.SvdOut, SVD_FIELDS, want, y, layout, B, rows, e._svd_dims(model), False)
            st, stp = e._status(y, B, True)
        self._ck(capi.load().bdlm_comm_svd_filter(self._h, pr, so, stp))
        res["status"] = st
        return res

    def loglik(self, model: Model, params: Dict, y, *, layout=SERIES_MAJOR):
        """Per-series log-likelihoods + their sums over every series of every rank."""
        e = self._eng0()
        with bound_engine(e):
            mem, _ = _mem_and_ptr(y)
            B = e._batch_of(model, y, layout)
            pr, keep = e._problem(model, params, y, layout, True, 0, B, mem)
            tr, inn = e._alloc(y, (B,)), e._alloc(y, (B,))
            st, stp = e._status(y, B, True)
        sums = np.zeros(2)
        self._ck(capi.load().bdlm_comm_loglik(self._h, pr, _mem_and_ptr(tr)[1], _mem_and_ptr(inn)[1],
                                              stp, sums.ctypes.data))
        return dict(transition=tr, innovations=inn, status=st, sum_transition=float(sums[0]),
                    sum_innovations=float(sums[1]))

    def ffbs(self, model: Model, params: Dict, y, z, *, layout=SERIES_MAJOR, svd=False,
             consistent_w=False):
        """FFBS over the devices with per-chain AND pooled Gibbs sufficient statistics."""
        e = self._eng0()
        n, p = model.n, model.p
        with bound_engine(e):
            mem, _ = _mem_and_ptr(y)
            B = e._batch_of(model, y, layout)
            rows = model.T + 1
            zptr = None if z is None else _mem_and_ptr(z)[1]
            compat = capi.SVD_CONSISTENT_W if (svd and consistent_w) else 0
            pr, keep = e._problem(model, params, y, layout, True, compat, B, mem)
            theta = e._alloc(y, e._shape(layout, B, rows, n))
            sout, gs = e._stats(y, layout, B, model, True)
            st, stp = e._status(y, B, True)
        pooled = dict(ssy=np.zeros(p), ny=np.zeros(p), ssw=np.zeros(n), scatter=np.zeros(n * n))
        pg = capi.GibbsStats()
        for k, v in pooled.items():
            setattr(pg, k, v.ctypes.data)
        lib = capi.load()
        if svd:
            self._ck(lib.bdlm_comm_svd_ffbs(self._h, pr, zptr, _mem_and_ptr(theta)[1], None, gs, stp, pg))
        else:
            self._ck(lib.bdlm_comm_ffbs(self._h, pr, zptr, _mem_and_ptr(theta)[1], None, gs, stp, pg))
        out = dict(theta=theta, status=st, pooled=pooled)
        out.update(sout)
        return out

    # ------------------------------------------------------------------ time-sharded scan
    def scan_setup(self, models: Sequence[Model], params: Dict, y_chunks: Sequence):
        """One entry per LOCAL device: the Model of that rank's chunk length and its CUDA slice of
        the series.  Returns a handle for ``scan_run`` (buffers are allocated once)."""
        import torch
        from .scan import _outputs, _problem
        nl = len(self.engines)
        assert len(models) == nl and len(y_chunks) == nl
        n = models[0].n
        probs = (capi.Problem * nl)()
        kfs, sms = (capi.KfOut * nl)(), (capi.SmoothOut * nl)()
        sts = (C.c_void_p * nl)()
        outs, keep, status = [], [], []
        for i, (eng, model, y) in enumerate(zip(self.engines, models, y_chunks)):
            rank = self.first_rank + i
            with torch.cuda.device(y.device), bound_engine(eng):
                pr, kp = _problem(model, params, y, keep_init=(rank == 0))
            probs[i] = pr
            keep.append((kp, model, y))
            o, kfs[i], sms[i] = _outputs(y, model.T + int(rank == 0), n)
            st = torch.zeros(1, dtype=torch.int32, device=y.device)
            sts[i] = st.data_ptr()
            outs.append(o)
            status.append(st)
        return dict(probs=probs, kfs=kfs, sms=sms, sts=sts, outs=outs, status=status, keep=keep)

    def scan_run(self, h):
        """Enqueue the whole time-sharded filter + smoother (``bdlm_comm_scan_filter_smooth``)."""
        self._ck(capi.load().bdlm_comm_scan_filter_smooth(self._h, h["probs"], h["kfs"], h["sms"],
                                                          h["sts"]))
        return h["outs"]

    def scan_loglik(self, h):
        """Enqueue the log-likelihoods and last filtered state of the series of ``scan_setup``
        (``bdlm_comm_scan_loglik``).  Per local device: transition [1], innovations [1], status [1]
        (the whole series', same bits on every rank) and, on global rank world - 1, m [n] / C [n*n]."""
        import torch
        nl = len(self.engines)
        outs, arrs = [], {k: (C.c_void_p * nl)() for k in ("m", "C", "transition", "innovations", "status")}
        for i, (kp, model, y) in enumerate(h["keep"]):
            n = model.n
            z = lambda k: torch.zeros(k, dtype=torch.float64, device=y.device)  # noqa: E731
            o = dict(transition=z(1), innovations=z(1), m=z(n), C=z(n * n),
                     status=torch.zeros(1, dtype=torch.int32, device=y.device))
            for k in arrs:
                arrs[k][i] = o[k].data_ptr()
            outs.append(o)
        self._ck(capi.load().bdlm_comm_scan_loglik(self._h, h["probs"], arrs["m"], arrs["C"], arrs["transition"],
                                                   arrs["innovations"], arrs["status"]))
        return outs

    def scan_ffbs(self, h, first_rows: Sequence[int], total_T: int, z: Optional[Sequence] = None):
        """Enqueue FFBS + Gibbs statistics of the series of ``scan_setup`` (``bdlm_comm_scan_ffbs``):
        the filter fields go to ``scan_setup``'s outputs, theta [rows, n] and ssy, ny, ssw, scatter,
        status (the whole series', same bits on every rank) to the returned per-device dicts.
        first_rows: global row of each local chunk's first row (``sharding.time_chunk``); z: per
        local device a CUDA tensor [rows, n] of injected normals, or None for Philox."""
        import torch
        nl = len(self.engines)
        theta, zs, sts = (C.c_void_p * nl)(), (C.c_void_p * nl)(), (C.c_void_p * nl)()
        gs = (capi.GibbsStats * nl)()
        outs = []
        for i, (kp, model, y) in enumerate(h["keep"]):
            n, rows = model.n, h["outs"][i]["m"].shape[0]
            o = dict(theta=torch.empty((rows, n), dtype=torch.float64, device=y.device),
                     status=torch.zeros(1, dtype=torch.int32, device=y.device))
            for k, d in (("ssy", 1), ("ny", 1), ("ssw", n), ("scatter", n * n)):
                o[k] = torch.zeros(d, dtype=torch.float64, device=y.device)
                setattr(gs[i], k, o[k].data_ptr())
            theta[i], sts[i] = o["theta"].data_ptr(), o["status"].data_ptr()
            if z is not None:
                zs[i] = z[i].data_ptr()
            outs.append(o)
        fr = (C.c_int64 * nl)(*[int(f) for f in first_rows])
        self._ck(capi.load().bdlm_comm_scan_ffbs(self._h, h["probs"], fr, int(total_T), None if z is None else zs,
                                                 theta, h["kfs"], gs, sts))
        return outs

"""GPU parity of the parallel-in-time (associative scan) filter / smoother, BASELINE config 5.

The reference has no parallel-in-time path, so the bar (SURVEY.md Appendix C) is: equal to the
sequential kernel in textbook-smoother mode to 1e-9 relative, which for n = 1 is the reference
itself (checked against the committed golden CSVs)."""
import numpy as np
import pytest

import helpers as H

pytestmark = pytest.mark.gpu
TOL = 1e-9


@pytest.fixture(scope="module")
def eng():
    import torch
    assert torch.cuda.is_available()
    from bayesian_dlms_b200 import default_engine
    return default_engine(0)


def _models():
    from bayesian_dlms_b200 import dlm
    return {
        1: (dlm.polynomial(1), np.array([[2.0]]), np.array([[3.0]]), np.zeros(1), np.array([[10.0]])),
        2: H.second_order(),
        3: (dlm.polynomial(3), np.array([[1.5]]), np.diag([1.0, 0.5, 0.1]), np.zeros(3), 10 * np.eye(3)),
    }


def _sequential(eng, model, params, y):
    from bayesian_dlms_b200 import TIME_MAJOR
    out = eng.filter_smooth(model, params, y.reshape(-1, 1, 1).contiguous(), layout=TIME_MAJOR,
                            keep_init=True, textbook=True)
    eng.sync()
    return {k: v[:, :, 0] for k, v in out.items() if k != "status"}


@pytest.mark.parametrize("n", [1, 2, 3])
@pytest.mark.parametrize("T", [1, 63, 64, 65, 1000, 40_001])
def test_scan_equals_sequential(eng, n, T):
    import torch
    from bayesian_dlms_b200 import Model
    from bayesian_dlms_b200.scan import scan_filter_smooth
    mod, V, W, m0, C0 = _models()[n]
    rng = np.random.default_rng(100 * n + T % 97)
    y = H.simulate(mod, V, W, m0, C0, np.arange(1, T + 1.0), rng, missing=0.05)[:, 0]
    yd = torch.from_numpy(y).cuda()
    model = Model.build(mod, T=T)
    params = dict(V=V, W=W, m0=m0, C0=C0)
    seq = _sequential(eng, model, params, yd)
    out = scan_filter_smooth(eng, model, params, yd)
    torch.cuda.synchronize()
    assert int(out["status"][0]) == 0
    for k in ("m", "C", "a", "R", "f", "Q", "s", "S"):
        a, b = out[k].cpu().numpy(), seq[k].cpu().numpy()
        if k in ("f", "Q"):
            a, b = a[1:], b[1:]
        assert H.rel_err(a, b) < TOL, (k, n, T, H.rel_err(a, b))


@pytest.mark.slow
@pytest.mark.parametrize("n", [1, 2])
def test_scan_full_config5_size_vs_cpu_oracle(eng, n):
    """BASELINE config 5 at its OWN size: one series, T = 2^24, against the CPU oracle's sequential
    recursion (Filter.scala:41-62 order; KalmanFilter.scala:64-118 + Smoothing.scala:31-47 with the
    textbook covariance, which for n = 1 is the reference itself) -- error growth of the scan over
    2^24 combines is bounded here, not extrapolated from short series.  Tolerance 1e-9 relative."""
    import oracle
    import torch
    from bayesian_dlms_b200 import Model, dlm
    from bayesian_dlms_b200.scan import scan_filter_smooth
    mod, V, W, m0, C0 = _models()[n]
    T = 1 << 24
    g = torch.Generator(device="cuda").manual_seed(20260105)
    yd = torch.randn(T, generator=g, device="cuda", dtype=torch.float64).cumsum(0) * 0.1
    yd[torch.rand(T, generator=g, device="cuda") < 0.001] = float("nan")   # missing observations too
    model = Model.build(mod, T=T)
    out = scan_filter_smooth(eng, model, dict(V=V, W=W, m0=m0, C0=C0), yd)
    torch.cuda.synchronize()
    assert int(out["status"][0]) == 0
    F, _, G, _, _, p = dlm.materialise(mod, np.arange(1, 9.0))
    y = yd.cpu().numpy()
    o = oracle.kf_filter(n, 1, F, G, dlm.cm(V), dlm.cm(W), m0, dlm.cm(C0), np.arange(1, T + 1.0), y)
    sm = oracle.rts_smooth(n, G, o, textbook=True)
    o.update(s=sm["s"], S=sm["S"])
    worst = {}
    for k in ("m", "C", "a", "R", "f", "Q", "s", "S"):
        a, b = out[k].cpu().numpy(), o[k]
        if k in ("f", "Q"):
            a, b = a[1:], b[1:]
        worst[k] = H.rel_err(a, b)
        del a
    print("config-5 full-size max relative error vs CPU oracle, n = %d:" % n, worst)
    assert max(worst.values()) < TOL, worst


def test_scan_reproduces_golden_csv(eng):
    import torch
    from bayesian_dlms_b200 import Model, dlm
    from bayesian_dlms_b200.scan import scan_filter_smooth
    times, y, g = H.first_order_golden()
    model = Model.build(dlm.polynomial(1), T=len(times))
    out = scan_filter_smooth(eng, model, dict(V=[[2.0]], W=[[3.0]], m0=[0.0], C0=[[10.0]]),
                             torch.from_numpy(y[:, 0].copy()).cuda())
    torch.cuda.synchronize()
    for key, ref in (("m", g["m"]), ("C", g["C"]), ("s", g["s"]), ("S", g["S"])):
        assert H.rel_err(out[key][:, 0].cpu().numpy(), ref) < TOL, key
    assert H.rel_err(out["f"][1:, 0].cpu().numpy(), g["f"]) < TOL
    assert H.rel_err(out["Q"][1:, 0].cpu().numpy(), g["Q"]) < TOL


def test_scan_rejects_unsupported_shapes(eng):
    import torch
    from bayesian_dlms_b200 import Model, _capi as capi
    from bayesian_dlms_b200.scan import scan_filter_smooth
    mod, V, W, m0, C0 = H.seasonal13()
    model = Model.build(mod, T=10)
    model.times = None
    with pytest.raises((capi.BdlmError, AssertionError)):
        scan_filter_smooth(eng, model, dict(V=V, W=W, m0=m0, C0=C0), torch.zeros(10, dtype=torch.float64).cuda())


@pytest.mark.parametrize("n", [1, 2, 3])
@pytest.mark.parametrize("world", [1, 2, 3, 5, 8])
def test_device_side_protocol_emulated_ranks(n, world):
    """bdlm_scan_dist_*: local -> all-gather (emulated by a device concat) -> finish, one context
    per emulated rank, nothing copied to the host between the phases."""
    import torch
    from bayesian_dlms_b200 import Engine, Model, default_engine
    from bayesian_dlms_b200.scan import DistScan
    from bayesian_dlms_b200.sharding import shard_range
    mod, V, W, m0, C0 = _models()[n]
    T = 7001
    rng = np.random.default_rng(31 + n)
    y = H.simulate(mod, V, W, m0, C0, np.arange(1, T + 1.0), rng, missing=0.02)[:, 0]
    yd = torch.from_numpy(y).cuda()
    params = dict(V=V, W=W, m0=m0, C0=C0)
    seq = _sequential(default_engine(0), Model.build(mod, T=T), params, yd)
    ranks = []
    for r in range(world):
        lo, hi = shard_range(T, r, world)
        e = Engine(0)
        e.use_torch_stream()   # every emulated rank on torch's stream, like the copies below
        ranks.append(DistScan(e, Model.build(mod, T=hi - lo), params, yd[lo:hi].contiguous(),
                              r, world))
    for d in ranks:
        d.forward_local()
    torch.cuda.synchronize()
    gathered = torch.cat([d.agg_f for d in ranks])
    for d in ranks:
        d.aggs_f.copy_(gathered)
        d.forward_finish()
        d.backward_local()
    torch.cuda.synchronize()
    gathered = torch.cat([d.agg_b for d in ranks])
    for d in ranks:
        d.aggs_b.copy_(gathered)
        d.backward_finish()
    torch.cuda.synchronize()
    for d in ranks:
        assert int(d.status[0]) == 0
    for k in ("m", "C", "a", "R", "s", "S"):
        got = torch.cat([d.out[k] for d in ranks]).cpu().numpy()
        assert got.shape == tuple(seq[k].shape)
        assert H.rel_err(got, seq[k].cpu().numpy()) < TOL, (k, world, H.rel_err(got, seq[k].cpu().numpy()))


@pytest.mark.parametrize("n", [1, 2])
@pytest.mark.parametrize("where", ["device", "host"])
def test_opt_in_dispatch_of_one_long_series_to_the_scan(eng, n, where):
    """BDLM_PARALLEL_IN_TIME on bdlm_kf_filter_smooth: one long series (here T = 50 000) takes the
    associative-scan kernels -- 1e-9 against the sequential recursion -- from device or host
    buffers; an ineligible problem (B = 3) silently keeps the sequential kernel, bit for bit."""
    import time
    import torch
    from bayesian_dlms_b200 import Model, SERIES_MAJOR
    mod, V, W, m0, C0 = _models()[n]
    T = 50_000
    rng = np.random.default_rng(3 + n)
    y = rng.standard_normal((1, T, 1)).cumsum(axis=1) * 0.1
    y[rng.random(y.shape) < 0.01] = np.nan
    model = Model.build(mod, T=T)
    params = dict(V=V, W=W, m0=m0, C0=C0)
    yy = torch.from_numpy(y).cuda() if where == "device" else y
    seq = eng.filter_smooth(model, params, yy, layout=SERIES_MAJOR, textbook=True)
    eng.sync()
    t0 = time.perf_counter()
    seq = eng.filter_smooth(model, params, yy, layout=SERIES_MAJOR, textbook=True)
    eng.sync()
    t_seq = time.perf_counter() - t0
    pit = eng.filter_smooth(model, params, yy, layout=SERIES_MAJOR, textbook=True, parallel_in_time=True)
    eng.sync()
    t0 = time.perf_counter()
    pit = eng.filter_smooth(model, params, yy, layout=SERIES_MAJOR, textbook=True, parallel_in_time=True)
    eng.sync()
    t_pit = time.perf_counter() - t0
    npy = lambda x: x.cpu().numpy() if hasattr(x, "cpu") else x  # noqa: E731
    assert int(npy(pit["status"])[0]) == 0
    for k in ("m", "C", "a", "R", "s", "S"):
        assert H.rel_err(npy(pit[k]), npy(seq[k])) < TOL, (k, H.rel_err(npy(pit[k]), npy(seq[k])))
    assert H.rel_err(npy(pit["f"])[:, 1:], npy(seq["f"])[:, 1:]) < TOL
    print("T = %d, n = %d, %s buffers: sequential %.2f ms, parallel in time %.2f ms" %
          (T, n, where, t_seq * 1e3, t_pit * 1e3))
    # (timings are informational: tools/scan_time.py and the bench's scan leg measure them)
    # not eligible (three series): the flag is ignored, results are those of the sequential kernel
    y3 = np.repeat(y[:, :5000], 3, axis=0).copy()
    m3 = Model.build(mod, T=5000)
    y3 = torch.from_numpy(y3).cuda() if where == "device" else y3
    a = eng.filter_smooth(m3, params, y3, layout=SERIES_MAJOR, textbook=True)
    b = eng.filter_smooth(m3, params, y3, layout=SERIES_MAJOR, textbook=True, parallel_in_time=True)
    eng.sync()
    assert np.array_equal(npy(a["S"]), npy(b["S"]))

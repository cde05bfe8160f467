"""The fused filter + smoother for n <= 2 rebuilds the backward pass's filtered (m, C) from every
K-th stored row by filtering again from it (kf_small.cu, kSeg = K), instead of re-reading every
row.  Whatever the segment edges fall on -- short series, a partial top segment, keep_init 0 or 1,
missing observations at checkpoint rows, dt = 0 on irregular grids, per-series F or G -- the
eight outputs and the status must be the oracle's bits, and the bits of separate filter and
smooth calls (whose smoother re-reads every row)."""
import numpy as np
import pytest

import helpers as H

pytestmark = pytest.mark.gpu

K = 4
FIELDS = ("m", "C", "a", "R", "f", "Q", "s", "S")


@pytest.fixture(scope="module")
def eng():
    import torch
    assert torch.cuda.is_available()
    from bayesian_dlms_b200 import default_engine
    return default_engine(0)


def _exact(a, b, what=""):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    ok = (a == b) | (np.isnan(a) & np.isnan(b))
    assert ok.all(), f"{what}: {np.sum(~ok)} of {a.size} differ, max rel {H.rel_err(a[~ok], b[~ok])}"


def _np(x):
    return x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)


def _sm(x, layout):
    """-> series-major (B, rows, k) numpy"""
    from bayesian_dlms_b200 import TIME_MAJOR
    x = _np(x)
    return x.transpose(2, 0, 1) if layout == TIME_MAJOR else x


def _params(n):
    if n == 1:
        return np.array([[3.0]]), np.array([[0.7]]), np.zeros(1), 100.0 * np.eye(1)
    _, V, W, m0, C0 = H.second_order()
    return V, W, m0, C0


def _missing(y, T, ki):
    """NaN at the first and last observation, and (odd series) at every checkpoint row."""
    y = y.copy()
    y[:, 0] = np.nan
    y[:, T - 1] = np.nan
    for r in range(0, T + ki, K):
        if r - ki >= 0:
            y[1::2, r - ki] = np.nan
    return y


def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _check(eng, model, mods, times, y, V, W, m0, C0, layout, to, keep_init, textbook=False,
           want=FIELDS):
    import oracle
    from bayesian_dlms_b200 import TIME_MAJOR, dlm
    B = y.shape[0]
    n, ki = len(m0), int(keep_init)
    params = dict(V=V, W=W, m0=m0, C0=C0)
    yy = to(y.transpose(1, 2, 0) if layout == TIME_MAJOR else y)
    fs = eng.filter_smooth(model, params, yy, layout=layout, keep_init=keep_init, textbook=textbook,
                           want=want)
    f = eng.filter(model, params, yy, layout=layout, keep_init=keep_init)
    s = eng.smooth(model, params, f, layout=layout, keep_init=keep_init, textbook=textbook)
    eng.sync()
    assert set(fs) == set(want) | {"status"}
    sep = dict(f)
    sep.update(s)
    assert int(_np(fs["status"]).max()) == 0
    for k in want:
        _exact(_sm(fs[k], layout), _sm(sep[k], layout), f"{k} vs filter + smooth")
    cm = oracle.oracle.cm
    for b in range(B):
        F, _, G, _, _, _ = dlm.materialise(mods[b], times[b])
        o = oracle.kf_filter(n, 1, F, G, cm(V), cm(W), m0, cm(C0), times[b], y[b], keep_init=keep_init)
        o.update(oracle.rts_smooth(n, G, o, keep_init=keep_init, textbook=textbook))
        for k in want:
            got, exp = _sm(fs[k], layout)[b], o[k]
            if k in ("f", "Q"):  # row 0 of keep_init holds no forecast
                got, exp = got[ki:], exp[ki:]
            _exact(got, exp, f"{k} series {b}")


@pytest.mark.parametrize("n", [1, 2])
@pytest.mark.parametrize("T", [1, 2, K - 1, K, K + 1, 2 * K + 1, 1000])
@pytest.mark.parametrize("keep_init", [True, False])
def test_fused_regular_grid(eng, n, T, keep_init):
    from bayesian_dlms_b200 import Model, TIME_MAJOR, dlm
    rng = np.random.default_rng(1000 * n + 10 * T + keep_init)
    B = 37
    V, W, m0, C0 = _params(n)
    mod = dlm.polynomial(n)
    times = np.tile(np.arange(1, T + 1, dtype=np.float64), (B, 1))
    y = np.stack([H.simulate(mod, V, W, m0, C0, times[b], rng, missing=0.1) for b in range(B)])
    y = _missing(y, T, int(keep_init))
    _check(eng, Model.build(mod, T=T), [mod] * B, times, y, V, W, m0, C0, TIME_MAJOR, _cuda, keep_init)


@pytest.mark.parametrize("T", [2 * K + 1, 1000])
def test_fused_textbook_smoother(eng, T):
    from bayesian_dlms_b200 import Model, TIME_MAJOR, dlm
    rng = np.random.default_rng(T)
    B = 19
    V, W, m0, C0 = _params(2)
    mod = dlm.polynomial(2)
    times = np.tile(np.arange(1, T + 1, dtype=np.float64), (B, 1))
    y = _missing(np.stack([H.simulate(mod, V, W, m0, C0, times[b], rng, missing=0.1) for b in range(B)]), T, 1)
    _check(eng, Model.build(mod, T=T), [mod] * B, times, y, V, W, m0, C0, TIME_MAJOR, _cuda, True,
           textbook=True)


@pytest.mark.parametrize("want", [("s", "S"), ("a", "R", "f", "Q", "s", "S")])
def test_fused_without_m_and_C(eng, want):
    """(m, C) not requested: the checkpoints come from the library's workspace."""
    from bayesian_dlms_b200 import Model, TIME_MAJOR, dlm
    rng = np.random.default_rng(len(want))
    B, T = 45, 4 * K + 2
    V, W, m0, C0 = _params(2)
    mod = dlm.polynomial(2)
    times = np.tile(np.arange(1, T + 1, dtype=np.float64), (B, 1))
    y = _missing(np.stack([H.simulate(mod, V, W, m0, C0, times[b], rng, missing=0.1) for b in range(B)]), T, 1)
    _check(eng, Model.build(mod, T=T), [mod] * B, times, y, V, W, m0, C0, TIME_MAJOR, _cuda, True,
           want=want)


def _irregular_times(rng, B, T):
    """Per-series grids with repeated times (dt = 0 passes the state through), one of them at
    the first observation after a checkpoint row."""
    dts = rng.choice([0.0, 0.5, 1.0, 2.0], (B, T))
    dts[:, K + 1] = 0.0
    return np.cumsum(dts, axis=1) + rng.uniform(1, 5, (B, 1))


@pytest.mark.parametrize("name", ["shared_times", "per_series_G", "per_series_F"])
@pytest.mark.parametrize("T", [2 * K + 1, 300])
@pytest.mark.parametrize("keep_init", [True, False])
def test_fused_irregular_grids(eng, name, T, keep_init):
    from bayesian_dlms_b200 import Model, TIME_MAJOR, build_batch_model, dlm, model_to_device
    rng = np.random.default_rng(sum(map(ord, name)) + T + keep_init)
    B = 29
    V, W, m0, C0 = _params(2)
    if name == "per_series_F":  # regression covariates: F_t = (1, x_t), G = I
        times = _irregular_times(rng, B, T)
        xs = rng.standard_normal((B, T, 1))
        mods = [dlm.Dlm(lambda t, xb=xs[b], tb=times[b]: np.r_[1.0, xb[np.searchsorted(tb, t)]].reshape(2, 1),
                        lambda dt: np.eye(2)) for b in range(B)]
    else:  # continuous-time trend: G(dt) = [[1, dt], [0, 1]]
        mods = [dlm.Dlm(lambda t: np.array([[1.0], [0.0]]),
                        lambda dt: np.array([[1.0, dt], [0.0, 1.0]]))] * B
        times = (np.tile(_irregular_times(rng, 1, T), (B, 1)) if name == "shared_times"
                 else _irregular_times(rng, B, T))
    y = _missing(np.stack([H.simulate(mods[b], V, W, m0, C0, times[b], rng, missing=0.1)
                           for b in range(B)]), T, int(keep_init))
    if name == "shared_times":
        model = Model.build(mods[0], times[0])
    else:
        model = model_to_device(build_batch_model(mods, times, layout=TIME_MAJOR), "cuda")
        assert ("G" if name == "per_series_G" else "F") in model.per_series
    _check(eng, model, mods, times, y, V, W, m0, C0, TIME_MAJOR, _cuda, keep_init)


@pytest.mark.parametrize("n", [1, 2])
def test_fused_series_major_host_buffers(eng, n):
    from bayesian_dlms_b200 import Model, SERIES_MAJOR, dlm
    rng = np.random.default_rng(7 + n)
    B, T = 33, 3 * K + 3
    V, W, m0, C0 = _params(n)
    mod = dlm.polynomial(n)
    times = np.tile(np.arange(1, T + 1, dtype=np.float64), (B, 1))
    y = _missing(np.stack([H.simulate(mod, V, W, m0, C0, times[b], rng, missing=0.1) for b in range(B)]), T, 1)
    _check(eng, Model.build(mod, T=T), [mod] * B, times, y, V, W, m0, C0, SERIES_MAJOR,
           np.ascontiguousarray, True)

"""Host-side model assembly (CPU): flattening the Dlm closures for a time grid."""
import numpy as np

from bayesian_dlms_b200 import dlm
from bayesian_dlms_b200.batch import Model


def _brute(mod, times, t_init=None):
    t0 = times.min() - 1.0 if t_init is None else t_init
    prev = np.concatenate([[t0], times[:-1]])
    F = np.stack([dlm.cm(mod.f(float(t))) for t in times])
    G = np.stack([dlm.cm(mod.g(float(dt))) for dt in times - prev])
    return F, G


def test_materialise_matches_per_step_evaluation():
    rng = np.random.default_rng(0)
    times = np.cumsum(rng.choice([0.5, 1.0, 2.0], 40))
    for mod in (dlm.polynomial(2), dlm.polynomial(1) + dlm.seasonal(24, 3),
                dlm.polynomial(1) * dlm.polynomial(1),
                dlm.regression([np.array([float(i)]) for i in range(60)])):
        tt = np.arange(1.0, 41.0) if not getattr(mod, "f_const", False) else times
        F, f_tv, G, g_tv, n, p = dlm.materialise(mod, tt)
        Fb, Gb = _brute(mod, tt)
        assert np.array_equal(F if f_tv else np.tile(F, (len(tt), 1)), Fb)
        assert np.array_equal(G if g_tv else np.tile(G, (len(tt), 1)), Gb)
    assert dlm.polynomial(3).f_const and (dlm.polynomial(1) + dlm.seasonal(12, 2)).f_const
    assert not dlm.regression([np.zeros(1)] * 3).f_const
    assert not (dlm.polynomial(1) * dlm.regression([np.zeros(1)] * 3)).f_const


def test_regular_grid_is_detected_and_long_grids_are_cheap():
    m = Model.build(dlm.polynomial(2), T=1 << 20)       # one f and one g evaluation
    assert m.times is None and not m.f_tv and not m.g_tv and m.T == 1 << 20
    m = Model.build(dlm.polynomial(1) + dlm.seasonal(24, 2), times=np.arange(1.0, 11.0))
    assert m.times is None and not m.g_tv
    m = Model.build(dlm.polynomial(1) + dlm.seasonal(24, 2), times=np.array([1.0, 2.0, 4.0]))
    assert m.times is not None and m.g_tv and m.G.size == 3 * 25


def test_resume_time_sets_the_first_increment():
    mod = dlm.polynomial(1) + dlm.seasonal(24, 2)
    times = np.array([10.0, 11.0, 13.0])
    F, f_tv, G, g_tv, n, p = dlm.materialise(mod, times, t_init=9.5)
    _, Gb = _brute(mod, times, 9.5)
    assert g_tv and np.array_equal(G, Gb)
    m = Model.build(mod, times, t_init=9.5)
    assert m.t_init is not None and m.t_init[0] == 9.5 and m.times is not None
    # forecast grid: first increment 0 (oneStepPrediction on the state itself)
    F, f_tv, G, g_tv, n, p = dlm.materialise(mod, 20.0 + np.arange(4.0), t_init=20.0)
    assert np.array_equal(G[0], dlm.cm(mod.g(0.0))) and np.array_equal(G[1], dlm.cm(mod.g(1.0)))


def test_build_batch_model_passes_per_series_only_what_differs():
    """Per-series grids (Data.time differs by series, Dlm.scala:94): times always travel per series;
    G only when g(dt) really differs (seasonal on irregular grids), F only with per-series closures
    (regression covariates); polynomial G and F stay shared."""
    import numpy as np
    from bayesian_dlms_b200 import SERIES_MAJOR, TIME_MAJOR, build_batch_model, dlm
    rng = np.random.default_rng(0)
    B, T = 5, 9
    times = np.cumsum(rng.choice([0.5, 1.0, 2.0], (B, T)), axis=1)
    m = build_batch_model(dlm.polynomial(2), times)
    assert m.per_series == ("times",) and not m.f_tv and not m.g_tv
    assert m.times.shape == (B, T, 1) and m.G.shape == (4,) and m.F.shape == (2,)
    seas = dlm.polynomial(1) + dlm.seasonal(24, 2)
    m = build_batch_model(seas, times, layout=TIME_MAJOR)
    assert m.per_series == ("times", "G") and m.g_tv and m.G.shape == (T, 25, B) and m.times.shape == (T, 1, B)
    # G of series b, step t is g(dt_t) of THAT series' grid, first dt = 1 (KalmanFilter.scala:116-117)
    b, t = 3, 4
    want = seas.g(times[b, t] - times[b, t - 1])
    assert np.array_equal(m.G[t, :, b], dlm.cm(want))
    assert np.array_equal(m.G[0, :, b], dlm.cm(seas.g(1.0)))
    xs = rng.standard_normal((B, T))
    mods = [dlm.Dlm(lambda t_, xb=xs[i], tb=times[i]: np.r_[1.0, xb[np.searchsorted(tb, t_)]].reshape(2, 1),
                    lambda dt: np.eye(2)) for i in range(B)]
    m = build_batch_model(mods, times, layout=SERIES_MAJOR)
    assert m.per_series == ("times", "F") and m.f_tv and m.F.shape == (B, T, 2)
    assert np.array_equal(m.F[2, 5], [1.0, xs[2, 5]])


def test_mirror_batch_padding_of_ragged_series():
    """_prep_batch pads a short series with None observations AT ITS LAST TIME (dt = 0: the state
    passes through) and keeps per-series DlmParameters column-major."""
    import numpy as np
    from bayesian_dlms_b200 import Data, DlmParameters, polynomial
    from bayesian_dlms_b200.reference_api import _prep_batch
    yss = [[Data(1.0, [0.5]), Data(2.5, [None]), Data(4.0, [1.5])], [Data(10.0, [2.0])]]
    ps = [DlmParameters(v=[[2.0]], w=[[1.0, 0.2], [0.3, 4.0]], m0=[0.0, 1.0], c0=np.eye(2)),
          DlmParameters(v=[[3.0]], w=np.eye(2), m0=[2.0, 3.0], c0=2 * np.eye(2))]
    model, params, times, y, lens = _prep_batch(polynomial(2), yss, ps)
    assert list(lens) == [3, 1] and y.shape == (2, 3, 1)
    assert np.array_equal(times[1], [10.0, 10.0, 10.0]) and np.isnan(y[1, 1:, 0]).all() and np.isnan(y[0, 1, 0])
    assert "times" in model.per_series and params["per_series"] == ("V", "W", "m0", "C0")
    assert np.array_equal(params["W"][0], [1.0, 0.3, 0.2, 4.0])   # column-major


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver times beside the CUDA arm) runs without
    a GPU and prints ONE JSON line with the contract's keys; its e2e repeats its own value (no
    copies on a CPU run) and its cpu_baseline says what was timed."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True
    assert d["metric"] == "filter+smoother series-steps/s" and d["unit"] == "series-steps/s"
    assert d["dtype"] == "f64" and d["n_gpus"] == 1 and d["value"] > 0
    assert d["config"]["workload"].startswith("config2: polynomial(2)")
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"]
    assert " x 1 passes " in d["cpu_baseline"]["sample"]     # --steps 1: one timed pass
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0}

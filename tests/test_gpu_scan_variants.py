"""The parallel-in-time scan (csrc/scan.cu) across its kernel variants, against the sequential
kernel (1e-9 relative, the scan's contract, DESIGN.md section 6) and, up to T = 5000, against the
extended-precision reference of tests/test_scan_reference_cpu.py (sequential kernel within 1e-12,
scan within 1e-9).

Every model here has a non-zero m0 and full SPD W and C0, and n = 2..4 use seasonal blocks
(rotation G, F != e1).  The cases reach what tests/test_gpu_scan.py does not: n = 4, keep_init = 0,
the scalar-store apply kernels behind unaligned outputs, level-2 block edges, missing values at
thread-range edges, output subsets, the context's model-table cache, the opt-in dispatch and the
status word."""
import numpy as np
import pytest

from test_scan_reference_cpu import (LEVEL2_EDGE_ROWS, MODEL_NAMES, TOL_LD, _ld_filter_smooth,
                                     close, ld_err, model_arrays, scan_model, simulate)

pytestmark = pytest.mark.gpu
TOL = 1e-9
LD_MAX_T = 5000
FIELDS = ("m", "C", "a", "R", "f", "Q", "s", "S")
DIMS = lambda n: dict(m=n, C=n * n, a=n, R=n * n, f=1, Q=1, s=n, S=n * n)  # noqa: E731


@pytest.fixture(scope="module")
def eng():
    import torch
    assert torch.cuda.is_available()
    from bayesian_dlms_b200 import default_engine
    return default_engine(0)


def _setup(name, T, seed, missing=0.02, **scale):
    from bayesian_dlms_b200 import Model
    mod, V, W, m0, C0 = scan_model(name, **scale)
    y = simulate(mod, V, W, m0, C0, T, seed, missing)
    return mod, Model.build(mod, T=T), dict(V=V, W=W, m0=m0, C0=C0), y


def _dev(y):
    import torch
    return torch.from_numpy(np.ascontiguousarray(y)).cuda()


def _np(out):
    return {k: v.cpu().numpy() for k, v in out.items() if k != "status"}


def _seq(eng, model, params, yd, keep_init):
    from bayesian_dlms_b200 import TIME_MAJOR
    out = eng.filter_smooth(model, params, yd.reshape(-1, 1, 1).contiguous(), layout=TIME_MAJOR,
                            keep_init=bool(keep_init), textbook=True)
    eng.sync()
    return {k: v[:, :, 0].cpu().numpy() for k, v in out.items() if k != "status"}


def _scan(eng, model, params, yd, keep_init, want=FIELDS):
    import torch
    from bayesian_dlms_b200.scan import scan_filter_smooth
    out = scan_filter_smooth(eng, model, params, yd, keep_init=bool(keep_init), want=want)
    torch.cuda.synchronize()
    st = int(out["status"][0])
    return _np(out), st


def _ld(mod, params, y, keep_init):
    F, G = model_arrays(mod, params["m0"].size)
    return _ld_filter_smooth(F, G, params["V"], params["W"], params["m0"], params["C0"], y, keep_init)


def _check(got, seq, ref=None, tag=()):
    for k in FIELDS:
        if k not in got:
            continue
        assert got[k].shape == seq[k].shape, (k, tag)
        e = close(got[k], seq[k])
        assert e < TOL, (k, tag, "scan vs sequential", e)
        if ref is not None:
            es, eg = ld_err(seq[k], ref[k]), ld_err(got[k], ref[k])
            assert es < TOL_LD, (k, tag, "sequential vs longdouble", es)
            assert eg < TOL, (k, tag, "scan vs longdouble", eg)


def _same(a, b, keys=FIELDS, tag=()):
    for k in keys:
        assert np.array_equal(a[k], b[k], equal_nan=True), (k, tag)


# ---------------------------------------------------------------------------- 1. shapes
@pytest.mark.parametrize("name", MODEL_NAMES)
@pytest.mark.parametrize("keep_init", [0, 1])
@pytest.mark.parametrize("T", [1, 2, 63, 64, 65, 1000, 40_001])
def test_shapes(eng, name, keep_init, T):
    mod, model, params, y = _setup(name, T, seed=T + 11 * keep_init)
    yd = _dev(y)
    got, st = _scan(eng, model, params, yd, keep_init)
    assert st == 0
    _check(got, _seq(eng, model, params, yd, keep_init),
           _ld(mod, params, y, keep_init) if T <= LD_MAX_T else None, (name, keep_init, T))


# ---------------------------------------------------------------------------- 2. level-2 edges
@pytest.mark.parametrize("name", ["n1", "n4"])
@pytest.mark.parametrize("keep_init", [0, 1])
@pytest.mark.parametrize("rows", LEVEL2_EDGE_ROWS)
def test_level2_block_edges(eng, name, keep_init, rows):
    """rows_per_thread is 16 at these T on any occupancy (test_scan_reference_cpu), so the forward
    pass has M + 1 = ceil(rows / 16) + 1 level-2 elements on both sides of 1024 and 2048, and the
    backward pass (one row fewer) too."""
    T = rows - keep_init
    _, model, params, y = _setup(name, T, seed=rows, missing=0.01)
    yd = _dev(y)
    got, st = _scan(eng, model, params, yd, keep_init)
    assert st == 0
    _check(got, _seq(eng, model, params, yd, keep_init), tag=(name, keep_init, rows))


# ---------------------------------------------------------------------------- 3. unaligned buffers
def _scan_views(eng, model, params, yd, keep_init, offset):
    """bdlm_scan_filter_smooth into views `offset` doubles into larger tensors, guards around."""
    import torch
    from bayesian_dlms_b200 import _capi as capi
    from bayesian_dlms_b200.batch import bound_engine
    from bayesian_dlms_b200.scan import _problem
    n, rows, guard = model.n, model.T + keep_init, 8
    with bound_engine(eng):
        pr, keep = _problem(model, params, yd, bool(keep_init))
    bufs, views = {}, {}
    for k, d in DIMS(n).items():
        bufs[k] = torch.full((offset + rows * d + guard,), -7.25, dtype=torch.float64, device="cuda")
        views[k] = bufs[k][offset:offset + rows * d]
    ko, so = capi.KfOut(), capi.SmoothOut()
    for k in ("m", "C", "a", "R", "f", "Q"):
        setattr(ko, k, views[k].data_ptr())
    for k in ("s", "S"):
        setattr(so, k, views[k].data_ptr())
    st = torch.zeros((1,), dtype=torch.int32, device="cuda")
    eng.ctx.check(capi.load().bdlm_scan_filter_smooth(eng.ctx.handle, pr, ko, so, st.data_ptr()))
    torch.cuda.synchronize()
    out = {}
    for k, d in DIMS(n).items():
        b = bufs[k].cpu().numpy()
        assert np.all(b[:offset] == -7.25) and np.all(b[offset + rows * d:] == -7.25), k
        out[k] = b[offset:offset + rows * d].reshape(rows, d)
    return out, int(st[0])


@pytest.mark.parametrize("name", ["n1", "n2", "n3", "n4"])
@pytest.mark.parametrize("y_aligned", [True, False])
@pytest.mark.parametrize("T,keep_init", [(1, 0), (4999, 1), (1003, 0)])
def test_unaligned_outputs_take_the_scalar_stores_bit_identically(eng, name, y_aligned, T, keep_init):
    """Outputs 8 bytes past a 32-byte boundary fail dense_aligned, so fwd_apply_kernel<N, false, *>
    and bwd_apply_kernel<N, false> write them; an offset y also runs fwd_reduce_kernel<N, false>.
    Same arithmetic as the 256-bit stores: the results must be the same bits."""
    import torch
    _, model, params, y = _setup(name, T, seed=T + 3)
    yd = _dev(y)
    if not y_aligned:
        yb = torch.empty(T + 5, dtype=torch.float64, device="cuda")
        yb[5:] = yd
        yd = yb[5:]
        assert yd.data_ptr() % 32 == 8
    ref, st_ref = _scan(eng, model, params, _dev(y), keep_init)
    got, st = _scan_views(eng, model, params, yd, keep_init, offset=5)
    assert st == st_ref == 0
    _same(got, ref, tag=(name, y_aligned, T))
    _check(got, _seq(eng, model, params, _dev(y), keep_init), tag=(name, T))


# ---------------------------------------------------------------------------- 4. output subsets
@pytest.mark.parametrize("name", ["n2", "n4s"])
@pytest.mark.parametrize("want", [("s", "S"), ("m", "C", "s", "S"), ("a", "R", "f", "Q", "s", "S")])
def test_output_subsets_are_bit_identical_to_the_full_call(eng, name, want):
    _, model, params, y = _setup(name, 20_000, seed=4)
    yd = _dev(y)
    full, _ = _scan(eng, model, params, yd, 1)
    part, st = _scan(eng, model, params, yd, 1, want=want)
    assert st == 0 and set(part) == set(want)
    _same(part, full, keys=want, tag=(name, want))


# ---------------------------------------------------------------------------- 5. missing data
def _missing(case, T, keep_init):
    """Observation indices (t = row - keep_init) to blank out."""
    if case == "first_and_last":
        return [0, T - 1]
    if case == "range_first_row":      # first row of two threads' 16-row ranges
        return [16 * 100 - keep_init, 16 * 250 - keep_init]
    if case == "range_last_row":
        return [16 * 100 + 15 - keep_init, 16 * 250 + 15 - keep_init]
    if case == "run_5000":             # crosses the level-2 edge at rows 16368-16384
        return slice(14_000, 19_000)
    return slice(None)


# A long gap inflates the state covariance by decades; the scan's combines then lose more than the
# sequential recursion does (5000 steps: 2.4e-7 against it on S, measured on B200; DESIGN.md
# section 6, "Conditioning").
TOL_GAP = 1e-6


@pytest.mark.parametrize("name", MODEL_NAMES)
@pytest.mark.parametrize("case", ["first_and_last", "range_first_row", "range_last_row", "run_5000", "all"])
@pytest.mark.parametrize("keep_init", [0, 1])
def test_missing_values(eng, name, case, keep_init):
    T = 40_001 if case == "run_5000" else 5000 if case != "all" else 1000
    mod, model, params, y = _setup(name, T, seed=17, missing=0.0)
    y[_missing(case, T, keep_init)] = np.nan
    yd = _dev(y)
    got, st = _scan(eng, model, params, yd, keep_init)
    seq = _seq(eng, model, params, yd, keep_init)
    assert st == 0
    if case == "run_5000":
        for k in FIELDS:
            e = close(got[k], seq[k])
            print(name, keep_init, k, "%.2e" % e)
            assert e < TOL_GAP, (k, e)
        return
    _check(got, seq, _ld(mod, params, y, keep_init) if T <= LD_MAX_T else None, (name, case, keep_init))


def test_all_missing_across_level2_blocks(eng):
    _, model, params, y = _setup("n3", 20_000, seed=18, missing=0.0)
    yd = _dev(np.full(20_000, np.nan))
    got, st = _scan(eng, model, params, yd, 1)
    seq = _seq(eng, model, params, yd, 1)
    assert st == 0
    for k in FIELDS:   # a 20 000-step gap: C measured 1.3e-8 from the sequential kernel
        assert close(got[k], seq[k]) < TOL_GAP, (k, close(got[k], seq[k]))


# ---------------------------------------------------------------------------- 6. table cache
def test_model_table_cache_follows_every_model_change():
    """The context keeps the level-1 table of the last (n, G, F, W, V).  Changing any one of them
    on the same context must give the bits a fresh context gives."""
    import torch
    from bayesian_dlms_b200 import Engine, Model
    mod, V, W, m0, C0 = scan_model("n2")
    T = 5000
    y = simulate(mod, V, W, m0, C0, T, seed=6)
    yd = _dev(y)
    base = Model.build(mod, T=T)
    W01 = W.copy()
    W01[0, 1] = W01[1, 0] = W[0, 1] * 0.5
    Fm = Model.build(mod, T=T)
    Fm.F = np.array([1.0, 0.25])
    Gm = Model.build(mod, T=T)
    Gm.G = base.G * 0.999
    pa = dict(V=V, W=W, m0=m0, C0=C0)
    seq = [("A", base, pa), ("V", base, dict(pa, V=V * 3.0)), ("W01", base, dict(pa, W=W01)),
           ("F", Fm, pa), ("G", Gm, pa), ("A again", base, pa)]
    e = Engine(0)
    fresh = {}
    for tag, model, params in seq:
        got, st = _scan(e, model, params, yd, 1)
        if tag not in fresh:
            fresh[tag] = _scan(Engine(0), model, params, yd, 1)[0]
        _same(got, fresh[tag if tag != "A again" else "A"], tag=(tag,))
    # a stream switch drops the table the old stream uploaded
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        e.use_torch_stream()
        for tag, model, params in (seq[1], seq[0]):
            got, _ = _scan(e, model, params, yd, 1)
            _same(got, fresh[tag], tag=("stream", tag))
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------- 7. opt-in dispatch
@pytest.mark.parametrize("T", [4095, 4096])
def test_opt_in_dispatch_threshold(eng, T):
    from bayesian_dlms_b200 import SERIES_MAJOR
    _, model, params, y = _setup("n2", T, seed=T)
    yd = _dev(y.reshape(1, T, 1))
    seq = _np(eng.filter_smooth(model, params, yd, layout=SERIES_MAJOR, textbook=True))
    pit = _np(eng.filter_smooth(model, params, yd, layout=SERIES_MAJOR, textbook=True,
                                parallel_in_time=True))
    eng.sync()
    if T < 4096:
        _same(pit, seq)
    else:
        for k in FIELDS:
            assert close(pit[k], seq[k]) < TOL, k


def test_opt_in_dispatch_n4_needs_textbook(eng):
    from bayesian_dlms_b200 import SERIES_MAJOR
    _, model, params, y = _setup("n4", 5000, seed=41)
    yd = _dev(y.reshape(1, 5000, 1))
    seq = _np(eng.filter_smooth(model, params, yd, layout=SERIES_MAJOR))
    pit = _np(eng.filter_smooth(model, params, yd, layout=SERIES_MAJOR, parallel_in_time=True))
    eng.sync()
    _same(pit, seq)


@pytest.mark.parametrize("name", ["n4", "n4s"])
@pytest.mark.parametrize("where", ["device", "host"])
@pytest.mark.parametrize("keep_init", [0, 1])
def test_opt_in_dispatch_n4_textbook(eng, name, where, keep_init):
    from bayesian_dlms_b200 import SERIES_MAJOR
    T = 5000
    mod, model, params, y = _setup(name, T, seed=42 + keep_init)
    yy = y.reshape(1, T, 1).copy()
    yy = _dev(yy) if where == "device" else yy
    kw = dict(layout=SERIES_MAJOR, keep_init=bool(keep_init), textbook=True)
    seq = eng.filter_smooth(model, params, yy, **kw)
    pit = eng.filter_smooth(model, params, yy, parallel_in_time=True, **kw)
    eng.sync()
    npy = lambda x: x.cpu().numpy() if hasattr(x, "cpu") else x  # noqa: E731
    assert int(npy(pit["status"])[0]) == 0
    ref = _ld(mod, params, y, keep_init)
    _check({k: npy(pit[k])[0] for k in FIELDS}, {k: npy(seq[k])[0] for k in FIELDS}, ref,
           (name, where, keep_init))


# ---------------------------------------------------------------------------- 8. status
@pytest.mark.parametrize("name", ["n1", "n2", "n4"])
@pytest.mark.parametrize("case", ["control", "inf", "zero_variances"])
def test_status_matches_the_sequential_route(eng, name, case):
    """Same bdlm_kf_filter_smooth call with and without BDLM_PARALLEL_IN_TIME: same status word.
    +inf in y makes the final (row-0 smoothed) state non-finite: BDLM_ST_NONFINITE.  V = W = C0 = 0
    gives Q = 0 (BDLM_ST_SINGULAR) and then 0/0 everywhere (BDLM_ST_NONFINITE)."""
    from bayesian_dlms_b200 import SERIES_MAJOR, _capi as capi
    T = 5000
    _, model, params, y = _setup(name, T, seed=8)
    if case == "inf":
        y[1234] = np.inf
    if case == "zero_variances":
        n = model.n
        params = dict(params, V=np.zeros((1, 1)), W=np.zeros((n, n)), C0=np.zeros((n, n)))
    yd = _dev(y.reshape(1, T, 1))
    kw = dict(layout=SERIES_MAJOR, textbook=True)
    seq = eng.filter_smooth(model, params, yd, **kw)
    pit = eng.filter_smooth(model, params, yd, parallel_in_time=True, **kw)
    eng.sync()
    s_seq, s_pit = int(seq["status"][0]), int(pit["status"][0])
    print(name, case, "sequential status", s_seq, "scan status", s_pit)
    assert s_pit == s_seq
    expect = {"control": 0, "inf": capi.ST_NONFINITE,
              "zero_variances": capi.ST_SINGULAR | capi.ST_NONFINITE}[case]
    assert s_seq == expect


@pytest.mark.parametrize("keep_init", [0, 1])
def test_status_nonfinite_single_row_and_short_series(eng, keep_init):
    """The scan's row 0 comes from the backward sweep, or, for a single row, from the terminal
    element itself: both flag a non-finite state like the sequential kernel."""
    from bayesian_dlms_b200 import Model, TIME_MAJOR
    mod, V, W, m0, C0 = scan_model("n2")
    params = dict(V=V, W=W, m0=m0, C0=C0)
    for T in (1, 2, 100):
        y = np.linspace(0.0, 1.0, T)
        y[-1] = np.inf
        model = Model.build(mod, T=T)
        yd = _dev(y)
        _, st = _scan(eng, model, params, yd, keep_init)
        seq = eng.filter_smooth(model, params, yd.reshape(-1, 1, 1).contiguous(), layout=TIME_MAJOR,
                                keep_init=bool(keep_init), textbook=True)
        eng.sync()
        assert st == int(seq["status"][0]) != 0, (T, st)


# ---------------------------------------------------------------------------- 9. emulated ranks
@pytest.mark.parametrize("name", ["n4", "n4s"])
@pytest.mark.parametrize("world", [2, 5])
def test_device_side_protocol_emulated_ranks_n4(eng, name, world):
    import torch
    from bayesian_dlms_b200 import Engine, Model
    from bayesian_dlms_b200.scan import DistScan
    from bayesian_dlms_b200.sharding import shard_range
    T = 7001
    mod, model, params, y = _setup(name, T, seed=31 + world)
    yd = _dev(y)
    seq = _seq(eng, model, params, yd, 1)
    ranks = []
    for r in range(world):
        lo, hi = shard_range(T, r, world)
        e = Engine(0)
        e.use_torch_stream()
        ranks.append(DistScan(e, Model.build(mod, T=hi - lo), params, yd[lo:hi].contiguous(), r, world))
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
    assert all(int(d.status[0]) == 0 for d in ranks)
    got = {k: torch.cat([d.out[k] for d in ranks]).cpu().numpy() for k in FIELDS}
    _check(got, seq, tag=(name, world))


# ---------------------------------------------------------------------------- 10. conditioning
@pytest.mark.parametrize("name", ["n2", "n4"])
@pytest.mark.parametrize("C0_scale", [10.0, 1e4, 1e6])
@pytest.mark.parametrize("ratio", [1e-4, 1.0, 1e4])
def test_conditioning_sweep(eng, name, C0_scale, ratio):
    """W / V and the prior scale over eight decades: wherever the sequential kernel is within
    1e-12 of the longdouble reference, the scan must be within 1e-9 of it.  Where the prior is
    large against V and W the scan loses more than the sequential recursion: measured on B200 up
    to 1.3e4 times its error (C0 1e6, W / V 1e-4: 1.8e-7 and 2.2e-3); that bound is pinned at 3e4."""
    T = 2000
    mod, model, params, y = _setup(name, T, seed=5, missing=0.0, W_scale=ratio, C0_scale=C0_scale, V=1.0)
    yd = _dev(y)
    got, st = _scan(eng, model, params, yd, 1)
    seq = _seq(eng, model, params, yd, 1)
    ref = _ld(mod, params, y, 1)
    es = max(ld_err(seq[k], ref[k]) for k in FIELDS)
    eg = max(ld_err(got[k], ref[k]) for k in FIELDS)
    print("%s C0 %.0e W/V %.0e: sequential %.2e, scan %.2e vs longdouble" % (name, C0_scale, ratio, es, eg))
    assert st == 0
    if es < TOL_LD:
        assert eg < TOL, (es, eg)
    assert eg < max(TOL, 3e4 * es), (es, eg)

"""Per-step F (f_tv: dynamic regression) on the parallel-in-time scan: filter + smoother,
log-likelihoods with the last state, FFBS with its Gibbs statistics, the time-sharded phases and the
BDLM_PARALLEL_IN_TIME routes, against the sequential kernels at the scan's 1e-9 contract (fields
relative to each row's largest entry, sums relative to sum_t |term_t|)."""
import numpy as np
import pytest

from test_gpu_scan_sharded import _concat_gather, _run_ffbs, _run_loglik, _same_on_every_rank
from test_scan_ffbs_reference_cpu import row_err
from test_scan_reference_cpu import LEVEL2_EDGE_ROWS, ld_err, model_arrays, scan_model, simulate
from test_scan_regression_cpu import REG_NAMES, ld_filter_smooth_tv, regression_model, simulate_tv

pytestmark = pytest.mark.gpu
TOL = 1e-9
TOL_GAP = 1e-6   # across a 5000-step gap, as the time-invariant scan's tests (DESIGN.md section 6)
LD_MAX_T = 5000
FIELDS = ("m", "C", "a", "R", "f", "Q", "s", "S")
STATS = ("ssy", "ny", "ssw", "scatter")


@pytest.fixture(scope="module")
def eng():
    import torch
    assert torch.cuda.is_available()
    from bayesian_dlms_b200 import default_engine
    return default_engine(0)


def _dev(x):
    import torch
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _npy(x):
    return x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)


def _model(F, G, per_series=False):
    """Model of a per-step F [T][n]: host (shared) or, per_series, a device tensor (1, T, n)."""
    from bayesian_dlms_b200 import Model, dlm
    T, n = F.shape
    Fm = _dev(F.reshape(1, T, n)) if per_series else np.ascontiguousarray(F.ravel())
    return Model(Fm, dlm.cm(G), True, False, n, 1, T, None, None, ("F",) if per_series else ())


def _case(name, T, seed, missing=0.02, gap=False, V=None):
    _, F, G, V0, W, m0, C0 = regression_model(name, T, seed)
    V = V0 if V is None else V
    y = simulate_tv(F, G, V0, W, m0, C0, seed + 1, missing)
    if gap:
        y[T // 3:T // 3 + 5000] = np.nan
    return F, G, dict(V=V, W=W, m0=m0, C0=C0), y


def _scan_fs(eng, model, params, yd):
    import torch
    from bayesian_dlms_b200.scan import scan_filter_smooth
    out = scan_filter_smooth(eng, model, params, yd)
    torch.cuda.synchronize()
    return {k: _npy(v) for k, v in out.items()}


def _seq_fs(eng, model, params, yd, pit=False):
    from bayesian_dlms_b200 import TIME_MAJOR
    out = eng.filter_smooth(model, params, yd.reshape(-1, 1, 1), layout=TIME_MAJOR, textbook=True,
                            parallel_in_time=pit)
    eng.sync()
    return {k: int(_npy(v).ravel()[0]) if k == "status" else _npy(v)[..., 0] for k, v in out.items()}


def _scan_ll(eng, model, params, yd):
    import torch
    from bayesian_dlms_b200.scan import scan_loglik
    out = scan_loglik(eng, model, params, yd, last=True)
    torch.cuda.synchronize()
    return {k: _npy(v) for k, v in out.items()}


def _seq_ll(eng, model, params, yd, pit=False):
    from bayesian_dlms_b200 import TIME_MAJOR
    out = eng.filter_last(model, params, yd.reshape(-1, 1, 1), layout=TIME_MAJOR, loglik=True,
                          parallel_in_time=pit)
    eng.sync()
    return {k: _npy(v).reshape(-1) for k, v in out.items()}


def _scan_fb(eng, model, params, yd, zd=None):
    import torch
    from bayesian_dlms_b200.scan import scan_ffbs
    out = scan_ffbs(eng, model, params, yd, zd, want_kf=("a", "R", "f", "Q"))
    torch.cuda.synchronize()
    return {k: _npy(v) for k, v in out.items()}


def _seq_fb(eng, model, params, yd, zd=None, pit=False):
    from bayesian_dlms_b200 import TIME_MAJOR
    T, n = model.T, model.n
    out = eng.ffbs(model, params, yd.reshape(T, 1, 1), None if zd is None else zd.reshape(T + 1, n, 1),
                   layout=TIME_MAJOR, want_kf=("a", "R", "f", "Q"), stats=True, parallel_in_time=pit)
    eng.sync()
    return {k: int(_npy(v).ravel()[0]) if k == "status" else _npy(v)[..., 0] for k, v in out.items()}


def _normals(eng, T, n, mode, seed):
    if mode == "z":
        return _dev(np.random.default_rng(seed).standard_normal((T + 1, n)))
    eng.ctx.set_rng(seed, 3, 0)
    return None


def _ll_scale(rows, y, W):
    """sum_t |term_t| of both log-likelihoods, from filter rows 1..T."""
    obs = ~np.isnan(y)
    sd = np.sqrt(rows["Q"][1:, 0][obs])
    dd = (y[obs] - rows["f"][1:, 0][obs]) / sd
    inn = np.sum(np.abs(-dd * dd / 2 - np.log(np.sqrt(2 * np.pi) * sd)))
    d = rows["m"][1:] - rows["a"][1:]
    Wi = np.linalg.inv(W)
    tr = np.sum(np.abs(-0.5 * np.einsum("ti,ij,tj->t", d, Wi, d) - 0.5 * np.log(np.linalg.det(2 * np.pi * W))))
    return tr, inn


def _stats_terms(F, G, y, theta):
    """Per-step terms of ssy (observed steps), ssw and scatter of a path."""
    e = y - np.einsum("ti,ti->t", F, theta[1:])
    d = theta[1:] - theta[:-1] @ G.T
    return dict(ssy=np.where(np.isnan(e), 0.0, e * e), ssw=d * d,
                scatter=np.einsum("ti,tj->tij", d, d).reshape(len(d), -1))


def _stats_err(got, ref, terms):
    out = {}
    for k in ("ssy", "ssw", "scatter"):
        scale = np.maximum(np.sum(np.abs(terms[k]), axis=0), 1e-300)
        out[k] = float(np.max(np.abs(np.ravel(got[k]) - np.ravel(ref[k])) / np.ravel(scale)))
    return out


def _fields_err(got, ref, rows=slice(None)):
    return {k: ld_err(got[k][rows], ref[k][rows]) for k in FIELDS}


# ---------------------------------------------------------------------------- filter + smoother
EDGE_T = [LEVEL2_EDGE_ROWS[0] - 1, LEVEL2_EDGE_ROWS[4] - 1, LEVEL2_EDGE_ROWS[-1] - 1]


@pytest.mark.parametrize("name", REG_NAMES)
@pytest.mark.parametrize("T", [1, 65, 4096, 50_000] + EDGE_T)
def test_filter_smoother_against_the_sequential_kernel(eng, name, T):
    F, G, params, y = _case(name, T, seed=T % 1000 + 11)
    model, yd = _model(F, G), _dev(y)
    got, seq = _scan_fs(eng, model, params, yd), _seq_fs(eng, model, params, yd)
    assert int(got["status"][0]) == seq["status"] == 0
    e = _fields_err(got, seq)
    assert max(e.values()) < TOL, e
    if T <= LD_MAX_T:
        ref = ld_filter_smooth_tv(F, G, params["V"], params["W"], params["m0"], params["C0"], y, 1)
        e = _fields_err(got, ref)
        assert max(e.values()) < TOL, e


@pytest.mark.parametrize("name", ["r1", "r1s", "r2w"])
def test_gap_of_5000_steps(eng, name):
    T = 20_000
    F, G, params, y = _case(name, T, seed=5, gap=True)
    model, yd = _model(F, G), _dev(y)
    got, seq = _scan_fs(eng, model, params, yd), _seq_fs(eng, model, params, yd)
    assert int(got["status"][0]) == seq["status"] == 0
    e = _fields_err(got, seq)
    assert max(e.values()) < TOL_GAP, e
    ll, sl = _scan_ll(eng, model, params, yd), _seq_ll(eng, model, params, yd)
    tr, inn = _ll_scale(got, y, params["W"])
    assert abs(ll["innovations"][0] - sl["innovations"][0]) / inn < TOL_GAP
    assert abs(ll["transition"][0] - sl["transition"][0]) / tr < TOL_GAP


# ---------------------------------------------------------------------------- log-likelihoods
@pytest.mark.parametrize("name", REG_NAMES)
@pytest.mark.parametrize("T", [1, 4096, 50_000, EDGE_T[1]])
def test_loglik_and_last_state_against_the_sequential_kernel(eng, name, T):
    F, G, params, y = _case(name, T, seed=T % 1000 + 23)
    model, yd = _model(F, G), _dev(y)
    got, seq = _scan_ll(eng, model, params, yd), _seq_ll(eng, model, params, yd)
    assert int(got["status"][0]) == seq["status"] == 0
    tr, inn = _ll_scale(_scan_fs(eng, model, params, yd), y, params["W"])
    assert abs(got["transition"][0] - seq["transition"][0]) / tr < TOL
    assert abs(got["innovations"][0] - seq["innovations"][0]) / inn < TOL
    for k in ("m", "C"):
        assert np.max(np.abs(got[k] - seq[k])) / np.max(np.abs(seq[k])) < TOL, k


# ---------------------------------------------------------------------------- FFBS
@pytest.mark.parametrize("mode", ["z", "philox"])
@pytest.mark.parametrize("name", REG_NAMES)
@pytest.mark.parametrize("T", [1, 4096, 50_000, EDGE_T[2]])
def test_ffbs_against_the_sequential_kernel(eng, name, T, mode):
    F, G, params, y = _case(name, T, seed=T % 1000 + 37)
    model, yd = _model(F, G), _dev(y)
    n = model.n
    seq = _seq_fb(eng, model, params, yd, _normals(eng, T, n, mode, seed=T))
    got = _scan_fb(eng, model, params, yd, _normals(eng, T, n, mode, seed=T))
    assert int(got["status"][0]) == seq["status"] == 0
    assert row_err(got["theta"], seq["theta"]) < TOL
    for k in ("a", "R", "f", "Q"):
        assert row_err(got[k][1:], seq[k][1:]) < TOL, k
    es = _stats_err(got, seq, _stats_terms(F, G, y, seq["theta"]))
    assert max(es.values()) < TOL, es
    assert got["ny"][0] == seq["ny"][0] == np.sum(~np.isnan(y))


# ---------------------------------------------------------------------------- F on host and device
def test_host_and_device_F_give_the_same_bits(eng):
    import torch
    T = 50_000
    F, G, params, y = _case("r1s", T, seed=3)
    yd = _dev(y)
    zd = _dev(np.random.default_rng(4).standard_normal((T + 1, 4)))
    outs = []
    for m in (_model(F, G), _model(F, G, per_series=True)):
        outs.append(dict(**{"fs_" + k: v for k, v in _scan_fs(eng, m, params, yd).items()},
                         **{"ll_" + k: v for k, v in _scan_ll(eng, m, params, yd).items()},
                         **{"fb_" + k: v for k, v in _scan_fb(eng, m, params, yd, zd).items()}))
    torch.cuda.synchronize()
    for k in outs[0]:
        assert np.array_equal(outs[0][k], outs[1][k], equal_nan=True), k


def test_constant_rows_agree_with_the_time_invariant_scan(eng):
    """polynomial(2) + seasonal(7, 1) given as f_tv with every row F_t = F: a constant F of a
    regression is not identifiable (only F beta is observed), so the scan tests' n = 4 model."""
    from bayesian_dlms_b200 import Model, dlm
    T = 50_000
    mod, V, W, m0, C0 = scan_model("n4")
    params = dict(V=V, W=W, m0=m0, C0=C0)
    y = simulate(mod, V, W, m0, C0, T, 9, 0.02)
    F1, G = model_arrays(mod, 4)
    F = np.ascontiguousarray(np.broadcast_to(F1, (T, 4)))
    yd = _dev(y)
    zd = _dev(np.random.default_rng(2).standard_normal((T + 1, 4)))
    tv = _model(F, G)
    ti = Model(np.ascontiguousarray(F1), dlm.cm(G), False, False, 4, 1, T, None)
    a, b = _scan_fs(eng, tv, params, yd), _scan_fs(eng, ti, params, yd)
    e = _fields_err(a, b)
    assert max(e.values()) < TOL, e
    la, lb = _scan_ll(eng, tv, params, yd), _scan_ll(eng, ti, params, yd)
    for k in ("transition", "innovations"):
        assert abs(la[k][0] - lb[k][0]) < TOL * abs(lb[k][0]), k
    fa, fb = _scan_fb(eng, tv, params, yd, zd), _scan_fb(eng, ti, params, yd, zd)
    assert row_err(fa["theta"], fb["theta"]) < TOL
    assert max(_stats_err(fa, fb, _stats_terms(F, G, y, fb["theta"])).values()) < TOL


def test_per_step_calls_leave_the_model_table_alone():
    """A time-invariant call after per-step-F calls on the same context gives a fresh context's bits."""
    from bayesian_dlms_b200 import Engine, Model, dlm
    T = 20_000
    F, G, params, y = _case("r2", T, seed=21)
    yd = _dev(y)
    ti = Model(np.ascontiguousarray(F[0]), dlm.cm(G), False, False, 3, 1, T, None)
    tv = _model(F, G)

    def both(e, m):
        return {**{"fs_" + k: v for k, v in _scan_fs(e, m, params, yd).items()},
                **{"ll_" + k: v for k, v in _scan_ll(e, m, params, yd).items()}}
    fresh = both(Engine(0), ti)
    e = Engine(0)
    for m in (tv, ti, tv, tv, ti, tv):
        out = both(e, m)
        if m is ti:
            for k in fresh:
                assert np.array_equal(out[k], fresh[k], equal_nan=True), k


# ---------------------------------------------------------------------------- opt-in routes
@pytest.mark.parametrize("where", ["device", "host"])
@pytest.mark.parametrize("ps", [False, True])
def test_opt_in_routes_give_the_direct_scan_bits(eng, where, ps):
    from bayesian_dlms_b200 import SERIES_MAJOR
    T = 50_000
    F, G, params, y = _case("r1", T, seed=31)
    n = 2
    yd = _dev(y)
    direct_model = _model(F, G)
    fs, ll = _scan_fs(eng, direct_model, params, yd), _scan_ll(eng, direct_model, params, yd)
    zd = _dev(np.random.default_rng(6).standard_normal((T + 1, n)))
    fb = _scan_fb(eng, direct_model, params, yd, zd)
    model = _model(F, G, per_series=ps)
    if where == "host":
        if ps:
            model.F = np.ascontiguousarray(F.reshape(1, T, n))
        yy, zz = y.reshape(1, T, 1).copy(), _npy(zd).reshape(1, T + 1, n).copy()
    else:
        yy, zz = yd.reshape(1, T, 1), zd.reshape(1, T + 1, n)
    row = lambda x: _npy(x)[0]  # noqa: E731
    for pit in (True, False):
        f = eng.filter_smooth(model, params, yy, layout=SERIES_MAJOR, textbook=True, parallel_in_time=pit)
        l = eng.loglik(model, params, yy, layout=SERIES_MAJOR, parallel_in_time=pit)  # noqa: E741
        la = eng.filter_last(model, params, yy, layout=SERIES_MAJOR, parallel_in_time=pit)
        b = eng.ffbs(model, params, yy, zz, layout=SERIES_MAJOR, stats=True, parallel_in_time=pit)
        eng.sync()
        same = [np.array_equal(row(f[k]), fs[k], equal_nan=True) for k in FIELDS]
        same += [np.array_equal(_npy(l[k]), ll[k]) for k in ("transition", "innovations")]
        same += [np.array_equal(row(la["m"]), ll["m"]), np.array_equal(row(la["C"]), ll["C"])]
        same += [np.array_equal(row(b["theta"]), fb["theta"])] + [np.array_equal(row(b[k]), fb[k]) for k in STATS]
        if pit:
            assert all(same), same
            assert int(row(f["status"])) == int(row(b["status"])) == 0
        else:  # the sequential kernels: other bits
            assert not same[0], same


@pytest.mark.parametrize("case", ["ok", "singular"])
def test_status_is_the_sequential_status_with_the_flag_on_and_off(eng, case):
    T = 8192
    F, G, params, y = _case("r1", T, seed=41)
    if case == "singular":  # V = 0 and F_t = 0: Q_t = 0
        params = dict(params, V=np.array([[0.0]]))
        F = F.copy()
        F[5000] = 0.0
        y[5000] = 1.0
    model, yd = _model(F, G), _dev(y)
    zd = _dev(np.random.default_rng(1).standard_normal((T + 1, 2)))
    st = {}
    for pit in (False, True):
        st[pit] = (_seq_fs(eng, model, params, yd, pit)["status"], int(_seq_ll(eng, model, params, yd, pit)["status"][0]),
                   _seq_fb(eng, model, params, yd, zd, pit)["status"])
    direct = (int(_scan_fs(eng, model, params, yd)["status"][0]), int(_scan_ll(eng, model, params, yd)["status"][0]),
              int(_scan_fb(eng, model, params, yd, zd)["status"][0]))
    print(case, st, direct)
    assert st[True] == st[False] == direct
    from bayesian_dlms_b200 import _capi as capi
    assert all((s & capi.ST_SINGULAR) != 0 for s in direct) == (case == "singular")


# ---------------------------------------------------------------------------- time-sharded
def _cuts(T, world):
    from bayesian_dlms_b200.sharding import time_chunk
    return [time_chunk(T, r, world)[0] for r in range(world)] + [T]


def _chunks(F, G, params, yd, cuts, cls, per_series=False, **kw):
    from bayesian_dlms_b200 import Engine
    ranks = []
    world = len(cuts) - 1
    for r in range(world):
        lo, hi = cuts[r], cuts[r + 1]
        e = Engine(0)
        e.use_torch_stream()
        args = dict(kw)
        if cls.__name__ == "DistFfbs":
            z = args.pop("z", None)
            first = 0 if r == 0 else lo + 1
            rows = hi - lo + (r == 0)
            args.update(first_row=first, total_T=cuts[-1], z=None if z is None else z[first:first + rows].contiguous())
        m = _model(np.ascontiguousarray(F[lo:hi]), G, per_series)
        ranks.append(cls(e, m, params, yd[lo:hi].contiguous(), r, world, **args))
    return ranks


@pytest.mark.parametrize("world", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("name", ["r1", "r3", "r1s"])
def test_emulated_ranks_match_the_single_gpu_call(eng, name, world):
    import torch
    from bayesian_dlms_b200.scan import DistFfbs, DistLoglik, DistScan
    T = 20_001
    F, G, params, y = _case(name, T, seed=world + 50)
    yd = _dev(y)
    cuts = _cuts(T, world)
    per_series = world % 2 == 0  # host F on odd worlds, device F on even ones
    model = _model(F, G)
    one_fs, one_ll = _scan_fs(eng, model, params, yd), _scan_ll(eng, model, params, yd)
    zd = _dev(np.random.default_rng(world).standard_normal((T + 1, model.n)))
    one_fb = _scan_fb(eng, model, params, yd, zd)
    # filter + smoother
    ranks = _chunks(F, G, params, yd, cuts, DistScan, per_series)
    for d in ranks:
        d.forward_local()
    _concat_gather(ranks, "agg_f", "aggs_f")
    for d in ranks:
        d.forward_finish()
        d.backward_local()
    _concat_gather(ranks, "agg_b", "aggs_b")
    for d in ranks:
        d.backward_finish()
    torch.cuda.synchronize()
    for k in FIELDS:
        got = np.concatenate([_npy(d.out[k]) for d in ranks])
        assert ld_err(got, one_fs[k]) < TOL, k
    # log-likelihoods
    outs = _run_loglik(_chunks(F, G, params, yd, cuts, DistLoglik, per_series))
    _same_on_every_rank(outs, ("transition", "innovations", "status"))
    tr, inn = _ll_scale(one_fs, y, params["W"])
    assert int(outs[0]["status"][0]) == 0
    assert abs(outs[0]["transition"][0] - one_ll["transition"][0]) / tr < TOL
    assert abs(outs[0]["innovations"][0] - one_ll["innovations"][0]) / inn < TOL
    for k in ("m", "C"):
        assert np.max(np.abs(outs[-1][k] - one_ll[k])) / np.max(np.abs(one_ll[k])) < TOL, k
    # FFBS
    outs = _run_ffbs(_chunks(F, G, params, yd, cuts, DistFfbs, per_series, z=zd))
    _same_on_every_rank(outs, STATS + ("status",))
    theta = np.concatenate([o["theta"] for o in outs])
    assert row_err(theta, one_fb["theta"]) < TOL
    assert int(outs[0]["status"][0]) == 0 and outs[0]["ny"][0] == one_fb["ny"][0]
    es = _stats_err(outs[0], one_fb, _stats_terms(F, G, y, one_fb["theta"]))
    assert max(es.values()) < TOL, es


@pytest.mark.parametrize("world", [1, 2])
def test_communicator(eng, world):
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    from bayesian_dlms_b200.comm import Comm
    from bayesian_dlms_b200.sharding import time_chunk
    T = 20_001
    F, G, params, y = _case("r1s", T, seed=60)
    yd = _dev(y)
    model = _model(F, G)
    one_fs, one_ll = _scan_fs(eng, model, params, yd), _scan_ll(eng, model, params, yd)
    comm = Comm.single_process(list(range(world)))
    try:
        models, chunks, firsts = [], [], []
        for i, d in enumerate(comm.devices):
            lo, hi, first = time_chunk(T, comm.first_rank + i, world)
            chunks.append(yd[lo:hi].to(f"cuda:{d}").contiguous())
            models.append(_model(np.ascontiguousarray(F[lo:hi]), G))
            firsts.append(first)
        h = comm.scan_setup(models, params, chunks)
        fs = comm.scan_run(h)
        comm.sync()
        for i, o in enumerate(fs):
            for k in ("m", "C", "s", "S"):
                ref = one_fs[k][firsts[i]:firsts[i] + o[k].shape[0]]
                assert row_err(_npy(o[k]), ref) < TOL, k
        ll = comm.scan_loglik(h)
        comm.sync()
        for o in ll:
            for k in ("transition", "innovations"):
                assert abs(float(o[k][0]) - one_ll[k][0]) < TOL * abs(one_ll[k][0]) + 1e-9, k
        fb = comm.scan_ffbs(h, firsts, T, None)
        comm.sync()
        assert all(int(o["status"][0]) == 0 for o in fb)
    finally:
        comm.close()


# ---------------------------------------------------------------------------- Gibbs
def test_gibbs_recovers_the_simulating_variances(eng):
    from bayesian_dlms_b200 import gibbs
    T, iters, burn = 1 << 18, 300, 50
    _, F, G, _, _, m0, C0 = regression_model("r1", T, seed=70)
    V, W = np.array([[1.0]]), np.diag([0.3, 0.1])
    y = simulate_tv(F, G, V, W, m0, C0, seed=71)
    prior = dict(v_shape=3.0, v_scale=3.0, w_shape=3.0, w_scale=3.0)
    init = dict(V=np.array([[1.0]]), W=np.eye(2), m0=m0, C0=C0)
    out = gibbs.sample(eng, _model(F, G), _dev(y.reshape(T, 1, 1)), prior, init, iters, seed=8,
                       parallel_in_time=True)
    eng.sync()
    v, w = _npy(out["V"])[burn:, 0, 0], _npy(out["W"])[burn:, :, 0]
    ev = abs(v.mean() / V[0, 0] - 1)
    ew = np.abs(w.mean(axis=0) / np.diag(W) - 1)
    print("posterior means V %.4f (true %.1f), W %s (true %s)" % (v.mean(), V[0, 0], w.mean(axis=0), np.diag(W)))
    assert ev < 0.05 and np.all(ew < 0.05), (ev, ew)
    assert int(_npy(out["status"])[0]) == 0

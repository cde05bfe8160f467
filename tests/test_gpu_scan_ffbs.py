"""The parallel-in-time FFBS (bdlm_scan_ffbs, csrc/scan.cu ffbs_*_kernel), its opt-in from bdlm_ffbs
and gibbs.sample(parallel_in_time=True).

Paths are compared with the sequential thread-per-chain kernel (bit-identical to the oracle) for the
same normals, relative to each row's largest |entry|.  That comparison is only well posed where the
eigen basis of each draw's covariance H_r is well determined, so the path tests assert a minimum
relative eigen gap of H_r over the compared rows; a model with repeated eigenvalues is checked by
distribution instead (the empirical mean and covariance of theta_r against the smoother's (s_r, S_r)).
The Gibbs statistics are checked against the sequential kernel's and, as bookkeeping, against the
longdouble terms of the scan's own path."""
import numpy as np
import pytest

from test_scan_ffbs_reference_cpu import joseph_cov, row_err, stats_terms
from test_scan_reference_cpu import LEVEL2_EDGE_ROWS, MODEL_NAMES, model_arrays, scan_model, simulate

pytestmark = pytest.mark.gpu
TOL = 1e-9
TOL_LD = 1e-12
MIN_EIGEN_GAP = 1e-2  # measured on the filter rows of MODEL_NAMES: 0.088 at least (n4s)


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


def _dev(x):
    import torch
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _npy(x):
    return x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)


STATS = ("ssy", "ny", "ssw", "scatter")


def _scan(eng, model, params, yd, zd=None, **kw):
    import torch
    from bayesian_dlms_b200.scan import scan_ffbs
    out = scan_ffbs(eng, model, params, yd, zd, **kw)
    torch.cuda.synchronize()
    res = {k: _npy(v) for k, v in out.items()}
    res["status"] = int(res["status"][0])
    return res


def _seq(eng, model, params, yd, zd=None, want_kf=(), parallel_in_time=False):
    """bdlm_ffbs (B = 1, time-major): the sequential kernel unless the flag routes it to the scan."""
    from bayesian_dlms_b200 import TIME_MAJOR
    T, n = model.T, model.n
    z3 = None if zd is None else zd.reshape(T + 1, n, 1)
    out = eng.ffbs(model, params, yd.reshape(T, 1, 1), z3, layout=TIME_MAJOR, want_kf=want_kf, stats=True,
                   parallel_in_time=parallel_in_time)
    eng.sync()
    res = {k: _npy(v)[..., 0] for k, v in out.items()}
    res["status"] = int(res["status"])
    return res


def _normals(eng, T, n, mode, seed):
    """Injected normals (device tensor) or None with the context's Philox key set."""
    if mode == "z":
        return _dev(np.random.default_rng(seed).standard_normal((T + 1, n)))
    eng.ctx.set_rng(seed, 3, 0)
    return None


def _min_eigen_gap(mod, params, m, C, rows):
    """Smallest relative gap between neighbouring eigenvalues of H_r over the given rows."""
    n = params["m0"].size
    if n == 1:
        return 1.0
    _, G = model_arrays(mod, n)
    gap = np.inf
    for r in rows:
        _, _, H = joseph_cov(G, params["W"], m[r], C[r].reshape(n, n).T)
        lam = np.linalg.eigvalsh(H)
        gap = min(gap, float(np.min(np.diff(lam)) / lam[-1]))
    return gap


def _gap_rows(T):
    return np.unique(np.r_[0:min(T, 200), max(T - 200, 0):T, np.linspace(0, T - 1, 200).astype(int)])


def _stats_err(got, ref, terms):
    """Per statistic: max |got - ref| / sum_t |term_t|."""
    out = {}
    for k in ("ssy", "ssw", "scatter"):
        scale = np.maximum(np.sum(np.abs(terms[k].astype(float)), axis=0), 1e-300)
        out[k] = float(np.max(np.abs(np.ravel(got[k]) - np.ravel(ref[k])) / np.ravel(scale)))
    return out


def _residual_rounding(F, G, y, theta):
    """Per statistic: the rounding a double evaluation of the residuals e_t = y_t - F theta_{t+1} and
    d_t = theta_{t+1} - G theta_t can carry, relative to sum_t |term_t|.  Each residual is a length-n
    dot product subtracted from a value, so its error is within (n + 1) eps of the sum of magnitudes
    it is formed from; where |theta| >> |d| (a trend next to unit innovations) that, not the
    bookkeeping, dominates the comparison with longdouble terms."""
    eps = np.finfo(float).eps
    n = theta.shape[1]
    cur, prev = np.abs(theta[1:]), np.abs(theta[:-1])
    obs = ~np.isnan(y)
    e = np.where(obs, np.where(obs, y, 0) - theta[1:] @ F, 0)
    de = (n + 1) * eps * np.where(obs, np.abs(np.where(obs, y, 0)) + cur @ np.abs(F), 0)
    d = theta[1:] - theta[:-1] @ G.T
    dd = (n + 1) * eps * (cur + prev @ np.abs(G).T)
    ad = np.abs(d)
    sc = ad[:, :, None] * dd[:, None, :] + dd[:, :, None] * ad[:, None, :]
    terms = stats_terms(F, G, y, theta)
    out = {}
    for k, r in (("ssy", 2 * np.abs(e) * de), ("ssw", 2 * ad * dd), ("scatter", sc.reshape(-1, n * n))):
        scale = np.maximum(np.sum(np.abs(terms[k]), axis=0), 1e-300)
        out[k] = float(np.max(np.sum(r, axis=0) / scale))
    return out


def _edge_missing(y):
    """NaN on the first and last row of a few 16-row thread ranges (step t = row r)."""
    for r in (16 * 3, 16 * 3 + 15, 16 * 200, 16 * 200 + 15):
        if r < y.size:
            y[r] = np.nan
    return y


# ---------------------------------------------------------------------------- 1. path
PATH_T = [1, 2, 63, 64, 65, 1000, 40_001] + [r - 1 for r in LEVEL2_EDGE_ROWS]


@pytest.mark.parametrize("mode", ["z", "philox"])
@pytest.mark.parametrize("name", MODEL_NAMES)
@pytest.mark.parametrize("T", PATH_T)
def test_path_and_statistics_against_the_sequential_kernel(eng, name, T, mode):
    mod, model, params, y = _setup(name, T, seed=T + 3, missing=0.03)
    y = _edge_missing(y)
    yd = _dev(y)
    n = model.n
    zd = _normals(eng, T, n, mode, seed=T)
    seq = _seq(eng, model, params, yd, zd, want_kf=("m", "C", "a", "R", "f", "Q"))
    zd2 = _normals(eng, T, n, mode, seed=T)
    got = _scan(eng, model, params, yd, zd2, want_kf=("a", "R", "f", "Q"))
    assert got["status"] == seq["status"] == 0
    gap = _min_eigen_gap(mod, params, seq["m"], seq["C"], _gap_rows(T))
    assert gap > MIN_EIGEN_GAP, gap
    e = row_err(got["theta"], seq["theta"])
    assert e < TOL, e
    for k in ("a", "R", "f", "Q"):
        a, b = got[k][1:], seq[k][1:]  # row 0: the prior (a, R) and NaN (f, Q)
        assert row_err(a, b) < TOL, k
        assert np.array_equal(np.isnan(got[k][0]), np.isnan(seq[k][0]))
    F, G = model_arrays(mod, n)
    terms = stats_terms(F, G, y, seq["theta"])
    es = _stats_err(got, seq, terms)
    assert max(es.values()) < TOL, es
    assert got["ny"][0] == seq["ny"][0] == np.sum(~np.isnan(y))
    # bookkeeping: the scan's sums against the longdouble terms of its own path, at 1e-12 plus the
    # double rounding of each residual (a step dropped or counted twice moves a sum by ~1 / T)
    own = stats_terms(F, G, y, got["theta"], dtype=np.longdouble)
    ref = {k: np.sum(v, axis=0) for k, v in own.items()}
    eb = _stats_err(got, ref, own)
    rb = _residual_rounding(F, G, y, got["theta"])
    for k in eb:
        assert eb[k] < TOL_LD + rb[k], (k, eb[k], rb[k])
    print("%s T %d %s: theta %.1e, stats %.1e, own-path stats %.1e, eigen gap %.2g" %
          (name, T, mode, e, max(es.values()), max(eb.values()), gap))


# A long gap inflates the state covariance by decades, where the scan's filter loses more than the
# sequential recursion (DESIGN.md section 6, "Conditioning"): held to the filter + smoother's bound
# across such gaps (measured on B200: theta 3.2e-10, statistics 7.8e-12 at most).
TOL_GAP = 1e-6


@pytest.mark.parametrize("name", MODEL_NAMES)
@pytest.mark.parametrize("case", ["gap5000", "all_missing"])
def test_missing_data(eng, name, case):
    T = 40_001 if case == "gap5000" else 20_000
    mod, model, params, y = _setup(name, T, seed=19, missing=0.0)
    if case == "gap5000":
        y[14_000:19_000] = np.nan
    else:
        y[:] = np.nan
    yd = _dev(y)
    zd = _normals(eng, T, model.n, "z", seed=7)
    seq = _seq(eng, model, params, yd, zd, want_kf=("m", "C"))
    got = _scan(eng, model, params, yd, zd)
    assert got["status"] == seq["status"] == 0
    gap = _min_eigen_gap(mod, params, seq["m"], seq["C"], _gap_rows(T))
    e = row_err(got["theta"], seq["theta"])
    F, G = model_arrays(mod, model.n)
    es = _stats_err(got, seq, stats_terms(F, G, y, seq["theta"]))
    print("%s %s: theta %.2e, stats %.2e, eigen gap %.2g" % (name, case, e, max(es.values()), gap))
    assert got["ny"][0] == seq["ny"][0] == np.sum(~np.isnan(y))
    if gap > MIN_EIGEN_GAP:
        assert e < TOL_GAP and max(es.values()) < TOL_GAP, (e, es)


# ---------------------------------------------------------------------------- 2. distribution
@pytest.mark.parametrize("case", ["seasonal_isotropic", "n4"])
def test_draws_follow_the_smoothing_distribution(eng, case):
    """theta_r | y ~ N(s_r, S_r): K Philox sweeps, mean within 5 standard errors, covariance
    entries within 5 standard errors of the Wishart spread sqrt((S_ii S_jj + S_ij^2) / K)."""
    import torch
    from bayesian_dlms_b200 import Model, dlm
    from bayesian_dlms_b200.scan import scan_ffbs, scan_filter_smooth
    T, K = 300, 3000
    if case == "seasonal_isotropic":  # repeated eigenvalues in H: no path comparison is possible
        mod = dlm.seasonal(12, 1)
        params = dict(V=np.array([[1.0]]), W=0.5 * np.eye(2), m0=np.array([1.0, -0.5]), C0=4.0 * np.eye(2))
        y = simulate(mod, params["V"], params["W"], params["m0"], params["C0"], T, seed=1)
    else:
        mod, model, params, y = _setup("n4", T, seed=2)
    model = Model.build(mod, T=T)
    yd = _dev(y)
    sm = scan_filter_smooth(eng, model, params, yd, want=("m", "C", "s", "S"))
    torch.cuda.synchronize()
    s, S = sm["s"].cpu().numpy(), sm["S"].cpu().numpy()
    n = model.n
    rows = [0, 1, T // 2, T - 1, T]
    draws = torch.empty((K, len(rows), n), dtype=torch.float64, device="cuda")
    idx = torch.tensor(rows, device="cuda")
    for k in range(K):
        eng.ctx.set_rng(77, k, 0)
        out = scan_ffbs(eng, model, params, yd, stats=False)
        draws[k] = out["theta"][idx]
    torch.cuda.synchronize()
    d = draws.cpu().numpy()
    worst_m = worst_c = 0.0
    for i, r in enumerate(rows):
        Sr = S[r].reshape(n, n).T
        mean = d[:, i].mean(axis=0)
        cov = np.cov(d[:, i].T, bias=False).reshape(n, n)
        zm = np.abs(mean - s[r]) / np.sqrt(np.diag(Sr) / K)
        zc = np.abs(cov - Sr) / np.sqrt((np.outer(np.diag(Sr), np.diag(Sr)) + Sr ** 2) / K)
        worst_m, worst_c = max(worst_m, float(zm.max())), max(worst_c, float(zc.max()))
    print("%s: worst mean %.2f, worst covariance %.2f standard errors" % (case, worst_m, worst_c))
    assert worst_m < 5 and worst_c < 5, (worst_m, worst_c)


# ---------------------------------------------------------------------------- 3. conditioning
@pytest.mark.parametrize("name", ["n2", "n4"])
@pytest.mark.parametrize("C0_scale", [10.0, 1e4, 1e6])
@pytest.mark.parametrize("ratio", [1e-4, 1.0, 1e4])
def test_conditioning_sweep(eng, name, C0_scale, ratio):
    """theta's error against the sequential kernel, pinned relative to the scan smoother's own error
    on s against the sequential textbook smoother for the same problem (DESIGN.md section 6)."""
    import torch
    from bayesian_dlms_b200 import TIME_MAJOR
    from bayesian_dlms_b200.scan import scan_filter_smooth
    T = 2000
    mod, model, params, y = _setup(name, T, seed=5, missing=0.0, W_scale=ratio, C0_scale=C0_scale, V=1.0)
    yd = _dev(y)
    zd = _normals(eng, T, model.n, "z", seed=9)
    seq, got = _seq(eng, model, params, yd, zd, want_kf=("m", "C")), _scan(eng, model, params, yd, zd)
    fs_seq = eng.filter_smooth(model, params, yd.reshape(T, 1, 1), layout=TIME_MAJOR, want=("s",), textbook=True)
    fs_pit = scan_filter_smooth(eng, model, params, yd, want=("s",))
    eng.sync()
    torch.cuda.synchronize()
    es = row_err(_npy(fs_pit["s"]), _npy(fs_seq["s"])[..., 0])
    e = row_err(got["theta"], seq["theta"])
    gap = _min_eigen_gap(mod, params, seq["m"], seq["C"], _gap_rows(T))
    print("%s C0 %.0e W/V %.0e: theta %.2e, smoother s %.2e, eigen gap %.2g" % (name, C0_scale, ratio, e, es, gap))
    assert got["status"] == seq["status"]
    if gap > MIN_EIGEN_GAP:
        assert e < COND_FACTOR * max(es, 1e-12), (e, es)


COND_FACTOR = 1e3


# ---------------------------------------------------------------------------- 4. determinism
def _same(a, b, tag=()):
    for k in a:
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k]), equal_nan=True), (k, tag)


def test_same_bits_on_every_call_context_and_stream(eng):
    import torch
    from bayesian_dlms_b200 import Engine
    _, model, params, y = _setup("n4", 100_003, seed=7)
    yd = _dev(y)

    def run(e):
        e.ctx.set_rng(5, 2, 0)
        return _scan(e, model, params, yd)
    first = run(eng)
    _same(first, run(eng), ("again",))
    _same(first, run(Engine(0)), ("context",))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        e = Engine(0)
        e.use_torch_stream()
        _same(first, run(e), ("stream",))
    torch.cuda.synchronize()


def test_model_table_cache_follows_every_model_change():
    from bayesian_dlms_b200 import Engine, Model
    mod, V, W, m0, C0 = scan_model("n2")
    T = 5000
    yd = _dev(simulate(mod, V, W, m0, C0, T, seed=6))
    zd = _dev(np.random.default_rng(6).standard_normal((T + 1, 2)))
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
        got = _scan(e, model, params, yd, zd)
        key = tag if tag != "A again" else "A"
        if key not in fresh:
            fresh[key] = _scan(Engine(0), model, params, yd, zd)
        _same(got, fresh[key], (tag,))


# ---------------------------------------------------------------------------- 5. status
@pytest.mark.parametrize("name", ["n1", "n2", "n4"])
@pytest.mark.parametrize("case", ["control", "inf", "zero_variances"])
def test_status_matches_the_sequential_kernel(eng, name, case):
    from bayesian_dlms_b200 import _capi as capi
    T = 5000
    _, model, params, y = _setup(name, T, seed=8)
    n = model.n
    if case == "inf":
        y[1234] = np.inf
    if case == "zero_variances":
        params = dict(params, V=np.zeros((1, 1)), W=np.zeros((n, n)), C0=np.zeros((n, n)))
    yd = _dev(y)
    zd = _normals(eng, T, n, "z", seed=1)
    s_seq = _seq(eng, model, params, yd, zd)["status"]
    s_pit = _seq(eng, model, params, yd, zd, parallel_in_time=True)["status"]
    s_scan = _scan(eng, model, params, yd, zd)["status"]
    print(name, case, "sequential", s_seq, "opt-in", s_pit, "scan", s_scan)
    assert s_pit == s_seq == s_scan
    if case == "control":
        assert s_seq == 0
    if case == "inf":
        assert s_seq & capi.ST_NONFINITE


# ---------------------------------------------------------------------------- 6. opt-in dispatch
@pytest.mark.parametrize("name", ["n1", "n2", "n4"])
@pytest.mark.parametrize("where", ["device", "host"])
@pytest.mark.parametrize("mode", ["z", "philox"])
def test_opt_in_dispatch(eng, name, where, mode):
    from bayesian_dlms_b200 import SERIES_MAJOR
    T = 50_000
    mod, model, params, y = _setup(name, T, seed=50)
    n = model.n
    z = np.random.default_rng(51).standard_normal((T + 1, n))
    yy, zz = y.reshape(1, T, 1).copy(), z.reshape(1, T + 1, n).copy()
    if where == "device":
        yy, zz = _dev(yy), _dev(zz)
    if mode == "philox":
        zz = None

    def call(pit):
        eng.ctx.set_rng(21, 4, 0)
        o = eng.ffbs(model, params, yy, zz, layout=SERIES_MAJOR, want_kf=("m", "C"), stats=True,
                     parallel_in_time=pit)
        eng.sync()
        return {k: _npy(v)[0] for k, v in o.items()}
    seq, pit = call(False), call(True)
    eng.ctx.set_rng(21, 4, 0)
    direct = _scan(eng, model, params, _dev(y), None if mode == "philox" else _dev(z), want_kf=("m", "C"))
    for k in ("theta", "m", "C") + STATS:
        assert np.array_equal(np.ravel(pit[k]), np.ravel(direct[k])), k
    assert int(pit["status"]) == direct["status"] == int(seq["status"]) == 0
    assert row_err(pit["theta"], seq["theta"]) < TOL
    # the flag did route to the scan: the path is not the sequential kernel's bits
    assert not np.array_equal(pit["theta"], seq["theta"])


@pytest.mark.parametrize("case", ["B3", "T4095", "irregular", "per_series", "v_tv"])
def test_ineligible_problems_keep_the_sequential_kernel(eng, case):
    from bayesian_dlms_b200 import TIME_MAJOR, Model
    mod, V, W, m0, C0 = scan_model("n2")
    B, T = (3, 5000) if case == "B3" else (1, 4095) if case == "T4095" else (1, 5000)
    ys = np.stack([simulate(mod, V, W, m0, C0, T, seed=60 + b, missing=0.02) for b in range(B)], axis=-1)
    yd = _dev(ys.reshape(T, 1, B))
    zd = _dev(np.random.default_rng(61).standard_normal((T + 1, 2, B)))
    times = np.cumsum(np.random.default_rng(3).uniform(0.5, 1.5, T)) if case == "irregular" else None
    model = Model.build(mod, times=times) if times is not None else Model.build(mod, T=T)
    params = dict(V=V, W=W, m0=m0, C0=C0)
    if case == "per_series":
        params = dict(params, V=_dev(V.reshape(1, 1)), W=_dev(W.T.reshape(4, 1)), per_series=("V", "W"))
    if case == "v_tv":
        params = dict(params, V=np.full((T, 1), float(V[0, 0])), v_tv=True)
    a = eng.ffbs(model, params, yd, zd, layout=TIME_MAJOR, stats=True)
    b = eng.ffbs(model, params, yd, zd, layout=TIME_MAJOR, stats=True, parallel_in_time=True)
    eng.sync()
    for k in a:
        assert np.array_equal(_npy(a[k]), _npy(b[k]), equal_nan=True), (case, k)


def test_outputs_left_null_and_launch_count(eng):
    _, model, params, y = _setup("n3", 50_000, seed=9)
    yd = _dev(y)
    zd = _normals(eng, 50_000, 3, "z", seed=9)
    full = _scan(eng, model, params, yd, zd, want_kf=("m", "C", "a", "R", "f", "Q"))
    counts = []
    for kw in (dict(stats=False), dict(want_kf=()), dict(want_kf=("a", "f"))):
        c0 = eng.ctx.launch_count()
        part = _scan(eng, model, params, yd, zd, **kw)
        counts.append(eng.ctx.launch_count() - c0)
        assert part["status"] == full["status"] == 0
        for k in part:
            if k != "status":
                assert np.array_equal(part[k], full[k], equal_nan=True), (kw, k)
    print("launches without statistics, with, with:", counts)
    # forward: reduce, level 2 (2 at this length), apply; sampler: reduce, level 2 (2), apply (+ finish)
    assert counts == [8, 9, 9], counts


# ---------------------------------------------------------------------------- 7. Gibbs
def _gibbs_setup(T, seed):
    mod, V, W, m0, C0 = scan_model("n1")
    y = simulate(mod, V, W, m0, C0, T, seed=seed)
    prior = dict(v_shape=3.0, v_scale=3.0, w_shape=3.0, w_scale=3.0)
    init = dict(V=np.array([[1.0]]), W=np.array([[1.0]]), m0=m0, C0=C0)
    return mod, V, W, y, prior, init


def test_gibbs_first_sweep_matches_the_sequential_sampler(eng):
    from bayesian_dlms_b200 import Model, gibbs
    T = 5000
    mod, _, _, y, prior, init = _gibbs_setup(T, seed=31)
    model = Model.build(mod, T=T)
    yd = _dev(y.reshape(T, 1, 1))
    a = gibbs.sample(eng, model, yd, prior, init, 2, seed=4)
    b = gibbs.sample(eng, model, yd, prior, init, 2, seed=4, parallel_in_time=True)
    eng.sync()
    for k in ("V", "W"):
        x, r = _npy(b[k])[0], _npy(a[k])[0]
        assert np.max(np.abs(x - r) / np.abs(r)) < TOL, (k, x, r)
    assert int(_npy(b["status"])[0]) == 0


def test_gibbs_recovers_the_simulating_variances(eng):
    from bayesian_dlms_b200 import Model, gibbs
    T, iters, burn = 1 << 18, 300, 50
    mod, V, W, y, prior, init = _gibbs_setup(T, seed=32)
    model = Model.build(mod, T=T)
    out = gibbs.sample(eng, model, _dev(y.reshape(T, 1, 1)), prior, init, iters, seed=8, parallel_in_time=True)
    eng.sync()
    v, w = _npy(out["V"])[burn:, 0, 0], _npy(out["W"])[burn:, 0, 0]
    ev, ew = abs(v.mean() / V[0, 0] - 1), abs(w.mean() / W[0, 0] - 1)
    print("posterior means V %.4f (true %.1f), W %.4f (true %.1f)" % (v.mean(), V[0, 0], w.mean(), W[0, 0]))
    # posterior sd at T = 2^18 is about 1 % of either variance: 5 % is five of them
    assert ev < 0.05 and ew < 0.05, (ev, ew)
    assert int(_npy(out["status"])[0]) == 0

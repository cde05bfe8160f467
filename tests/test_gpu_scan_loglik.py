"""The parallel-in-time log-likelihood (bdlm_scan_loglik, csrc/scan.cu fwd_loglik_kernel) and its
opt-in from bdlm_loglik / bdlm_kf_filter_last.

Errors of a sum are measured as |x - ref| / sum_t |term_t| (sum_err): the per-step terms can cancel,
which makes the sum itself a poor denominator.  The checks are
  - bookkeeping: the scan's sums against the longdouble terms of bdlm_scan_filter_smooth's own
    (m, f, Q) rows at 1e-12, and its last state against that call's row T -- a term dropped or
    counted twice at a thread-range or level-2 edge, a wrong m_{t-1} at a thread start or a missing
    observation summed shows here, free of the scan's state rounding;
  - the sequential kernel (1e-9), the longdouble reference up to T = 5000 and the oracle at 2^24;
  - determinism, the model-table cache, the status word and the opt-in dispatch."""
import numpy as np
import pytest

from test_scan_loglik_reference_cpu import TOL_LD, _ld_loglik, ld_terms, sum_err
from test_scan_reference_cpu import LEVEL2_EDGE_ROWS, MODEL_NAMES, model_arrays, scan_model, simulate

pytestmark = pytest.mark.gpu
TOL = 1e-9
LD_MAX_T = 5000


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


def _scan_ll(eng, model, params, yd, **kw):
    import torch
    from bayesian_dlms_b200.scan import scan_loglik
    kw.setdefault("last", True)
    out = scan_loglik(eng, model, params, yd, **kw)
    torch.cuda.synchronize()
    res = {k: v.cpu().numpy() for k, v in out.items()}
    for k in ("transition", "innovations"):
        if k in res:
            res[k] = float(res[k][0])
    res["status"] = int(res["status"][0])
    return res


def _seq_ll(eng, model, params, yd, parallel_in_time=False):
    """bdlm_kf_filter_last (B = 1) with both log-likelihoods: the sequential kernel unless the flag
    routes it to the scan."""
    from bayesian_dlms_b200 import TIME_MAJOR
    out = eng.filter_last(model, params, yd.reshape(-1, 1, 1).contiguous(), layout=TIME_MAJOR, loglik=True,
                          parallel_in_time=parallel_in_time)
    eng.sync()
    npy = lambda x: x.cpu().numpy() if hasattr(x, "cpu") else x  # noqa: E731
    return dict(transition=float(npy(out["transition"])[0]), innovations=float(npy(out["innovations"])[0]),
                m=npy(out["m"])[:, 0], C=npy(out["C"])[:, 0], status=int(npy(out["status"])[0]))


def _rows(eng, model, params, yd):
    """bdlm_scan_filter_smooth's own rows 1..T of (m, C, f, Q) (keep_init = 1)."""
    import torch
    from bayesian_dlms_b200.scan import scan_filter_smooth
    out = scan_filter_smooth(eng, model, params, yd, keep_init=True, want=("m", "C", "a", "f", "Q", "s"))
    torch.cuda.synchronize()
    return {k: out[k].cpu().numpy()[1:] for k in ("m", "C", "a", "f", "Q")}


def _terms(mod, params, rows, y, own_a=False):
    """Longdouble terms of the rows; own_a: with the rows' own predictions a_t as the transition mean."""
    _, G = model_arrays(mod, params["m0"].size)
    return ld_terms(G, params["W"], params["m0"], rows["m"], rows["f"], rows["Q"], y,
                    a=rows["a"] if own_a else None)


def _state_err(a, b):
    """Last state against a reference, relative to the reference's largest entry."""
    a, b = np.asarray(a, float).ravel(), np.asarray(b, float).ravel()
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def _edge_missing(y, keep_init=1):
    """NaN on the first and last row of a few 16-row thread ranges (row = t + 1)."""
    for r in (16 * 3, 16 * 3 + 15, 16 * 200, 16 * 200 + 15):
        if r - keep_init < y.size:
            y[r - keep_init] = np.nan
    return y


# ---------------------------------------------------------------------------- 1. bookkeeping
BOOK_T = [1, 2, 63, 64, 65, 1000, 40_001] + [r - 1 for r in LEVEL2_EDGE_ROWS[::3]]


@pytest.mark.parametrize("name", MODEL_NAMES)
@pytest.mark.parametrize("T", BOOK_T)
def test_sums_match_the_terms_of_the_scans_own_rows(eng, name, T):
    mod, model, params, y = _setup(name, T, seed=T + 5, missing=0.05)
    y = _edge_missing(y)
    yd = _dev(y)
    got = _scan_ll(eng, model, params, yd)
    rows = _rows(eng, model, params, yd)
    # the rows' predictions are G m_{t-1} up to the rounding of that product
    _, G = model_arrays(mod, params["m0"].size)
    prev = np.concatenate([params["m0"].reshape(1, -1), rows["m"][:-1]])
    scale = np.maximum(np.max(np.abs(rows["a"]), axis=1), 1e-300)
    ea = float(np.max(np.max(np.abs(rows["a"] - prev @ G.T), axis=1) / scale))
    assert ea < 1e-14, ea
    tr, inn = _terms(mod, params, rows, y, own_a=True)
    assert got["status"] == 0
    et, ei = sum_err(got["transition"], tr), sum_err(got["innovations"], inn)
    assert et < TOL_LD and ei < TOL_LD, (et, ei)
    em, eC = _state_err(got["m"], rows["m"][-1]), _state_err(got["C"], rows["C"][-1])
    same = np.array_equal(got["m"], rows["m"][-1]) and np.array_equal(got["C"], rows["C"][-1])
    print("%s T %d: transition %.1e innovations %.1e, last state %s" %
          (name, T, et, ei, "bit-identical" if same else "m %.1e C %.1e" % (em, eC)))
    assert em < 1e-13 and eC < 1e-13, (em, eC)


# ---------------------------------------------------------------------------- 2. sequential kernel
SEQ_T = [1, 2, 63, 64, 65, 1000, 40_001] + [r - 1 for r in LEVEL2_EDGE_ROWS]


@pytest.mark.parametrize("name", MODEL_NAMES)
@pytest.mark.parametrize("T", SEQ_T)
def test_against_the_sequential_kernel(eng, name, T):
    mod, model, params, y = _setup(name, T, seed=T + 17, missing=0.02)
    yd = _dev(y)
    got = _scan_ll(eng, model, params, yd)
    seq = _seq_ll(eng, model, params, yd)
    assert got["status"] == seq["status"] == 0
    if T <= LD_MAX_T:
        F, G = model_arrays(mod, params["m0"].size)
        tr, inn, mT, _ = _ld_loglik(F, G, params["V"], params["W"], params["m0"], params["C0"], y)
        for k, terms in (("transition", tr), ("innovations", inn)):
            es, eg = sum_err(seq[k], terms), sum_err(got[k], terms)
            assert es < TOL_LD, (k, "sequential vs longdouble", es)
            assert eg < TOL, (k, "scan vs longdouble", eg)
    else:
        tr, inn = _terms(mod, params, _rows(eng, model, params, yd), y)
    for k, terms in (("transition", tr), ("innovations", inn)):
        e = abs(got[k] - seq[k]) / float(np.sum(np.abs(terms)))
        assert e < TOL, (k, e)
    assert _state_err(got["m"], seq["m"]) < TOL and _state_err(got["C"], seq["C"]) < TOL


@pytest.mark.parametrize("name", ["n1", "n2"])
def test_long_series_against_the_oracle(eng, name):
    import oracle
    from bayesian_dlms_b200 import dlm
    T = 1 << 24
    mod, model, params, y = _setup(name, T, seed=24, missing=0.01)
    yd = _dev(y)
    got = _scan_ll(eng, model, params, yd)
    n = params["m0"].size
    F, G = model_arrays(mod, n)
    o = oracle.loglik(n, 1, F, dlm.cm(G), dlm.cm(params["V"]), dlm.cm(params["W"]), params["m0"],
                      dlm.cm(params["C0"]), np.arange(1, T + 1.0), y.reshape(T, 1))
    # scale sum_t |term_t| from the scan's own rows, in double (a scale, not a reference)
    import torch
    from bayesian_dlms_b200.scan import scan_filter_smooth
    out = scan_filter_smooth(eng, model, params, yd, want=("m", "f", "Q"))
    torch.cuda.synchronize()
    m, f, Q = (out[k].cpu().numpy()[1:] for k in ("m", "f", "Q"))
    del out
    prev = np.concatenate([params["m0"].reshape(1, n), m[:-1]])
    d = m - prev @ G.T
    tr_abs = np.sum(np.abs(-0.5 * np.sum(d * np.linalg.solve(params["W"], d.T).T, axis=1)
                           - 0.5 * (n * np.log(2 * np.pi) + np.linalg.slogdet(params["W"])[1])))
    obs = ~np.isnan(y)
    sd = np.sqrt(Q[obs, 0])
    dd = (y[obs] - f[obs, 0]) / sd
    in_abs = np.sum(np.abs(-dd * dd / 2 - np.log(np.sqrt(2 * np.pi) * sd)))
    et = abs(got["transition"] - o["transition"]) / tr_abs
    ei = abs(got["innovations"] - o["innovations"]) / in_abs
    print("%s T 2^24 vs oracle: transition %.2e innovations %.2e" % (name, et, ei))
    assert got["status"] == o["status"] == 0
    assert et < TOL and ei < TOL, (et, ei)


# ---------------------------------------------------------------------------- 3. inputs
# A long gap inflates the state covariance by decades, and the scan's combines then lose more than the
# sequential recursion (DESIGN.md section 6, "Conditioning").  The sums and m_T still hold 1e-9 across
# 5000 missing steps (measured on B200: 7.1e-13 at most); C_T of an all-missing series is held to the
# filter + smoother's bound across such gaps.
TOL_GAP = 1e-6


@pytest.mark.parametrize("name", MODEL_NAMES)
def test_gap_of_5000_steps(eng, name):
    mod, model, params, y = _setup(name, 40_001, seed=19, missing=0.0)
    y[14_000:19_000] = np.nan
    yd = _dev(y)
    got, seq = _scan_ll(eng, model, params, yd), _seq_ll(eng, model, params, yd)
    tr, inn = _terms(mod, params, _rows(eng, model, params, yd), y)
    et = abs(got["transition"] - seq["transition"]) / float(np.sum(np.abs(tr)))
    ei = abs(got["innovations"] - seq["innovations"]) / float(np.sum(np.abs(inn)))
    print("%s gap 5000: transition %.2e innovations %.2e, m %.2e" % (name, et, ei, _state_err(got["m"], seq["m"])))
    assert got["status"] == seq["status"] == 0
    assert et < TOL and ei < TOL and _state_err(got["m"], seq["m"]) < TOL


@pytest.mark.parametrize("name", ["n1", "n3", "n4"])
@pytest.mark.parametrize("T", [1, 20_000])
def test_all_missing(eng, name, T):
    mod, model, params, _ = _setup(name, T, seed=1, missing=0.0)
    yd = _dev(np.full(T, np.nan))
    got, seq = _scan_ll(eng, model, params, yd), _seq_ll(eng, model, params, yd)
    assert got["innovations"] == 0.0 and seq["innovations"] == 0.0
    assert got["status"] == seq["status"] == 0
    F, G = model_arrays(mod, params["m0"].size)
    tr = _ld_loglik(F, G, params["V"], params["W"], params["m0"], params["C0"], np.full(min(T, 50), np.nan))[0]
    # pure prediction: every transition term is the same constant
    assert abs(got["transition"] - seq["transition"]) <= TOL * abs(float(tr[0])) * T
    assert _state_err(got["m"], seq["m"]) < TOL_GAP and _state_err(got["C"], seq["C"]) < TOL_GAP


@pytest.mark.parametrize("name", ["n2", "n4"])
@pytest.mark.parametrize("C0_scale", [10.0, 1e4, 1e6])
@pytest.mark.parametrize("ratio", [1e-4, 1.0, 1e4])
def test_conditioning_sweep(eng, name, C0_scale, ratio):
    """W / V and the prior scale over eight decades, against the longdouble reference: where the
    sequential kernel is within 1e-12 the scan must be within 1e-9, and everywhere within a measured
    multiple of the sequential kernel's error, floored at 1e-14 (measured on B200: at most 21 times,
    n = 4, C0 1e6, W / V 1e-4: 3.4e-14 / 7.1e-13; DESIGN.md section 6)."""
    T = 2000
    mod, model, params, y = _setup(name, T, seed=5, missing=0.0, W_scale=ratio, C0_scale=C0_scale, V=1.0)
    yd = _dev(y)
    got, seq = _scan_ll(eng, model, params, yd), _seq_ll(eng, model, params, yd)
    F, G = model_arrays(mod, params["m0"].size)
    tr, inn, _, _ = _ld_loglik(F, G, params["V"], params["W"], params["m0"], params["C0"], y)
    es = max(sum_err(seq["transition"], tr), sum_err(seq["innovations"], inn))
    eg = max(sum_err(got["transition"], tr), sum_err(got["innovations"], inn))
    print("%s C0 %.0e W/V %.0e: sequential %.2e, scan %.2e vs longdouble" % (name, C0_scale, ratio, es, eg))
    assert got["status"] == seq["status"] == 0
    if es < TOL_LD:
        assert eg < TOL, (es, eg)
    assert eg < COND_FACTOR * max(es, 1e-14), (es, eg)


COND_FACTOR = 100


# ---------------------------------------------------------------------------- 4. determinism
def _same(a, b, tag=()):
    for k in a:
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k]), equal_nan=True), (k, tag)


def test_same_bits_on_every_call_context_and_stream(eng):
    import torch
    from bayesian_dlms_b200 import Engine
    _, model, params, y = _setup("n4", 100_003, seed=7)
    yd = _dev(y)
    first = _scan_ll(eng, model, params, yd)
    _same(first, _scan_ll(eng, model, params, yd), ("again",))
    _same(first, _scan_ll(Engine(0), model, params, yd), ("context",))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        e = Engine(0)
        e.use_torch_stream()
        _same(first, _scan_ll(e, model, params, yd), ("stream",))
    torch.cuda.synchronize()


def test_model_table_cache_follows_every_model_change():
    from bayesian_dlms_b200 import Engine, Model
    mod, V, W, m0, C0 = scan_model("n2")
    T = 5000
    yd = _dev(simulate(mod, V, W, m0, C0, T, seed=6))
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
        got = _scan_ll(e, model, params, yd)
        key = tag if tag != "A again" else "A"
        if key not in fresh:
            fresh[key] = _scan_ll(Engine(0), model, params, yd)
        _same(got, fresh[key], (tag,))


# ---------------------------------------------------------------------------- 5. status
def _ll_call(eng, model, params, yd, *, flag, transition):
    """bdlm_loglik on a device series with the transition form requested or not."""
    import torch
    from bayesian_dlms_b200 import SERIES_MAJOR, _capi as capi
    from bayesian_dlms_b200.batch import bound_engine
    y3 = yd.reshape(1, -1, 1).contiguous()
    with bound_engine(eng):  # the engine runs on torch's current stream, after the fills below
        pr, keep = eng._problem(model, params, y3, SERIES_MAJOR, True, capi.PARALLEL_IN_TIME if flag else 0, 1,
                                capi.DEVICE)
    tr = torch.zeros(1, dtype=torch.float64, device="cuda")
    inn = torch.zeros(1, dtype=torch.float64, device="cuda")
    st = torch.full((1,), -1, dtype=torch.int32, device="cuda")
    eng.ctx.check(capi.load().bdlm_loglik(eng.ctx.handle, pr, tr.data_ptr() if transition else None,
                                          inn.data_ptr(), st.data_ptr()))
    eng.sync()
    return int(st[0]), float(tr[0]), float(inn[0])


@pytest.mark.parametrize("name", ["n1", "n2", "n4"])
@pytest.mark.parametrize("case", ["control", "inf", "zero_variances", "singular_W", "singular_W_transition"])
def test_status_matches_the_sequential_route(eng, name, case):
    from bayesian_dlms_b200 import _capi as capi
    T = 5000
    _, model, params, y = _setup(name, T, seed=8)
    n = model.n
    if case == "inf":
        y[1234] = np.inf
    if case == "zero_variances":
        params = dict(params, V=np.zeros((1, 1)), W=np.zeros((n, n)), C0=np.zeros((n, n)))
    if case.startswith("singular_W"):
        W = np.zeros((n, n))
        W[0, 0] = 0.5
        params = dict(params, W=W)
    yd = _dev(y)
    want_tr = case != "singular_W"
    s_seq = _ll_call(eng, model, params, yd, flag=False, transition=want_tr)[0]
    s_pit = _ll_call(eng, model, params, yd, flag=True, transition=want_tr)[0]
    last_seq = _seq_ll(eng, model, params, yd)["status"]
    last_pit = _seq_ll(eng, model, params, yd, parallel_in_time=True)["status"]
    print(name, case, "sequential", s_seq, last_seq, "scan", s_pit, last_pit)
    assert s_pit == s_seq and last_pit == last_seq
    if case == "control":
        assert s_seq == 0
    if case == "inf":
        assert s_seq & capi.ST_NONFINITE
    if case == "zero_variances":
        assert s_seq & capi.ST_SINGULAR
    if case == "singular_W":
        assert s_seq == 0
    if case == "singular_W_transition" and n > 1:
        assert s_seq & (capi.ST_SINGULAR | capi.ST_NOTPD)


# ---------------------------------------------------------------------------- 6. opt-in dispatch
@pytest.mark.parametrize("name", ["n1", "n2", "n4"])
@pytest.mark.parametrize("where", ["device", "host"])
def test_opt_in_dispatch(eng, name, where):
    from bayesian_dlms_b200 import SERIES_MAJOR
    T = 50_000
    mod, model, params, y = _setup(name, T, seed=50)
    yy = y.reshape(1, T, 1).copy()
    yy = _dev(yy) if where == "device" else yy
    npy = lambda x: x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)  # noqa: E731
    seq = eng.loglik(model, params, yy, layout=SERIES_MAJOR)
    pit = eng.loglik(model, params, yy, layout=SERIES_MAJOR, parallel_in_time=True)
    lseq = eng.filter_last(model, params, yy, layout=SERIES_MAJOR, loglik=True)
    lpit = eng.filter_last(model, params, yy, layout=SERIES_MAJOR, loglik=True, parallel_in_time=True)
    eng.sync()
    tr, inn = _terms(mod, params, _rows(eng, model, params, _dev(y)), y)
    scale = dict(transition=float(np.sum(np.abs(tr))), innovations=float(np.sum(np.abs(inn))))
    for a, b in ((seq, pit), (lseq, lpit)):
        assert int(npy(a["status"])[0]) == int(npy(b["status"])[0]) == 0
        for k in ("transition", "innovations"):
            x, r = float(npy(b[k])[0]), float(npy(a[k])[0])
            assert abs(x - r) / scale[k] < TOL, (k, abs(x - r) / scale[k])
    assert _state_err(npy(lpit["m"]), npy(lseq["m"])) < TOL and _state_err(npy(lpit["C"]), npy(lseq["C"])) < TOL
    # the flag did route to the scan: the sums are not the sequential kernel's bits
    assert float(npy(pit["transition"])[0]) != float(npy(seq["transition"])[0])


@pytest.mark.parametrize("case", ["B3", "T4095", "irregular"])
def test_ineligible_problems_keep_the_sequential_kernel(eng, case):
    from bayesian_dlms_b200 import TIME_MAJOR, Model
    mod, V, W, m0, C0 = scan_model("n2")
    params = dict(V=V, W=W, m0=m0, C0=C0)
    B, T = (3, 5000) if case == "B3" else (1, 4095) if case == "T4095" else (1, 5000)
    ys = np.stack([simulate(mod, V, W, m0, C0, T, seed=60 + b, missing=0.02) for b in range(B)], axis=-1)
    yd = _dev(ys.reshape(T, 1, B))
    times = np.cumsum(np.random.default_rng(3).uniform(0.5, 1.5, T)) if case == "irregular" else None
    model = Model.build(mod, times=times) if times is not None else Model.build(mod, T=T)
    for call in ("loglik", "filter_last"):
        kw = dict(layout=TIME_MAJOR)
        if call == "filter_last":
            kw["loglik"] = True
        a = getattr(eng, call)(model, params, yd, **kw)
        b = getattr(eng, call)(model, params, yd, parallel_in_time=True, **kw)
        eng.sync()
        for k in a:
            assert np.array_equal(a[k].cpu().numpy(), b[k].cpu().numpy(), equal_nan=True), (case, call, k)


def test_outputs_left_null_and_launch_count(eng):
    _, model, params, y = _setup("n3", 50_000, seed=9)
    yd = _dev(y)
    full = _scan_ll(eng, model, params, yd)
    for kw in (dict(transition=False), dict(innovations=False), dict(transition=False, innovations=False),
               dict(last=False)):
        c0 = eng.ctx.launch_count()
        part = _scan_ll(eng, model, params, yd, **kw)
        assert eng.ctx.launch_count() - c0 <= 6
        assert part["status"] == full["status"] == 0
        for k in part:
            if k != "status":
                assert np.array_equal(part[k], full[k]), (kw, k)
    # bdlm_kf_filter_last with only m_last: no log-likelihood, no C
    import torch
    from bayesian_dlms_b200 import SERIES_MAJOR, _capi as capi
    from bayesian_dlms_b200.batch import bound_engine
    y3 = yd.reshape(1, -1, 1).contiguous()
    with bound_engine(eng):
        pr, keep = eng._problem(model, params, y3, SERIES_MAJOR, True, capi.PARALLEL_IN_TIME, 1, capi.DEVICE)
    m = torch.zeros(3, dtype=torch.float64, device="cuda")
    c0 = eng.ctx.launch_count()
    eng.ctx.check(capi.load().bdlm_kf_filter_last(eng.ctx.handle, pr, m.data_ptr(), None, None, None, None))
    assert eng.ctx.launch_count() - c0 <= 6
    eng.sync()
    assert np.array_equal(m.cpu().numpy(), full["m"])

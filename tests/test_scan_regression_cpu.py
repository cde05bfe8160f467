"""Per-step observation vectors (f_tv: dynamic regression, F_t = (1, x_t)) on the parallel-in-time scan,
host side: an extended-precision filter + textbook smoother with per-step F pinned to the oracle, the
filtering elements built with F_t composed in random bracketings, and the argument rules of the
time-sharded phases, which need no device.  The regression models of
tests/test_gpu_scan_regression.py are built here."""
import math

import numpy as np
import pytest

import oracle
from bayesian_dlms_b200 import _capi as capi, dlm
from test_scan_combine_cpu import _cm, _comb, _f_element, _pack_f, _unpack_f
from test_scan_reference_cpu import LD, TOL_LD, _ld_inv, ld_err

REG_NAMES = ("r1", "r2", "r3", "r1s", "r2w")  # n = 2, 3, 4, 4 (with a rotation G), 3 (wide covariates)


def covariates(name, T, seed):
    """x_t of the model (T, k): standard normal, or for 'r2w' magnitudes spanning 1e-3 .. 1e3 with
    stretches of x_t = 0."""
    rng = np.random.default_rng(seed)
    k = {"r1": 1, "r2": 2, "r3": 3, "r1s": 1, "r2w": 2}[name]
    x = rng.standard_normal((T, k))
    if name == "r2w":
        x *= 10.0 ** rng.uniform(-3, 3, size=(T, k))
        for lo in range(T // 7, T, max(T // 3, 1)):
            x[lo:lo + max(T // 50, 3)] = 0.0
    return x


def regression_model(name, T, seed=0):
    """name -> (Dlm, F [T][n], G (n, n), V, W, m0, C0): dlm.regression of the covariates, alone or
    composed with seasonal(12, 1)."""
    x = covariates(name, T, seed)
    mod = dlm.regression(list(x))
    if name == "r1s":
        mod = mod + dlm.seasonal(12, 1)
    F, f_tv, G, g_tv, n, p = dlm.materialise(mod, np.arange(1, T + 1.0))
    assert p == 1 and not g_tv
    F = np.ascontiguousarray(np.asarray(F, float).reshape(-1, n) * np.ones((T, 1)))
    G = dlm.from_cm(np.asarray(G, float), n, n)
    W = np.diag(np.linspace(0.05, 0.01, n))
    V = np.array([[1.0]])
    m0, C0 = np.zeros(n), 10.0 * np.eye(n)
    return mod, F, G, V, W, m0, C0


def simulate_tv(F, G, V, W, m0, C0, seed, missing=0.0):
    """Dlm.simStep with per-step F on the regular grid."""
    rng = np.random.default_rng(seed)
    T, n = F.shape
    x = m0 + np.linalg.cholesky(C0) @ rng.standard_normal(n)
    w = rng.standard_normal((T, n)) @ np.linalg.cholesky(W).T
    v = rng.standard_normal(T) * math.sqrt(float(V[0, 0]))
    y = np.empty(T)
    for t in range(T):
        x = G @ x + w[t]
        y[t] = F[t] @ x + v[t]
    if missing > 0:
        y[rng.random(T) < missing] = np.nan
    return y


def ld_filter_smooth_tv(F, G, V, W, m0, C0, y, keep_init):
    """As test_scan_reference_cpu._ld_filter_smooth with F_t = F[t] (F [T][n]), in np.longdouble."""
    F = np.asarray(F, float).astype(LD)
    G, W, C0 = (np.asarray(a, float).astype(LD) for a in (G, W, C0))
    m0 = np.asarray(m0, float).ravel().astype(LD)
    V = LD(float(np.asarray(V, float).ravel()[0]))
    y = np.asarray(y, float).ravel()
    n, T = m0.size, y.size
    I = np.eye(n, dtype=LD)
    a, R, m, C, f, Q = [], [], [], [], [], []
    if keep_init:
        a.append(m0); R.append(C0); m.append(m0); C.append(C0)
        f.append(LD(np.nan)); Q.append(LD(np.nan))
    mt, Ct = m0, C0
    for t in range(T):
        at = G @ mt
        Rt = G @ Ct @ G.T + W
        ft = F[t] @ at
        Qt = F[t] @ Rt @ F[t] + V
        if np.isnan(y[t]):
            mt, Ct = at, Rt
        else:
            K = Rt @ F[t] / Qt
            mt = at + K * (LD(y[t]) - ft)
            IKF = I - np.outer(K, F[t])
            Ct = IKF @ Rt @ IKF.T + V * np.outer(K, K)
        a.append(at); R.append(Rt); f.append(ft); Q.append(Qt); m.append(mt); C.append(Ct)
    rows = len(m)
    s, S = [None] * rows, [None] * rows
    s[-1], S[-1] = m[-1], C[-1]
    for r in range(rows - 2, -1, -1):
        B = C[r] @ G.T @ _ld_inv(R[r + 1])
        s[r] = m[r] + B @ (s[r + 1] - a[r + 1])
        S[r] = C[r] - B @ (R[r + 1] - S[r + 1]) @ B.T
    vec = lambda xs: np.array([np.asarray(x, LD).ravel() for x in xs], float)  # noqa: E731
    mat = lambda xs: np.array([np.asarray(x, LD).T.ravel() for x in xs], float)  # noqa: E731
    return dict(m=vec(m), C=mat(C), a=vec(a), R=mat(R), f=np.array(f, float).reshape(rows, 1),
                Q=np.array(Q, float).reshape(rows, 1), s=vec(s), S=mat(S))


def oracle_filter_smooth_tv(F, G, V, W, m0, C0, y, keep_init):
    n, T = m0.size, y.size
    o = oracle.kf_filter(n, 1, np.ascontiguousarray(F), dlm.cm(G), dlm.cm(V), dlm.cm(W), m0, dlm.cm(C0),
                         np.arange(1, T + 1.0), y.reshape(T, 1), keep_init=keep_init)
    sm = oracle.rts_smooth(n, dlm.cm(G), o, keep_init=keep_init, textbook=True)
    o.update(s=sm["s"], S=sm["S"])
    return o


@pytest.mark.parametrize("name", REG_NAMES)
@pytest.mark.parametrize("keep_init", [0, 1])
@pytest.mark.parametrize("T", [2, 37, 400])
def test_longdouble_reference_with_per_step_F_matches_the_oracle(name, keep_init, T):
    _, F, G, V, W, m0, C0 = regression_model(name, T, seed=T)
    y = simulate_tv(F, G, V, W, m0, C0, seed=T + 1, missing=0.1)
    ref = ld_filter_smooth_tv(F, G, V, W, m0, C0, y, keep_init)
    o = oracle_filter_smooth_tv(F, G, V, W, m0, C0, y, keep_init)
    for k in ("m", "C", "a", "R", "f", "Q", "s", "S"):
        assert ref[k].shape == o[k].shape, k
        assert ld_err(o[k], ref[k]) < TOL_LD, (k, ld_err(o[k], ref[k]))


def _bracketed(lib, n, elems, rng):
    """elems[0] (x) ... (x) elems[-1] with a random bracketing."""
    if len(elems) == 1:
        return elems[0]
    cut = int(rng.integers(1, len(elems)))
    return _comb(lib, n, 0, _bracketed(lib, n, elems[:cut], rng), _bracketed(lib, n, elems[cut:], rng))


@pytest.mark.parametrize("name", REG_NAMES)
def test_elements_with_per_step_F_compose_in_any_bracketing(name):
    lib = capi.load()
    T = 120
    _, F, G, V, W, m0, C0 = regression_model(name, T, seed=3)
    y = simulate_tv(F, G, V, W, m0, C0, seed=4, missing=0.1)
    n = m0.size
    ref = ld_filter_smooth_tv(F, G, V, W, m0, C0, y, keep_init=1)
    start = _pack_f(np.zeros((n, n)), m0, C0, np.zeros(n), np.zeros((n, n)))
    elems = [_pack_f(*_f_element(G, F[t], W, float(V[0, 0]), y[t])) for t in range(T)]
    rng = np.random.default_rng(5)
    for cut in (1, 17, 64, T):
        for _ in range(3):
            _, b, Cm, _, _ = _unpack_f(_bracketed(lib, n, [start] + elems[:cut], rng), n)
            assert ld_err(b[None], ref["m"][cut][None]) < 1e-9, (cut, b, ref["m"][cut])
            assert ld_err(_cm(Cm)[None], ref["C"][cut][None]) < 1e-9, cut


def _problem(n=2, T=10, keep_init=1, f_tv=1, g_tv=0, per_series=0):
    p = capi.Problem()
    p.B, p.T, p.n, p.p, p.keep_init = 1, T, n, 1, keep_init
    p.layout, p.mem = 1, capi.DEVICE
    p.f_tv, p.g_tv, p.per_series = f_tv, g_tv, per_series
    return p


def _err():
    return capi.load().bdlm_last_error(None).decode()


def test_argument_rules_of_a_per_step_F_without_a_context():
    lib = capi.load()
    x = np.zeros(64)
    d = x.ctypes.data
    kf = capi.KfOut(m=d, C=d)
    phases = (lambda p: lib.bdlm_scan_dist_forward_local(None, p, 0, 1, d),
              lambda p: lib.bdlm_scan_dist_forward_finish(None, p, 0, 1, d, kf, None),
              lambda p: lib.bdlm_scan_dist_loglik_partial(None, p, 0, 1, d, None, None, d),
              lambda p: lib.bdlm_scan_dist_ffbs_local(None, p, 0, 1, 0, 10, d, None, d, kf, d, None))
    refused = (_problem(per_series=capi.PS_F | capi.PS_V),  # a per-step F with a per-series V
               _problem(g_tv=1),                             # a per-step G
               _problem(f_tv=0, per_series=capi.PS_F))       # a per-series F that does not vary with t
    for p in refused:
        for call in phases:
            assert call(p) == capi.E_ARG
            assert "n <= 4" in _err() and "v_tv" in _err(), _err()
    # f_tv alone, or with BDLM_PS_F alone, passes the shape check: what stops the call is the context
    for p in (_problem(), _problem(per_series=capi.PS_F)):
        for call in phases:
            assert call(p) == capi.E_ARG
            assert "null context" in _err(), _err()

"""Extended-precision reference for the parallel-in-time scan's tests, and the models they run.

``_ld_filter_smooth`` restates the Kalman filter (KalmanFilter.scala:64-118) and the textbook RTS
smoother (Smoothing.scala:31-47 with S = C - B (R1 - S) B^T) for p = 1, n <= 4, in np.longdouble
(80-bit extended precision on x86-64): an answer whose own rounding is ~1e-19, against which both
the bit-exact sequential kernel and the scan can be measured.  It shares no code with the oracle or
the kernels.  Here it is pinned to the oracle at 1e-12 relative; tests/test_gpu_scan_variants.py
imports it, the model builders and ``rows_per_thread`` from this module.
"""
import math

import numpy as np
import pytest

import helpers as H
from bayesian_dlms_b200 import dlm

LD = np.longdouble
TOL_LD = 1e-12


def _ld_inv(A):
    """Gauss-Jordan inverse with partial pivoting (np.linalg has no longdouble)."""
    n = A.shape[0]
    M = np.concatenate([np.asarray(A, LD), np.eye(n, dtype=LD)], axis=1)
    for j in range(n):
        p = j + int(np.argmax(np.abs(M[j:, j])))
        if M[p, j] == 0:
            raise ZeroDivisionError("singular matrix")
        M[[j, p]] = M[[p, j]]
        M[j] = M[j] / M[j, j]
        for i in range(n):
            if i != j:
                M[i] = M[i] - M[i, j] * M[j]
    return M[:, n:]


def _ld_filter_smooth(F, G, V, W, m0, C0, y, keep_init):
    """F (n,), G (n, n), V scalar, W (n, n), m0 (n,), C0 (n, n), y (T,) with NaN = missing.

    Returns float64 arrays [rows, k] laid out like the library's outputs (matrices column-major
    within a row), rows = T + keep_init.  Row 0 of a keep_init run is the prior, f and Q NaN."""
    F, G, W, C0 = (np.asarray(x, float).astype(LD) for x in (F, G, W, C0))
    m0 = np.asarray(m0, float).ravel().astype(LD)
    V = LD(float(np.asarray(V, float).ravel()[0]))
    y = np.asarray(y, float).ravel()
    n, T = m0.size, y.size
    F = F.ravel()
    I = np.eye(n, dtype=LD)
    rows = T + int(bool(keep_init))
    a, R, m, C = [], [], [], []
    f, Q = [], []
    if keep_init:
        a.append(m0); R.append(C0); m.append(m0); C.append(C0)
        f.append(LD(np.nan)); Q.append(LD(np.nan))
    mt, Ct = m0, C0
    for t in range(T):
        at = G @ mt
        Rt = G @ Ct @ G.T + W
        ft = F @ at
        Qt = F @ Rt @ F + V
        if np.isnan(y[t]):
            mt, Ct = at, Rt
        else:
            K = Rt @ F / Qt
            mt = at + K * (LD(y[t]) - ft)
            IKF = I - np.outer(K, F)
            Ct = IKF @ Rt @ IKF.T + V * np.outer(K, K)
        a.append(at); R.append(Rt); f.append(ft); Q.append(Qt); m.append(mt); C.append(Ct)
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


# ----------------------------------------------------------------------------- models
# p = 1, regular grid.  Every model has a non-zero m0 and full SPD C0 and W, so that an m0, an
# off-diagonal of W or an F other than e1 that the scan dropped would change its answer.
MODEL_NAMES = ("n1", "n2", "n3", "n4", "n4s")


def scan_model(name, W_scale=None, C0_scale=None, V=None):
    """name -> (Dlm, V, W, m0, C0).  ``*_scale`` rescale the full SPD W and C0 (conditioning)."""
    rng = np.random.default_rng(sum(map(ord, name)))
    if name == "n1":
        mod = dlm.polynomial(1)
        Vv, W, m0, C0 = 2.0, np.array([[3.0]]), np.array([1.5]), np.array([[10.0]])
    else:
        mod = {"n2": dlm.seasonal(12, 1),                       # G a rotation, F = (1, 0)
               "n3": dlm.polynomial(1) + dlm.seasonal(12, 1),
               "n4": dlm.polynomial(2) + dlm.seasonal(7, 1),
               "n4s": dlm.seasonal(12, 2)}[name]                 # F = (1, 0, 1, 0)
        n = int(name[1])
        Vv = 1.5
        W = H.spd(rng, n, 0.5)
        m0 = rng.standard_normal(n) + 1.0
        C0 = H.spd(rng, n, 10.0)
    if W_scale is not None:
        W = W / np.max(np.abs(W)) * W_scale
    if C0_scale is not None:
        C0 = C0 / np.max(np.abs(C0)) * C0_scale
    if V is not None:
        Vv = V
    return mod, np.array([[float(Vv)]]), W, m0, C0


def model_arrays(mod, n):
    """(F (n,), G (n, n)) of a time-invariant p = 1 model."""
    F = np.asarray(mod.f(1.0), float).reshape(n)
    G = np.asarray(mod.g(1.0), float)
    return F, G


def simulate(mod, V, W, m0, C0, T, seed, missing=0.0):
    """Dlm.simStep on the regular grid 1..T (as helpers.simulate, vectorised draws)."""
    rng = np.random.default_rng(seed)
    n = m0.size
    F, G = model_arrays(mod, n)
    x = m0 + np.linalg.cholesky(C0) @ rng.standard_normal(n)
    w = rng.standard_normal((T, n)) @ np.linalg.cholesky(W).T
    v = rng.standard_normal(T) * math.sqrt(float(V[0, 0]))
    y = np.empty(T)
    for t in range(T):
        x = G @ x + w[t]
        y[t] = F @ x + v[t]
    if missing > 0:
        y[rng.random(T) < missing] = np.nan
    return y


def rows_per_thread(T, slots):
    """scan.cu scan_rows_per_thread's cost model: level-1 rows per thread for a series of T
    observations when `slots` blocks of the apply sweeps are resident on the device."""
    rows = T + 1.0
    best, best_cost = 64, 1e300
    for sub in range(16, 65, 16):
        blocks = math.ceil(rows / (sub * 128.0))
        waves = blocks / slots
        cost = 3.1 * sub * 0.5 * (math.ceil(waves) + waves) + 0.00057 * rows / sub
        if cost < best_cost:
            best_cost, best = cost, sub
    return best


def close(a, b):
    """H.rel_err over the entries that are not NaN in both; NaN positions must agree."""
    a, b = np.asarray(a, float), np.asarray(b, float)
    na, nb = np.isnan(a), np.isnan(b)
    if not np.array_equal(na, nb):
        return math.inf
    return H.rel_err(a[~na], b[~nb])


def ld_err(a, b):
    """Error of a [rows, k] field against the longdouble reference b, relative to each row's
    largest entry, floored at 1e-3 of the field's largest entry.  Entrywise relative error is no
    measure of the double kernels here: a seasonal component of 0.02 next to a trend of 8000
    carries the trend's absolute rounding (the oracle itself is 6e-12 off on such entries), and
    so does a forecast f near 0.  NaN positions must agree."""
    a, b = np.asarray(a, float), np.asarray(b, float)
    na, nb = np.isnan(a), np.isnan(b)
    if not np.array_equal(na, nb):
        return math.inf
    a, b = np.where(na, 0.0, a), np.where(nb, 0.0, b)
    scale = np.maximum(np.max(np.abs(b), axis=1, keepdims=True), 1e-3 * np.max(np.abs(b), initial=0.0))
    return float(np.max(np.abs(a - b) / np.maximum(scale, 1e-300))) if a.size else 0.0


# ----------------------------------------------------------------------------- tests
def _oracle(mod, V, W, m0, C0, y, keep_init):
    import oracle
    n = m0.size
    F, G = model_arrays(mod, n)
    T = y.size
    o = oracle.kf_filter(n, 1, F, dlm.cm(G), dlm.cm(V), dlm.cm(W), m0, dlm.cm(C0),
                         np.arange(1, T + 1.0), y.reshape(T, 1), keep_init=keep_init)
    sm = oracle.rts_smooth(n, dlm.cm(G), o, keep_init=keep_init, textbook=True)
    o.update(s=sm["s"], S=sm["S"])
    return o


def test_longdouble_is_extended():
    if np.finfo(LD).eps > 1e-18:
        pytest.skip("np.longdouble is IEEE double on this platform")
    assert _ld_inv(np.array([[4.0, 1.0], [2.0, 3.0]])) @ np.array([[4.0, 1.0], [2.0, 3.0]]).astype(LD) \
        == pytest.approx(np.eye(2), abs=1e-18)


@pytest.mark.parametrize("name", MODEL_NAMES)
@pytest.mark.parametrize("keep_init", [0, 1])
@pytest.mark.parametrize("T", [1, 2, 37, 500])
def test_longdouble_reference_matches_the_oracle(name, keep_init, T):
    mod, V, W, m0, C0 = scan_model(name)
    y = simulate(mod, V, W, m0, C0, T, seed=T + 7 * keep_init, missing=0.1)
    if T > 2:
        y[0] = y[-1] = np.nan
    F, G = model_arrays(mod, m0.size)
    ref = _ld_filter_smooth(F, G, V, W, m0, C0, y, keep_init)
    o = _oracle(mod, V, W, m0, C0, y, keep_init)
    for k in ("m", "C", "a", "R", "f", "Q", "s", "S"):
        assert ref[k].shape == o[k].shape, k
        assert ld_err(o[k], ref[k]) < TOL_LD, (k, ld_err(o[k], ref[k]))


def test_longdouble_reference_all_missing():
    mod, V, W, m0, C0 = scan_model("n4")
    y = np.full(50, np.nan)
    F, G = model_arrays(mod, 4)
    ref = _ld_filter_smooth(F, G, V, W, m0, C0, y, 1)
    o = _oracle(mod, V, W, m0, C0, y, 1)
    for k in ("m", "C", "a", "R", "f", "Q", "s", "S"):
        assert ld_err(o[k], ref[k]) < TOL_LD, k
    # pure prediction: the smoothed states are the filtered ones
    assert close(ref["s"], ref["m"]) < TOL_LD and close(ref["S"], ref["C"]) < TOL_LD


@pytest.mark.parametrize("name", MODEL_NAMES)
def test_models_have_the_structure_the_scan_tests_rely_on(name):
    mod, V, W, m0, C0 = scan_model(name)
    n = m0.size
    F, G = model_arrays(mod, n)
    assert np.all(m0 != 0)
    for M in (W, C0):
        assert np.all(np.linalg.eigvalsh(M) > 0)
        assert n == 1 or np.all(M[~np.eye(n, dtype=bool)] != 0)
    if n > 1:
        assert not np.allclose(G, np.triu(G))   # not an upper-triangular (polynomial) G
    if n > 2:
        assert not np.array_equal(F, np.eye(n)[0])
    if name == "n4s":
        assert np.array_equal(F, [1.0, 0.0, 1.0, 0.0])


# forward rows = T + keep_init on both sides of M + 1 = 1024 and 2048 level-2 elements with 16 rows
# per thread; the backward pass has one row fewer, so one more row puts it on the same edges
LEVEL2_EDGE_ROWS = (16368, 16369, 16370, 16384, 16385, 16386, 32752, 32753, 32754, 32768, 32769, 32770)


def test_level2_edges_use_16_rows_per_thread_on_any_occupancy():
    for rows in LEVEL2_EDGE_ROWS:
        for keep_init in (0, 1):
            T = rows - keep_init
            for slots in range(148, 148 * 16 + 1):
                assert rows_per_thread(T, slots) == 16, (T, slots)

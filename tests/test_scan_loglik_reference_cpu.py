"""Extended-precision reference for the parallel-in-time log-likelihood (bdlm_scan_loglik).

``_ld_loglik`` restates both log-likelihood forms of bdlm_loglik for p = 1, n <= 4 in np.longdouble:
the transition form log N(m_t; G m_{t-1}, W) over the filtered means (KalmanFilter.likelihood,
KalmanFilter.scala:299-306) and the innovations form -dd^2/2 - log(sqrt(2 pi) sd) over the observed
steps (conditionalLikelihood, :138-153).  The Cholesky log-determinant and the solve are written out
by hand (np.linalg has no longdouble).  It returns the per-step terms, so that a test can measure a
sum against sum_t |term_t|: the terms can cancel, which makes the sum itself a poor denominator.
Here it is pinned to the oracle at 1e-12 of that scale; tests/test_gpu_scan_loglik.py imports it.
"""
import numpy as np
import pytest

from test_scan_reference_cpu import MODEL_NAMES, model_arrays, scan_model, simulate

LD = np.longdouble
TOL_LD = 1e-12
_LOG_2PI = np.log(2 * np.arccos(LD(-1)))


def _ld_chol(A):
    """Lower Cholesky factor of a symmetric positive definite matrix, in longdouble."""
    n = A.shape[0]
    L = np.zeros((n, n), dtype=LD)
    for j in range(n):
        d = A[j, j] - sum(L[j, k] * L[j, k] for k in range(j))
        if not d > 0:
            raise ValueError("W is not positive definite")
        L[j, j] = np.sqrt(d)
        for i in range(j + 1, n):
            L[i, j] = (A[i, j] - sum(L[i, k] * L[j, k] for k in range(j))) / L[j, j]
    return L


def _ld_solve_chol(L, b):
    """Rows x of X with L L^T x = b for every row b of B (forward then back substitution)."""
    n = L.shape[0]
    z = np.zeros_like(b)
    for i in range(n):
        z[:, i] = (b[:, i] - sum((L[i, k] * z[:, k] for k in range(i)), LD(0))) / L[i, i]
    x = np.zeros_like(b)
    for i in range(n - 1, -1, -1):
        x[:, i] = (z[:, i] - sum((L[k, i] * x[:, k] for k in range(i + 1, n)), LD(0))) / L[i, i]
    return x


def ld_terms(G, W, m0, m, f, Q, y, a=None):
    """Per-step terms from given filtered rows: m (T, n) = m_1..m_T, f, Q (T,) the one-step forecast
    and its variance, y (T,) with NaN = missing.  The transition density's mean is G m_{t-1}, or the
    given prediction rows a (T, n) -- the double a_t = G m_{t-1} a kernel carried, which takes the
    rounding of G m_{t-1} (eps |a_t|, large against m_t - a_t when the state is large) out of a
    comparison with that kernel.  Returns (transition (T,), innovations (T,)) as longdouble; an
    unobserved step's innovations term is 0."""
    G, W = np.asarray(G, LD), np.asarray(W, LD)
    y = np.asarray(y, float).ravel()
    m = np.asarray(m, LD).reshape(y.size, -1)
    f, Q = np.asarray(f, LD).ravel(), np.asarray(Q, LD).ravel()
    n = m.shape[1]
    L = _ld_chol(W)
    half_logdet = sum(np.log(L[k, k]) for k in range(n))
    if a is None:
        a = np.concatenate([np.asarray(m0, LD).reshape(1, n), m[:-1]]) @ G.T
    d = m - np.asarray(a, LD).reshape(y.size, n)
    tr = -np.sum(d * _ld_solve_chol(L, d), axis=1) / 2 - (LD(n) / 2 * _LOG_2PI + half_logdet)
    obs = ~np.isnan(y)
    inn = np.zeros(y.size, dtype=LD)
    sd = np.sqrt(Q[obs])
    dd = (y[obs].astype(LD) - f[obs]) / sd
    inn[obs] = -dd * dd / 2 - (_LOG_2PI / 2 + np.log(sd))
    return tr, inn


def _ld_loglik(F, G, V, W, m0, C0, y):
    """F (n,), G (n, n), V scalar, W (n, n), m0 (n,), C0 (n, n), y (T,) with NaN = missing.
    Returns (transition terms (T,), innovations terms (T,), m_T (n,), C_T (n, n)), longdouble."""
    F = np.asarray(F, float).ravel().astype(LD)
    G, W, C0 = (np.asarray(x, float).astype(LD) for x in (G, W, C0))
    mt = np.asarray(m0, float).ravel().astype(LD)
    V = LD(float(np.asarray(V, float).ravel()[0]))
    y = np.asarray(y, float).ravel()
    n, T = mt.size, y.size
    I = np.eye(n, dtype=LD)
    Ct = C0
    m, f, Q = np.zeros((T, n), dtype=LD), np.zeros(T, dtype=LD), np.zeros(T, dtype=LD)
    for t in range(T):
        at = G @ mt
        Rt = G @ Ct @ G.T + W
        f[t] = F @ at
        Q[t] = F @ Rt @ F + V
        if np.isnan(y[t]):
            mt, Ct = at, Rt
        else:
            K = Rt @ F / Q[t]
            mt = at + K * (LD(y[t]) - f[t])
            IKF = I - np.outer(K, F)
            Ct = IKF @ Rt @ IKF.T + V * np.outer(K, K)
        m[t] = mt
    tr, inn = ld_terms(G, W, m0, m, f, Q, y)
    return tr, inn, mt, Ct


def sum_err(x, terms):
    """|x - sum(terms)| / sum |terms| (0 / 0 = 0: an all-missing innovations sum)."""
    ref = np.sum(terms)
    scale = np.sum(np.abs(terms))
    if scale == 0:
        return 0.0 if x == 0 else np.inf
    return float(abs(LD(x) - ref) / scale)


def _oracle(mod, V, W, m0, C0, y):
    import oracle
    from bayesian_dlms_b200 import dlm
    F, G = model_arrays(mod, m0.size)
    return oracle.loglik(m0.size, 1, F, dlm.cm(G), dlm.cm(V), dlm.cm(W), m0, dlm.cm(C0),
                         np.arange(1, y.size + 1.0), y.reshape(-1, 1))


@pytest.mark.parametrize("name", MODEL_NAMES)
@pytest.mark.parametrize("T", [1, 2, 37, 500])
def test_longdouble_loglik_matches_the_oracle(name, T):
    mod, V, W, m0, C0 = scan_model(name)
    y = simulate(mod, V, W, m0, C0, T, seed=T + 3, missing=0.1)
    if T > 2:
        y[0] = y[-1] = np.nan
    F, G = model_arrays(mod, m0.size)
    tr, inn, mT, CT = _ld_loglik(F, G, V, W, m0, C0, y)
    o = _oracle(mod, V, W, m0, C0, y)
    assert o["status"] == 0
    assert sum_err(o["transition"], tr) < TOL_LD, sum_err(o["transition"], tr)
    assert sum_err(o["innovations"], inn) < TOL_LD, sum_err(o["innovations"], inn)


@pytest.mark.parametrize("name", ["n1", "n4"])
def test_longdouble_loglik_all_missing(name):
    mod, V, W, m0, C0 = scan_model(name)
    y = np.full(50, np.nan)
    F, G = model_arrays(mod, m0.size)
    tr, inn, _, _ = _ld_loglik(F, G, V, W, m0, C0, y)
    o = _oracle(mod, V, W, m0, C0, y)
    assert np.all(inn == 0) and o["innovations"] == 0.0
    assert sum_err(o["transition"], tr) < TOL_LD


def test_terms_from_rows_restate_the_filter():
    """ld_terms on the longdouble filter's own rows is what _ld_loglik returns (the GPU test feeds
    it the scan's rows instead)."""
    mod, V, W, m0, C0 = scan_model("n3")
    y = simulate(mod, V, W, m0, C0, 200, seed=9, missing=0.1)
    F, G = model_arrays(mod, 3)
    from test_scan_reference_cpu import _ld_filter_smooth
    rows = _ld_filter_smooth(F, G, V, W, m0, C0, y, 0)
    tr, inn = ld_terms(G, W, m0, rows["m"], rows["f"], rows["Q"], y)
    tr2, inn2, _, _ = _ld_loglik(F, G, V, W, m0, C0, y)
    assert sum_err(float(np.sum(tr)), tr2) < TOL_LD and sum_err(float(np.sum(inn)), inn2) < TOL_LD

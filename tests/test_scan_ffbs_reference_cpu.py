"""CPU restatement of the parallel-in-time backward sampler (csrc/scan.cu ffbs_*_kernel).

On the regular grid Smoothing.step's draw is affine in the successor draw,
    theta_r = B_r theta_{r+1} + c_r,   c_r = m_r - B_r a_{r+1} + M_r z_r,   theta_T = m_T + M_T z_T,
with M_r = V diag(sqrt(lam)) from the oracle's eigSym of the symmetrised Joseph-form covariance H_r.
Elements (E, g) = (B_r, c_r) compose as E = E_i E_j, g = E_i g_j + g_i (i earlier), so theta_r is the
g of the composition of rows r .. T in ANY bracketing.  These tests pin that restatement to the
oracle's sequential sampler, and the Gibbs statistics summed in the kernels' thread-range order to
the oracle's ascending sum."""
import numpy as np
import pytest

from bayesian_dlms_b200 import dlm
from test_scan_reference_cpu import MODEL_NAMES, model_arrays, scan_model, simulate

TOL = 1e-12
LD = np.longdouble


def filter_rows(mod, V, W, m0, C0, y):
    import oracle
    n, T = m0.size, y.size
    F, G = model_arrays(mod, n)
    return oracle.kf_filter(n, 1, F, dlm.cm(G), dlm.cm(V), dlm.cm(W), m0, dlm.cm(C0),
                            np.arange(1, T + 1.0), y.reshape(T, 1))


def joseph_cov(G, W, m, C):
    """(B, a1, H_r symmetrised) of a filtered row: B = C G^T R1^-1, H = (I - B G) C (I - B G)^T + B W B^T."""
    n = m.size
    a1, R1 = G @ m, G @ C @ G.T + W
    B = np.linalg.solve(R1.T, G @ C.T).T
    D = np.eye(n) - B @ G
    Hm = D @ C @ D.T + B @ W @ B.T
    return B, a1, (Hm + Hm.T) / 2


def eig_sqrt(H):
    """V diag(sqrt(lam)) with the oracle's eigSym (ascending, largest-|component| positive)."""
    import oracle
    n = H.shape[0]
    lam, Vm, _ = oracle.eigsym(dlm.cm(H))
    return Vm * np.sqrt(lam).reshape(1, n)


def elements(G, W, filt, z):
    """(E, g) of rows 0 .. T (row T: the terminal element (0, m_T + M_T z_T))."""
    rows, n = filt["m"].shape
    out = []
    for r in range(rows - 1):
        m, C = filt["m"][r], filt["C"][r].reshape(n, n).T
        B, a1, H = joseph_cov(G, W, m, C)
        out.append((B, m - B @ a1 + eig_sqrt(H) @ z[r]))
    mT, CT = filt["m"][-1], filt["C"][-1].reshape(n, n).T
    out.append((np.zeros((n, n)), mT + eig_sqrt(CT) @ z[-1]))
    return out


def combine(ei, ej):
    """ei (x) ej, ei earlier in time."""
    return ei[0] @ ej[0], ei[0] @ ej[1] + ei[1]


def compose(elems, how, rng=None):
    if len(elems) == 1:
        return elems[0]
    if how == "left":
        acc = elems[0]
        for e in elems[1:]:
            acc = combine(acc, e)
        return acc
    if how == "right":
        acc = elems[-1]
        for e in elems[-2::-1]:
            acc = combine(e, acc)
        return acc
    k = int(rng.integers(1, len(elems)))
    return combine(compose(elems[:k], how, rng), compose(elems[k:], how, rng))


def row_err(a, b):
    """Error relative to each row's largest |entry| of the reference."""
    scale = np.maximum(np.max(np.abs(b), axis=1, keepdims=True), 1e-300)
    return float(np.max(np.abs(a - b) / scale))


@pytest.mark.parametrize("name", MODEL_NAMES)
@pytest.mark.parametrize("how", ["left", "right", "tree"])
def test_composition_in_any_bracketing_is_the_oracles_draw(name, how):
    import oracle
    T = 40
    mod, V, W, m0, C0 = scan_model(name)
    n = m0.size
    y = simulate(mod, V, W, m0, C0, T, seed=3, missing=0.1)
    z = np.random.default_rng(4).standard_normal((T + 1, n))
    filt = filter_rows(mod, V, W, m0, C0, y)
    _, G = model_arrays(mod, n)
    ref = oracle.backward_sample(n, dlm.cm(G), dlm.cm(W), filt, z)
    assert ref["status"] == 0
    el = elements(G, W, filt, z)
    rng = np.random.default_rng(5)
    theta = np.array([compose(el[r:], how, rng)[1] for r in range(T + 1)])
    for r in range(T + 1):  # the composition of a suffix that ends in the terminal element has E = 0
        assert not np.any(compose(el[r:], how, rng)[0])
    e = row_err(theta, ref["theta"])
    assert e < TOL, e


def stats_terms(F, G, y, theta, dtype=float):
    """Per-step terms (t = 0 .. T-1) of oracle_gibbs_stats on the regular grid:
    ssy (y_t - F theta_{t+1})^2 where observed, ny 1 where observed, ssw / scatter of
    d_t = theta_{t+1} - G theta_t."""
    th = np.asarray(theta, dtype)
    F, G = np.asarray(F, dtype), np.asarray(G, dtype)
    obs = ~np.isnan(y)
    f = th[1:] @ F
    res = np.where(obs, (np.where(obs, y, 0).astype(dtype) - f) ** 2, 0)
    d = th[1:] - th[:-1] @ G.T
    n = th.shape[1]
    sc = (d[:, :, None] * d[:, None, :]).transpose(0, 2, 1).reshape(-1, n * n)  # column-major
    return dict(ssy=res, ny=obs.astype(dtype), ssw=d * d, scatter=sc)


def thread_order_sum(terms, sub=16):
    """Sum as the apply sweep does: each thread adds its steps in descending order, threads'
    sums go through a pairwise tree."""
    T = terms.shape[0]
    parts = [np.sum(terms[r0:min(r0 + sub, T)][::-1], axis=0) for r0 in range(0, T, sub)]
    while len(parts) > 1:
        parts = [parts[i] + parts[i + 1] if i + 1 < len(parts) else parts[i] for i in range(0, len(parts), 2)]
    return parts[0]


@pytest.mark.parametrize("name", MODEL_NAMES)
@pytest.mark.parametrize("T", [1, 15, 16, 17, 1000])
def test_gibbs_statistics_in_thread_range_order(name, T):
    import oracle
    mod, V, W, m0, C0 = scan_model(name)
    n = m0.size
    y = simulate(mod, V, W, m0, C0, T, seed=T, missing=0.1)
    z = np.random.default_rng(T + 1).standard_normal((T + 1, n))
    F, G = model_arrays(mod, n)
    o = oracle.ffbs(n, 1, F, dlm.cm(G), dlm.cm(V), dlm.cm(W), m0, dlm.cm(C0), np.arange(1, T + 1.0),
                    y.reshape(T, 1), z)
    ref = oracle.gibbs_stats(n, 1, F, dlm.cm(G), o["time"], y.reshape(T, 1), o["theta"])
    terms = stats_terms(F, G, y, o["theta"])
    for k in ("ssy", "ssw", "scatter"):
        got = np.atleast_1d(thread_order_sum(terms[k]))
        scale = np.maximum(np.sum(np.abs(terms[k]), axis=0), 1e-300)
        e = float(np.max(np.abs(got - ref[k]) / scale))
        assert e < TOL, (k, e)
    assert thread_order_sum(terms["ny"]) == ref["ny"][0] == np.sum(~np.isnan(y))

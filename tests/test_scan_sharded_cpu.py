"""Host side of the time-sharded log-likelihoods and FFBS (bdlm_scan_dist_loglik_* / _ffbs_*,
bdlm_comm_scan_loglik / _ffbs): argument checks that need no device, exchange sizes, the chunk
helper, and a numpy restatement of how the Gibbs statistics of one path split over the ranks."""
import ctypes as C

import numpy as np
import pytest

from bayesian_dlms_b200 import _capi as capi
from bayesian_dlms_b200.sharding import time_chunk
from test_scan_ffbs_reference_cpu import stats_terms
from test_scan_reference_cpu import MODEL_NAMES, model_arrays, scan_model, simulate


def _problem(n=2, T=10, keep_init=0):
    p = capi.Problem()
    p.B, p.T, p.n, p.p, p.keep_init = 1, T, n, 1, keep_init
    p.layout, p.mem = 1, capi.DEVICE
    return p


def _err():
    return capi.load().bdlm_last_error(None).decode()


def test_bad_arguments_are_codes_with_their_reason_even_without_a_context():
    lib = capi.load()
    x = np.zeros(64)
    d = x.ctypes.data
    kf = capi.KfOut(m=d, C=d)
    # rank out of range
    assert lib.bdlm_scan_dist_loglik_partial(None, _problem(), 2, 2, d, None, None, d) == capi.E_ARG
    assert "rank" in _err()
    assert lib.bdlm_scan_dist_ffbs_local(None, _problem(), -1, 2, 5, 20, d, None, d, kf, d, None) == capi.E_ARG
    assert "rank" in _err()
    # keep_init on a rank other than 0, and missing on rank 0
    assert lib.bdlm_scan_dist_loglik_partial(None, _problem(keep_init=1), 1, 2, d, None, None, d) == capi.E_ARG
    assert "keep_init" in _err()
    assert lib.bdlm_scan_dist_ffbs_finish(None, _problem(keep_init=0), 0, 2, d, d, kf, d, None) == capi.E_ARG
    assert "keep_init" in _err()
    # first_row + rows > total_T + 1 (rank 1 of T = 20: rows 11 .. 20 fit, 12 .. 21 do not)
    assert lib.bdlm_scan_dist_ffbs_local(None, _problem(T=10), 1, 2, 12, 20, d, None, d, kf, d, None) == capi.E_ARG
    assert "first_row + rows" in _err()
    assert lib.bdlm_scan_dist_ffbs_local(None, _problem(T=10, keep_init=1), 0, 2, 1, 20, d, None, d, kf, d,
                                         None) == capi.E_ARG
    assert "first_row = 0 on rank 0" in _err()
    # n = 5 is not a scan model
    assert lib.bdlm_scan_dist_loglik_partial(None, _problem(n=5, keep_init=1), 0, 1, d, None, None, d) == capi.E_ARG
    assert "n <= 4" in _err()
    assert lib.bdlm_scan_dist_ffbs_local(None, _problem(n=5), 1, 2, 11, 20, d, None, d, kf, d, None) == capi.E_ARG
    assert "n <= 4" in _err()
    # a per-step V or W is not a scan model: the filter / smoother phases refuse it too
    sm = capi.SmoothOut(s=d, S=d)
    for tv in ("v_tv", "w_tv"):
        p = _problem(keep_init=1)
        setattr(p, tv, 1)
        assert lib.bdlm_scan_dist_forward_local(None, p, 0, 1, d) == capi.E_ARG
        assert tv in _err()
        assert lib.bdlm_scan_dist_forward_finish(None, p, 0, 1, d, kf, None) == capi.E_ARG
        assert tv in _err()
        assert lib.bdlm_scan_dist_backward_local(None, p, 0, 1, kf, sm, d) == capi.E_ARG
        assert tv in _err()
        assert lib.bdlm_scan_dist_backward_finish(None, p, 0, 1, d, kf, sm, None) == capi.E_ARG
        assert tv in _err()
    # null problem / context; the well-formed call still needs a context
    assert lib.bdlm_scan_dist_loglik_partial(None, None, 0, 1, d, None, None, d) == capi.E_ARG
    assert lib.bdlm_scan_dist_ffbs_local(None, _problem(T=10), 1, 2, 11, 20, d, None, d, kf, d, None) == capi.E_ARG
    assert lib.bdlm_scan_dist_loglik_finish(None, 2, d, d, d, None) == capi.E_ARG
    assert lib.bdlm_scan_dist_ffbs_stats_finish(None, 2, 2, d, None, None) == capi.E_ARG
    assert "null context" in _err()
    # communicator calls
    arr = (C.c_void_p * 1)(d)
    fr = (C.c_int64 * 1)(0)
    probs = (capi.Problem * 1)(_problem(keep_init=1))
    assert lib.bdlm_comm_scan_loglik(None, probs, None, None, arr, arr, None) == capi.E_ARG
    assert lib.bdlm_comm_scan_ffbs(None, probs, fr, 10, None, arr, None, None, None) == capi.E_ARG
    assert "null communicator" in lib.bdlm_comm_last_error(None).decode()


@pytest.mark.parametrize("n", [1, 2, 3, 4])
def test_exchange_sizes(n):
    lib = capi.load()
    assert lib.bdlm_scan_dist_doubles(n, capi.SCAN_DIST_SAMPLER_ELEM) == n * n + n
    assert lib.bdlm_scan_dist_doubles(n, capi.SCAN_DIST_LOGLIK_PART) == 3
    assert lib.bdlm_scan_dist_doubles(n, capi.SCAN_DIST_FFBS_PART) == 2 + n + n * n + 1
    # every exchange fits the communicator's 56-double slots (the forward element at n = 4)
    assert max(lib.bdlm_scan_dist_doubles(n, w) for w in range(3)) <= lib.bdlm_scan_elem_doubles(4, 0)
    assert lib.bdlm_scan_dist_doubles(n, 3) == capi.E_ARG
    assert lib.bdlm_scan_dist_doubles(0, 0) == capi.E_ARG and lib.bdlm_scan_dist_doubles(5, 1) == capi.E_ARG


@pytest.mark.parametrize("T", [1, 2, 7, 8, 1000, 2 ** 24])
@pytest.mark.parametrize("world", [1, 2, 3, 5, 8])
def test_time_chunks_tile_the_series(T, world):
    if world > T:
        with pytest.raises(ValueError):
            time_chunk(T, 0, world)
        return
    rows, obs = [], []
    for r in range(world):
        lo, hi, first = time_chunk(T, r, world)
        assert hi > lo
        n_rows = hi - lo + (r == 0)
        rows.extend(range(first, first + n_rows))
        obs.extend(range(lo, hi))
        assert first == (0 if r == 0 else lo + 1)   # global row of observation y[lo] is lo + 1
    assert rows == list(range(T + 1)) and obs == list(range(T))


def chunk_statistics(F, G, y, theta, cuts):
    """Restatement of the per-rank bookkeeping of the time-sharded sampler (ffbs_apply_kernel): rank k
    owns observations y[cuts[k]:cuts[k+1]] and sees only its own rows of theta plus, unless it is last,
    the carry's theta (the next chunk's first row).  Returns each rank's summed terms and the global
    step indices it counted, for observation and transition terms separately."""
    world = len(cuts) - 1
    sums, counted = [], []
    for k in range(world):
        lo, hi = cuts[k], cuts[k + 1]
        keep = k == 0
        first = 0 if keep else lo + 1
        rows = hi - lo + keep
        th = theta[first:first + rows]
        last = k == world - 1
        carry = None if last else theta[first + rows]
        yl = y[lo:hi]
        n = theta.shape[1]
        acc = dict(ssy=0.0, ny=0.0, ssw=np.zeros(n), scatter=np.zeros(n * n))
        obs_steps, trans_steps = [], []

        def add(key_terms, step, which):
            for key, v in key_terms.items():
                acc[key] = acc[key] + v
            (obs_steps if which == "obs" else trans_steps).append(step)

        def obs(cur, yt, step):
            if np.isnan(yt):
                obs_steps.append(step)
                return
            e = yt - cur @ F
            add(dict(ssy=e * e, ny=1.0), step, "obs")

        def trans(cur, prev, step):
            dd = cur - G @ prev
            add(dict(ssw=dd * dd, scatter=np.outer(dd, dd).T.ravel()), step, "trans")

        nsucc = rows - 1 if last else rows
        if not keep and last:
            obs(th[rows - 1], yl[rows - 1], first + rows - 2)   # the terminal row's own observation
        for r in range(nsucc - 1, -1, -1):                      # descending, as the sweep
            cur = th[r + 1] if r + 1 < rows else carry
            step = first + r                                    # step t pairs theta_{t+1}, theta_t
            if keep:
                if r < yl.size:
                    obs(cur, yl[r], step)
            else:
                obs(th[r], yl[r], step - 1)
            trans(cur, th[r], step)
        sums.append(acc)
        counted.append((obs_steps, trans_steps))
    return sums, counted


@pytest.mark.parametrize("name", MODEL_NAMES)
@pytest.mark.parametrize("cuts", [(0, 1, 2, 3), (0, 37), (0, 1, 37), (0, 36, 37), (0, 5, 6, 20, 21, 37),
                                  (0, 16, 32, 37), (0, 12, 13, 14, 30, 37)])
def test_per_rank_statistics_add_up_to_the_whole_path(name, cuts):
    """Chunks of one observation, boundaries inside a run of missing values (y[10:16]) and on thread-
    range edges: the ranks' sums equal stats_terms of the whole path, every step counted once."""
    mod, V, W, m0, C0 = scan_model(name)
    n = m0.size
    T = cuts[-1]
    y = simulate(mod, V, W, m0, C0, T, seed=T + len(cuts), missing=0.1)
    y[10:16] = np.nan
    F, G = model_arrays(mod, n)
    theta = np.random.default_rng(len(cuts)).standard_normal((T + 1, n)) * 3.0
    sums, counted = chunk_statistics(F, G, y, theta, list(cuts))
    for which in (0, 1):
        steps = sorted(s for c in counted for s in c[which])
        assert steps == list(range(T)), (which, steps)
    terms = stats_terms(F, G, y, theta)
    for key in ("ssy", "ny", "ssw", "scatter"):
        got = np.sum([np.atleast_1d(s[key]) for s in sums], axis=0)
        ref = np.sum(terms[key], axis=0)
        scale = np.maximum(np.sum(np.abs(terms[key]), axis=0), 1e-300)
        assert np.max(np.abs(got - ref) / scale) < 1e-13, key
    assert np.sum([s["ny"] for s in sums]) == np.sum(~np.isnan(y))

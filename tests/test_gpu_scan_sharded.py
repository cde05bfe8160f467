"""Time-sharded log-likelihoods and FFBS of one long series (bdlm_scan_dist_loglik_* / _ffbs_*,
bdlm_comm_scan_loglik / _ffbs).

Ranks are emulated on one GPU: one context each, with the all-gathers done by a device
concatenation, as in test_gpu_scan.py::test_device_side_protocol_emulated_ranks.  Every rank must
end with the single-GPU call's results for the whole series: the sums, statistics and status with
the same bits on every rank, theta concatenated over the ranks, and the filter fields of its rows."""
import numpy as np
import pytest

from test_gpu_scan_ffbs import STATS, _gap_rows, _min_eigen_gap, _normals, _scan, _seq, _stats_err
from test_gpu_scan_loglik import _rows, _scan_ll, _seq_ll, _state_err, _terms
from test_scan_ffbs_reference_cpu import row_err, stats_terms
from test_scan_reference_cpu import LEVEL2_EDGE_ROWS, MODEL_NAMES, model_arrays, scan_model, simulate

pytestmark = pytest.mark.gpu
TOL = 1e-9
MIN_EIGEN_GAP = 1e-2


@pytest.fixture(scope="module")
def eng():
    import torch
    assert torch.cuda.is_available()
    from bayesian_dlms_b200 import default_engine
    return default_engine(0)


def _setup(name, T, seed, missing=0.02):
    from bayesian_dlms_b200 import Model
    mod, V, W, m0, C0 = scan_model(name)
    y = simulate(mod, V, W, m0, C0, T, seed, missing)
    return mod, Model.build(mod, T=T), dict(V=V, W=W, m0=m0, C0=C0), y


def _dev(x):
    import torch
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _cuts(T, world):
    from bayesian_dlms_b200.sharding import time_chunk
    return [time_chunk(T, r, world)[0] for r in range(world)] + [T]


def _chunks(mod, params, yd, cuts, cls, **kw):
    """One engine per emulated rank on torch's stream; kw['z'] (whole-series normals) is cut by rows."""
    from bayesian_dlms_b200 import Engine, Model
    ranks = []
    world = len(cuts) - 1
    for r in range(world):
        lo, hi = cuts[r], cuts[r + 1]
        first = 0 if r == 0 else lo + 1
        e = Engine(0)
        e.use_torch_stream()
        args = dict(kw)
        if cls.__name__ == "DistFfbs":
            z = args.pop("z", None)
            rows = hi - lo + (r == 0)
            args.update(first_row=first, total_T=cuts[-1], z=None if z is None else z[first:first + rows].contiguous())
        ranks.append(cls(e, Model.build(mod, T=hi - lo), params, yd[lo:hi].contiguous(), r, world, **args))
    return ranks


def _concat_gather(ranks, src, dst):
    """all-gather emulated: every rank's dst = the concatenation of the ranks' src, in rank order."""
    import torch
    torch.cuda.synchronize()
    g = torch.cat([getattr(d, src) for d in ranks])
    for d in ranks:
        getattr(d, dst).copy_(g)


def _run_loglik(ranks):
    import torch
    for d in ranks:
        d.forward_local()
    _concat_gather(ranks, "agg_f", "aggs_f")
    for d in ranks:
        d.partial()
    _concat_gather(ranks, "part", "parts")
    for d in ranks:
        d.finish()
    torch.cuda.synchronize()
    return [{k: v.cpu().numpy() for k, v in d.out.items()} for d in ranks]


def _run_ffbs(ranks, seed=None):
    import torch
    if seed is not None:
        for d in ranks:
            d.eng.ctx.set_rng(seed, 3, 0)
    for d in ranks:
        d.forward_local()
    _concat_gather(ranks, "agg_f", "aggs_f")
    for d in ranks:
        d.local()
    _concat_gather(ranks, "agg_s", "aggs_s")
    for d in ranks:
        d.finish()
    _concat_gather(ranks, "part", "parts")
    for d in ranks:
        d.stats_finish()
    torch.cuda.synchronize()
    return [{k: v.cpu().numpy() for k, v in d.out.items()} for d in ranks]


def _same_on_every_rank(outs, keys):
    for k in keys:
        for o in outs[1:]:
            assert np.array_equal(o[k], outs[0][k], equal_nan=True), k


def _edge_cuts(T):
    """A chunk of one observation, a boundary on a 16-row thread-range edge (global row 16 * 5) and one
    inside the run of missing values y[3000:3010]."""
    return [0, 1, 2, 16 * 5 - 1, 3005, T]


# ---------------------------------------------------------------------------- log-likelihoods
def _check_loglik(eng, mod, model, params, y, cuts):
    from bayesian_dlms_b200.scan import DistLoglik
    yd = _dev(y)
    one = _scan_ll(eng, model, params, yd)
    seq = _seq_ll(eng, model, params, yd)
    tr, inn = _terms(mod, params, _rows(eng, model, params, yd), y)
    outs = _run_loglik(_chunks(mod, params, yd, cuts, DistLoglik))
    _same_on_every_rank(outs, ("transition", "innovations", "status"))
    got = outs[0]
    assert int(got["status"][0]) == one["status"] == seq["status"] == 0
    for k, terms in (("transition", tr), ("innovations", inn)):
        scale = float(np.sum(np.abs(terms)))
        for ref in (one, seq):
            e = abs(float(got[k][0]) - ref[k]) / scale
            assert e < TOL, (k, e)
    last = outs[-1]
    assert _state_err(last["m"], one["m"]) < TOL and _state_err(last["C"], one["C"]) < TOL
    assert _state_err(last["m"], seq["m"]) < TOL and _state_err(last["C"], seq["C"]) < TOL


@pytest.mark.parametrize("name", MODEL_NAMES)
@pytest.mark.parametrize("world", [1, 2, 3, 5, 8])
def test_loglik_equals_the_single_gpu_call(eng, name, world):
    T = 40_001
    mod, model, params, y = _setup(name, T, seed=world + 11)
    _check_loglik(eng, mod, model, params, y, _cuts(T, world))


@pytest.mark.parametrize("name", MODEL_NAMES)
@pytest.mark.parametrize("T", [2, 8, 65] + [r - 1 for r in LEVEL2_EDGE_ROWS[::3]] + ["edges"])
def test_loglik_short_series_and_edges(eng, name, T):
    if T == "edges":
        T = 40_001
        mod, model, params, y = _setup(name, T, seed=3)
        y[3000:3010] = np.nan
        cuts = _edge_cuts(T)
    else:
        mod, model, params, y = _setup(name, T, seed=T)
        cuts = _cuts(T, min(T, 3))
    _check_loglik(eng, mod, model, params, y, cuts)


# ---------------------------------------------------------------------------- FFBS
def _check_ffbs(eng, mod, model, params, y, cuts, mode, seed):
    from bayesian_dlms_b200.scan import DistFfbs
    T, n = model.T, model.n
    yd = _dev(y)
    zd = _normals(eng, T, n, mode, seed)
    seq = _seq(eng, model, params, yd, zd, want_kf=("m", "C"))
    zd = _normals(eng, T, n, mode, seed)
    one = _scan(eng, model, params, yd, zd, want_kf=("a", "R", "f", "Q"))
    kf = ("a", "R", "f", "Q")
    outs = _run_ffbs(_chunks(mod, params, yd, cuts, DistFfbs, z=zd, want_kf=kf),
                     seed=seed if mode == "philox" else None)
    _same_on_every_rank(outs, STATS + ("status",))
    got = {k: np.concatenate([o[k] for o in outs]) for k in ("theta",) + kf}
    got.update({k: outs[0][k] for k in STATS})
    assert int(outs[0]["status"][0]) == one["status"] == seq["status"] == 0
    gap = _min_eigen_gap(mod, params, seq["m"], seq["C"], _gap_rows(T))
    assert gap > MIN_EIGEN_GAP, gap
    assert got["theta"].shape == one["theta"].shape
    e1, es = row_err(got["theta"], one["theta"]), row_err(got["theta"], seq["theta"])
    assert e1 < TOL and es < TOL, (e1, es)
    for k in kf:
        assert row_err(got[k][1:], one[k][1:]) < TOL, k
        assert np.array_equal(np.isnan(got[k][0]), np.isnan(one[k][0]))
    F, G = model_arrays(mod, n)
    terms = stats_terms(F, G, y, one["theta"])
    e = _stats_err(got, one, terms)
    assert max(e.values()) < TOL, e
    assert got["ny"][0] == np.sum(~np.isnan(y))
    return outs


@pytest.mark.parametrize("mode", ["z", "philox"])
@pytest.mark.parametrize("name", MODEL_NAMES)
@pytest.mark.parametrize("world", [1, 2, 3, 5, 8])
def test_ffbs_equals_the_single_gpu_call(eng, name, world, mode):
    T = 40_001
    mod, model, params, y = _setup(name, T, seed=world + 23, missing=0.03)
    _check_ffbs(eng, mod, model, params, y, _cuts(T, world), mode, seed=world)


@pytest.mark.parametrize("mode", ["z", "philox"])
@pytest.mark.parametrize("name", MODEL_NAMES)
@pytest.mark.parametrize("T", [2, 8, 65] + [r - 1 for r in LEVEL2_EDGE_ROWS[::3]] + ["edges"])
def test_ffbs_short_series_and_edges(eng, name, T, mode):
    if T == "edges":
        T = 40_001
        mod, model, params, y = _setup(name, T, seed=5)
        y[3000:3010] = np.nan
        cuts = _edge_cuts(T)
    else:
        mod, model, params, y = _setup(name, T, seed=T + 1)
        cuts = _cuts(T, min(T, 3))
    _check_ffbs(eng, mod, model, params, y, cuts, mode, seed=7)


# ---------------------------------------------------------------------------- bits, status, draws
def test_same_bits_on_every_rank_and_call(eng):
    from bayesian_dlms_b200.scan import DistFfbs, DistLoglik
    T = 20_000
    mod, model, params, y = _setup("n4", T, seed=2)
    yd = _dev(y)
    cuts = _cuts(T, 5)
    ll, fb = _chunks(mod, params, yd, cuts, DistLoglik), _chunks(mod, params, yd, cuts, DistFfbs)
    first_ll, first_fb = _run_loglik(ll), _run_ffbs(fb, seed=9)
    for _ in range(2):
        for a, b in zip(first_ll, _run_loglik(ll)):
            for k in a:
                assert np.array_equal(a[k], b[k], equal_nan=True), k
        for a, b in zip(first_fb, _run_ffbs(fb, seed=9)):
            for k in a:
                assert np.array_equal(a[k], b[k], equal_nan=True), k


@pytest.mark.parametrize("name", ["n1", "n2", "n4"])
@pytest.mark.parametrize("case", ["control", "inf", "zero_variances"])
def test_status_of_every_rank_is_the_single_gpu_status(eng, name, case):
    from bayesian_dlms_b200 import _capi as capi
    from bayesian_dlms_b200.scan import DistFfbs, DistLoglik
    T = 5000
    mod, model, params, y = _setup(name, T, seed=8)
    n = model.n
    if case == "inf":
        y[1234] = np.inf
    if case == "zero_variances":
        params = dict(params, V=np.zeros((1, 1)), W=np.zeros((n, n)), C0=np.zeros((n, n)))
    yd = _dev(y)
    zd = _normals(eng, T, n, "z", seed=1)
    want_ll = _scan_ll(eng, model, params, yd)["status"]
    want_fb = _scan(eng, model, params, yd, zd)["status"]
    cuts = _cuts(T, 3)
    got_ll = {int(o["status"][0]) for o in _run_loglik(_chunks(mod, params, yd, cuts, DistLoglik))}
    got_fb = {int(o["status"][0]) for o in _run_ffbs(_chunks(mod, params, yd, cuts, DistFfbs, z=zd))}
    print(name, case, "loglik", want_ll, got_ll, "ffbs", want_fb, got_fb)
    assert got_ll == {want_ll} and got_fb == {want_fb}
    assert want_fb == {"control": 0, "inf": 8, "zero_variances": 9}[case]
    # the log-likelihoods include the transition form, whose W = 0 is not positive definite: + NOTPD
    assert want_ll == {"control": 0, "inf": 8, "zero_variances": 9 | capi.ST_NOTPD}[case]


def test_gibbs_draws_are_the_same_on_every_rank(eng):
    import torch
    from bayesian_dlms_b200 import SERIES_MAJOR, _capi as capi
    from bayesian_dlms_b200.scan import DistFfbs
    T = 30_000
    mod, model, params, y = _setup("n2", T, seed=4)
    ranks = _chunks(mod, params, _dev(y), _cuts(T, 5), DistFfbs)
    _run_ffbs(ranks, seed=3)
    draws = []
    for d in ranks:
        n = d.n
        prob = capi.Problem()
        prob.B, prob.T, prob.n, prob.p, prob.layout, prob.mem = 1, T, n, 1, SERIES_MAJOR, capi.DEVICE
        prob.keep_init = 1
        gs = capi.GibbsStats(**{k: d.out[k].data_ptr() for k in STATS})
        prior = capi.GibbsPrior(3.0, 3.0, 3.0, 3.0, 0.0, None)
        rng = capi.GibbsRng(11, 2, None, None, None)
        V, W = (torch.empty(k, dtype=torch.float64, device="cuda") for k in (1, n * n))
        d.eng.ctx.check(capi.load().bdlm_gibbs_draw(d.eng.ctx.handle, prob, gs, prior, rng, V.data_ptr(),
                                                    W.data_ptr(), None, None, None))
        torch.cuda.synchronize()
        draws.append((V.cpu().numpy(), W.cpu().numpy()))
    for V, W in draws[1:]:
        assert np.array_equal(V, draws[0][0]) and np.array_equal(W, draws[0][1])
    assert np.all(np.isfinite(draws[0][0])) and np.all(draws[0][0] > 0)


def test_launch_counts_per_phase(eng):
    from bayesian_dlms_b200.scan import DistFfbs, DistLoglik
    T = 200_000  # two chunks of 100 000: two level-2 launches each
    mod, model, params, y = _setup("n3", T, seed=9)
    yd = _dev(y)
    cuts = _cuts(T, 2)
    ll, fb = _chunks(mod, params, yd, cuts, DistLoglik), _chunks(mod, params, yd, cuts, DistFfbs)
    _run_loglik(ll)
    _run_ffbs(fb)

    def count(d, phase):
        c0 = d.eng.ctx.launch_count()
        getattr(d, phase)()
        return d.eng.ctx.launch_count() - c0
    # loglik: fold + sweep + block sum; one kernel for the rank-order sum
    assert [count(d, "partial") for d in ll] == [3, 3]
    assert [count(d, "finish") for d in ll] == [1, 1]
    # FFBS local: forward fold + apply, sampler reduce (+ identity terminal on rank 0), level 2 (2 here)
    assert [count(d, "local") for d in fb] == [6, 5]
    # finish: carry fold (rank 0 only) + apply + block sum; stats: one kernel
    assert [count(d, "finish") for d in fb] == [3, 2]
    assert [count(d, "stats_finish") for d in fb] == [1, 1]


# ---------------------------------------------------------------------------- communicator
def _comm_case(comm, T, name="n2", mode="z"):
    """Single-GPU references and the communicator's per-device handles for one series."""
    import torch
    from bayesian_dlms_b200.sharding import time_chunk
    mod, model, params, y = _setup(name, T, seed=13)
    world = comm.world
    yd = _dev(y)
    models, chunks, firsts = [], [], []
    for i, d in enumerate(comm.devices):
        lo, hi, first = time_chunk(T, comm.first_rank + i, world)
        with torch.cuda.device(d):
            chunks.append(yd[lo:hi].to(f"cuda:{d}").contiguous())
        from bayesian_dlms_b200 import Model
        models.append(Model.build(mod, T=hi - lo))
        firsts.append(first)
    return mod, model, params, y, yd, models, chunks, firsts


def _comm_check(eng, comm, T, mode):
    import torch
    from bayesian_dlms_b200.scan import scan_filter_smooth
    mod, model, params, y, yd, models, chunks, firsts = _comm_case(comm, T)
    n = model.n
    z = np.random.default_rng(5).standard_normal((T + 1, n))
    zd = _dev(z) if mode == "z" else None
    if mode == "philox":
        eng.ctx.set_rng(17, 1, 0)
        for e in comm.engines:
            e.ctx.set_rng(17, 1, 0)
    one_fs = scan_filter_smooth(eng, model, params, yd)
    one_ll = _scan_ll(eng, model, params, yd)
    one_fb = _scan(eng, model, params, yd, zd)
    torch.cuda.synchronize()
    h = comm.scan_setup(models, params, chunks)
    zs = None
    if mode == "z":
        zs = []
        for i, d in enumerate(comm.devices):
            rows = models[i].T + int(firsts[i] == 0)
            zs.append(zd[firsts[i]:firsts[i] + rows].to(f"cuda:{d}").contiguous())
    for rep in range(2):   # filter_smooth -> loglik -> ffbs -> filter_smooth on one communicator
        fs = comm.scan_run(h)
        comm.sync()
        for i, o in enumerate(fs):
            lo = firsts[i]
            for k in ("m", "C", "s", "S"):
                ref = one_fs[k][lo:lo + o[k].shape[0]].cpu().numpy()
                assert row_err(o[k].cpu().numpy(), ref) < TOL, (rep, k)
        if rep == 1:
            break
        ll = comm.scan_loglik(h)
        comm.sync()
        for o in ll:
            assert int(o["status"][0]) == one_ll["status"] == 0
            for k in ("transition", "innovations"):
                assert abs(float(o[k][0]) - one_ll[k]) < TOL * abs(one_ll[k]) + 1e-9, k
        if comm.first_rank + len(comm.devices) == comm.world:
            assert _state_err(ll[-1]["m"].cpu().numpy(), one_ll["m"]) < TOL
        fb = comm.scan_ffbs(h, firsts, T, zs)
        comm.sync()
        theta = np.concatenate([o["theta"].cpu().numpy() for o in fb])
        if len(theta) == T + 1:
            assert row_err(theta, one_fb["theta"]) < TOL
        for o in fb:
            assert int(o["status"][0]) == one_fb["status"] == 0
            assert o["ny"][0].item() == one_fb["ny"][0]
            for k in ("ssy", "ssw", "scatter"):
                assert np.allclose(o[k].cpu().numpy(), one_fb[k], rtol=TOL, atol=0), k
        _same_on_every_rank([{k: o[k].cpu().numpy() for k in STATS + ("status",)} for o in fb],
                            STATS + ("status",))


@pytest.mark.parametrize("mode", ["z", "philox"])
def test_world_one_communicator(eng, mode):
    from bayesian_dlms_b200.comm import Comm
    comm = Comm.single_process([0])
    try:
        _comm_check(eng, comm, 20_001, mode)
    finally:
        comm.close()


@pytest.mark.parametrize("peer", [True, False])
def test_world_two_communicator_interleaved_with_the_filter_smoother(eng, peer, monkeypatch):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    if not peer:
        monkeypatch.setenv("BDLM_COMM_NO_PEER", "1")
    from bayesian_dlms_b200.comm import Comm
    comm = Comm.single_process([0, 1])
    try:
        if peer and not comm.uses_peer_exchange:
            pytest.skip("no peer access between the two GPUs")
        _comm_check(eng, comm, 20_001, "z")
    finally:
        comm.close()

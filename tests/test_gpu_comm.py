"""The multi-GPU communicator of the C ABI (bdlm_comm_*): per-device contexts + NCCL behind one
object.  With one visible GPU the world-1 communicator still runs every code path (host threads,
sub-range dispatch, ncclAllReduce / all-gather on one rank); the world-2 cases need two visible
GPUs and are skipped otherwise."""
import os

import numpy as np
import pytest

import helpers as H

pytestmark = pytest.mark.gpu


def _ngpu():
    import torch
    return torch.cuda.device_count()


def _devices(world):
    if _ngpu() < world:
        pytest.skip("needs %d GPUs" % world)
    return list(range(world))


@pytest.fixture(scope="module")
def eng():
    from bayesian_dlms_b200 import default_engine
    return default_engine(0)


@pytest.mark.parametrize("world", [1, 2])
def test_sharded_host_batch_equals_one_call(eng, world):
    """A host batch cut over the communicator's devices gives exactly the results of one
    bdlm_kf_filter_smooth / bdlm_loglik / bdlm_ffbs call, and the NCCL-reduced sums equal the sums
    of the per-series values."""
    from bayesian_dlms_b200 import Model, SERIES_MAJOR, TIME_MAJOR
    from bayesian_dlms_b200.comm import Comm
    comm = Comm.single_process(_devices(world))
    try:
        mod, V, W, m0, C0 = H.second_order()
        rng = np.random.default_rng(8)
        B, T = 1001, 60
        y = rng.standard_normal((B, T, 1)).cumsum(axis=1)
        y[rng.random(y.shape) < 0.05] = np.nan
        model = Model.build(mod, T=T)
        params = dict(V=V, W=W, m0=m0, C0=C0)
        for layout in (SERIES_MAJOR, TIME_MAJOR):
            yy = y if layout == SERIES_MAJOR else np.ascontiguousarray(y.transpose(1, 2, 0))
            one = eng.filter_smooth(model, params, yy, layout=layout)
            many = comm.filter_smooth(model, params, yy, layout=layout)
            for k in ("m", "C", "a", "R", "f", "Q", "s", "S"):
                assert np.array_equal(one[k], many[k], equal_nan=True), (k, layout)
            ll1 = eng.loglik(model, params, yy, layout=layout)
            ll = comm.loglik(model, params, yy, layout=layout)
            assert np.array_equal(ll1["transition"], ll["transition"])
            assert abs(ll["sum_transition"] - ll1["transition"].sum()) <= 1e-9 * abs(ll1["transition"].sum())
            assert abs(ll["sum_innovations"] - ll1["innovations"].sum()) <= 1e-9 * abs(ll1["innovations"].sum())
        f1 = eng.filter(model, params, y, layout=SERIES_MAJOR, keep_init=False)
        fN = comm.filter(model, params, y, layout=SERIES_MAJOR, keep_init=False)
        assert np.array_equal(f1["C"], fN["C"]) and np.array_equal(f1["f"], fN["f"], equal_nan=True)
        s1 = eng.svd_filter(model, params, y, layout=SERIES_MAJOR)
        sN = comm.svd_filter(model, params, y, layout=SERIES_MAJOR)
        assert np.array_equal(s1["uc"], sN["uc"]) and np.array_equal(s1["dc"], sN["dc"])
        # FFBS with injected normals: chains identical whatever the cut; pooled statistics
        mod13, V, W, m0, C0 = H.seasonal13()
        B, T = 37, 30
        y = rng.standard_normal((B, T, 1)) * 2
        z = rng.standard_normal((B, T + 1, 13))
        model = Model.build(mod13, T=T)
        params = dict(V=V, W=W, m0=m0, C0=C0)
        one = eng.ffbs(model, params, y, z, layout=SERIES_MAJOR, stats=True)
        many = comm.ffbs(model, params, y, z, layout=SERIES_MAJOR)
        assert np.array_equal(one["theta"], many["theta"])
        for k in ("ssy", "ny", "ssw", "scatter"):
            assert np.array_equal(one[k], many[k]), k
            assert np.allclose(many["pooled"][k], one[k].sum(axis=0), rtol=1e-12), k
        v = comm.allreduce_sum(np.array([1.5, -2.0, 3.0]))
        assert np.array_equal(v, [1.5, -2.0, 3.0])      # one process contributes once
    finally:
        comm.close()


@pytest.mark.parametrize("world,peer", [(1, True), (2, True), (2, False)])
@pytest.mark.parametrize("n", [1, 2])
def test_time_sharded_scan_through_the_communicator(eng, world, peer, n):
    """bdlm_comm_scan_filter_smooth on real devices: NCCL all-gathers (peer = False) or peer
    mailboxes over NVLink (peer = True, when the devices can address each other) -- both equal the
    single-GPU scan of the whole series to 1e-9."""
    import torch
    from bayesian_dlms_b200 import Model, dlm
    from bayesian_dlms_b200.comm import Comm
    from bayesian_dlms_b200.scan import scan_filter_smooth
    from bayesian_dlms_b200.sharding import shard_range
    devs = _devices(world)
    if peer:
        os.environ.pop("BDLM_COMM_NO_PEER", None)
    else:
        os.environ["BDLM_COMM_NO_PEER"] = "1"
    comm = Comm.single_process(devs)
    os.environ.pop("BDLM_COMM_NO_PEER", None)
    try:
        if world > 1 and not peer:
            assert not comm.uses_peer_exchange
        mod = dlm.polynomial(n)
        V, W = np.array([[3.0]]), np.diag([2.0, 1.0][:n])
        m0, C0 = np.zeros(n), 100.0 * np.eye(n)
        T = 200_003
        rng = np.random.default_rng(5)
        y = rng.standard_normal(T).cumsum() * 0.1
        y[rng.random(T) < 0.01] = np.nan
        params = dict(V=V, W=W, m0=m0, C0=C0)
        yd0 = torch.from_numpy(y).cuda(0)
        ref = scan_filter_smooth(eng, Model.build(mod, T=T), params, yd0)
        torch.cuda.synchronize(0)
        models, chunks = [], []
        for r in range(world):
            lo, hi = shard_range(T, r, world)
            models.append(Model.build(mod, T=hi - lo))
            chunks.append(torch.from_numpy(y[lo:hi].copy()).cuda(devs[r]))
        h = comm.scan_setup(models, params, chunks)
        for _ in range(3):          # repeated calls reuse the mailboxes (epoch flags)
            outs = comm.scan_run(h)
        comm.sync()
        assert all(int(s.item()) == 0 for s in h["status"])
        for k in ("m", "C", "a", "R", "s", "S"):
            got = np.concatenate([o[k].cpu().numpy() for o in outs])
            want = ref[k].cpu().numpy()
            assert got.shape == want.shape
            assert H.rel_err(got, want) < 1e-9, (k, world, peer, H.rel_err(got, want))
    finally:
        comm.close()

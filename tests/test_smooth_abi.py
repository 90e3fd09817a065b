"""Argument checks of the ensemble Kalman smoother of recorded hydrographs (txh_enks_smooth, txh_set_transform_history,
Muskingum.run_assimilating(smooth_lag=...)) and the self-consistency of its gain-form reference: bad input is refused
before any device work, so these run without a GPU."""
import ctypes
import types

import numpy as np
import pytest

from enks_oracle import enks_gain


def test_enks_gain_is_the_filter_gain_for_the_current_forecast(oracle):
    """Applied to the forecast the update started from, with Q = 0, the smoother gain is the filter gain K dz of
    oracle.enkf_update (its cross-covariance P[:, s] is then the sample one alone)."""
    from tx_fast_hydrology_b200 import synthetic as S
    n, M, m, seed = 300, 24, 12, 5
    net = S.make_network(n, seed)
    prm = S.make_params(n, seed)
    rng = np.random.default_rng(seed)
    O = prm["o_t"][:, None] * rng.uniform(0.5, 1.5, size=(n, M))
    gauges = np.asarray(S.make_gauges(net["endnodes"], m, seed=seed), dtype=np.int64)
    m = gauges.size
    Zp = rng.uniform(0.5, 8.0, size=(m, 1)) + 0.1 * rng.standard_normal((m, M))
    R = 1e-2 * np.eye(m)
    ind = oracle.compute_indegree(net["startnodes"], net["endnodes"])
    onet = {"startnodes": net["startnodes"], "endnodes": net["endnodes"], "indegree": ind}
    _, _, K = oracle.enkf_update(onet, O, O, gauges, Zp, np.zeros(n), R)
    A = O - O.mean(axis=1, keepdims=True)
    HA = A[gauges]
    S_ = HA @ HA.T / (M - 1) + R
    want = K @ (Zp - O[gauges])
    got = enks_gain(A, HA, Zp - O[gauges], S_)
    assert float(np.abs(got - want).max()) <= 1e-12 * float(np.abs(want).max())


_BUF = (ctypes.c_double * 4096)()


def _smooth(libtxh, M=4, nupd=3, every=2, T=True, nslots=3, k=5, rec_every=2, lag=3, rec=True, out=True, work=True,
            out_offset=None):
    base = ctypes.addressof(_BUF)
    o = base + 8 * (out_offset if out_offset is not None else 2048)
    return libtxh.txh_enks_smooth(M, nupd, every, base + 8 * 3000 if T else None, nslots, k, rec_every, lag,
                                  base if rec else None, o if out else None, base + 8 * 3500 if work else None, None)


@pytest.mark.parametrize("kw,msg", [
    (dict(M=1), b"member count"), (dict(M=0), b"member count"), (dict(nupd=-1), b"update count"),
    (dict(every=0), b"cadence"), (dict(rec_every=0), b"recording shape"), (dict(nslots=-1), b"recording shape"),
    (dict(lag=-1), b"lag"), (dict(T=False), b"null"), (dict(rec=False), b"null"), (dict(out=False), b"null"),
    (dict(work=False), b"null"), (dict(out_offset=10), b"overlaps"), (dict(out_offset=0), b"overlaps")])
def test_enks_smooth_rejects_bad_arguments(libtxh, kw, msg):
    assert _smooth(libtxh, **kw) == -1
    assert msg in libtxh.txh_last_error()


def test_enks_smooth_needs_a_device(libtxh):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present")
    assert _smooth(libtxh) == -4
    assert _smooth(libtxh, out_offset=60) == -4          # out right behind rec: no overlap
    assert _smooth(libtxh, M=2, lag=0) == -4
    assert libtxh.txh_enks_work_size(64, 168) == 6 * 168 * 64 * 64


def _net():
    from tx_fast_hydrology_b200.network import RiverNetwork
    net = RiverNetwork(np.array([1, 2, 2], dtype=np.int64))
    net.compute_coeffs(np.full(3, 600.0), np.full(3, 0.2), 300.0)
    return net


def _assim(libtxh, net, nsteps, every, M=2):
    buf = (ctypes.c_double * 8)()
    obs = (ctypes.c_int64 * 1)(1)
    rr = (ctypes.c_int64 * 1)(0)
    return libtxh.txh_run_assimilating_rec(net.handle, buf, buf, M, None, 0, 1, nsteps, every, 1, obs, 1, buf, buf, buf,
                                           buf, 1, buf, buf, buf, buf, buf, buf, 0, None, rr, 1, 1, buf, None, None)


def test_transform_history_arguments(libtxh):
    net = _net()
    hist = (ctypes.c_double * 16)()
    assert libtxh.txh_set_transform_history(None, hist, 16) == -1
    assert libtxh.txh_set_transform_history(net.handle, hist, -1) == -1
    assert b"capacity" in libtxh.txh_last_error()
    # 3 updates of 2 x 2 need 12 doubles: 11 is refused before any device work
    assert libtxh.txh_set_transform_history(net.handle, hist, 11) == 0
    assert _assim(libtxh, net, 6, 2) == -1
    assert b"transform history" in libtxh.txh_last_error()
    assert libtxh.txh_set_transform_history(net.handle, None, 0) == 0   # off again


def test_transform_history_call_needs_a_device(libtxh):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present")
    net = _net()
    hist = (ctypes.c_double * 16)()
    assert libtxh.txh_set_transform_history(net.handle, hist, 12) == 0
    assert _assim(libtxh, net, 6, 2) == -4                # the capacity suffices: on to the device
    assert _assim(libtxh, net, 7, 2) == -4                # remainder steps add no update
    assert libtxh.txh_set_transform_history(net.handle, None, 0) == 0


@pytest.mark.parametrize("lag,reaches,enkf,msg", [
    (-1, [0], None, "non-negative"), (2.5, [0], None, "non-negative"), (True, [0], None, "non-negative"),
    ("3", [0], None, "non-negative"), (3, None, None, "record_reaches"),
    (3, [0], types.SimpleNamespace(world=2), "member-sharded")])
def test_python_smoothing_arguments_raise_value_error(libtxh, lag, reaches, enkf, msg):
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.muskingum import Muskingum
    nd = S.make_network(10, 1)
    m = Muskingum(S.model_dict(nd, S.make_params(10, 1)))
    with pytest.raises(ValueError, match=msg):
        m.run_assimilating(None, 12, enkf, 6, None, record_reaches=reaches, smooth_lag=lag)

"""Argument checks of the hydrograph recording of the assimilation loop (txh_run_assimilating_rec,
Muskingum.run_assimilating(record_reaches=...)): bad input is refused before any device work, so these run without
a GPU."""
import ctypes

import numpy as np
import pytest


def _net():
    from tx_fast_hydrology_b200.network import RiverNetwork
    net = RiverNetwork(np.array([1, 2, 2], dtype=np.int64))
    net.compute_coeffs(np.full(3, 600.0), np.full(3, 0.2), 300.0)
    return net


def _call(libtxh, net, reaches, rec_every, rec_out=True):
    buf = (ctypes.c_double * 8)()
    obs = (ctypes.c_int64 * 1)(1)
    rr = (ctypes.c_int64 * max(1, len(reaches)))(*reaches)
    return libtxh.txh_run_assimilating_rec(net.handle, buf, buf, 2, None, 0, 1, 2, 1, 1, obs, 1, buf, buf, buf, buf, 1,
                                           buf, buf, buf, buf, buf, buf, 0, None, rr, len(reaches), rec_every,
                                           buf if rec_out else None, None, None)


def test_rec_entry_point_rejects_bad_recording_arguments(libtxh):
    net = _net()
    assert _call(libtxh, net, [0, 2, 0], 1) == -1                   # duplicate
    assert b"twice" in libtxh.txh_last_error()
    assert _call(libtxh, net, [0, 3], 1) == -1                      # out of range
    assert _call(libtxh, net, [-1], 1) == -1
    assert _call(libtxh, net, [1], 0) == -1                         # rec_every < 1
    assert _call(libtxh, net, [1], 1, rec_out=False) == -1          # no output buffer


def test_rec_entry_point_needs_a_device(libtxh):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present")
    net = _net()
    assert _call(libtxh, net, [0, 2], 2) == -4
    assert _call(libtxh, net, [], 1) == -4                          # rec_count == 0: txh_run_assimilating


@pytest.mark.parametrize("reaches,every,msg", [([0, 1, 1], 1, "twice"), ([0, 10], 1, "out of range"),
                                               ([-1], 1, "out of range"), ([[0, 1]], 1, "1-D"), ([], 1, "1-D"),
                                               ([0.5], 1, "integer"), ([0], 0, "positive"), ([0], 2.5, "positive"),
                                               ([0], 100, "records nothing")])
def test_python_recording_arguments_raise_value_error(libtxh, reaches, every, msg):
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.muskingum import Muskingum
    nd = S.make_network(10, 1)
    m = Muskingum(S.model_dict(nd, S.make_params(10, 1)))
    with pytest.raises(ValueError, match=msg):
        m.run_assimilating(None, 12, None, 6, None, record_reaches=reaches, record_every=every)

"""A network handle stays usable after a CUDA call on it fails.

A refused allocation is an ordinary (non-sticky) runtime error.  The call that met it reports TXH_E_CUDA; the next
call on the same handle must neither fail with that stale error nor compute anything different.  Both requests below
exceed the device's memory, so the driver refuses them at once without reserving anything.
"""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N, M, SEED = 10_000, 4, 7
TXH_E_CUDA = -3


def _handle():
    """A 10,000-reach synthetic network with coefficients and a seeded 4-member state on the device."""
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.network import RiverNetwork
    nd, prm = S.make_network(N, SEED), S.make_params(N, SEED)
    net = RiverNetwork(nd["endnodes"])
    net.compute_coeffs(prm["K"], prm["X"], 300.0)
    o = prm["o_t"][:, None] * np.random.default_rng(SEED).uniform(0.5, 1.5, size=(N, M))
    O, I = net.alloc_state(M), net.alloc_state(M)
    net.pack_host(o, M, O)
    net.init_inflows(O, I, M)
    return net, O, I


def _pack_host_too_large(lib, net, O, stream):
    # stages 2**24 members of every reach, about 1.3 TB; the pointers are never read
    src = np.zeros(8)
    return lib.txh_pack_host(net.handle, src.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), 2**24, 0,
                             ctypes.c_void_p(O.data_ptr()), stream)


def _forcing_create_too_large(lib, net, O, stream):
    # a table of 2**22 rows, about 335 GB; the times are read (checked ascending) before the allocation, the table not
    from tx_fast_hydrology_b200 import _lib as L
    R = 2**22
    times = np.arange(R, dtype=np.float64)
    table = np.zeros(8)
    out = ctypes.c_void_p()
    return lib.txh_forcing_create(net.handle, R, L.ptr_f64(times), ctypes.c_void_p(table.ctypes.data), 0, None, stream,
                                  ctypes.byref(out))


@pytest.mark.parametrize("failing", [_pack_host_too_large, _forcing_create_too_large], ids=["pack_host", "forcing_create"])
def test_handle_usable_after_failed_call(libtxh, failing):
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (no CPU fallback exists)"
    from tx_fast_hydrology_b200.network import _stream_ptr
    net, O, I = _handle()
    stream = _stream_ptr()
    assert failing(libtxh, net, O, stream) == TXH_E_CUDA, libtxh.txh_last_error()

    net.route_step(O, I, M)
    ref, O_ref, I_ref = _handle()
    ref.route_step(O_ref, I_ref, M)
    assert np.array_equal(net.unpack_host(O, M), ref.unpack_host(O_ref, M))
    assert np.array_equal(net.unpack_host(I, M), ref.unpack_host(I_ref, M))
    assert libtxh.txh_check(net.handle, stream) == 0, libtxh.txh_last_error()

"""GPU parity tests of the routing kernels, through the C ABI (libtxh.so), against the
CPU oracle and the golden vectors produced by the unmodified reference.

Tolerance: FP64, element-wise relative error <= 1e-9 with an absolute floor of 1e-12 of the largest
element (tests/parity.py; BASELINE.json north_star); the kernels re-associate the confluence sums and
contract to FMA, so results are not bit-identical (observed ~1e-15).  Integer artefacts are compared exactly elsewhere (test_topology.py).
"""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RTOL = 1e-9


from parity import relerr, normerr        # element-wise |a-b| / max(|b|, 1e-12 max|b|); max-norm


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (no CPU fallback exists)"
    return torch


def _setup(endnodes, K, X, dt, sched_params=None):
    from tx_fast_hydrology_b200.network import RiverNetwork
    net = RiverNetwork(endnodes, sched_params)
    coef = net.compute_coeffs(K, X, dt)
    return net, coef


def _upload(torch, net, o, i, M):
    """o, i: [n] or [n][M] host arrays in reach order -> device schedule-order tensors."""
    O = net.alloc_state(M); I = net.alloc_state(M)
    net.pack_host(np.asarray(o, dtype=np.float64).reshape(net.n, M), M, O)
    net.pack_host(np.asarray(i, dtype=np.float64).reshape(net.n, M), M, I)
    return O, I


@pytest.mark.parametrize("kernel", ["lane", "window", "dataflow"])
@pytest.mark.parametrize("fname", ["kernels_n60.npz", "kernels_n160.npz"])
def test_golden_kernels(torch_cuda, libtxh, golden_dir, monkeypatch, fname, kernel):
    """Outputs of the unmodified reference's kernels; single steps and operator applications run on the
    window kernel (the default) and on the dataflow kernel."""
    monkeypatch.setenv("TXH_ROUTE_KERNEL", kernel)
    torch = torch_cuda
    g = np.load(os.path.join(golden_dir, fname))
    n = g["endnodes"].size
    net, coef = _setup(g["endnodes"], g["K"], g["X"], float(g["dt"]))
    for c, k in zip(coef, ("alpha", "beta", "chi", "gamma")):
        assert (c == g[k]).all()                       # coefficient arithmetic is bit-exact
    q = torch.from_numpy(g["q"]).cuda()
    # _ax_bu (nutils.py:64-89): dataflow kernel and level-scheduled kernel
    for levels in (False, True):
        O, I = _upload(torch, net, g["o_init"], g["i_init"], 1)
        net.route_step(O, I, 1, q, levels=levels)
        o = net.unpack_host(O, 1)[:, 0]; i = net.unpack_host(I, 1)[:, 0]
        assert relerr(o, g["axbu_o"]) < RTOL and relerr(i, g["axbu_i"]) < RTOL
    # _ax (nutils.py:91-114): no forcing
    O, I = _upload(torch, net, g["o_init"], g["i_init"], 1)
    net.route_step(O, I, 1, None)
    assert relerr(net.unpack_host(O, 1)[:, 0], g["ax_o"]) < RTOL
    assert relerr(net.unpack_host(I, 1)[:, 0], g["ax_i"]) < RTOL
    # init_states (muskingum.py:410-419): self-loop inflow included
    O, I = _upload(torch, net, g["o_init"], np.zeros(n), 1)
    net.init_inflows(O, I, 1)
    assert relerr(net.unpack_host(I, 1)[:, 0], g["i_init"]) < RTOL
    # _apply_gain (nutils.py:116-134) as the in-place update of da.py:124-126
    G, _ = _upload(torch, net, g["gain"], g["gain"], 1)
    O, I = _upload(torch, net, g["o_init"], g["i_init"], 1)
    net.apply_gain(G, O, I, 1)
    assert relerr(net.unpack_host(O, 1)[:, 0], g["o_init"] + g["gain_o"]) < RTOL
    assert relerr(net.unpack_host(I, 1)[:, 0], g["i_init"] + g["gain_i"]) < RTOL
    # _ap_par (nutils.py:157-169): the columns of P are the members
    X = net.alloc_state(n); scr = net.alloc_state(n)
    net.pack_host(g["P_sym"], n, X)
    net.route_apply(X, scr, n)
    assert relerr(net.unpack_host(X, n), g["ap"]) < RTOL
    # _aqat_par (nutils.py:194-214): A (A P)^T, returned as the transposed view
    for key in ("sym", "gen"):
        net.pack_host(g["P_" + key], n, X)
        net.route_apply(X, scr, n)
        first = net.unpack_host(X, n)
        net.pack_host(np.ascontiguousarray(first.T), n, X)
        net.route_apply(X, scr, n)
        assert relerr(net.unpack_host(X, n), g["aqat_" + key]) < RTOL
    net.check()


def test_golden_model_c1(torch_cuda, libtxh, golden_dir):
    """BASELINE.json configs[0]: 1,000 reaches x 288 steps of Muskingum.simulate, one launch."""
    torch = torch_cuda
    from tx_fast_hydrology_b200.network import Forcing
    g = np.load(os.path.join(golden_dir, "model_c1.npz"))
    n = g["endnodes"].size
    net, _ = _setup(g["endnodes"], g["K"], g["X"], float(g["dt"]))
    f = Forcing(net, g["times"], g["table"])
    o0 = g["o_init"]
    O, I = _upload(torch, net, o0, np.zeros(n), 1)
    net.init_inflows(O, I, 1)
    T = 288
    rec = torch.zeros((T, n, 1), dtype=torch.float64, device="cuda")
    net.route_run(O, I, 1, f, int(g["t0_ns"]), int(300e9), T, rec_reach=np.arange(n), rec_every=1, rec_out=rec)
    net.check()
    traj = rec.cpu().numpy()[:, :, 0]
    keep = g["keep"]
    assert relerr(traj[keep], g["O"]) < RTOL
    assert relerr(traj.sum(axis=0), g["o_sum"]) < RTOL
    assert relerr(net.unpack_host(O, 1)[:, 0], g["O"][-1]) < RTOL
    assert relerr(net.unpack_host(I, 1)[:, 0], g["I"][-1]) < RTOL


@pytest.mark.parametrize("kernel", ["lane", "window", "dataflow"])
@pytest.mark.parametrize("n,seed,M,sched", [
    (1000, 1, 1, None), (1000, 1, 3, None), (2500, 6, 64, None), (2500, 6, 70, None),
    (1500, 9, 130, None), (3000, 4, 5, (8, 4, 6, 3)), (300, 5, 2, (4, 8, 8, 1)), (7, 12, 2, None),
    (1, 13, 1, None), (4000, 21, 8, (16, 8, 12, 2, 4))])
def test_members_vs_oracle(torch_cuda, libtxh, oracle, monkeypatch, n, seed, M, sched, kernel):
    """Member-batched multi-step run == _ax_bu looped per member (SURVEY.md 8c (i)), through both device
    paths: the window-resident kernel (state in shared memory across the steps of a launch) and the
    dataflow kernel (state streamed every step)."""
    monkeypatch.setenv("TXH_ROUTE_KERNEL", kernel)
    torch = torch_cuda
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.network import Forcing
    net_d = S.make_network(n, seed, n_basins=3 if n >= 1000 else 1)
    prm = S.make_params(n, seed)
    net, (al, be, ch, ga) = _setup(net_d["endnodes"], prm["K"], prm["X"], 300.0, sched)
    T = 30
    t0 = 1_700_000_000 * 10**9
    times, table = S.make_forcing(n, T, 300.0, seed, t0_ns=t0, rows_every=4)
    mul = S.make_member_multipliers(times.size, M, seed) if M > 1 else None
    rng = np.random.default_rng(seed)
    o0 = prm["o_t"][:, None] * rng.uniform(0.5, 1.5, size=(n, M))
    i0 = np.stack([oracle.init_states(net_d["startnodes"], net_d["endnodes"], o0[:, k]) for k in range(M)], 1)
    f = Forcing(net, times, table, mul)
    O, I = _upload(torch, net, o0, i0, M)
    net.route_run(O, I, M, f, t0, int(300e9), T)
    net.check()
    o_gpu = net.unpack_host(O, M); i_gpu = net.unpack_host(I, M)
    ref = {"startnodes": net_d["startnodes"], "endnodes": net_d["endnodes"],
           "indegree": oracle.compute_indegree(net_d["startnodes"], net_d["endnodes"]),
           "alpha": al, "beta": be, "chi": ch, "gamma": ga}
    o_ref = np.ascontiguousarray(o0.T); i_ref = np.ascontiguousarray(i0.T)
    oracle.run_members(ref, o_ref, i_ref, T, times.astype(np.float64), table, float(t0), 300e9, wmul=mul)
    assert relerr(o_gpu, o_ref.T) < RTOL
    assert relerr(i_gpu, i_ref.T) < RTOL
    # member-major download agrees with reach-major
    assert (net.unpack_host(O, M, member_major=True) == o_gpu.T).all()


@pytest.mark.parametrize("n,seed,M,T", [(600, 31, 2, 150), (2000, 32, 1, 70)])
def test_long_launches_vs_oracle(torch_cuda, libtxh, oracle, n, seed, M, T):
    """Runs longer than one launch holds: with few members a launch covers up to 64 steps (interpolation records
    read in place instead of staged), and the run continues in the next launch from the state in HBM."""
    torch = torch_cuda
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.network import Forcing
    net_d = S.make_network(n, seed)
    prm = S.make_params(n, seed)
    net, (al, be, ch, ga) = _setup(net_d["endnodes"], prm["K"], prm["X"], 300.0)
    t0 = 1_700_000_000 * 10**9
    times, table = S.make_forcing(n, T, 300.0, seed, t0_ns=t0, rows_every=5)
    mul = S.make_member_multipliers(times.size, M, seed) if M > 1 else None
    rng = np.random.default_rng(seed)
    o0 = prm["o_t"][:, None] * rng.uniform(0.5, 1.5, size=(n, M))
    i0 = np.stack([oracle.init_states(net_d["startnodes"], net_d["endnodes"], o0[:, k]) for k in range(M)], 1)
    O, I = _upload(torch, net, o0, i0, M)
    net.route_run(O, I, M, Forcing(net, times, table, mul), t0, int(300e9), T)
    net.check()
    ref = {"startnodes": net_d["startnodes"], "endnodes": net_d["endnodes"],
           "indegree": oracle.compute_indegree(net_d["startnodes"], net_d["endnodes"]),
           "alpha": al, "beta": be, "chi": ch, "gamma": ga}
    o_ref = np.ascontiguousarray(o0.T); i_ref = np.ascontiguousarray(i0.T)
    oracle.run_members(ref, o_ref, i_ref, T, times.astype(np.float64), table, float(t0), 300e9, wmul=mul)
    assert relerr(net.unpack_host(O, M), o_ref.T) < RTOL
    assert relerr(net.unpack_host(I, M), i_ref.T) < RTOL


def test_texas_scale_short(torch_cuda, libtxh, oracle):
    """~100k reaches, ~1k levels (BASELINE.json configs[1] network), 24 steps, 2 members."""
    torch = torch_cuda
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.network import Forcing
    n, seed, M, T = 100_000, 2, 2, 24
    net_d = S.make_network(n, seed)
    prm = S.make_params(n, seed)
    net, (al, be, ch, ga) = _setup(net_d["endnodes"], prm["K"], prm["X"], 300.0)
    lev, nl = net.levels()
    assert 900 <= nl <= 1100
    t0 = 1_700_000_000 * 10**9
    times, table = S.make_forcing(n, T, 300.0, seed, t0_ns=t0)
    mul = S.make_member_multipliers(times.size, M, seed)
    o0 = np.stack([prm["o_t"], prm["o_t"][::-1]], 1)
    i0 = np.stack([oracle.init_states(net_d["startnodes"], net_d["endnodes"], o0[:, k]) for k in range(M)], 1)
    f = Forcing(net, times, table, mul)
    O, I = _upload(torch, net, o0, i0, M)
    net.route_run(O, I, M, f, t0, int(300e9), T)
    net.check()
    ref = {"startnodes": net_d["startnodes"], "endnodes": net_d["endnodes"],
           "indegree": oracle.compute_indegree(net_d["startnodes"], net_d["endnodes"]),
           "alpha": al, "beta": be, "chi": ch, "gamma": ga}
    o_ref = np.ascontiguousarray(o0.T); i_ref = np.ascontiguousarray(i0.T)
    oracle.run_members(ref, o_ref, i_ref, T, times.astype(np.float64), table, float(t0), 300e9, wmul=mul)
    assert relerr(net.unpack_host(O, M), o_ref.T) < RTOL
    assert relerr(net.unpack_host(I, M), i_ref.T) < RTOL
    # linearity (size-independent property): route(a x + b y) == a route(x) + b route(y), no forcing
    X = net.alloc_state(3); scr = net.alloc_state(3)
    x = np.stack([o0[:, 0], o0[:, 1], 2.0 * o0[:, 0] - 0.5 * o0[:, 1]], 1)
    net.pack_host(x, 3, X)
    net.route_apply(X, scr, 3)
    y = net.unpack_host(X, 3)
    # (max-norm: the combination cancels, its small elements carry the rounding of the large ones)
    assert normerr(y[:, 2], 2.0 * y[:, 0] - 0.5 * y[:, 1]) < 1e-12


def test_dataflow_equals_levels(torch_cuda, libtxh):
    """Two independent device paths (persistent dataflow vs one launch per level) agree."""
    torch = torch_cuda
    from tx_fast_hydrology_b200 import synthetic as S
    n, seed, M = 20_000, 17, 8
    net_d = S.make_network(n, seed, n_basins=5)
    prm = S.make_params(n, seed)
    net, _ = _setup(net_d["endnodes"], prm["K"], prm["X"], 300.0)
    rng = np.random.default_rng(1)
    o0 = rng.uniform(0.1, 10.0, size=(n, M)); i0 = rng.uniform(0.1, 10.0, size=(n, M))
    q = torch.from_numpy(rng.gamma(0.5, 2.0, size=n)).cuda()
    Oa, Ia = _upload(torch, net, o0, i0, M)
    Ob, Ib = _upload(torch, net, o0, i0, M)
    for _ in range(3):
        net.route_step(Oa, Ia, M, q)
        net.route_step(Ob, Ib, M, q, levels=True)
    net.check()
    # (random, inconsistent o / i: elements cancel, so the tight bound is in the max-norm)
    assert normerr(net.unpack_host(Oa, M), net.unpack_host(Ob, M)) < 1e-13
    assert normerr(net.unpack_host(Ia, M), net.unpack_host(Ib, M)) < 1e-13
    assert relerr(net.unpack_host(Oa, M), net.unpack_host(Ob, M)) < RTOL


def test_no_coeffs_is_an_error(torch_cuda, libtxh):
    from tx_fast_hydrology_b200.network import RiverNetwork
    from tx_fast_hydrology_b200._lib import TxhError
    net = RiverNetwork(np.array([1, 2, 2], dtype=np.int64))
    O = net.alloc_state(1); I = net.alloc_state(1)
    with pytest.raises(TxhError):
        net.route_step(O, I, 1, None)


def test_forcing_update_in_place(torch_cuda, libtxh):
    """txh_forcing_update refreshes a resident table: the run equals one with a freshly created forcing."""
    torch = torch_cuda
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.network import Forcing
    n, seed, M, T = 3000, 17, 6, 20
    net_d = S.make_network(n, seed)
    prm = S.make_params(n, seed)
    net, _ = _setup(net_d["endnodes"], prm["K"], prm["X"], 300.0)
    t0 = 1_700_000_000 * 10**9
    times, table = S.make_forcing(n, T, 300.0, seed, t0_ns=t0, rows_every=4)
    mul = S.make_member_multipliers(times.size, M, seed)
    rng = np.random.default_rng(seed)
    o0 = prm["o_t"][:, None] * rng.uniform(0.5, 1.5, size=(n, M))
    i0 = np.zeros_like(o0)
    f = Forcing(net, times, 0.5 * table, 2.0 * mul)
    f.update(times, table, mul)
    O, I = _upload(torch, net, o0, i0, M)
    net.route_run(O, I, M, f, t0, int(300e9), T)
    g = Forcing(net, times, table, mul)
    O2, I2 = _upload(torch, net, o0, i0, M)
    net.route_run(O2, I2, M, g, t0, int(300e9), T)
    net.check()
    assert torch.equal(O, O2) and torch.equal(I, I2)
    with pytest.raises(ValueError):
        f.update(times[:-1], table[:-1], mul[:-1])


def test_forcing_update_overlapped(torch_cuda, libtxh):
    """txh_forcing_update_async: the table arrives in row chunks on the handle's copy stream while routing calls
    that read only its first hours already run; window by window the result equals the synchronous upload.
    (A 40 MB table: several chunks.)  The rows sit at irregular times off the step grid, so the rows a call waits
    for come from the search of its last step, and the first pass interpolates the nearest row."""
    torch = torch_cuda
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.network import Forcing
    n, seed, M, every, nwin = 60000, 19, 2, 12, 80
    net_d = S.make_network(n, seed)
    prm = S.make_params(n, seed)
    net, _ = _setup(net_d["endnodes"], prm["K"], prm["X"], 300.0)
    t0 = 1_700_000_000 * 10**9
    times, table = S.make_forcing(n, every * nwin, 300.0, seed, t0_ns=t0)
    # gaps of 1 s to 2 h (mean one hour) from 7 min before t0: some calls need no new row, some several
    gaps = np.random.default_rng(seed).uniform(1.0 / 3600, 2.0, size=times.size - 1) * 3600 * 10**9
    times = t0 - 420 * 10**9 + np.concatenate([[0], np.cumsum(gaps.astype(np.int64))])
    mul = S.make_member_multipliers(times.size, M, seed)
    tp = torch.from_numpy(np.ascontiguousarray(table)).pin_memory()
    mp = torch.from_numpy(np.ascontiguousarray(mul)).pin_memory()
    rng = np.random.default_rng(seed)
    o0 = prm["o_t"][:, None] * rng.uniform(0.5, 1.5, size=(n, M))
    f = Forcing(net, times, torch.zeros_like(tp), torch.ones_like(mp))
    g = Forcing(net, times, tp, mp)
    for rep, method in enumerate((0, 1)):                  # the second pass re-uses the table while it may be in use
        O, I = _upload(torch, net, o0, np.zeros_like(o0), M)
        O2, I2 = _upload(torch, net, o0, np.zeros_like(o0), M)
        f.update(times, tp, mp, overlap=True)
        for k in range(nwin):
            net.route_run(O, I, M, f, t0 + k * every * int(300e9), int(300e9), every, method=method)
        for k in range(nwin):
            net.route_run(O2, I2, M, g, t0 + k * every * int(300e9), int(300e9), every, method=method)
        net.check()
        assert torch.equal(O, O2) and torch.equal(I, I2)
    f.wait()

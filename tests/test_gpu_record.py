"""Ensemble hydrographs: recording in the window-resident routing kernel (route_window_kernel, REC variant) and in the
assimilation loop (Muskingum.run_assimilating(record_reaches=...), txh_run_assimilating_rec), against the CPU oracle.

Tolerance: FP64, element-wise relative error <= 1e-9 (tests/parity.py); after an ensemble update relative to
max(|posterior|, |forecast|) and the eps * cond(S) bound of the update (parity.enkf_tolerance)."""
import os

import numpy as np
import pandas as pd
import pytest

pytestmark = pytest.mark.gpu

RTOL = 1e-9

from parity import relerr, normerr, enkf_tolerance        # noqa: E402


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (no CPU fallback exists)"
    return torch


def _upload(net, o, i, M):
    O = net.alloc_state(M); I = net.alloc_state(M)
    net.pack_host(np.asarray(o, dtype=np.float64).reshape(net.n, M), M, O)
    net.pack_host(np.asarray(i, dtype=np.float64).reshape(net.n, M), M, I)
    return O, I


def _record_set(net, endnodes, rng, extra=40):
    """Reaches that cover every way the window kernel forms an outflow: pocket roots and interiors, segment first /
    interior / last rows, headwaters, confluences and outlets."""
    n = endnodes.size
    ws = net.window_schedule()
    pos_of_reach = net.schedule()["pos_of_reach"]
    reach_of_pos = np.empty(n, dtype=np.int64); reach_of_pos[pos_of_reach] = np.arange(n)
    pick = set()
    segs = [t for t in ws["tasks"] if t[2] == 1 and t[1] >= 3][:6]
    pockets = [t for t in ws["tasks"] if t[2] == 0 and t[1] >= 3][:6]
    assert segs and pockets, "the network has no long segments / pockets to record from"
    for t in segs:
        b, ln = int(t[0]), int(t[1])
        pick.update(int(reach_of_pos[p]) for p in (b, b + ln // 2, b + ln - 1))
    for t in pockets:
        b, ln = int(t[0]), int(t[1])
        pick.update(int(reach_of_pos[p]) for p in (b, b + ln // 2, b + ln - 1))
    start = np.arange(n)
    indeg = np.bincount(endnodes[endnodes != start], minlength=n)
    pick.update(int(x) for x in np.flatnonzero(indeg == 0)[:5])
    pick.update(int(x) for x in np.flatnonzero(indeg >= 2)[:5])
    pick.update(int(x) for x in np.flatnonzero(endnodes == start)[:3])
    pick.update(int(x) for x in rng.choice(n, size=extra, replace=False))
    return rng.permutation(np.array(sorted(pick), dtype=np.int64))


def _route_case(torch, oracle, monkeypatch, kernel, n, seed, M, T, every):
    monkeypatch.setenv("TXH_ROUTE_KERNEL", kernel)
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.network import Forcing, RiverNetwork
    net_d = S.make_network(n, seed, n_basins=2)
    prm = S.make_params(n, seed)
    net = RiverNetwork(net_d["endnodes"])
    al, be, ch, ga = net.compute_coeffs(prm["K"], prm["X"], 300.0)
    t0 = 1_700_000_000 * 10**9
    times, table = S.make_forcing(n, T, 300.0, seed, t0_ns=t0, rows_every=4)
    mul = S.make_member_multipliers(times.size, M, seed)
    rng = np.random.default_rng(seed)
    o0 = prm["o_t"][:, None] * rng.uniform(0.5, 1.5, size=(n, M))
    i0 = np.stack([oracle.init_states(net_d["startnodes"], net_d["endnodes"], o0[:, k]) for k in range(M)], 1)
    f = Forcing(net, times, table, mul)
    reaches = _record_set(net, net_d["endnodes"], rng)
    O, I = _upload(net, o0, i0, M)
    rec = torch.full((T // every, reaches.size, M), np.nan, dtype=torch.float64, device="cuda")
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        net.route_run(O, I, M, f, t0, int(300e9), T, rec_reach=reaches, rec_every=every, rec_out=rec)
        torch.cuda.synchronize()
    net.check()
    # the kernel asked for ran (run_routing falls back to the dataflow kernel where the window kernel declines)
    names = " ".join(e.name for e in prof.events())
    assert ("route_" + kernel + "_kernel") in names, f"route_{kernel}_kernel did not run"
    ref = {"startnodes": net_d["startnodes"], "endnodes": net_d["endnodes"],
           "indegree": oracle.compute_indegree(net_d["startnodes"], net_d["endnodes"]),
           "alpha": al, "beta": be, "chi": ch, "gamma": ga}
    o = np.ascontiguousarray(o0.T); i = np.ascontiguousarray(i0.T)
    want = np.empty((T // every, reaches.size, M))
    for s in range(1, T + 1):
        oracle.run_members(ref, o, i, 1, times.astype(np.float64), table, float(t0 + (s - 1) * 300e9), 300e9, wmul=mul)
        if s % every == 0:
            want[s // every - 1] = o[:, reaches].T
    return rec.cpu().numpy(), want, net.unpack_host(O, M), net.unpack_host(I, M), o.T, i.T


@pytest.mark.parametrize("n,seed,M,T,every", [(3000, 41, 64, 40, 1), (2500, 42, 33, 45, 5), (4000, 43, 8, 70, 7),
                                              (2000, 44, 70, 40, 7), (5000, 45, 64, 100, 7)])
def test_window_recording_vs_oracle(torch_cuda, oracle, monkeypatch, n, seed, M, T, every):
    """route_window_kernel<REC>: the outflow of every recorded reach after every `every`-th step, pocket and segment
    rows alike, equals the oracle's; 7 does not divide the 16- / 64-step launches, 70 members take two member
    blocks, odd M leaves a padding column that must not be written."""
    got, want, o, i, o_ref, i_ref = _route_case(torch_cuda, oracle, monkeypatch, "window", n, seed, M, T, every)
    assert not np.isnan(got).any()
    assert relerr(got, want) < RTOL
    assert relerr(o, o_ref) < RTOL and relerr(i, i_ref) < RTOL


@pytest.mark.parametrize("n,seed,M,T,every", [(2500, 46, 64, 30, 1), (2000, 47, 70, 28, 7)])
def test_window_recording_equals_dataflow(torch_cuda, oracle, monkeypatch, n, seed, M, T, every):
    """The same recording through the window kernel and the dataflow kernel (the former recording path)."""
    a = _route_case(torch_cuda, oracle, monkeypatch, "window", n, seed, M, T, every)
    b = _route_case(torch_cuda, oracle, monkeypatch, "dataflow", n, seed, M, T, every)
    assert relerr(a[0], b[0]) < RTOL
    assert relerr(b[0], b[1]) < RTOL


@pytest.mark.parametrize("M", [64, 70, 3])
def test_recording_leaves_route_state_alone(torch_cuda, monkeypatch, M):
    """route_run with and without recording end in the bit-identical state."""
    torch = torch_cuda
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.network import Forcing, RiverNetwork
    n, seed, T = 3000, 48, 37
    net_d = S.make_network(n, seed)
    prm = S.make_params(n, seed)
    net = RiverNetwork(net_d["endnodes"])
    net.compute_coeffs(prm["K"], prm["X"], 300.0)
    t0 = 1_700_000_000 * 10**9
    times, table = S.make_forcing(n, T, 300.0, seed, t0_ns=t0, rows_every=4)
    f = Forcing(net, times, table, S.make_member_multipliers(times.size, M, seed))
    rng = np.random.default_rng(seed)
    o0 = prm["o_t"][:, None] * rng.uniform(0.5, 1.5, size=(n, M))
    out = []
    for record in (False, True):
        O, I = _upload(net, o0, o0, M)
        net.init_inflows(O, I, M)
        if record:
            r = rng.choice(n, size=500, replace=False)
            rec = torch.zeros((T // 3, r.size, M), dtype=torch.float64, device="cuda")
            net.route_run(O, I, M, f, t0, int(300e9), T, rec_reach=r, rec_every=3, rec_out=rec)
        else:
            net.route_run(O, I, M, f, t0, int(300e9), T)
        out.append((net.unpack_host(O, M), net.unpack_host(I, M)))
    assert (out[0][0] == out[1][0]).all() and (out[0][1] == out[1][1]).all()


def _assim_case(oracle, n, M, m, seed, in_library, every, nwin, rest=0, dense_R=False, record_every=1, reaches=None):
    """_run_assimilating_case of test_gpu_model.py with recording: returns the device's (rec, prior, final state) and
    the oracle's hydrographs at every step (posterior at update steps), its priors and tolerances."""
    import torch
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.muskingum import Muskingum
    from tx_fast_hydrology_b200.da import EnsembleKalmanFilter
    nsteps = every * nwin + rest
    net_d = S.make_network(n, seed)
    prm = S.make_params(n, seed, well_posed=True)
    rng = np.random.default_rng(seed)
    o0 = prm["o_t"][:, None] * rng.uniform(0.5, 1.5, size=(n, M))
    d = S.model_dict(net_d, prm, dt_s=300.0)
    d["o_t"] = o0
    mdl = Muskingum(d, members=M)
    t0 = int(mdl.datetime.value)
    times, table = S.make_forcing(n, nsteps, 300.0, seed, t0_ns=t0, rows_every=4)
    mul = S.make_member_multipliers(times.size, M, seed)
    gidx = np.asarray(S.make_gauges(net_d["endnodes"], m, seed=seed), dtype=np.int64)
    m = gidx.size
    mt = t0 + (np.arange(nwin, dtype=np.int64) + 1) * int(every * 300e9)
    meas = rng.uniform(0.5, 8.0, size=(nwin, m))
    mdf = pd.DataFrame(meas, index=pd.DatetimeIndex(pd.to_datetime(mt, unit="ns", utc=True)).as_unit("ns"),
                       columns=[d["reach_ids"][j] for j in gidx])
    R = 1e-2 * np.eye(m)
    if dense_R:
        Bm = rng.standard_normal((m, m))
        R = 1e-2 * (np.eye(m) + 0.5 * (Bm @ Bm.T) / m)
    q = rng.uniform(0.5, 2.0, size=n)
    enkf = EnsembleKalmanFilter(mdl, mdf, q, R)
    Zp = meas[:, :, None] + 0.1 * rng.standard_normal((nwin, m, M))
    f = mdl.make_forcing(times_ns=times, table=table, member_mul=mul)
    if reaches is None:                      # gauged and ungauged reaches, in no particular order
        ung = np.setdiff1d(np.arange(n), gidx)
        reaches = rng.permutation(np.concatenate([gidx[:max(3, m // 2)], rng.choice(ung, size=60, replace=False)]))
    Zd = torch.as_tensor(np.ascontiguousarray(Zp), device="cuda")
    rec, prior = mdl.run_assimilating(f, nsteps, enkf, every, Zd if in_library else list(Zd), record_reaches=reaches,
                                      record_every=record_every, record_prior=True)
    mdl.network.check()
    ind = oracle.compute_indegree(net_d["startnodes"], net_d["endnodes"])
    al, be, ch, ga = oracle.compute_coeffs(prm["K"], prm["X"], 300.0)
    onet = {"startnodes": net_d["startnodes"], "endnodes": net_d["endnodes"], "indegree": ind,
            "alpha": al, "beta": be, "chi": ch, "gamma": ga}
    o = np.ascontiguousarray(o0.T)
    i = np.stack([oracle.init_states(net_d["startnodes"], net_d["endnodes"], x) for x in o])
    hyd = np.empty((nsteps, reaches.size, M))
    pri = np.empty((nwin, reaches.size, M))
    tol = RTOL
    for s in range(1, nsteps + 1):
        oracle.run_members(onet, o, i, 1, times.astype(np.float64), table, float(t0 + (s - 1) * 300e9), 300e9, wmul=mul)
        hyd[s - 1] = o[:, reaches].T
        if s % every == 0 and s // every <= nwin:
            k = s // every - 1
            pri[k] = o[:, reaches].T
            tol = max(tol, enkf_tolerance(o.T, gidx, q, R))
            Op, Ip, _ = oracle.enkf_update(onet, o.T, i.T, gidx, Zp[k], q, R)
            o = np.ascontiguousarray(Op.T); i = np.ascontiguousarray(Ip.T)
            hyd[s - 1] = o[:, reaches].T
    sel = np.arange(record_every, nsteps + 1, record_every) - 1
    return rec.cpu().numpy(), prior.cpu().numpy(), mdl.o_t_next[reaches], hyd[sel], pri, tol, sel


@pytest.mark.parametrize("n,M,m,seed,every,nwin,rest,record_every,dense_R", [
    (2000, 64, 50, 51, 6, 3, 0, 1, False),
    (1200, 20, 30, 52, 6, 3, 4, 4, False),       # 4 does not divide 6; remainder steps
    (900, 70, 40, 53, 5, 3, 2, 1, False),        # two member blocks: the transform kernel applies the update
    (1400, 48, 90, 54, 5, 3, 0, 5, True),        # dense R: the general launches of the ensemble-space system
    (1500, 64, 25, 55, 5, 2, 3, 3, False)])
@pytest.mark.parametrize("in_library", [True, False])
def test_run_assimilating_recording_vs_oracle(oracle, n, M, m, seed, every, nwin, rest, record_every, dense_R,
                                              in_library):
    """rec = the forecast at non-update steps and the posterior at update steps; prior = the forecast every update
    started from; the last slot is the final state when record_every divides nsteps."""
    rec, prior, final, want, pri, tol, sel = _assim_case(oracle, n, M, m, seed, in_library, every, nwin, rest, dense_R,
                                                         record_every)
    assert rec.shape == want.shape and prior.shape == pri.shape
    assert relerr(prior, pri) < tol
    assert relerr(rec, want, scale=_update_scale(want, pri, sel, every)) < tol
    if (every * nwin + rest) % record_every == 0:
        assert relerr(rec[-1], final, scale=np.abs(pri[-1])) < tol


def _update_scale(want, pri, sel, every):
    """max(|posterior|, |its forecast|) at update steps (tests/parity.py), |value| elsewhere."""
    sc = np.abs(want).copy()
    for j, s in enumerate(sel + 1):
        if s % every == 0 and s // every <= pri.shape[0]:
            sc[j] = np.maximum(sc[j], np.abs(pri[s // every - 1]))
    return sc


def test_run_assimilating_recording_leaves_state_alone():
    """run_assimilating with and without recording end in the bit-identical state (in-library loop, M = 64)."""
    import torch
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.muskingum import Muskingum
    from tx_fast_hydrology_b200.da import EnsembleKalmanFilter
    n, M, m, seed, every, nwin = 2500, 64, 40, 56, 6, 3
    out = []
    for record in (False, True):
        net = S.make_network(n, seed); prm = S.make_params(n, seed, well_posed=True)
        rng = np.random.default_rng(seed)
        d = S.model_dict(net, prm, dt_s=300.0); d["o_t"] = prm["o_t"][:, None] * rng.uniform(0.5, 1.5, size=(n, M))
        mdl = Muskingum(d, members=M); t0 = int(mdl.datetime.value)
        times, table = S.make_forcing(n, every * nwin, 300.0, seed, t0_ns=t0, rows_every=4)
        g = S.make_gauges(net["endnodes"], m, seed=seed)
        mt = t0 + (np.arange(nwin, dtype=np.int64) + 1) * int(every * 300e9)
        meas = rng.uniform(0.5, 8.0, size=(nwin, m))
        mdf = pd.DataFrame(meas, index=pd.DatetimeIndex(pd.to_datetime(mt, unit="ns", utc=True)).as_unit("ns"),
                           columns=[d["reach_ids"][j] for j in g])
        enkf = EnsembleKalmanFilter(mdl, mdf, rng.uniform(0.5, 2.0, size=n), 1e-2 * np.eye(m))
        Zp = torch.as_tensor(meas[:, :, None] + 0.1 * rng.standard_normal((nwin, m, M)), device="cuda")
        f = mdl.make_forcing(times_ns=times, table=table, member_mul=S.make_member_multipliers(times.size, M, seed))
        r = mdl.run_assimilating(f, every * nwin, enkf, every, Zp,
                                 record_reaches=np.arange(0, n, 7) if record else None, record_prior=record)
        assert (r is None) == (not record)
        mdl.network.check()
        out.append((mdl.o_t_next, mdl.i_t_next))
    assert (out[0][0] == out[1][0]).all() and (out[0][1] == out[1][1]).all()


def test_run_assimilating_recording_refuses_multipliers_for_another_M():
    """A forcing whose member multipliers were made for another member count is refused with TXH_E_INVALID before
    any device work when the in-library loop records, as it is without recording: state and clock stay as they were."""
    import torch
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200._lib import TxhError
    from tx_fast_hydrology_b200.muskingum import Muskingum
    from tx_fast_hydrology_b200.da import EnsembleKalmanFilter
    n, M, m, seed, every, nwin = 1500, 16, 20, 57, 6, 2
    net = S.make_network(n, seed); prm = S.make_params(n, seed, well_posed=True)
    rng = np.random.default_rng(seed)
    d = S.model_dict(net, prm, dt_s=300.0); d["o_t"] = prm["o_t"][:, None] * rng.uniform(0.5, 1.5, size=(n, M))
    mdl = Muskingum(d, members=M); t0 = mdl.datetime
    times, table = S.make_forcing(n, every * nwin, 300.0, seed, t0_ns=int(t0.value), rows_every=4)
    g = S.make_gauges(net["endnodes"], m, seed=seed)
    mt = int(t0.value) + (np.arange(nwin, dtype=np.int64) + 1) * int(every * 300e9)
    meas = rng.uniform(0.5, 8.0, size=(nwin, m))
    mdf = pd.DataFrame(meas, index=pd.DatetimeIndex(pd.to_datetime(mt, unit="ns", utc=True)).as_unit("ns"),
                       columns=[d["reach_ids"][j] for j in g])
    enkf = EnsembleKalmanFilter(mdl, mdf, rng.uniform(0.5, 2.0, size=n), 1e-2 * np.eye(m))
    Zp = torch.as_tensor(meas[:, :, None] + 0.1 * rng.standard_normal((nwin, m, M)), device="cuda")
    # multipliers of M + 3 members: a run that went ahead would read them inside the table, with the wrong stride
    f = mdl.make_forcing(times_ns=times, table=table, member_mul=S.make_member_multipliers(times.size, M + 3, seed))
    O, I = mdl.device_state
    O0, I0 = O.clone(), I.clone()
    for record in (None, np.arange(0, n, 7)):
        with pytest.raises(TxhError, match="do not match M") as err:
            mdl.run_assimilating(f, every * nwin, enkf, every, Zp, record_reaches=record, record_prior=record is not None)
        assert err.value.code == -1                             # TXH_E_INVALID
        torch.cuda.synchronize()
        assert torch.equal(O, O0) and torch.equal(I, I0)
        assert mdl.datetime == t0 and enkf.n_updates == 0


def test_run_assimilating_recording_variants_agree():
    """With the fused stages switched off (TXH_ENKF_FUSED=0 TXH_ENKF_FUSE_LOAD=0 TXH_PDL=0, read once per process: a
    child process), the recorded hydrographs and priors agree with the default path to 1e-10."""
    import subprocess
    import sys
    import tempfile
    code = (
        "import sys, numpy as np, torch\n"
        "sys.path.insert(0, %r)\n"
        "from tx_fast_hydrology_b200 import synthetic as S\n"
        "from tx_fast_hydrology_b200.muskingum import Muskingum\n"
        "from tx_fast_hydrology_b200.da import EnsembleKalmanFilter\n"
        "import pandas as pd\n"
        "n, M, m, seed, every, nwin = 2500, 64, 40, 57, 6, 4\n"
        "net = S.make_network(n, seed); prm = S.make_params(n, seed, well_posed=True)\n"
        "rng = np.random.default_rng(seed)\n"
        "d = S.model_dict(net, prm, dt_s=300.0); d['o_t'] = prm['o_t'][:, None] * rng.uniform(0.5, 1.5, size=(n, M))\n"
        "mdl = Muskingum(d, members=M); t0 = int(mdl.datetime.value)\n"
        "times, table = S.make_forcing(n, every * nwin + 3, 300.0, seed, t0_ns=t0, rows_every=4)\n"
        "mul = S.make_member_multipliers(times.size, M, seed)\n"
        "g = S.make_gauges(net['endnodes'], m, seed=seed)\n"
        "mt = t0 + (np.arange(nwin, dtype=np.int64) + 1) * int(every * 300e9)\n"
        "meas = rng.uniform(0.5, 8.0, size=(nwin, m))\n"
        "idx = pd.DatetimeIndex(pd.to_datetime(mt, unit='ns', utc=True)).as_unit('ns')\n"
        "mdf = pd.DataFrame(meas, index=idx, columns=[d['reach_ids'][j] for j in g])\n"
        "enkf = EnsembleKalmanFilter(mdl, mdf, rng.uniform(0.5, 2.0, size=n), 1e-2 * np.eye(m))\n"
        "Zp = torch.as_tensor(meas[:, :, None] + 0.1 * rng.standard_normal((nwin, m, M)), device='cuda')\n"
        "f = mdl.make_forcing(times_ns=times, table=table, member_mul=mul)\n"
        "r = np.concatenate([g[:10], np.arange(1, n, 37)])\n"
        "rec, pri = mdl.run_assimilating(f, every * nwin + 3, enkf, every, Zp, record_reaches=np.unique(r),\n"
        "                                record_every=2, record_prior=True)\n"
        "mdl.network.check()\n"
        "np.savez(sys.argv[1], rec=rec.cpu().numpy(), pri=pri.cpu().numpy())\n"
    ) % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        for name, env in (("fused", {}), ("plain", {"TXH_ENKF_FUSED": "0", "TXH_ENKF_FUSE_LOAD": "0", "TXH_PDL": "0"})):
            path = os.path.join(tmp, name + ".npz")
            e = dict(os.environ); e.update(env)
            subprocess.run([sys.executable, "-c", code, path], check=True, env=e, timeout=600)
            z = np.load(path)
            out[name] = (z["rec"], z["pri"])
    assert normerr(out["fused"][0], out["plain"][0]) < 1e-10
    assert normerr(out["fused"][1], out["plain"][1]) < 1e-10


@pytest.mark.parametrize("in_library", [True, False])
def test_run_assimilating_recording_equals_simulate(in_library):
    """Against the consumer path the hydrographs stand for: the same case through `simulate()` with an
    EnsembleKalmanFilter(every=...) bound (the filter fires in the step-end hook, before the state is yielded), keeping
    `state.o_t_next[reaches]` after every step.  The filter also fires at the start of the simulation (t0 is on the
    cadence), so the recorded run gets that same update by hand first.  Agreement within 1e-10, relative to
    max(|value|, |forecast|) at update steps."""
    import torch
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.muskingum import Muskingum
    from tx_fast_hydrology_b200.da import EnsembleKalmanFilter
    n, M, m, seed, every, nwin, rest = 1200, 64, 30, 58, 6, 3, 2
    nsteps = every * nwin + rest
    net_d = S.make_network(n, seed)
    prm = S.make_params(n, seed, well_posed=True)
    rng = np.random.default_rng(seed)
    d = S.model_dict(net_d, prm, dt_s=300.0)
    d["o_t"] = prm["o_t"][:, None] * rng.uniform(0.5, 1.5, size=(n, M))
    t0 = int(pd.Timestamp(d["datetime"]).value)
    assert t0 % int(every * 300e9) == 0
    times, table = S.make_forcing(n, nsteps, 300.0, seed, t0_ns=t0, rows_every=4)
    fdf = pd.DataFrame(table, index=pd.DatetimeIndex(pd.to_datetime(times, unit="ns", utc=True)).as_unit("ns"),
                       columns=d["reach_ids"])
    gidx = np.asarray(S.make_gauges(net_d["endnodes"], m, seed=seed), dtype=np.int64)
    m = gidx.size
    mt = t0 + (np.arange(nwin + 1, dtype=np.int64)) * int(every * 300e9)
    meas = pd.DataFrame(rng.uniform(0.5, 8.0, size=(nwin + 1, m)),
                        index=pd.DatetimeIndex(pd.to_datetime(mt, unit="ns", utc=True)).as_unit("ns"),
                        columns=[d["reach_ids"][j] for j in gidx])
    noise = 0.1 * rng.standard_normal((nwin + 1, m, M))
    q = rng.uniform(0.5, 2.0, size=n)
    R = 1e-2 * np.eye(m)
    cadence = pd.Timedelta(seconds=every * 300)
    ung = np.setdiff1d(np.arange(n), gidx)
    reaches = rng.permutation(np.concatenate([gidx[:10], rng.choice(ung, size=30, replace=False)]))

    # the consumer loop
    sim = Muskingum(dict(d), members=M)
    sim.bind_callback(EnsembleKalmanFilter(sim, meas, q, R, obs_noise=noise, every=cadence), key="enkf")
    got = [state.o_t_next[reaches] for state in sim.simulate(fdf, end_time=pd.Timestamp(t0 + int(nsteps * 300e9),
                                                                                         tz="UTC"))]
    assert len(got) == nsteps
    want = np.stack(got)

    # the recorded run
    mdl = Muskingum(dict(d), members=M)
    enkf = EnsembleKalmanFilter(mdl, meas, q, R, obs_noise=noise, every=cadence)
    enkf.filter()                                                  # the simulation-start update
    Zp = torch.as_tensor(np.stack([enkf.perturbed_observations(pd.Timestamp(int(t), tz="UTC")) for t in mt[1:]]),
                         device="cuda").contiguous()
    f = mdl.make_forcing(fdf)
    rec, prior = mdl.run_assimilating(f, nsteps, enkf, every, Zp if in_library else list(Zp), record_reaches=reaches,
                                      record_prior=True)
    mdl.network.check()
    rec = rec.cpu().numpy(); prior = prior.cpu().numpy()
    assert rec.shape == want.shape
    assert relerr(rec, want, scale=_update_scale(want, prior, np.arange(nsteps), every)) < 1e-10

"""Every dispatch path of the ensemble Kalman update against the extended-precision reference
(tests/enkf_reference.py) and the CPU oracle, at odd and boundary member and gauge counts.

The paths (txh_capi.cu: enkf_solve_impl, txh_enkf_apply, txh_run_assimilating_rec; txh_da.cu: launch_enkf_update,
launch_chol_solve_small):
  solve  cluster        M < m, M <= 64, diagonal D: enkf_small_system_kernel (one cluster launch)
         woodbury       M < m, M <= 128, dense D^-1 or M > 64: innovation_cat, dgemm, chol_solve_blocked_kernel<64/96/128>
         woodbury_big   M < m, M > 128: ... woodbury_assemble, blocked spd_solve (chol_panel_kernel)
         direct         M >= m or no D^-1: innov_cov_finish, spd_solve
  apply  ld <= 64 unsharded: enkf_update64_kernel + inflow_gain; ld > 64: enkf_update_kernel + apply_gain;
         sharded (Xall or peer blocks): enkf_update_kernel
  loop   window kernel, ld <= 64: the update applied by the next window launch (route_window_kernel<.., UPD, REC>);
         lane / dataflow kernel: enkf_record_kernel + enkf_update64_kernel + inflow_rebuild_kernel

Every case names the kernels of its path and checks with torch.profiler that they ran, so that a change of the
dispatch cannot move a case off the path it pins.  No state that is routed ever holds a NaN or an Inf: the pad
sentinels are finite (1e6) and only the solve and apply cases, which route nothing, use them."""
import numpy as np
import pandas as pd
import pytest

import enkf_reference as E
from parity import relerr, normerr, enkf_tolerance

pytestmark = pytest.mark.gpu

SENTINEL = 1e6
RTOL = 1e-9


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (no CPU fallback exists)"
    return torch


@pytest.fixture(scope="module")
def fnet(torch_cuda):
    """The network of the shared forecast (tests/enkf_reference.py) and its reach -> schedule position map."""
    from tx_fast_hydrology_b200.network import RiverNetwork
    fc = E.forecast()
    net = RiverNetwork(fc["endnodes"])
    n = net.n
    net.set_coeffs(np.zeros(n), np.zeros(n), np.zeros(n), np.zeros(n))
    return net, net.schedule()["pos_of_reach"], fc


def _kernels(torch, fn):
    """Run `fn` under the profiler; the names of the CUDA kernels it launched, in one string."""
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return " ".join(e.name for e in prof.events())


def _expect(names, want, absent=()):
    for k in want:
        assert k in names, f"{k} did not run (kernels: {sorted(set(names.split()))[:40]})"
    for k in absent:
        assert k not in names, f"{k} ran, but this case is meant to take another path"


def _dev(torch, a):
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device="cuda")


def _sched(vec, pos):
    out = np.empty_like(vec)
    out[pos] = vec
    return out


def _f64(a):
    return np.asarray(a, dtype=np.float64)


# ---- (a) the solve --------------------------------------------------------------------------------------------
def _solve_kernels(M, m, dinv_kind, path):
    if path == "cluster":
        return ["enkf_small_system_kernel"], ["innovation_cat_kernel", "spd_solve_kernel", "chol_panel_kernel"]
    if path == "woodbury":
        mt = 64 if M <= 64 else (96 if M <= 96 else 128)
        return ["innovation_cat_kernel", "dgemm_kernel", f"chol_solve_blocked_kernel<{mt}>"], \
               ["enkf_small_system_kernel", "woodbury_assemble_kernel"]
    if path == "woodbury_big":
        return ["innovation_cat_kernel", "woodbury_assemble_kernel", "chol_panel_kernel"], \
               ["enkf_small_system_kernel", "chol_solve_blocked_kernel"]
    return ["innov_cov_finish_kernel", "spd_solve_kernel" if m <= 48 else "chol_panel_kernel"], \
           ["enkf_small_system_kernel", "innovation_cat_kernel"]


def _solve_dev(torch, net, pos, inp, M, dinv_kind, R=None):
    m = inp["HX"].shape[0]
    R = inp["R"] if R is None else R
    D = np.diag(inp["qs"]) + R
    Dinv = None if dinv_kind == 0 else _dev(torch, 1.0 / np.diagonal(D) if dinv_kind == 1 else np.linalg.inv(D))
    args = dict(HX=_dev(torch, inp["HX"]), Zp=_dev(torch, inp["Zp"]), mean=_dev(torch, _sched(inp["mean_all"], pos)),
                qs=_dev(torch, inp["qs"]), R=_dev(torch, R), Dinv=Dinv,
                work=torch.empty(net.enkf_work_size(m, M), dtype=torch.float64, device="cuda"),
                W=torch.full((m, M), np.nan, dtype=torch.float64, device="cuda"),
                T=torch.full((M, M), np.nan, dtype=torch.float64, device="cuda"))

    def run():
        net.enkf_solve(m, M, args["HX"], args["Zp"], args["mean"], inp["gauges"], args["qs"], args["R"], args["work"],
                       args["W"], args["T"], args["Dinv"], dinv_kind)
    return run, args


@pytest.mark.parametrize("M,m,dense_R,dinv_kind,path", E.SOLVE_CASES)
def test_solve_paths_vs_reference(torch_cuda, fnet, record_property, M, m, dense_R, dinv_kind, path):
    """T and W of RiverNetwork.enkf_solve against the longdouble reference, max-norm relative error within
    max(1e-12, 64 eps cond) (tests/enkf_reference.py:solve_tolerance)."""
    torch = torch_cuda
    net, pos, _ = fnet
    inp, T, W, tol = E.case_reference(M, m, dense_R, dinv_kind, path)
    run, a = _solve_dev(torch, net, pos, inp, M, dinv_kind)
    names = _kernels(torch, run)
    net.check()
    want, absent = _solve_kernels(M, m, dinv_kind, path)
    _expect(names, want, absent)
    eT = normerr(a["T"].cpu().numpy(), _f64(T))
    eW = normerr(a["W"].cpu().numpy(), _f64(W))
    record_property("path", path)
    record_property("T_err", eT)
    record_property("W_err", eW)
    record_property("bound", tol)
    assert eT <= tol and eW <= tol, f"T error {eT:.2e}, W error {eW:.2e}, bound {tol:.2e}"


def test_failed_direct_solve_is_reported_then_cleared(torch_cuda, fnet):
    """An indefinite S (negative R) on the direct path: net.check() raises; the next correct solve on the same
    handle passes and is right.  Nothing is routed afterwards."""
    torch = torch_cuda
    from tx_fast_hydrology_b200._lib import TxhError
    net, pos, _ = fnet
    M, m = 64, 20
    inp, T, W, tol = E.case_reference(M, m, False, 1, "direct")
    run, _ = _solve_dev(torch, net, pos, inp, M, 1, R=-1e6 * np.eye(m))
    run()
    with pytest.raises(TxhError, match="not positive definite"):
        net.check()
    run, a = _solve_dev(torch, net, pos, inp, M, 1)
    run()
    net.check()
    assert normerr(a["T"].cpu().numpy(), _f64(T)) <= tol
    assert normerr(a["W"].cpu().numpy(), _f64(W)) <= tol


# ---- (b) stats and apply ----------------------------------------------------------------------------------------
APPLY_M = [2, 3, 5, 31, 33, 63, 64, 65, 127, 128, 129, 200, 257]
APPLY_GAUGES = 90


def _apply_setup(Mtot):
    """Forecast columns 0 .. Mtot, the gauges, and a real transform of that ensemble (the reference solve, FP64)."""
    fc = E.forecast()
    inp = E.solve_inputs(Mtot, APPLY_GAUGES, E.case_seed(Mtot, APPLY_GAUGES))
    T, W, _ = E.solve_ref(inp["HX"], inp["Zp"], inp["mean"], inp["qs"], inp["R"])
    return fc, inp, _f64(T), _f64(W)


def _state(torch, net, x, M):
    """alloc_state(M) holding x [n][M] (reach order), its pad column (odd M) set to the sentinel."""
    X = net.alloc_state(M)
    net.pack_host(np.ascontiguousarray(x), M, X)
    if X.shape[1] > M:
        X[:, M:] = SENTINEL
    return X


@pytest.mark.parametrize("M", APPLY_M)
def test_stats_and_apply_vs_reference(torch_cuda, fnet, M):
    """enkf_stats (row sums, gauge rows) and enkf_apply (posterior O, I) of an unsharded ensemble; the pad columns
    of O, I and all of G hold a finite sentinel before the calls."""
    torch = torch_cuda
    net, pos, fc = fnet
    fc, inp, T, W = _apply_setup(M)
    n, g = net.n, inp["gauges"]
    O0, I0 = fc["O"][:, :M], fc["I"][:, :M]
    O, I = _state(torch, net, O0, M), _state(torch, net, I0, M)
    G = torch.full_like(O, SENTINEL)
    rowsum = torch.full((n,), np.nan, dtype=torch.float64, device="cuda")
    HX = torch.full((g.size, M), np.nan, dtype=torch.float64, device="cuda")
    Td, Wd, qs = _dev(torch, T), _dev(torch, W), _dev(torch, inp["qs"])

    def run():
        net.enkf_stats(O, M, g, rowsum, HX, scale=1.0 / M)
        net.enkf_apply(O, I, M, None, 0, M, 0, rowsum, Td, g, qs, Wd, G)
    names = _kernels(torch, run)
    net.check()
    ld = net.row_stride(M)
    _expect(names, ["enkf_stats_kernel"] + (["enkf_update64_kernel", "inflow_gain_kernel"] if ld <= 64 else
                                            ["enkf_update_kernel", "apply_gain_kernel"]))
    assert (HX.cpu().numpy() == O0[g]).all()
    mean = rowsum.cpu().numpy()[pos]                           # reach order
    exact = np.asarray(np.asarray(O0, dtype=E.LD).sum(axis=1) / M, dtype=np.float64)
    assert relerr(mean, exact) <= M * E.EPS64
    Op, Ip = E.apply_ref(O0, I0, mean, T, W, g, inp["qs"], fc["endnodes"])
    assert normerr(net.unpack_host(O, M), _f64(Op)) < 1e-12
    assert normerr(net.unpack_host(I, M), _f64(Ip)) < 1e-12
    if ld > M:                                                # pads stay finite: the routing kernels carry them
        assert torch.isfinite(O[:, M:]).all() and torch.isfinite(I[:, M:]).all()


@pytest.mark.parametrize("world,Mloc", [(2, 32), (2, 33), (4, 16), (2, 64), (3, 64)])
def test_sharded_apply_on_one_gpu(torch_cuda, fnet, world, Mloc):
    """A member-sharded update emulated on one GPU: every shard's state as its own buffer, Xall = [world][n][ldx] (the
    all-gather), enkf_apply once per shard (col0 = r Mloc, x_block_stride = n ldx), and enkf_apply_peers with every
    shard tensor on this device.  Each shard's posterior equals the reference update of the whole ensemble restricted
    to its columns, to 1e-12 (max-norm)."""
    torch = torch_cuda
    net, pos, fc = fnet
    Mtot = world * Mloc
    fc, inp, T, W = _apply_setup(Mtot)
    n, g = net.n, inp["gauges"]
    mean = inp["mean_all"]
    md, Td, Wd, qs = _dev(torch, _sched(mean, pos)), _dev(torch, T), _dev(torch, W), _dev(torch, inp["qs"])
    X = [_state(torch, net, fc["O"][:, r * Mloc:(r + 1) * Mloc], Mloc) for r in range(world)]
    ldx = X[0].shape[1]
    Xall = torch.stack(X).contiguous()
    for r in range(world):
        cols = slice(r * Mloc, (r + 1) * Mloc)
        Op, Ip = E.apply_ref_shard(fc["O"][:, :Mtot], fc["I"][:, cols], mean, T, W, g, inp["qs"], fc["endnodes"],
                                   r * Mloc, Mloc)
        O, I = X[r].clone(), _state(torch, net, fc["I"][:, cols], Mloc)
        G = torch.full_like(O, SENTINEL)
        names = _kernels(torch, lambda: net.enkf_apply(O, I, Mloc, Xall, ldx, Mtot, r * Mloc, md, Td, g, qs, Wd, G,
                                                       x_block_stride=n * ldx))
        net.check()
        _expect(names, ["enkf_update_kernel", "inflow_gain_kernel"], ["enkf_update64_kernel"])
        assert normerr(net.unpack_host(O, Mloc), _f64(Op)) < 1e-12, f"shard {r}, all-gathered ensemble"
        assert normerr(net.unpack_host(I, Mloc), _f64(Ip)) < 1e-12, f"shard {r}, all-gathered ensemble"
        Oout = torch.full_like(O, SENTINEL)
        I2 = _state(torch, net, fc["I"][:, cols], Mloc)
        names = _kernels(torch, lambda: net.enkf_apply_peers(X[r], Oout, I2, Mloc, [x.data_ptr() for x in X], Mtot,
                                                             r * Mloc, md, Td, g, qs, Wd, G))
        net.check()
        _expect(names, ["enkf_update_kernel", "inflow_gain_kernel"], ["enkf_update64_kernel"])
        assert normerr(net.unpack_host(Oout, Mloc), _f64(Op)) < 1e-12, f"shard {r}, peer blocks"
        assert normerr(net.unpack_host(I2, Mloc), _f64(Ip)) < 1e-12, f"shard {r}, peer blocks"
        assert (net.unpack_host(X[r], Mloc) == fc["O"][:, cols]).all(), "the peer path wrote its input"


# ---- (c) the assimilation loop against the oracle, step by step ------------------------------------------------
def _loop_case(torch, oracle, monkeypatch, n, M, m, seed, every, nwin, rest, kernel, in_library):
    """test_gpu_record.py:_assim_case with the routing kernel chosen by TXH_ROUTE_KERNEL (set before the model's
    device state exists) and the kernels of the run returned."""
    if kernel is not None:
        monkeypatch.setenv("TXH_ROUTE_KERNEL", kernel)
    else:
        monkeypatch.delenv("TXH_ROUTE_KERNEL", raising=False)
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
    gidx = E.gauge_set(net_d["endnodes"], m, seed)
    mt = t0 + (np.arange(nwin, dtype=np.int64) + 1) * int(every * 300e9)
    meas = rng.uniform(0.5, 8.0, size=(nwin, m))
    mdf = pd.DataFrame(meas, index=pd.DatetimeIndex(pd.to_datetime(mt, unit="ns", utc=True)).as_unit("ns"),
                       columns=[d["reach_ids"][j] for j in gidx])
    R = 1e-2 * np.eye(m)
    q = rng.uniform(0.5, 2.0, size=n)
    enkf = EnsembleKalmanFilter(mdl, mdf, q, R)
    Zp = meas[:, :, None] + 0.1 * rng.standard_normal((nwin, m, M))
    f = mdl.make_forcing(times_ns=times, table=table, member_mul=mul)
    ung = np.setdiff1d(np.arange(n), gidx)
    reaches = rng.permutation(np.concatenate([gidx[:max(3, m // 2)], rng.choice(ung, size=40, replace=False)]))
    Zd = torch.as_tensor(np.ascontiguousarray(Zp), device="cuda")
    out = {}

    def run():
        out["r"] = mdl.run_assimilating(f, nsteps, enkf, every, Zd if in_library else list(Zd), record_reaches=reaches,
                                        record_prior=True)
    names = _kernels(torch, run)
    mdl.network.check()
    rec, prior = out["r"]
    ind = oracle.compute_indegree(net_d["startnodes"], net_d["endnodes"])
    al, be, ch, ga = oracle.compute_coeffs(prm["K"], prm["X"], 300.0)
    onet = {"startnodes": net_d["startnodes"], "endnodes": net_d["endnodes"], "indegree": ind,
            "alpha": al, "beta": be, "chi": ch, "gamma": ga}
    o = np.ascontiguousarray(o0.T)
    i = np.stack([oracle.init_states(net_d["startnodes"], net_d["endnodes"], x) for x in o])
    hyd = np.empty((nsteps, reaches.size, M))
    pri = np.empty((nwin, reaches.size, M))
    # Error scales.  An update forms o + gain; where the gain cancels most of the forecast (here down to 1e-6 of it)
    # no FP64 implementation holds the posterior to 1e-9 of its own size, only to 1e-9 of the forecast
    # (parity.relerr).  Routing is linear, so that absolute error travels on with the state: e' = A e, and
    # |A e| <= |A| |e|.  The scale of every later step is therefore max(|post|, |forecast|) routed with the absolute
    # values of the coefficients and no forcing (om, im), and the value's own size where that is larger.  (Measured
    # on these cases: the FP64 oracle's update, against the extended-precision one, stays within 4e-12 of this scale
    # and exceeds 1e-9 of |value| by up to 20x a few steps after an update.)
    om = np.zeros_like(o); im = np.zeros_like(i)
    anet = dict(onet, alpha=np.abs(al), beta=np.abs(be), chi=np.abs(ch), gamma=np.zeros(n))
    zero = np.zeros_like(table)
    sc = np.empty_like(hyd)
    sc_pri = np.empty_like(pri)
    tol, oracle_err = RTOL, 0.0
    for s in range(1, nsteps + 1):
        t = float(t0 + (s - 1) * 300e9)
        oracle.run_members(onet, o, i, 1, times.astype(np.float64), table, t, 300e9, wmul=mul)
        oracle.run_members(anet, om, im, 1, times.astype(np.float64), zero, t, 300e9)
        hyd[s - 1] = o[:, reaches].T
        sc[s - 1] = om[:, reaches].T
        if s % every == 0 and s // every <= nwin:
            k = s // every - 1
            pri[k] = o[:, reaches].T
            sc_pri[k] = om[:, reaches].T
            tol = max(tol, enkf_tolerance(o.T, gidx, q, R))
            # the update in extended precision (the routing between updates is exact enough in FP64); the FP64
            # oracle's explicit-inverse update is kept for comparison only
            O, I = o.T, i.T
            mean = np.asarray(np.asarray(O, dtype=E.LD).sum(axis=1) / M, dtype=np.float64)
            T, W, _ = E.solve_ref(O[gidx], Zp[k], mean[gidx], q[gidx], R)
            Op, Ip = E.apply_ref(O, I, mean, T, W, gidx, q[gidx], net_d["endnodes"])
            Op, Ip = _f64(Op), _f64(Ip)
            Oo, _, _ = oracle.enkf_update(onet, O, I, gidx, Zp[k], q, R)
            oracle_err = max(oracle_err, relerr(Oo, Op, scale=np.abs(O)))
            om = np.ascontiguousarray(np.maximum(np.abs(Op), np.abs(O)).T)
            im = np.ascontiguousarray(np.maximum(np.abs(Ip), np.abs(I)).T)
            o = np.ascontiguousarray(Op.T); i = np.ascontiguousarray(Ip.T)
            hyd[s - 1] = o[:, reaches].T
            sc[s - 1] = om[:, reaches].T
    return names, rec.cpu().numpy(), prior.cpu().numpy(), mdl.o_t_next[reaches], hyd, pri, sc, sc_pri, tol, oracle_err


def _loop_kernels(M, m, kernel, in_library):
    ld = M + (M & 1)
    solve = ["enkf_small_system_kernel"] if (M < m and M <= 64) else \
            ["chol_solve_blocked_kernel<128>"] if M < m and M <= 128 else ["woodbury_assemble_kernel"]
    route = {"lane": "route_lane_kernel", "dataflow": "route_dataflow_kernel"}.get(kernel, "route_window_kernel")
    want = [route] + solve
    if ld > 64:
        return want + ["enkf_update_kernel", "apply_gain_kernel"] + (["enkf_record_kernel"] if in_library else [])
    if kernel in ("lane", "dataflow"):
        # the row sums: enkf_stats after the routing launch
        return want + ["enkf_stats_kernel", "enkf_update64_kernel"] + (
            ["enkf_record_kernel", "inflow_rebuild_kernel"] if in_library else ["inflow_gain_kernel"])
    if in_library:                                     # the next window applies the update and records its rows
        return want + ["route_window_kernel<true, true, true, true>"]
    return want + ["enkf_update64_kernel"]


LOOP_CASES = [  # n, M, m, seed, every, nwin, rest, route kernel, also with the Python loop
    (2500, 64, 120, 81, 6, 3, 0, None, True),       # cluster kernel + UPD window + record_posterior at M = 64
    (2500, 63, 90, 82, 6, 3, 0, None, False),       # pad column on the TMA bulk path (ld = 64)
    (2500, 33, 70, 83, 6, 3, 4, None, True),        # odd M on cp.async; the remainder launch applies the last update
    (2000, 5, 12, 84, 6, 3, 0, None, False),        # smallest window-kernel ensemble; most cluster CTAs empty
    (2000, 2, 6, 85, 6, 3, 0, "lane", True),        # lane kernel + stand-alone update + enkf_record_kernel
    (2000, 3, 8, 86, 6, 3, 2, "lane", False),
    (2000, 16, 40, 87, 12, 3, 0, "lane", True),     # lane kernel at its largest M, hourly updates
    (2000, 40, 60, 88, 6, 3, 0, "dataflow", True),  # stand-alone update after the dataflow kernel
    (2500, 97, 200, 89, 6, 3, 0, None, True),       # partial Cholesky panel (chol<128>)
    (2500, 129, 300, 90, 6, 3, 3, None, False),     # three member blocks with a pad; M > 128 solve
    (4000, 64, 1100, 91, 6, 3, 0, None, False),     # cluster kernel with more than one gauge tile per CTA
]


def _loop_params():
    out = []
    for c in LOOP_CASES:
        out.append(pytest.param(*c[:8], True, id=f"M{c[1]}-m{c[2]}-{c[7] or 'default'}-lib"))
        if c[8]:
            out.append(pytest.param(*c[:8], False, id=f"M{c[1]}-m{c[2]}-{c[7] or 'default'}-py"))
    return out


@pytest.mark.parametrize("n,M,m,seed,every,nwin,rest,kernel,in_library", _loop_params())
def test_assimilation_loop_paths_vs_oracle(torch_cuda, oracle, monkeypatch, record_property, n, M, m, seed, every,
                                           nwin, rest, kernel, in_library):
    """run_assimilating with record_reaches and record_prior: hydrographs (forecast, posterior at update steps),
    priors and final state against the oracle's routing and the extended-precision update, with the tolerance of
    test_gpu_record.py (1e-9, or 64 eps cond(S) after an update) relative to the error scale of _loop_case."""
    names, rec, prior, final, hyd, pri, sc, sc_pri, tol, oracle_err = _loop_case(
        torch_cuda, oracle, monkeypatch, n, M, m, seed, every, nwin, rest, kernel, in_library)
    _expect(names, _loop_kernels(M, m, kernel, in_library))
    nsteps = every * nwin + rest
    assert rec.shape == hyd.shape and prior.shape == pri.shape
    assert not np.isnan(rec).any() and not np.isnan(prior).any()
    e_pri, e_rec = relerr(prior, pri, scale=sc_pri), relerr(rec, hyd, scale=sc)
    record_property("tol", tol)
    record_property("rec_err", e_rec)
    record_property("oracle_fp64_update_err", oracle_err)
    assert e_pri < tol, f"priors: {e_pri:.2e}, bound {tol:.2e}"
    per_step = [relerr(rec[j], hyd[j], scale=sc[j]) for j in range(nsteps)]
    assert e_rec < tol, f"hydrographs: {e_rec:.2e}, bound {tol:.2e}; worst step {int(np.argmax(per_step)) + 1}"
    assert relerr(final, hyd[nsteps - 1], scale=sc[nsteps - 1]) < tol


# ---- ensembles too small for a sample covariance ----------------------------------------------------------------
def test_one_member_filter_refused_on_device(torch_cuda):
    """EnsembleKalmanFilter refuses Muskingum(members=1) before any device work: the model's device state and clock
    are those it had before the call."""
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.muskingum import Muskingum
    from tx_fast_hydrology_b200.da import EnsembleKalmanFilter
    n = 300
    net_d = S.make_network(n, 5)
    d = S.model_dict(net_d, S.make_params(n, 5, well_posed=True))
    mdl = Muskingum(d, members=1)
    mdl._ensure_device()
    O, I = (x.clone() for x in mdl.device_state)
    t = mdl.datetime
    g = E.gauge_set(net_d["endnodes"], 4, 5)
    mdf = pd.DataFrame(np.ones((2, 4)), columns=[d["reach_ids"][j] for j in g],
                       index=pd.DatetimeIndex([t + mdl.timedelta * 6, t + mdl.timedelta * 12]))
    with pytest.raises(ValueError, match="at least 2 members"):
        EnsembleKalmanFilter(mdl, mdf, 1.0, 1e-2 * np.eye(4))
    torch_cuda.cuda.synchronize()
    assert mdl.datetime == t
    O2, I2 = mdl.device_state
    assert torch_cuda.equal(O, O2) and torch_cuda.equal(I, I2)

"""The harness the GPU tests of the ensemble filter share (tests/test_gpu_enkf_paths.py, test_gpu_enkf_missing.py,
test_gpu_etkf.py, test_gpu_record.py, test_gpu_smooth.py, test_gpu_model.py): fixtures, the kernel-name capture, the
solve-path helpers and the assimilation loop -- a synthetic case (numpy only), its run on the device, and the same
run on the CPU oracle with an extended-precision or FP64 reference update."""
import numpy as np
import pandas as pd
import pytest

import enkf_reference as E
import enkf_missing_reference as X
import etkf_reference as K
from parity import relerr, enkf_tolerance

RTOL = 1e-9
SENTINEL = 1e6


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


def _f64(a):
    return np.asarray(a, dtype=np.float64)


def _sched(vec, pos):
    out = np.empty_like(vec)
    out[pos] = vec
    return out


def _state(torch, net, x, M):
    """alloc_state(M) holding x [n][M] (reach order), its pad column (odd M) set to the sentinel."""
    X = net.alloc_state(M)
    net.pack_host(np.ascontiguousarray(x), M, X)
    if X.shape[1] > M:
        X[:, M:] = SENTINEL
    return X


# ---- the solve paths ------------------------------------------------------------------------------------------------
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


# ---- the assimilation loop: the case ----------------------------------------------------------------------------------
def make_case(n, M, m, seed, every, nwin, rest, *, gauges, dense_R=False, extra_reaches=40, observations="perturbed"):
    """`nwin` windows of `every` 300 s routing steps, one ensemble update at the end of each, then `rest` more steps,
    on a synthetic network of n reaches and M members.  Numpy only: nothing here touches the device.

    gauges: "reference" (enkf_reference.gauge_set: outlets and confluences first), "synthetic" (synthetic.make_gauges)
    or the gauged reaches themselves; m becomes their count.  dense_R: a correlated observation error covariance
    instead of 1e-2 I.  observations: "perturbed" (the measurement plus noise of 0.1 in every member) or "identical"
    (the measurement in every member, as a square-root filter takes it).  The recorded reaches are the first half of
    the gauges and `extra_reaches` ungauged ones, in no particular order; None records nothing.

    The draws from default_rng(seed) come in one order, so that a case is the same whichever options it leaves out:
    initial outflows, measurements, dense R, q, observation noise, recorded reaches."""
    from tx_fast_hydrology_b200 import synthetic as S
    net = S.make_network(n, seed)
    prm = S.make_params(n, seed, well_posed=True)
    rng = np.random.default_rng(seed)
    o0 = prm["o_t"][:, None] * rng.uniform(0.5, 1.5, size=(n, M))
    d = S.model_dict(net, prm, dt_s=300.0)
    d["o_t"] = o0
    t0 = int(d["datetime"].value)
    nsteps = every * nwin + rest
    times, table = S.make_forcing(n, nsteps, 300.0, seed, t0_ns=t0, rows_every=4)
    mul = S.make_member_multipliers(times.size, M, seed)
    if isinstance(gauges, str):
        gauges = {"reference": E.gauge_set, "synthetic": S.make_gauges}[gauges](net["endnodes"], m, seed)
    gidx = np.asarray(gauges, dtype=np.int64)
    m = gidx.size
    mt = t0 + (np.arange(nwin, dtype=np.int64) + 1) * int(every * 300e9)
    meas = rng.uniform(0.5, 8.0, size=(nwin, m))
    mdf = pd.DataFrame(meas, index=pd.DatetimeIndex(pd.to_datetime(mt, unit="ns", utc=True)).as_unit("ns"),
                       columns=[d["reach_ids"][j] for j in gidx])
    R = 1e-2 * np.eye(m)
    if dense_R:                                                   # correlated observation errors: SPD, not diagonal
        Bm = rng.standard_normal((m, m))
        R = 1e-2 * (np.eye(m) + 0.5 * (Bm @ Bm.T) / m)
    q = rng.uniform(0.5, 2.0, size=n)
    if observations == "perturbed":
        Zp = meas[:, :, None] + 0.1 * rng.standard_normal((nwin, m, M))
    else:
        assert observations == "identical", observations
        Zp = np.repeat(meas[:, :, None], M, axis=2)
    reaches = None
    if extra_reaches is not None:
        ung = np.setdiff1d(np.arange(n), gidx)
        reaches = rng.permutation(np.concatenate([gidx[:max(3, m // 2)],
                                                  rng.choice(ung, size=extra_reaches, replace=False)]))
    return dict(n=n, M=M, every=every, nwin=nwin, nsteps=nsteps, net=net, prm=prm, d=d, o0=o0, t0=t0, times=times,
                table=table, mul=mul, gidx=gidx, meas=meas, mdf=mdf, R=R, q=q, Zp=Zp, reaches=reaches)


def model(c, **filter_kw):
    """The case's Muskingum model, its EnsembleKalmanFilter (`filter_kw`: method, rtpp) and its forcing."""
    from tx_fast_hydrology_b200.muskingum import Muskingum
    from tx_fast_hydrology_b200.da import EnsembleKalmanFilter
    mdl = Muskingum(c["d"], members=c["M"])
    enkf = EnsembleKalmanFilter(mdl, c["mdf"], c["q"], c["R"], **filter_kw)
    return mdl, enkf, mdl.make_forcing(times_ns=c["times"], table=c["table"], member_mul=c["mul"])


# ---- the assimilation loop on the device ------------------------------------------------------------------------------
def run_device(c, in_library, *, monkeypatch=None, kernel=None, record_every=1, lag=None, **filter_kw):
    """run_assimilating of case c with record_reaches and record_prior, the observations as one tensor (`in_library`:
    the loop runs inside libtxh) or as a list of tensors (the Python loop); `lag` smooths.

    With `monkeypatch` the routing kernel is pinned to `kernel` (TXH_ROUTE_KERNEL, None: the default; set before the
    model's device state exists) and the run is profiled: `names` holds the kernels it launched.  Returns those names,
    the results of the run as numpy (rec, prior[, smoothed]), the final state at the recorded reaches, the model and
    the filter."""
    import torch
    if monkeypatch is not None:
        if kernel is not None:
            monkeypatch.setenv("TXH_ROUTE_KERNEL", kernel)
        else:
            monkeypatch.delenv("TXH_ROUTE_KERNEL", raising=False)
    mdl, enkf, f = model(c, **filter_kw)
    Zd = torch.as_tensor(np.ascontiguousarray(c["Zp"]), device="cuda")
    out = {}

    def run():
        out["r"] = mdl.run_assimilating(f, c["nsteps"], enkf, c["every"], Zd if in_library else list(Zd),
                                        record_reaches=c["reaches"], record_every=record_every, record_prior=True,
                                        smooth_lag=lag)
    names = None
    if monkeypatch is not None:
        names = _kernels(torch, run)
    else:
        run()
    mdl.network.check()
    return dict(names=names, res=[x.cpu().numpy() for x in out["r"]], final=mdl.o_t_next[c["reaches"]], mdl=mdl,
                enkf=enkf)


# ---- the assimilation loop on the CPU oracle --------------------------------------------------------------------------
def oracle_start(oracle, c):
    """The case's network for the oracle and its initial outflows and inflows [M][n]."""
    net, prm = c["net"], c["prm"]
    al, be, ch, ga = oracle.compute_coeffs(prm["K"], prm["X"], 300.0)
    onet = {"startnodes": net["startnodes"], "endnodes": net["endnodes"],
            "indegree": oracle.compute_indegree(net["startnodes"], net["endnodes"]),
            "alpha": al, "beta": be, "chi": ch, "gamma": ga}
    o = np.ascontiguousarray(c["o0"].T)
    i = np.stack([oracle.init_states(net["startnodes"], net["endnodes"], x) for x in o])
    return onet, o, i


def reference_loop(oracle, c, update, record_every=1):
    """Case c step by step on the oracle, with `update` at the end of every window.

    update(c, k, O, I, oracle, onet) takes the forecast O, I [n][M] of update k and returns the posterior (Op, Ip), what
    the test keeps of the update (in `kept`), the update's tolerance and an amplification of it.  Returns the
    hydrographs at the recorded reaches after every `record_every`-th step (`sel`: their steps - 1; the posterior at
    update steps), the priors, the error scales of both, the tolerance (the largest of RTOL and the updates', times
    the largest amplification), the updates' tolerances and what was kept."""
    onet, o, i = oracle_start(oracle, c)
    M, every, nwin, nsteps, reaches = c["M"], c["every"], c["nwin"], c["nsteps"], c["reaches"]
    times, table = c["times"].astype(np.float64), c["table"]
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
    anet = dict(onet, alpha=np.abs(onet["alpha"]), beta=np.abs(onet["beta"]), chi=np.abs(onet["chi"]),
                gamma=np.zeros(c["n"]))
    zero = np.zeros_like(table)
    sc = np.empty_like(hyd)
    sc_pri = np.empty_like(pri)
    tols, amps, kept = [], [], []
    for s in range(1, nsteps + 1):
        t = float(c["t0"] + (s - 1) * 300e9)
        oracle.run_members(onet, o, i, 1, times, table, t, 300e9, wmul=c["mul"])
        oracle.run_members(anet, om, im, 1, times, zero, t, 300e9)
        hyd[s - 1] = o[:, reaches].T
        sc[s - 1] = om[:, reaches].T
        if s % every == 0 and s // every <= nwin:
            k = s // every - 1
            pri[k] = o[:, reaches].T
            sc_pri[k] = om[:, reaches].T
            O, I = o.T, i.T
            Op, Ip, keep, tol, amp = update(c, k, O, I, oracle, onet)
            kept.append(keep); tols.append(tol); amps.append(amp)
            om = np.ascontiguousarray(np.maximum(np.abs(Op), np.abs(O)).T)
            im = np.ascontiguousarray(np.maximum(np.abs(Ip), np.abs(I)).T)
            o = np.ascontiguousarray(Op.T); i = np.ascontiguousarray(Ip.T)
            hyd[s - 1] = o[:, reaches].T
            sc[s - 1] = om[:, reaches].T
    sel = np.arange(record_every, nsteps + 1, record_every) - 1
    return dict(hyd=hyd[sel], sc=sc[sel], sel=sel, pri=pri, sc_pri=sc_pri, tol=max(RTOL, *tols) * max(1.0, *amps),
                tols=tols, kept=kept)


def _ld_mean(O):
    return np.asarray(np.asarray(O, dtype=E.LD).sum(axis=1) / O.shape[1], dtype=np.float64)


def update_ref(c, k, O, I, oracle, onet):
    """The update in extended precision (the routing between updates is exact enough in FP64).  Keeps the error of the
    FP64 oracle's explicit-inverse update against it, relative to the forecast, for comparison only."""
    g, q, R, Z = c["gidx"], c["q"], c["R"], c["Zp"][k]
    tol = enkf_tolerance(O, g, q, R)
    mean = _ld_mean(O)
    T, W, _ = E.solve_ref(O[g], Z, mean[g], q[g], R)
    Op, Ip = E.apply_ref(O, I, mean, T, W, g, q[g], c["net"]["endnodes"])
    Op, Ip = _f64(Op), _f64(Ip)
    Oo, _, _ = oracle.enkf_update(onet, O, I, g, Z, q, R)
    return Op, Ip, relerr(Oo, Op, scale=np.abs(O)), tol, 1.0


def _solve_masked(c, k, O):
    """The masked solve of update k in extended precision, the ensemble mean and the tolerance over the kept gauges
    (0 with every gauge missing: the update changes nothing)."""
    g, q, R, Z = c["gidx"], c["q"], c["R"], c["Zp"][k]
    keep = ~X.missing_rows(Z)
    tol = enkf_tolerance(O, g[keep], q, R[np.ix_(keep, keep)]) if keep.any() else 0.0
    mean = _ld_mean(O)
    T, W, _, _ = X.solve_masked(O[g], Z, mean[g], q[g], R)
    return T, W, mean, tol


def update_masked(c, k, O, I, oracle, onet):
    """The update with missing gauges (NaN rows of Zp[k]) in extended precision; keeps its transform."""
    T, W, mean, tol = _solve_masked(c, k, O)
    Op, Ip = E.apply_ref(O, I, mean, T, W, c["gidx"], c["q"][c["gidx"]], c["net"]["endnodes"])
    return _f64(Op), _f64(Ip), _f64(T), tol, 1.0


def update_etkf(c, k, O, I, oracle, onet, rho=0.0):
    """The square-root update (ETKF, relaxed to the prior perturbations by `rho`) of the masked solve in extended
    precision; keeps its transform.  The tolerance is amplified by M / (2 sqrt(lambda_min(G))), the conditioning of
    the matrix square root."""
    T, W, mean, tol = _solve_masked(c, k, O)
    amp = c["M"] / (2.0 * np.sqrt(K.lambda_min(T)))
    Tp, Wp = K.etkf_post(T, W, rho)
    Op, Ip = E.apply_ref(O, I, mean, Tp, Wp, c["gidx"], c["q"][c["gidx"]], c["net"]["endnodes"])
    return _f64(Op), _f64(Ip), _f64(Tp), tol, amp


def update_fp64(c, k, O, I, oracle, onet):
    """The FP64 oracle's update (da.py's explicit inverse).  Keeps what the smoother needs of it: the forecast anomalies
    at the gauges, the innovations and the innovation covariance."""
    g, q, R, Z = c["gidx"], c["q"], c["R"], c["Zp"][k]
    HA = O[g] - O[g].mean(axis=1, keepdims=True)
    dz = Z - O[g]
    S = HA @ HA.T / (c["M"] - 1) + np.diag(q[g]) + R
    tol = enkf_tolerance(O, g, q, R)
    Op, Ip, _ = oracle.enkf_update(onet, O, I, g, Z, q, R)
    return Op, Ip, (HA, dz, S), tol, 1.0


# ---- the loop cases of the dispatch paths -----------------------------------------------------------------------------
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


def loop_params(cases):
    """pytest parameters (n, M, m, seed, every, nwin, rest, kernel, in_library) of loop cases: each in the library,
    and in the Python loop too where the case asks for it."""
    out = []
    for c in cases:
        out.append(pytest.param(*c[:8], True, id=f"M{c[1]}-m{c[2]}-{c[7] or 'default'}-lib"))
        if c[8]:
            out.append(pytest.param(*c[:8], False, id=f"M{c[1]}-m{c[2]}-{c[7] or 'default'}-py"))
    return out

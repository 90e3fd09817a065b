"""The square-root ensemble update (ETKF) and relaxation to prior perturbations (RTPP) on the GPU: every solve path
followed by enkf_transform_post_kernel / enkf_rtpp_kernel against the extended-precision reference
(tests/etkf_reference.py), missing gauges, the assimilation loops (in the library and in Python, with the update
applied by the next window launch and by the stand-alone kernels), the smoother on an ETKF run, the default left
bit for bit as it was, and the refusals.  Every case checks with torch.profiler which kernels ran, as
tests/test_gpu_enkf_paths.py does.

Tolerances: T' and W' against the reference at etkf_reference.case's bounds -- the solve tolerance of
enkf_reference.solve_tolerance (64 eps cond), for T' of the ETKF amplified by M / (2 sqrt(lambda_min(G))), the
conditioning of the matrix square root, plus the Jacobi stop (1e-14 ||G||_F).  The loops use the tolerance of
test_gpu_enkf_paths.py times the same amplification of the worst update."""
import functools

import numpy as np
import pandas as pd
import pytest

import enkf_reference as E
import enkf_missing_reference as X
import etkf_reference as K
from assim_case import (torch_cuda, fnet, _kernels, _expect, _f64, _solve_dev, _solve_kernels,  # noqa: F401
                        make_case, run_device, reference_loop, update_etkf)
from enks_oracle import smooth_transforms
from parity import relerr, normerr

pytestmark = pytest.mark.gpu

POST, RTPP = "enkf_transform_post_kernel", "enkf_rtpp_kernel"
FUSED = "route_window_kernel<true, true, true, true>"           # the window launch that applies an owed update


def _launches():
    from tx_fast_hydrology_b200 import _lib
    return int(_lib.load().txh_launch_count())


# ---- (a) the solve paths ---------------------------------------------------------------------------------------------
ETKF_M = (2, 3, 5, 33, 63, 64)
ETKF_CASES = ([(M, 100, False, 1, "cluster") for M in ETKF_M] +
              [(M, 80, True, 2, "woodbury") for M in ETKF_M] +
              [(M, max(1, M // 2) if M < 64 else 64, False, 1, "direct") for M in ETKF_M])


def _run_case(torch, fnet, M, m, dense_R, dinv_kind, path, rho, mask="none", method="etkf"):
    net, pos, _ = fnet
    inp, miss, Tp, Wp, tolT, tolW = K.case(M, m, dense_R, path, rho=rho, mask=mask, method=method)
    run, a = _solve_dev(torch, net, pos, inp, M, dinv_kind)
    net.set_enkf_transform(method, rho)
    try:
        names = _kernels(torch, run)
    finally:
        net.set_enkf_transform()
    net.check()
    want, absent = _solve_kernels(M, m, dinv_kind, path)
    post = POST if method == "etkf" else RTPP
    _expect(names, want + [post], absent + [RTPP if method == "etkf" else POST])
    return a["T"].cpu().numpy(), a["W"].cpu().numpy(), miss, _f64(Tp), _f64(Wp), tolT, tolW


@pytest.mark.parametrize("rho", [0.0, 0.5])
@pytest.mark.parametrize("M,m,dense_R,dinv_kind,path", ETKF_CASES)
def test_etkf_solve_paths_vs_reference(torch_cuda, fnet, record_property, M, m, dense_R, dinv_kind, path, rho):
    """T' and W' of every solve path with the ETKF set on the handle, against the longdouble reference."""
    Td, Wd, _, Tp, Wp, tolT, tolW = _run_case(torch_cuda, fnet, M, m, dense_R, dinv_kind, path, rho)
    eT, eW = normerr(Td, Tp), normerr(Wd, Wp)
    record_property("ratio", max(eT / tolT, eW / tolW))
    assert eT <= tolT and eW <= tolW, f"T' error {eT:.2e} (bound {tolT:.2e}), W' error {eW:.2e} (bound {tolW:.2e})"
    assert (Wd == Wd[:, :1]).all(), "W' is not one column repeated"


@pytest.mark.parametrize("M,m,dense_R,dinv_kind,path", [(5, 100, False, 1, "cluster"), (64, 100, False, 1, "cluster"),
                                                       (33, 80, True, 2, "woodbury"), (97, 300, False, 1, "woodbury"),
                                                       (129, 450, False, 1, "woodbury_big"),
                                                       (64, 64, False, 1, "direct")])
def test_rtpp_solve_paths_vs_reference(torch_cuda, fnet, M, m, dense_R, dinv_kind, path):
    """The stochastic update relaxed with rtpp = 0.5 (enkf_rtpp_kernel, any member count) against the reference."""
    Td, Wd, _, Tp, Wp, tolT, tolW = _run_case(torch_cuda, fnet, M, m, dense_R, dinv_kind, path, 0.5, method="stochastic")
    eT, eW = normerr(Td, Tp), normerr(Wd, Wp)
    assert eT <= tolT and eW <= tolW, f"T' error {eT:.2e} (bound {tolT:.2e}), W' error {eW:.2e} (bound {tolW:.2e})"


@pytest.mark.parametrize("mask", X.MASKS)
@pytest.mark.parametrize("M", [33, 64])
def test_etkf_with_missing_gauges(torch_cuda, fnet, M, mask):
    """NaN rows on the cluster path: T', W' of the filter without the missing gauges; W' exactly 0 at them; with every
    gauge missing T' = 0 and W' = 0 exactly (G = I)."""
    Td, Wd, miss, Tp, Wp, tolT, tolW = _run_case(torch_cuda, fnet, M, 100, False, 1, "cluster", 0.0, mask=mask)
    assert np.isfinite(Td).all() and np.isfinite(Wd).all()
    assert (Wd[miss] == 0.0).all()
    if miss.all():
        assert not Td.any() and not Wd.any()
        return
    assert normerr(Td, Tp) <= tolT and normerr(Wd, Wp) <= tolW


def test_default_transform_is_bitwise_unchanged(torch_cuda, fnet):
    """After an ETKF solve and a reset, the default solve gives the same bits with the same launch count as before any
    setting; the reset costs no launch."""
    torch = torch_cuda
    net, pos, _ = fnet
    inp = E.solve_inputs(33, 100, E.case_seed(33, 100))
    run, a = _solve_dev(torch, net, pos, inp, 33, 1)
    out = []
    for step in ("before", "etkf", "after"):
        if step == "etkf":
            net.set_enkf_transform("etkf", 0.3)
        n0 = _launches()
        run()
        torch.cuda.synchronize()
        out.append((a["T"].clone(), a["W"].clone(), _launches() - n0))
        net.set_enkf_transform()
    net.check()
    (T0, W0, n0), (T1, _, n1), (T2, W2, n2) = out
    assert torch.equal(T0, T2) and torch.equal(W0, W2) and n0 == n2
    assert n1 == n0 + 1 and not torch.equal(T0, T1)


def test_member_sharded_ranks_solve_the_same_transform(torch_cuda, fnet):
    """A member-sharded filter has every rank solve the same Mtot x Mtot system: two solves of it on two handles give
    the same bits, so every rank post-processes the same transform."""
    torch = torch_cuda
    from tx_fast_hydrology_b200.network import RiverNetwork
    net, pos, fc = fnet
    net2 = RiverNetwork(fc["endnodes"])
    inp = E.solve_inputs(64, 100, E.case_seed(64, 100))
    inp = dict(inp, Zp=K.identical_columns(inp["Zp"]))
    res = []
    for h in (net, net2):
        run, a = _solve_dev(torch, h, pos, inp, 64, 1)
        h.set_enkf_transform("etkf", 0.0)
        run()
        h.set_enkf_transform()
        h.check()
        res.append((a["T"], a["W"]))
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])
    net2.close()


# ---- (b) refusals ----------------------------------------------------------------------------------------------------
def _small_filter_inputs(torch, M=8):
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.muskingum import Muskingum
    n, m = 400, 6
    net_d = S.make_network(n, 9)
    d = S.model_dict(net_d, S.make_params(n, 9, well_posed=True))
    mdl = Muskingum(d, members=M)
    mdl._ensure_device()
    g = E.gauge_set(net_d["endnodes"], m, 9)
    t = mdl.datetime
    idx = pd.DatetimeIndex([t + mdl.timedelta * 6, t + mdl.timedelta * 12])
    mdf = pd.DataFrame(np.ones((2, m)), columns=[d["reach_ids"][j] for j in g], index=idx)
    return mdl, mdf, 1e-2 * np.eye(m)


def test_refusals(torch_cuda):
    """ValueError before any device work: an ETKF with obs_noise or more than 64 members, rtpp outside [0, 1), an
    unknown method, run_assimilating observations whose members differ on a row without NaN; TxhError from the C ABI
    for another kind, a bad rtpp, and an ETKF solve of more than 64 members."""
    torch = torch_cuda
    from tx_fast_hydrology_b200 import _lib
    from tx_fast_hydrology_b200.da import EnsembleKalmanFilter
    mdl, mdf, R = _small_filter_inputs(torch)
    m = R.shape[0]
    noise = np.zeros((2, m, 8))
    with pytest.raises(ValueError, match="obs_noise"):
        EnsembleKalmanFilter(mdl, mdf, 1.0, R, obs_noise=noise, group=False, method="etkf")
    for bad in (-0.1, 1.0, float("nan"), True, "0.5"):
        with pytest.raises(ValueError, match="rtpp"):
            EnsembleKalmanFilter(mdl, mdf, 1.0, R, group=False, rtpp=bad)
    with pytest.raises(ValueError, match="method"):
        EnsembleKalmanFilter(mdl, mdf, 1.0, R, group=False, method="eakf")
    big, bdf, bR = _small_filter_inputs(torch, M=65)
    with pytest.raises(ValueError, match="64 members"):
        EnsembleKalmanFilter(big, bdf, 1.0, bR, group=False, method="etkf")
    EnsembleKalmanFilter(big, bdf, 1.0, bR, group=False, rtpp=0.5)           # RTPP alone takes any member count
    enkf = EnsembleKalmanFilter(mdl, mdf, 1.0, R, group=False, method="etkf", rtpp=0.2)
    O0 = mdl.device_state[0].clone()
    t0 = mdl.datetime
    f = mdl.make_forcing(times_ns=np.array([int(t0.value)]), table=np.ones((1, mdl.n)))
    obs = torch.full((2, m, 8), 2.0, dtype=torch.float64, device="cuda")
    obs[1, 3, 5] = 2.5
    for o in (obs, list(obs)):
        with pytest.raises(ValueError, match="same observation in every member"):
            mdl.run_assimilating(f, 12, enkf, 6, o)
    assert mdl.datetime == t0 and torch.equal(mdl.device_state[0], O0)
    obs[1, 3, 4] = float("nan")                                              # a NaN row: the gauge is missing
    mdl.run_assimilating(f, 12, enkf, 6, obs)
    mdl.network.check()
    net = mdl.network
    lib = _lib.load()
    with pytest.raises(_lib.TxhError):
        _lib.check(lib.txh_set_enkf_transform(net.handle, 2, 0.0))
    for bad in (-1e-3, 1.0, float("nan")):
        with pytest.raises(_lib.TxhError):
            _lib.check(lib.txh_set_enkf_transform(net.handle, 1, bad))
    # an ETKF solve of 65 members: refused before any device work, the outputs untouched
    mb = 65
    args = dict(HX=torch.zeros((m, mb), dtype=torch.float64, device="cuda"),
                W=torch.full((m, mb), 7.0, dtype=torch.float64, device="cuda"),
                T=torch.full((mb, mb), 7.0, dtype=torch.float64, device="cuda"))
    bn = big.network
    big._ensure_device()
    bn.set_enkf_transform("etkf")
    try:
        with pytest.raises(_lib.TxhError, match="64 members"):
            bn.enkf_solve(m, mb, args["HX"], args["HX"], torch.zeros(big.n, dtype=torch.float64, device="cuda"),
                          np.arange(m), torch.ones(m, dtype=torch.float64, device="cuda"),
                          torch.as_tensor(bR, device="cuda"), torch.empty(bn.enkf_work_size(m, mb), dtype=torch.float64,
                                                                           device="cuda"),
                          args["W"], args["T"], torch.ones(m, dtype=torch.float64, device="cuda"), 1)
    finally:
        bn.set_enkf_transform()
    torch.cuda.synchronize()
    assert (args["T"] == 7.0).all() and (args["W"] == 7.0).all()


# ---- (c) the loops and the smoother ----------------------------------------------------------------------------------
def _etkf_case(n, M, m, seed, every, nwin, rest):
    """A loop case for the ETKF: identical observation columns, an outlet gauge missing at every update and every gauge
    missing at update 1."""
    c = make_case(n, M, m, seed, every, nwin, rest, gauges="reference", observations="identical")
    end = np.asarray(c["net"]["endnodes"])
    c["Zp"][:, np.flatnonzero(end[c["gidx"]] == c["gidx"])[0]] = np.nan
    if nwin > 1:
        c["Zp"][1] = np.nan
    return c


ETKF_LOOPS = [  # n, M, m, seed, every, nwin, rest, route kernel, in the library
    pytest.param(2500, 64, 120, 81, 6, 3, 0, None, True, id="M64-window-fused-lib"),
    pytest.param(2500, 64, 120, 81, 6, 3, 0, None, False, id="M64-window-py"),
    pytest.param(2500, 33, 70, 83, 6, 3, 4, None, True, id="M33-window-fused-rest-lib"),
    pytest.param(2000, 40, 60, 88, 6, 3, 0, "dataflow", True, id="M40-dataflow-standalone-lib"),
    pytest.param(2000, 16, 40, 87, 12, 3, 0, "lane", True, id="M16-lane-standalone-lib"),
    pytest.param(2000, 5, 12, 84, 6, 3, 0, None, True, id="M5-window-lib"),
]


@pytest.mark.parametrize("rho", [0.0, 0.4])
@pytest.mark.parametrize("n,M,m,seed,every,nwin,rest,kernel,in_library", ETKF_LOOPS)
def test_etkf_assimilation_loop_vs_reference(torch_cuda, oracle, monkeypatch, record_property, n, M, m, seed, every,
                                             nwin, rest, kernel, in_library, rho):
    """Hydrographs, priors and final state of an ETKF run (with an outage) against the extended-precision loop; the
    post kernel runs once per update; the update with every gauge missing leaves the state as it was."""
    c = _etkf_case(n, M, m, seed, every, nwin, rest)
    d = run_device(c, in_library, monkeypatch=monkeypatch, kernel=kernel, method="etkf", rtpp=rho)
    r = reference_loop(oracle, c, functools.partial(update_etkf, rho=rho))
    assert d["names"].count(POST + "(") == nwin
    if kernel is None and in_library:
        _expect(d["names"], [FUSED])                                                  # applied by the next window
    elif kernel is not None:
        _expect(d["names"], ["enkf_update64_kernel"])                                 # the stand-alone kernels
    rec, prior = d["res"]
    e_pri, e_rec = relerr(prior, r["pri"], scale=r["sc_pri"]), relerr(rec, r["hyd"], scale=r["sc"])
    record_property("rec_ratio", e_rec / r["tol"])
    assert e_pri < r["tol"], f"priors: {e_pri:.2e}, bound {r['tol']:.2e}"
    assert e_rec < r["tol"], f"hydrographs: {e_rec:.2e}, bound {r['tol']:.2e}"
    nsteps = every * nwin + rest
    assert relerr(d["final"], r["hyd"][nsteps - 1], scale=r["sc"][nsteps - 1]) < r["tol"]
    assert np.array_equal(rec[2 * every - 1], prior[1]), "the update with every gauge missing changed the state"


def test_fused_load_matches_standalone_apply(torch_cuda, oracle, monkeypatch):
    """The same ETKF run with the update applied by the next window launch and by the stand-alone kernels (dataflow
    routing): the hydrographs agree to the loop tolerance."""
    c = _etkf_case(2000, 40, 60, 88, 6, 3, 0)
    a = run_device(c, True, monkeypatch=monkeypatch, method="etkf", rtpp=0.2)
    r = reference_loop(oracle, c, functools.partial(update_etkf, rho=0.2))
    b = run_device(_etkf_case(2000, 40, 60, 88, 6, 3, 0), True, monkeypatch=monkeypatch, kernel="dataflow",
                   method="etkf", rtpp=0.2)
    _expect(a["names"], [FUSED])
    _expect(b["names"], ["route_dataflow_kernel", "enkf_update64_kernel"])
    assert relerr(a["res"][0], b["res"][0], scale=r["sc"]) < r["tol"]


@pytest.mark.parametrize("in_library", [True, False])
def test_smoother_on_an_etkf_run(torch_cuda, oracle, monkeypatch, in_library):
    """smooth_lag on an ETKF run is the ETKS: enks_oracle.smooth_transforms of the reference hydrographs with the
    reference ETKF transforms."""
    n, M, m, seed, every, nwin, rest = 2500, 64, 120, 81, 6, 3, 0
    lag = every + 2
    c = _etkf_case(n, M, m, seed, every, nwin, rest)
    rec, prior, sm = run_device(c, in_library, monkeypatch=monkeypatch, lag=lag, method="etkf")["res"]
    r = reference_loop(oracle, c, update_etkf)
    want = smooth_transforms(r["hyd"], np.stack(r["kept"]), nwin, every, 1, lag)
    sc = np.maximum(np.maximum(np.abs(want), r["sc"]), np.abs(rec))
    assert np.isfinite(sm).all()
    assert relerr(sm, want, scale=sc) < r["tol"] * (nwin + 1)

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
from assim_case import (torch_cuda, fnet, _kernels, _expect, _dev, _f64, _sched, _state, SENTINEL,  # noqa: F401
                        _solve_kernels, _solve_dev, _loop_kernels, LOOP_CASES, loop_params, make_case, run_device,
                        reference_loop, update_ref)
from parity import relerr, normerr

pytestmark = pytest.mark.gpu


# ---- (a) the solve --------------------------------------------------------------------------------------------
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
@pytest.mark.parametrize("n,M,m,seed,every,nwin,rest,kernel,in_library", loop_params(LOOP_CASES))
def test_assimilation_loop_paths_vs_oracle(torch_cuda, oracle, monkeypatch, record_property, n, M, m, seed, every,
                                           nwin, rest, kernel, in_library):
    """run_assimilating with record_reaches and record_prior: hydrographs (forecast, posterior at update steps),
    priors and final state against the oracle's routing and the extended-precision update, with the tolerance of
    test_gpu_record.py (1e-9, or 64 eps cond(S) after an update) relative to the error scale of
    assim_case.reference_loop."""
    c = make_case(n, M, m, seed, every, nwin, rest, gauges="reference")
    d = run_device(c, in_library, monkeypatch=monkeypatch, kernel=kernel)
    r = reference_loop(oracle, c, update_ref)
    _expect(d["names"], _loop_kernels(M, m, kernel, in_library))
    (rec, prior), final = d["res"], d["final"]
    hyd, pri, sc, sc_pri, tol, oracle_err = r["hyd"], r["pri"], r["sc"], r["sc_pri"], r["tol"], max(r["kept"])
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

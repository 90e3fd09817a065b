"""Missing gauge observations (NaN in a row of Zp) on every solve path, in the assimilation loops and the smoother,
against the masked extended-precision reference (tests/enkf_missing_reference.py): the update equals that of a filter
without the missing gauges, W is exactly 0 at them, and nothing downstream sees a NaN.  With a dense D the NaN is
reported (net.check()) or refused before any device work.  Every case checks with torch.profiler which kernels ran,
as tests/test_gpu_enkf_paths.py does."""
import functools

import numpy as np
import pandas as pd
import pytest

import enkf_reference as E
import enkf_missing_reference as X
from assim_case import (torch_cuda, fnet, _kernels, _expect, _dev, _f64, _solve_dev, _solve_kernels,  # noqa: F401
                        _loop_kernels, _state, LOOP_CASES, loop_params, make_case, run_device, reference_loop,
                        update_masked)
from enks_oracle import smooth_transforms
from parity import relerr, normerr

pytestmark = pytest.mark.gpu


# ---- (a) the solve paths ---------------------------------------------------------------------------------------------
DIAG_CASES = [c for c in E.SOLVE_CASES if c[3] == 1] + [(64, 1100, False, 1, "cluster")]   # several tiles per CTA
DENSE_CASES = [c for c in E.SOLVE_CASES if c[3] != 1]


@functools.lru_cache(maxsize=None)
def _masked_case(M, m, dense_R, path, kind):
    inp = E.solve_inputs(M, m, E.case_seed(M, m), dense_R)
    Zp, miss = X.plant(inp["Zp"], kind)
    T, W, condS, ce = X.solve_masked(inp["HX"], Zp, inp["mean"], inp["qs"], inp["R"])
    return dict(inp, Zp=Zp), miss, _f64(T), _f64(W), X.masked_tolerance(condS, ce, path)


@pytest.mark.parametrize("kind", X.MASKS)
@pytest.mark.parametrize("M,m,dense_R,dinv_kind,path", DIAG_CASES)
def test_solve_paths_with_missing_gauges(torch_cuda, fnet, record_property, M, m, dense_R, dinv_kind, path, kind):
    """T and W against the masked reference at its solve tolerance; W exactly 0.0 at the missing gauges."""
    torch = torch_cuda
    net, pos, _ = fnet
    inp, miss, T, W, tol = _masked_case(M, m, dense_R, path, kind)
    run, a = _solve_dev(torch, net, pos, inp, M, dinv_kind)
    names = _kernels(torch, run)
    net.check()
    _expect(names, *_solve_kernels(M, m, dinv_kind, path))
    Td, Wd = a["T"].cpu().numpy(), a["W"].cpu().numpy()
    assert np.isfinite(Td).all() and np.isfinite(Wd).all()
    assert (Wd[miss] == 0.0).all()
    if miss.all():
        assert (Td == 0.0).all()
        return
    eT, eW = normerr(Td, T), normerr(Wd, W)
    record_property("path", path)
    record_property("ratio", max(eT, eW) / tol)
    assert eT <= tol and eW <= tol, f"T error {eT:.2e}, W error {eW:.2e}, bound {tol:.2e}"


@pytest.mark.parametrize("M,m,dense_R,dinv_kind,path", DENSE_CASES)
def test_dense_D_reports_a_missing_gauge_then_clears(torch_cuda, fnet, M, m, dense_R, dinv_kind, path):
    """dinv_kind 2 (dense D^-1) or 0 (none): a NaN row is reported by net.check() with its own message; the next solve
    without NaN on the same handle is right."""
    torch = torch_cuda
    from tx_fast_hydrology_b200._lib import TxhError
    net, pos, _ = fnet
    inp, T, W, tol = E.case_reference(M, m, dense_R, dinv_kind, path)
    Zp, _ = X.plant(inp["Zp"], "one")
    run, _ = _solve_dev(torch, net, pos, dict(inp, Zp=Zp), M, dinv_kind)
    names = _kernels(torch, run)
    _expect(names, *_solve_kernels(M, m, dinv_kind, path))
    with pytest.raises(TxhError, match="missing observation .* non-diagonal observation covariance"):
        net.check()
    run, a = _solve_dev(torch, net, pos, inp, M, dinv_kind)
    run()
    net.check()
    assert normerr(a["T"].cpu().numpy(), _f64(T)) <= tol
    assert normerr(a["W"].cpu().numpy(), _f64(W)) <= tol


def test_member_sharded_solve_with_missing_gauges(torch_cuda, fnet):
    """A member-sharded update emulated on one GPU (test_gpu_enkf_paths.py:test_sharded_apply_on_one_gpu) with a
    masked solve of the whole ensemble: every shard's posterior equals the whole ensemble's, to 1e-12."""
    torch = torch_cuda
    net, pos, fc = fnet
    world, Mloc = 2, 32
    Mtot, m = world * Mloc, 120
    inp, miss, Tr, Wr, tol = _masked_case(Mtot, m, False, "cluster", "edges")
    run, a = _solve_dev(torch, net, pos, inp, Mtot, 1)
    names = _kernels(torch, run)
    net.check()
    _expect(names, ["enkf_small_system_kernel"])
    assert normerr(a["T"].cpu().numpy(), Tr) <= tol and normerr(a["W"].cpu().numpy(), Wr) <= tol
    n, g = net.n, inp["gauges"]
    md = a["mean"]
    qs = _dev(torch, inp["qs"])
    O_all, I_all = _state(torch, net, fc["O"][:, :Mtot], Mtot), _state(torch, net, fc["I"][:, :Mtot], Mtot)
    net.enkf_apply(O_all, I_all, Mtot, None, 0, Mtot, 0, md, a["T"], g, qs, a["W"], torch.empty_like(O_all))
    O_whole, I_whole = net.unpack_host(O_all, Mtot), net.unpack_host(I_all, Mtot)
    assert np.isfinite(O_whole).all()
    X_ = [_state(torch, net, fc["O"][:, r * Mloc:(r + 1) * Mloc], Mloc) for r in range(world)]
    ldx = X_[0].shape[1]
    Xall = torch.stack(X_).contiguous()
    for r in range(world):
        cols = slice(r * Mloc, (r + 1) * Mloc)
        O, I = X_[r].clone(), _state(torch, net, fc["I"][:, cols], Mloc)
        net.enkf_apply(O, I, Mloc, Xall, ldx, Mtot, r * Mloc, md, a["T"], g, qs, a["W"], torch.empty_like(O),
                       x_block_stride=n * ldx)
        net.check()
        assert normerr(net.unpack_host(O, Mloc), O_whole[:, cols]) < 1e-12
        assert normerr(net.unpack_host(I, Mloc), I_whole[:, cols]) < 1e-12


# ---- (b) refusals before any device work ----------------------------------------------------------------------------
def _small_model(torch):
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.muskingum import Muskingum
    n, M, m = 400, 8, 6
    net_d = S.make_network(n, 9)
    d = S.model_dict(net_d, S.make_params(n, 9, well_posed=True))
    mdl = Muskingum(d, members=M)
    mdl._ensure_device()
    g = E.gauge_set(net_d["endnodes"], m, 9)
    t = mdl.datetime
    idx = pd.DatetimeIndex([t + mdl.timedelta * 6, t + mdl.timedelta * 12])
    meas = np.ones((2, m))
    mdf = pd.DataFrame(meas, columns=[d["reach_ids"][j] for j in g], index=idx)
    rng = np.random.default_rng(9)
    B = rng.standard_normal((m, m))
    R_dense = 1e-2 * (np.eye(m) + 0.5 * (B @ B.T) / m)
    return mdl, mdf, R_dense


def _unchanged(torch, mdl, before):
    torch.cuda.synchronize()
    O, I = mdl.device_state
    assert mdl.datetime == before[0]
    assert torch.equal(O, before[1]) and torch.equal(I, before[2])


def test_dense_R_filter_refuses_measurements_with_gaps(torch_cuda):
    """EnsembleKalmanFilter with a non-diagonal R_cov: a frame holding a NaN raises ValueError at construction and on
    assignment, before any device work; a diagonal R_cov takes the same frame."""
    torch = torch_cuda
    from tx_fast_hydrology_b200.da import EnsembleKalmanFilter
    mdl, mdf, R_dense = _small_model(torch)
    before = (mdl.datetime,) + tuple(x.clone() for x in mdl.device_state)
    gap = mdf.copy()
    gap.iloc[1, 2] = np.nan
    with pytest.raises(ValueError, match="missing values"):
        EnsembleKalmanFilter(mdl, gap, 1.0, R_dense)
    _unchanged(torch, mdl, before)
    enkf = EnsembleKalmanFilter(mdl, mdf, 1.0, R_dense)
    with pytest.raises(ValueError, match="missing values"):
        enkf.measurements = gap
    assert not np.isnan(enkf._meas_values).any()
    diag = EnsembleKalmanFilter(mdl, gap, 1.0, 1e-2 * np.eye(mdf.shape[1]))
    Zp = diag.perturbed_observations(gap.index[1])
    assert np.isnan(Zp[2]).all() and np.isfinite(np.delete(Zp, 2, axis=0)).all()
    _unchanged(torch, mdl, before)


@pytest.mark.parametrize("in_library", [True, False])
def test_dense_R_run_assimilating_refuses_nan_observations(torch_cuda, in_library):
    torch = torch_cuda
    from tx_fast_hydrology_b200.da import EnsembleKalmanFilter
    mdl, mdf, R_dense = _small_model(torch)
    enkf = EnsembleKalmanFilter(mdl, mdf, 1.0, R_dense)
    before = (mdl.datetime,) + tuple(x.clone() for x in mdl.device_state)
    obs = torch.ones((2, mdf.shape[1], mdl.members), dtype=torch.float64, device="cuda")
    obs[1, 3, 5] = float("nan")
    f = mdl.make_forcing(times_ns=np.array([float(mdl.datetime.value)]), table=np.zeros((1, mdl.n)))
    with pytest.raises(ValueError, match="missing values"):
        mdl.run_assimilating(f, 12, enkf, 6, obs if in_library else list(obs))
    _unchanged(torch, mdl, before)
    assert enkf.n_updates == 0


# ---- (c) the loops and the smoother ----------------------------------------------------------------------------------
def outage(endnodes, gidx, nwin, seed):
    """Seeded outage pattern [nwin][m] (True: missing) and the one-member NaN: an outlet gauge and a confluence gauge
    down for every update, a quarter of the rest down at random, every gauge missing at update 1, and at the last
    update one otherwise observed gauge with a NaN in its last member only."""
    end = np.asarray(endnodes, dtype=np.int64)
    n, m = end.size, gidx.size
    rng = np.random.default_rng(seed + 977)
    indeg = np.bincount(end[end != np.arange(n)], minlength=n)
    miss = rng.random((nwin, m)) < 0.25
    outlet = np.flatnonzero(end[gidx] == gidx)
    conf = np.flatnonzero(indeg[gidx] >= 2)
    assert outlet.size and conf.size
    miss[:, [outlet[0], conf[0]]] = True
    miss[1] = True
    last = nwin - 1
    free = np.flatnonzero(~miss[last])
    assert free.size >= 2
    one = int(free[0])
    return miss, (last, one)


def _outage_case(n, M, m, seed, every, nwin, rest):
    """A loop case with the outage pattern planted in its observations, and the pattern."""
    c = make_case(n, M, m, seed, every, nwin, rest, gauges="reference")
    miss, (k1, g1) = outage(c["net"]["endnodes"], c["gidx"], nwin, seed)
    for k in range(nwin):
        c["Zp"][k][miss[k]] = np.nan
    c["Zp"][k1, g1, M - 1] = np.nan
    return c, miss


MISSING_LOOP_CASES = [c for c in LOOP_CASES
                      if (c[7] is None and c[1] in (64, 63, 33, 5, 97, 129)) or c[2] == 1100
                      or (c[7] == "lane" and c[1] == 16) or c[7] == "dataflow"]


@pytest.mark.parametrize("n,M,m,seed,every,nwin,rest,kernel,in_library", loop_params(MISSING_LOOP_CASES))
def test_assimilation_loop_with_outages(torch_cuda, oracle, monkeypatch, record_property, n, M, m, seed, every, nwin,
                                        rest, kernel, in_library):
    """Hydrographs, priors and final state of an outage run against the masked extended-precision loop, at the
    tolerance and error scale of test_gpu_enkf_paths.py; at the update with every gauge missing the recorded posterior
    equals the prior element-wise.  (Without the masking the run comes out all NaN.)"""
    c, miss = _outage_case(n, M, m, seed, every, nwin, rest)
    d = run_device(c, in_library, monkeypatch=monkeypatch, kernel=kernel)
    r = reference_loop(oracle, c, update_masked)
    _expect(d["names"], _loop_kernels(M, m, kernel, in_library))
    rec, prior = d["res"]
    assert not np.isnan(rec).any() and not np.isnan(prior).any()
    e_pri, e_rec = relerr(prior, r["pri"], scale=r["sc_pri"]), relerr(rec, r["hyd"], scale=r["sc"])
    record_property("rec_ratio", e_rec / r["tol"])
    assert e_pri < r["tol"], f"priors: {e_pri:.2e}, bound {r['tol']:.2e}"
    assert e_rec < r["tol"], f"hydrographs: {e_rec:.2e}, bound {r['tol']:.2e}"
    nsteps = every * nwin + rest
    assert relerr(d["final"], r["hyd"][nsteps - 1], scale=r["sc"][nsteps - 1]) < r["tol"]
    assert miss[1].all()
    assert np.array_equal(rec[2 * every - 1], prior[1]), "the update with every gauge missing changed the state"


@pytest.mark.parametrize("in_library", [True, False])
def test_smoother_on_an_outage_run(torch_cuda, oracle, monkeypatch, in_library):
    """smooth_lag on an outage run: the smoothed hydrographs equal enks_oracle.smooth_transforms applied to the
    reference hydrographs with the masked reference transforms."""
    n, M, m, seed, every, nwin, rest = 2500, 64, 120, 81, 6, 3, 0
    lag = every + 2
    c, _ = _outage_case(n, M, m, seed, every, nwin, rest)
    rec, prior, sm = run_device(c, in_library, monkeypatch=monkeypatch, lag=lag)["res"]
    r = reference_loop(oracle, c, update_masked)
    want = smooth_transforms(r["hyd"], np.stack(r["kept"]), nwin, every, 1, lag)
    sc = np.maximum(np.maximum(np.abs(want), r["sc"]), np.abs(rec))
    assert not np.isnan(sm).any()
    assert relerr(sm, want, scale=sc) < r["tol"] * (nwin + 1)

"""The dense Kalman filter, the RTS smoother, the batched filters of a generation of sub-models and the dense kernels
under them (Gauss-Jordan inverse, DMMA GEMM) against the extended-precision reference of tests/kf_reference.py.

Every bound comes from a condition number or is an exact identity, and every case prints its measured error next to
its bound.  Each group checks with torch.profiler that the kernels it targets ran."""
import asyncio
import json
import os
import tempfile

import numpy as np
import pandas as pd
import pytest

import kf_reference as R
from parity import relerr, normerr

pytestmark = pytest.mark.gpu
EPS = R.EPS64


@pytest.fixture(scope="module", autouse=True)
def _cuda(libtxh):
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (no CPU fallback exists)"


def _kernels(fn):
    """Run `fn` under the profiler; [(kernel name, trace args)] of the CUDA kernels it launched."""
    import torch
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    return [(e["name"], e.get("args", {})) for e in events if e.get("cat") == "kernel"]


def _expect(kernels, *names):
    ran = " ".join(k for k, _ in kernels)
    for name in names:
        assert name in ran, f"{name} did not run (kernels: {sorted(set(k for k, _ in kernels))[:30]})"


def _report(what, err, bound):
    print(f"{what}: error {err:.3e}  bound {bound:.3e}  ratio {err / bound:.3e}")
    assert err <= bound, f"{what}: error {err:.3e} exceeds its bound {bound:.3e}"


def _dev(a):
    import torch
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device="cuda")


def _f64(x):
    return np.asarray(x, dtype=np.float64)


# ---- inverse_smem_kernel ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("m", R.INVERSE_SIZES)
def test_inverse(m):
    """txh_inverse at sizes on both sides of the shared / global memory switch (158 | 159) and past one element per
    thread (1025), on inputs that pivot: a permutation is inverted exactly, the others within m eps cond(A) of the
    longdouble inverse (FP64 residuals A X - I and X A - I past 400)."""
    from tx_fast_hydrology_b200.network import inverse
    in_smem = (4 * m + m * m) * 8 <= 200 * 1024
    for kind in R.INVERSE_KINDS:
        if m == 1 and kind == "zero_leading_diagonal":
            continue
        A = R.inverse_input(kind, m)
        Ad = _dev(A)
        kernels = _kernels(lambda: inverse(Ad))
        _expect(kernels, "inverse_smem_kernel")
        smem = [a.get("shared memory") for k, a in kernels if "inverse_smem_kernel" in k]
        assert smem and smem[0] is not None, "the trace does not record the kernel's shared memory"
        assert (smem[0] >= (4 * m + m * m) * 8) if in_smem else (smem[0] < (4 * m + m * m) * 8), (m, smem[0])
        X = Ad.cpu().numpy()
        if kind == "permutation":
            assert (X == A.T).all(), "the inverse of a permutation is its transpose, exactly"
            continue
        cond = np.linalg.cond(A)
        tol = R.inverse_tolerance(m, cond)
        if m <= R.LD_INVERSE_MAX:
            Xr, piv = R.inverse_ref(A)
            if kind in ("permuted_dominant", "spd_1e8") and m > 1:
                assert (piv != np.arange(m)).any(), "the case was meant to pivot"
            _report(f"inverse m={m} {kind} cond={cond:.1e} vs longdouble", normerr(X, _f64(Xr)), tol)
        res = max(np.abs(A @ X - np.eye(m)).max(), np.abs(X @ A - np.eye(m)).max())
        _report(f"inverse m={m} {kind} cond={cond:.1e} residual", res, tol)


def test_singular_inverse_is_reported_and_the_next_call_is_right():
    from tx_fast_hydrology_b200._lib import TxhError
    from tx_fast_hydrology_b200.network import inverse
    for m in (5, 200):
        with pytest.raises(TxhError):
            inverse(_dev(np.zeros((m, m))))
        A = R.inverse_input("permuted_dominant", m)
        Ad = _dev(A)
        inverse(Ad)
        _report(f"inverse m={m} after a singular one", normerr(Ad.cpu().numpy(), _f64(R.inverse_ref(A)[0])),
                R.inverse_tolerance(m, np.linalg.cond(A)))


# ---- dgemm_kernel -----------------------------------------------------------------------------------------------
GEMM_SHAPES = [(1, 1, 1), (15, 17, 63), (17, 15, 65), (63, 65, 129), (65, 129, 17), (129, 63, 15), (65, 65, 0),
               (1, 129, 65), (129, 1, 17), (64, 64, 16)]


@pytest.mark.parametrize("ta,tb", [(False, False), (True, False), (False, True), (True, True)])
def test_dgemm(ta, tb):
    """C = alpha op(A) op(B) + beta C against longdouble, element-wise within 2 (K + 2) eps (|alpha| |A| |B| +
    |beta| |C|), at sizes off the 64 x 64 x 16 tiles, K = 0, alpha = 0, beta = 0 over a C full of NaN, and row slices
    of wider matrices (leading dimension > row); the columns beyond a sliced C stay untouched."""
    import torch
    from tx_fast_hydrology_b200.network import dgemm
    rng = np.random.default_rng(11 + 2 * ta + tb)
    worst = 0.0
    for (M, N, K) in GEMM_SHAPES:
        for alpha, beta, sliced in ((1.0, 0.0, False), (-0.7, 1.3, True), (0.0, 2.0, False), (1.5, 0.0, True)):
            A = rng.standard_normal((K, M) if ta else (M, K))
            B = rng.standard_normal((N, K) if tb else (K, N))
            C0 = rng.standard_normal((M, N))
            pad = 3 if sliced or K == 0 else 0           # an empty operand still needs an address
            Ab, Bb, Cb = (np.full((x.shape[0], x.shape[1] + pad), 7.0) for x in (A, B, C0))
            Ab[:, :A.shape[1]], Bb[:, :B.shape[1]], Cb[:, :N] = A, B, C0
            if beta == 0.0:
                Cb[:, :N] = np.nan                      # beta = 0: C is not read
            Ad, Bd, Cd = _dev(Ab), _dev(Bb), _dev(Cb)
            Av, Bv, Cv = Ad[:, :A.shape[1]], Bd[:, :B.shape[1]], Cd[:, :N]
            kernels = _kernels(lambda: dgemm(Av, Bv, Cv, ta, tb, alpha, beta))
            if M and N:
                _expect(kernels, "dgemm_kernel")
            out = Cd.cpu().numpy()
            if sliced:
                assert (out[:, N:] == 7.0).all(), "dgemm wrote past the columns of a sliced C"
            opA = np.asarray(A.T if ta else A, dtype=R.LD)
            opB = np.asarray(B.T if tb else B, dtype=R.LD)
            c_in = np.zeros((M, N)) if beta == 0.0 else C0
            ref = R.LD(alpha) * (opA @ opB) + R.LD(beta) * np.asarray(c_in, dtype=R.LD)
            scale = abs(alpha) * (np.abs(opA) @ np.abs(opB)) + abs(beta) * np.abs(np.asarray(c_in, dtype=R.LD))
            bound = 2 * (K + 2) * EPS * _f64(scale) + 1e-300
            err = np.abs(out[:, :N] - _f64(ref))
            assert np.isfinite(out[:, :N]).all()
            assert (err <= bound).all(), f"M={M} N={N} K={K} alpha={alpha} beta={beta}: {(err / bound).max():.2e}"
            worst = max(worst, float((err / bound).max()) if err.size else 0.0)
    print(f"dgemm transA={ta} transB={tb}: worst element-wise error / bound {worst:.3e}")


def test_dense_kernels_refuse_bad_matrices():
    """Device tensors of the wrong shape, a transposed view, a non-float64 tensor: ValueError before the C ABI."""
    import torch
    from tx_fast_hydrology_b200.network import dgemm, inverse, spd_solve
    A, B, C = _dev(np.ones((4, 3))), _dev(np.ones((3, 5))), _dev(np.ones((4, 5)))
    for call in (lambda: inverse(_dev(np.ones((4, 3)))), lambda: inverse(_dev(np.eye(4)).t()),
                 lambda: inverse(_dev(np.eye(4)).float()),
                 lambda: spd_solve(_dev(np.eye(4)), _dev(np.ones((3, 2)))),
                 lambda: dgemm(A, B, _dev(np.ones((4, 4)))), lambda: dgemm(A, _dev(np.ones((2, 5))), C),
                 lambda: dgemm(_dev(np.ones((3, 4))).t(), B, C), lambda: dgemm(A, B, C, transA=True)):
        with pytest.raises(ValueError):
            call()
    dgemm(A, B, C)
    assert (C.cpu().numpy() == 3.0).all()


# ---- dense filter: txh_kf_filter through KalmanFilter -----------------------------------------------------------
def _model(net, prm, name="kf", prefix=""):
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.muskingum import Muskingum
    d = S.model_dict(net, prm, dt_s=R.DT_S, name=name)
    d["reach_ids"] = [f"{prefix}{r}" for r in d["reach_ids"]]
    return Muskingum(d)


def _frame(times_ns, values, cols):
    idx = pd.DatetimeIndex(pd.to_datetime(np.asarray(times_ns, dtype=np.int64), unit="ns", utc=True)).as_unit("ns")
    return pd.DataFrame(values, index=idx, columns=cols)


def _check_update(tag, kf, mdl, r, o_pr, i_pr, indeg_max):
    condS = np.linalg.cond(_f64(r["S"]))
    tol = R.kf_tolerance(condS)
    gmax = float(np.abs(_f64(r["gain"])).max())
    _report(f"{tag} cond(S)={condS:.1e} K", normerr(kf.K, _f64(r["K"])), tol)
    _report(f"{tag} gain", normerr(kf.gain, _f64(r["gain"])), tol)
    # P+ = P- - K P-[s] can cancel to ~1e-8 of P- (cond(S) ~ 1e9): its error is measured against the terms it is
    # summed from; the FP64 oracle misses a bound relative to |P+| just as the device does
    _report(f"{tag} P", float(np.abs(kf.P_t_next - _f64(r["P"])).max()) / float(np.abs(_f64(r["Pm"])).max()), tol)
    _report(f"{tag} dz", float(np.abs(kf.dz - _f64(r["dz"])).max()) / max(1e-300, float(np.abs(_f64(r["dz"])).max())
                                                                             + float(np.abs(o_pr).max())), tol)
    _report(f"{tag} o", relerr(mdl.o_t_next, _f64(r["o"]), scale=np.abs(o_pr) + gmax), tol)
    _report(f"{tag} i", relerr(mdl.i_t_next, _f64(r["i"]), scale=np.abs(i_pr) + indeg_max * gmax), tol)


@pytest.mark.parametrize("case", R.FILTER_CASES, ids=[c["id"] for c in R.FILTER_CASES])
def test_dense_filter(case):
    """KalmanFilter.filter at the start and after each of FILTER_STEPS routing steps, every update against
    kf_update_ref from the same prior (P, o, i read back from the device): K, gain, P+ and dz in the max-norm within
    64 eps cond(S), o and i element-wise relative to what they were summed from.  The measurement columns arrive
    unsorted."""
    from tx_fast_hydrology_b200.da import KalmanFilter
    c = R.filter_case(case)
    end, g, m = c["net"]["endnodes"], c["gauges"], case["m"]
    mdl = _model(c["net"], c["prm"])
    perm = np.random.default_rng(case["n"]).permutation(m)
    times = R.T0_NS + np.arange(R.FILTER_STEPS + 1, dtype=np.int64) * int(R.DT_S * 1e9)
    mdf = _frame(times, c["z"][:, perm], [mdl.reach_ids[j] for j in g[perm]])
    kf = KalmanFilter(mdl, mdf, c["Q"], c["R"][np.ix_(perm, perm)], c["P0"])
    assert (kf.reach_indices == g).all()
    indeg_max = max(1, int(np.bincount(end[end != np.arange(end.size)], minlength=end.size).max()))
    for k in range(R.FILTER_STEPS + 1):
        if k:
            mdl.step(c["q"][k - 1])
        P, o_pr, i_pr = kf.P_t_next, mdl.o_t_next.copy(), mdl.i_t_next.copy()
        kernels = _kernels(kf.filter)
        mdl.network.check()
        _expect(kernels, "inverse_smem_kernel", "dgemm_kernel", "kf_prior_finish_kernel", "kf_gain_kernel")
        r = R.kf_update_ref(P, c["Q"], c["R"], g, c["z"][k], o_pr, i_pr, end, mdl.alpha, mdl.beta, mdl.chi)
        _check_update(f"filter {case['id']} step {k}", kf, mdl, r, o_pr, i_pr, indeg_max)


def test_singular_innovation_covariance_is_reported_and_the_next_update_is_right():
    """P0 = Q = R = 0 makes S = 0: check() reports it; a filter with proper covariances on the same network handle
    then updates correctly."""
    from tx_fast_hydrology_b200._lib import TxhError
    from tx_fast_hydrology_b200.da import KalmanFilter
    case = R.FILTER_CASES[1]
    c = R.filter_case(case)
    end, g = c["net"]["endnodes"], c["gauges"]
    n, m = end.size, g.size
    mdl = _model(c["net"], c["prm"])
    mdf = _frame([R.T0_NS], c["z"][:1], [mdl.reach_ids[j] for j in g])
    zero = KalmanFilter(mdl, mdf, np.zeros((n, n)), np.zeros((m, m)), np.zeros((n, n)))
    zero.filter()
    with pytest.raises(TxhError):
        mdl.network.check()
    mdl.network.check()                                            # reported once
    kf = KalmanFilter(mdl, mdf, c["Q"], c["R"], c["P0"])
    o_pr, i_pr = mdl.o_t_next.copy(), mdl.i_t_next.copy()
    kf.filter()
    mdl.network.check()
    r = R.kf_update_ref(c["P0"], c["Q"], c["R"], g, c["z"][0], o_pr, i_pr, end, mdl.alpha, mdl.beta, mdl.chi)
    _check_update("filter after a singular S", kf, mdl, r, o_pr, i_pr, 4)


# ---- KalmanSmoother ---------------------------------------------------------------------------------------------
SMOOTH_STEPS = 4


@pytest.mark.parametrize("n", [60, 158, 159, 300])
def test_smoother(n):
    """KalmanSmoother (forward filter at exact measurement times, backward pass on the device) against rts_ref run on
    the forward quantities the smoother stored.  Q has eigenvalues from 1 down to 1e-6, which leaves cond(P_p) above
    1e4 (about 3e4 on these networks).
    Bound: each of the N backward steps inverts P_p (n eps cond(P_p), as the inverse) and carries the error of the
    step after it, so N n eps max cond(P_p)."""
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.da import KalmanSmoother
    seed = 40 + n
    net = S.make_network(n, seed, n_basins=2)
    prm = S.make_params(n, seed, well_posed=True)
    end = net["endnodes"]
    g = R.special_gauges(end, max(2, n // 10), seed)
    rng = np.random.default_rng(seed)
    U, _ = np.linalg.qr(rng.standard_normal((n, n)))
    Q = (U * np.logspace(0, -6, n)) @ U.T
    Q = (Q + Q.T) / 2
    mdl = _model(net, prm)
    times = R.T0_NS + np.arange(SMOOTH_STEPS + 1, dtype=np.int64) * int(R.DT_S * 1e9)
    mdf = _frame(times, prm["o_t"][g][None, :] * rng.uniform(0.8, 1.2, size=(times.size, g.size)),
                 [mdl.reach_ids[j] for j in g])
    ks = KalmanSmoother(mdl, mdf, Q, 1e-2 * np.eye(g.size), Q.copy())
    mdl.bind_callback(ks, key="ks")
    df = _frame(times[[0, -1]], np.tile(rng.uniform(0, 1, n), (2, 1)), mdl.reach_ids)
    kernels = _kernels(lambda: [None for _ in mdl.simulate(df)])
    _expect(kernels, "inverse_smem_kernel", "dgemm_kernel")
    ts = ks.datetimes
    host = lambda d: {t: (v.cpu().numpy() if hasattr(v, "cpu") else v) for t, v in d.items()}
    P_f, P_p = host(ks.P_f), host(ks.P_p)
    x_f = {t: np.stack([ks.i_hat_f[t], ks.o_hat_f[t]], axis=1) for t in ks.i_hat_f}
    x_p = {t: np.stack([ks.i_hat_p[t], ks.o_hat_p[t]], axis=1) for t in ks.i_hat_p}
    x_s, P_s = R.rts_ref(ts, P_f, P_p, x_f, x_p, end, mdl.alpha, mdl.beta, mdl.chi)
    cond = max(np.linalg.cond(P_p[t]) for t in ts[1:])
    assert cond > 1e4, f"cond(P_p) = {cond:.1e}: the case was meant to be ill-conditioned"
    tol = max(1e-12, (len(ts) - 1) * n * EPS * cond)
    t_all = sorted(x_s)
    _report(f"smoother n={n} max cond(P_p)={cond:.1e} o_hat_s",
            normerr(ks.o_hat_s.loc[t_all].values, np.stack([_f64(x_s[t][:, 1]) for t in t_all])), tol)
    _report(f"smoother n={n} i_hat_s",
            normerr(ks.i_hat_s.loc[t_all].values, np.stack([_f64(x_s[t][:, 0]) for t in t_all])), tol)
    _report(f"smoother n={n} P_s", max(normerr(ks.P_s[t].cpu().numpy(), _f64(P_s[t])) for t in t_all), tol)


# ---- batched filters: txh_kfb_* ---------------------------------------------------------------------------------
def _batch_models(blocks, gauges=None):
    """Fresh sub-models (reach ids prefixed per block), a KalmanFilter bound to each, one forcing frame.  `gauges`:
    {block: number of gauges} in place of the blocks' own."""
    from tx_fast_hydrology_b200.da import KalmanFilter
    models, filters, cols, q = [], [], [], []
    for k in blocks:
        c = R.batch_block(k, (gauges or {}).get(k))
        stop = R.BATCH_BLOCKS[k]["stop"]
        mdl = _model(c["net"], c["prm"], name=f"b{k}", prefix=f"b{k}:")
        times = R.T0_NS + np.arange(stop + 1, dtype=np.int64) * int(R.DT_S * 1e9)
        kf = KalmanFilter(mdl, _frame(times, c["z"], [mdl.reach_ids[j] for j in c["gauges"]]), c["Q"], c["R"],
                          c["P0"])
        mdl.bind_callback(kf, key="kf")
        models.append(mdl); filters.append(kf); cols += mdl.reach_ids; q.append(c["q"])
    ends = R.T0_NS + np.array([0, R.BATCH_STEPS], dtype=np.int64) * int(R.DT_S * 1e9)
    return models, filters, _frame(ends, np.tile(np.concatenate(q), (2, 1)), cols)


def _run_collection(blocks, batched):
    from tx_fast_hydrology_b200.muskingum import ModelCollection
    from tx_fast_hydrology_b200.simulation import AsyncSimulation
    models, filters, df = _batch_models(blocks)
    sim = AsyncSimulation(ModelCollection(models), df)
    sim.batch_filters = batched
    holder = {}
    kernels = _kernels(lambda: holder.update(out=asyncio.run(sim.simulate())))
    return models, filters, holder["out"], kernels


def test_batched_filters_that_stop_at_different_times():
    """A generation of sub-models whose measurement tables end at different steps (blocks of 1 reach, every reach
    gauged, 158 gauges, ...): the batched chain leaves every filter as the per-model path does -- P_t_next,
    P_t_prev, K, dz and gain of its LAST update, also for the filters that stopped early -- and the hydrographs and
    final states agree.  P_t_next and K are also checked against kf_update_ref from the per-model P_t_prev."""
    blocks = list(range(len(R.BATCH_BLOCKS)))
    mb, fb, outb, kb = _run_collection(blocks, True)
    mp, fp, outp, _ = _run_collection(blocks, False)
    _expect(kb, "kfb_inverse_kernel", "kfb_gain_kernel", "kfb_post_kernel")
    for k, (a, b, ma, mp_) in enumerate(zip(fb, fp, mb, mp)):
        c = R.batch_block(k)
        end, g = c["net"]["endnodes"], c["gauges"]
        Pm = R.aqat_ref(b.P_t_prev, end, mp_.alpha, mp_.beta, mp_.chi) + np.asarray(c["Q"], dtype=R.LD)
        condS = np.linalg.cond(_f64(Pm[np.ix_(g, g)]) + c["R"])
        tol = R.kf_tolerance(condS)
        tag = f"batched block {k} (n={end.size} m={g.size} stop={R.BATCH_BLOCKS[k]['stop']})"
        assert a.K is not None and a.gain is not None and a.dz is not None, f"{tag}: K / dz / gain missing"
        for name in ("P_t_next", "P_t_prev", "K", "dz", "gain"):
            _report(f"{tag} {name} vs per-model", normerr(getattr(a, name), getattr(b, name)), tol)
        Sinv = R.inverse_ref(Pm[np.ix_(g, g)] + np.asarray(c["R"], dtype=R.LD))[0]
        Kr = Pm[:, g] @ Sinv
        _report(f"{tag} K vs longdouble", normerr(a.K, _f64(Kr)), tol)
        _report(f"{tag} P_t_next vs longdouble", normerr(a.P_t_next, _f64(Pm - Kr @ Pm[g])), tol)
        _report(f"{tag} hydrographs", relerr(outb[ma.name].values, outp[mp_.name].values), max(1e-9, tol))
        _report(f"{tag} o", relerr(ma.o_t_next, mp_.o_t_next), max(1e-9, tol))
        _report(f"{tag} i", relerr(ma.i_t_next, mp_.i_t_next), max(1e-9, tol))
        assert ma.datetime == mp_.datetime and a.datetime == b.datetime


def test_batched_block_gauge_limit():
    """The library reports how many gauges a batched block may have and refuses one more; a generation with a
    sub-model over the limit still runs (that sub-model on the per-model path) and matches the per-model run."""
    from tx_fast_hydrology_b200 import _lib
    from tx_fast_hydrology_b200._lib import TxhError
    from tx_fast_hydrology_b200.da import BatchedKalmanFilters
    from tx_fast_hydrology_b200.muskingum import ModelCollection
    from tx_fast_hydrology_b200.simulation import AsyncSimulation
    limit = _lib.load().txh_kfb_max_gauges()
    assert limit == 158 and (4 * limit + limit ** 2) * 8 <= 200 * 1024 < (4 * (limit + 1) + (limit + 1) ** 2) * 8
    over = {2: limit + 1}
    models, _, _ = _batch_models([2, 1], over)
    with pytest.raises(TxhError):
        BatchedKalmanFilters(models)
    out = {}
    for batched in (True, False):
        models, filters, df = _batch_models([2, 1, 3], over)
        sim = AsyncSimulation(ModelCollection(models), df)
        sim.batch_filters = batched
        out[batched] = (asyncio.run(sim.simulate()), models, filters)
    (ob, mb, fb), (op, mp, fp) = out[True], out[False]
    for a, b in zip(mb, mp):
        _report(f"gauge-limit generation {a.name} hydrographs", relerr(ob[a.name].values, op[b.name].values), 1e-9)
    for a, b in zip(fb, fp):
        _report(f"gauge-limit generation P_t_next", normerr(a.P_t_next, b.P_t_next), 1e-9)

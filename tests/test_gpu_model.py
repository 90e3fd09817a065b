"""GPU parity tests of the Python drop-in layer (Muskingum, callbacks, KalmanFilter, nutils names,
EnsembleKalmanFilter) against the golden vectors of the unmodified reference and the CPU oracle.
Tolerance: FP64 max relative error <= 1e-9 (BASELINE.json north_star)."""
import os

import numpy as np
import pandas as pd
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
RTOL = 1e-9
# Dense filter / smoother quantities are held to the same 1e-9 as the states.  Measured on B200 against the
# reference goldens (tests/perf/kf_error_budget.py, profiles/r02_kf_error_budget.json): gains 6e-16, P 2.4e-16,
# K 4.4e-16, smoothed states 8e-16, smoothed covariance 7e-16 (max-norm); cond(P[s][:,s] + R) = 3.7 and
# cond(P_p) <= 12.3 in these fixtures, so nothing here needs a looser bound.
GAIN_TOL = RTOL
SMOOTH_X_TOL = RTOL
SMOOTH_P_TOL = RTOL


from assim_case import make_case, model, oracle_start
from parity import relerr, normerr, enkf_tolerance        # element-wise with a floor / max-norm (dense matrices)


def frame(times_ns, table, cols):
    idx = pd.DatetimeIndex(pd.to_datetime(times_ns, unit="ns", utc=True)).as_unit("ns")
    return pd.DataFrame(table, index=idx, columns=cols)


def model_from(g, **kw):
    from tx_fast_hydrology_b200.muskingum import Muskingum
    n = g["endnodes"].size
    d = {"name": "golden", "datetime": pd.Timestamp(int(g["t0_ns"]), tz="UTC"),
         "timedelta": pd.to_timedelta(float(g["dt"]), unit="s"), "reach_ids": [str(i) for i in range(n)],
         "startnodes": np.arange(n, dtype=np.int64), "endnodes": g["endnodes"].astype(np.int64),
         "K": g["K"].astype(np.float64), "X": g["X"].astype(np.float64), "o_t": g["o_init"].astype(np.float64)}
    return Muskingum(d, **kw), d


@pytest.fixture(scope="module", autouse=True)
def _cuda(libtxh):
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (no CPU fallback exists)"


def test_simulate_matches_reference_c1(golden_dir):
    """Muskingum.simulate (generator, callbacks hooks, per-step launches) on BASELINE configs[0]."""
    g = np.load(os.path.join(golden_dir, "model_c1.npz"))
    mdl, d = model_from(g)
    df = frame(g["times"], g["table"], d["reach_ids"])
    keep = set(int(k) for k in g["keep"])
    O, I = [], []
    total = np.zeros(mdl.n)
    for k, state in enumerate(mdl.simulate(df)):
        total += state.o_t_next
        if k in keep:
            O.append(state.o_t_next.copy()); I.append(state.i_t_next.copy())
    assert k == 287 and mdl.datetime.value == int(g["final_time_ns"])
    assert relerr(np.stack(O), g["O"]) < RTOL and relerr(np.stack(I), g["I"]) < RTOL
    assert relerr(total, g["o_sum"]) < RTOL
    # o_t_prev / i_t_prev hold the state before the last step (muskingum.py:458-461)
    assert relerr(mdl.o_t_prev + 0 * total, mdl.o_t_prev) == 0.0


def test_run_fast_path_equals_simulate(golden_dir):
    g = np.load(os.path.join(golden_dir, "model_c1.npz"))
    mdl, d = model_from(g)
    f = mdl.make_forcing(times_ns=g["times"], table=g["table"])
    rec = mdl.run(f, 288, record_reaches=np.arange(mdl.n), record_every=1)
    traj = rec.cpu().numpy()[:, :, 0]
    assert relerr(traj[g["keep"]], g["O"]) < RTOL and relerr(traj.sum(axis=0), g["o_sum"]) < RTOL
    assert relerr(mdl.o_t_next, g["O"][-1]) < RTOL and relerr(mdl.i_t_next, g["I"][-1]) < RTOL
    assert mdl.datetime.value == int(g["final_time_ns"])


def test_kalman_filter_matches_reference(golden_dir):
    """KalmanFilter bound as a callback (da.py:14-136): unsorted gauge columns, dense R, filter at
    simulation start and after every step while measurements last."""
    from tx_fast_hydrology_b200.da import KalmanFilter
    g = np.load(os.path.join(golden_dir, "kalman_n120.npz"))
    mdl, d = model_from(g)
    df = frame(g["times"], g["table"], d["reach_ids"])
    mdf = frame(g["meas_times"], g["meas"], [d["reach_ids"][j] for j in g["gauge_cols"]])
    kf = KalmanFilter(mdl, mdf, g["Q"], g["R"], g["P0"])
    assert (kf.reach_indices == g["sorted_idx"]).all()
    mdl.bind_callback(kf, key="kf")
    O, I, Pd, gains = [], [], [], []
    for state in mdl.simulate(df):
        O.append(state.o_t_next.copy()); I.append(state.i_t_next.copy())
        Pd.append(np.diag(kf.P_t_next).copy()); gains.append(kf.gain.copy())
    assert relerr(np.stack(O), g["O"]) < RTOL and relerr(np.stack(I), g["I"]) < RTOL
    assert normerr(np.stack(Pd), g["P_diag"]) < RTOL
    assert normerr(np.stack(gains), g["gains"]) < GAIN_TOL
    assert normerr(kf.P_t_next, g["P_final"]) < RTOL and normerr(kf.K, g["K_final"]) < RTOL


def test_kalman_smoother_matches_reference(golden_dir):
    """KalmanSmoother (da.py:139-264): forward filter at exact measurement times + RTS backward pass."""
    from tx_fast_hydrology_b200.da import KalmanSmoother
    g = np.load(os.path.join(golden_dir, "smoother_n60.npz"))
    mdl, d = model_from(g)
    df = frame(g["times"], g["table"], d["reach_ids"])
    mdf = frame(g["meas_times"], g["meas"], [d["reach_ids"][j] for j in g["gauge_idx"]])
    ks = KalmanSmoother(mdl, mdf, g["Q"], g["R"], g["P0"])
    mdl.bind_callback(ks, key="ks")
    for _ in mdl.simulate(df):
        pass
    assert len(ks.datetimes) == int(g["n_times"])
    assert relerr(mdl.o_t_next, g["o_final"]) < RTOL and relerr(mdl.i_t_next, g["i_final"]) < RTOL
    ts = sorted(ks.o_hat_s.index)
    assert [pd.Timestamp(t).value for t in ts] == [int(x) for x in g["smooth_times"]]
    assert normerr(ks.o_hat_s.loc[ts].values, g["o_hat_s"]) < SMOOTH_X_TOL
    assert normerr(ks.i_hat_s.loc[ts].values, g["i_hat_s"]) < SMOOTH_X_TOL
    assert normerr(ks.P_f[ts[-1]].cpu().numpy(), g["P_f_last"]) < RTOL
    assert normerr(ks.P_s[ts[0]].cpu().numpy(), g["P_s_first"]) < SMOOTH_P_TOL


def test_checkpoint_rewind(golden_dir):
    """CheckPoint + save_state / load_state (simulation.py:169-211, muskingum.py:573-588)."""
    from tx_fast_hydrology_b200.simulation import CheckPoint
    g = np.load(os.path.join(golden_dir, "checkpoint_n80.npz"))
    mdl, d = model_from(g)
    df = frame(g["times"], g["table"], d["reach_ids"])
    mdl.bind_callback(CheckPoint(mdl, timedelta=3600), key="checkpoint")
    for _ in mdl.simulate(df):
        pass
    assert relerr(mdl.o_t_next, g["o_end"]) < RTOL and mdl.datetime.value == int(g["t_end"])
    assert relerr(mdl.saved_states["o_t_next"], g["saved_o"]) < RTOL
    assert relerr(mdl.saved_states["i_t_next"], g["saved_i"]) < RTOL
    assert mdl.saved_states["datetime"].value == int(g["saved_t"])
    mdl.load_state()
    assert relerr(mdl.o_t_next, g["o_loaded"]) < RTOL and mdl.datetime.value == int(g["t_loaded"])
    for _ in mdl.simulate(df):
        pass
    assert relerr(mdl.o_t_next, g["o_end2"]) < RTOL and mdl.datetime.value == int(g["t_end2"])
    assert mdl.saved_states["datetime"].value == int(g["saved_t2"])


def test_transmissive_boundary_and_variable_timestep(golden_dir):
    """User-mutated coefficients (set_transmissive_boundary, muskingum.py:567-571) reach the device copies in the
    middle of a run, and step(p, timedelta=dt2) followed by default steps keeps the dt2 coefficients
    (muskingum.py:447-449; SURVEY.md A.5) -- both against the unmodified reference."""
    g = np.load(os.path.join(golden_dir, "quirks_n90.npz"))
    q = g["q"]
    mdl, d = model_from(g)
    for s in range(5):
        mdl.step(q[s])
    assert relerr(mdl.o_t_next, g["o_a5"]) < RTOL and relerr(mdl.i_t_next, g["i_a5"]) < RTOL
    mdl.set_transmissive_boundary(g["tb"])
    for s in range(5, 10):
        mdl.step(q[s])
    assert (np.stack([mdl.alpha, mdl.beta, mdl.chi, mdl.gamma]) == g["coef_a"]).all()
    assert relerr(mdl.o_t_next, g["o_a10"]) < RTOL and relerr(mdl.i_t_next, g["i_a10"]) < RTOL
    # a pass-through reach hands its inflow on unchanged
    assert relerr(mdl.o_t_next[g["tb"]], mdl.i_t_next[g["tb"]]) < 1e-15
    # the device fast path sees the mutated coefficients too: 3 more steps through run() == 3 step() calls
    twin = mdl.copy()
    for s in range(10, 13):
        mdl.step(q[s])
    times = int(g["t0_ns"]) + np.arange(11, 14, dtype=np.int64) * int(300e9)      # sampled at the END of a step
    f = twin.make_forcing(times_ns=times, table=np.ascontiguousarray(q[10:13]))
    twin.run(f, 3)
    assert relerr(twin.o_t_next, mdl.o_t_next) < 1e-13 and twin.datetime == mdl.datetime

    mdl, d = model_from(g)
    mdl.step(q[0])
    mdl.step(q[1], timedelta=pd.to_timedelta(600, unit="s"))
    assert mdl.datetime.value == int(g["t_b2"]) and relerr(mdl.o_t_next, g["o_b2"]) < RTOL
    assert (np.stack([mdl.alpha, mdl.beta, mdl.chi, mdl.gamma]) == g["coef_b2"]).all()
    mdl.step(q[2]); mdl.step(q[3])
    assert mdl.datetime.value == int(g["t_b4"])
    assert (np.stack([mdl.alpha, mdl.beta, mdl.chi, mdl.gamma]) == g["coef_b4"]).all()
    assert relerr(mdl.o_t_next, g["o_b4"]) < RTOL and relerr(mdl.i_t_next, g["i_b4"]) < RTOL


def test_checkpoint_with_kalman_filter_and_new_measurements(golden_dir):
    """The service loop of app/app.py:56-80,125-141 against the unmodified reference: 'checkpoint' bound before
    'kf' (SURVEY.md A.7), a run, load_state -- model state, clock AND the filter's covariance rewind through
    CheckPoint's fan-out (simulation.py:196-206, da.py:83-89) -- then the measurement table is REASSIGNED
    (app.py:75-80) and the next cycle must assimilate the new frame, not the one the filter was built with."""
    from tx_fast_hydrology_b200.da import KalmanFilter
    from tx_fast_hydrology_b200.simulation import CheckPoint
    g = np.load(os.path.join(golden_dir, "checkpoint_kf_n70.npz"))
    mdl, d = model_from(g)
    cols = d["reach_ids"]
    T, t0 = int(g["T"]), int(g["t0_ns"])
    times, table = g["times"], g["table"]
    sel = times <= t0 + T * int(300e9)
    df1 = frame(times[sel], table[sel], cols)
    gcols = g["gauge_cols"]
    mdf1 = frame(g["meas_times1"], g["meas1"], [cols[j] for j in gcols])
    mdl.bind_callback(CheckPoint(mdl, timedelta=3600), key="checkpoint")
    kf = KalmanFilter(mdl, mdf1, g["Q"], g["R"], g["P0"])
    mdl.bind_callback(kf, key="kf")
    for _ in mdl.simulate(df1):
        pass
    assert mdl.datetime.value == int(g["t_end"]) and relerr(mdl.o_t_next, g["o_end"]) < RTOL
    # covariances: max-norm (entries between far-apart reaches are differences of O(1) products)
    assert normerr(kf.P_t_next, g["P_end"]) < RTOL
    assert mdl.saved_states["datetime"].value == int(g["saved_t"])
    assert relerr(mdl.saved_states["o_t_next"], g["saved_o"]) < RTOL
    assert relerr(mdl.saved_states["i_t_next"], g["saved_i"]) < RTOL
    assert normerr(kf.saved_states["P_t_next"].cpu().numpy(), g["saved_P"]) < RTOL
    mdl.load_state()
    assert mdl.datetime.value == int(g["t_loaded"]) and relerr(mdl.o_t_next, g["o_loaded"]) < RTOL
    assert normerr(kf.P_t_next, g["P_loaded"]) < RTOL
    t1 = mdl.datetime.value
    sel = (times >= t1) & (times <= t1 + T * int(300e9))
    df2 = frame(times[sel], table[sel], cols)
    new = frame(g["meas_times2"], g["meas2"], [cols[j] for j in gcols])
    kf.measurements = new                      # columns in the caller's order: re-ordered by label
    assert list(kf.measurements.columns) == [cols[j] for j in np.sort(gcols)]
    assert kf.latest_timestamp.value == int(g["meas_times2"][-1])
    O2 = [state.o_t_next.copy() for state in mdl.simulate(df2)]
    assert relerr(np.stack(O2), g["O2"]) < RTOL
    assert relerr(mdl.o_t_next, g["o_end2"]) < RTOL and relerr(mdl.i_t_next, g["i_end2"]) < RTOL
    assert mdl.datetime.value == int(g["t_end2"]) and mdl.saved_states["datetime"].value == int(g["saved_t2"])
    assert normerr(kf.P_t_next, g["P_end2"]) < RTOL
    with pytest.raises(ValueError):
        kf.measurements = new.iloc[:, :-1]


def test_bad_shapes_are_rejected_before_the_c_abi(golden_dir):
    """Raw pointers cross the boundary: sizes are checked on the Python side (no out-of-bounds device reads)."""
    from tx_fast_hydrology_b200.da import KalmanFilter
    g = np.load(os.path.join(golden_dir, "checkpoint_kf_n70.npz"))
    mdl, d = model_from(g)
    cols = d["reach_ids"]
    n, m = mdl.n, g["gauge_cols"].size
    mdf = frame(g["meas_times1"], g["meas1"], [cols[j] for j in g["gauge_cols"]])
    with pytest.raises(ValueError):
        mdl.step(np.zeros(n - 1))
    with pytest.raises(ValueError):
        KalmanFilter(mdl, mdf, g["Q"], g["R"][:-1, :-1], g["P0"])
    with pytest.raises(ValueError):
        KalmanFilter(mdl, mdf, g["Q"], g["R"], g["P0"][:-1])
    with pytest.raises(ValueError):
        KalmanFilter(mdl, mdf, np.ones(n - 1), g["R"], g["P0"])
    # what the reference accepts through numpy broadcasting (da.py:115-116) is accepted here: scalar Q
    kf = KalmanFilter(mdl, mdf, 2.0, g["R"], g["P0"])
    mdl.bind_callback(kf, key="kf")
    kf.filter()
    ref_mdl, _ = model_from(g)
    kf2 = KalmanFilter(ref_mdl, mdf, 2.0 * np.ones((n, n)), g["R"], g["P0"])
    kf2.filter()
    assert (kf.P_t_next == kf2.P_t_next).all() and (mdl.o_t_next == ref_mdl.o_t_next).all()
    with pytest.raises(ValueError):
        mdl.network.unpack_host(mdl.device_state[0], 1, out=np.empty(n - 1))


def test_nutils_names(golden_dir):
    """The free functions da.py / muskingum.py import by name (muskingum.py:10, da.py:8-9)."""
    from tx_fast_hydrology_b200 import nutils as NU
    g = np.load(os.path.join(golden_dir, "kernels_n60.npz"))
    en = g["endnodes"]; n = en.size; sn = np.arange(n)
    ind = g["indegree"]; heads = sn[ind == 0]
    a, b, c, ga = g["alpha"], g["beta"], g["chi"], g["gamma"]
    i1, o1 = NU._ax_bu(heads, en, a, b, c, ga, g["i_init"], g["o_init"], g["q"], ind)
    assert relerr(o1, g["axbu_o"]) < RTOL and relerr(i1, g["axbu_i"]) < RTOL
    i2, o2 = NU._ax(heads, en, a, b, c, g["i_init"], g["o_init"], ind)
    assert relerr(o2, g["ax_o"]) < RTOL and relerr(i2, g["ax_i"]) < RTOL
    ig, og = NU._apply_gain(heads, en, g["gain"], ind)
    assert relerr(og, g["gain_o"]) < RTOL and relerr(ig, g["gain_i"]) < RTOL
    out = np.empty((n, n))
    res = NU._ap_par(g["P_sym"], out, heads, en, a, b, c, ind)
    assert res is out and relerr(out, g["ap"]) < RTOL
    out2 = np.empty((n, n))
    res2 = NU._aqat_par(g["P_gen"], out2, heads, en, a, b, c, ind)
    assert relerr(np.ascontiguousarray(res2), g["aqat_gen"]) < RTOL and res2.base is out2
    lin = np.stack([NU.interpolate_sample(float(x), g["xp"], g["fp"], 1) for x in g["xs"]])
    near = np.stack([NU.interpolate_sample(float(x), g["xp"], g["fp"], 0) for x in g["xs"]])
    assert (lin == g["interp_lin"]).all() and (near == g["interp_near"]).all()


def test_dense_linear_algebra():
    """FP64 tensor-core GEMM, SPD solve and inverse against numpy."""
    import torch
    from tx_fast_hydrology_b200.network import dgemm, spd_solve, inverse
    rng = np.random.default_rng(3)
    for (M, N, K, ta, tb) in [(70, 33, 50, False, False), (64, 64, 64, True, False), (129, 7, 200, False, True),
                              (5, 300, 3, True, True)]:
        A = rng.standard_normal((K, M) if ta else (M, K)); B = rng.standard_normal((N, K) if tb else (K, N))
        C0 = rng.standard_normal((M, N))
        ref = 0.5 * (A.T if ta else A) @ (B.T if tb else B) - 2.0 * C0
        C = torch.as_tensor(C0, device="cuda").clone()
        dgemm(torch.as_tensor(A, device="cuda"), torch.as_tensor(B, device="cuda"), C, ta, tb, 0.5, -2.0)
        assert normerr(C.cpu().numpy(), ref) < 1e-13       # matrix results: max-norm (backward-stable, not element-wise)
    for m, k in [(7, 3), (130, 64), (500, 64)]:
        X = rng.standard_normal((m, m)); S = X @ X.T + m * np.eye(m); B = rng.standard_normal((m, k))
        Sd = torch.as_tensor(S, device="cuda").clone(); Bd = torch.as_tensor(B, device="cuda").clone()
        spd_solve(Sd, Bd)
        assert normerr(Bd.cpu().numpy(), np.linalg.solve(S, B)) < 1e-11
        Ad = torch.as_tensor(S + 0.1 * X, device="cuda").clone()
        inverse(Ad)
        assert normerr(Ad.cpu().numpy(), np.linalg.inv(S + 0.1 * X)) < 1e-10


@pytest.mark.parametrize("n,M,m,seed,diag", [(400, 16, 12, 1, False), (1500, 64, 40, 2, False), (900, 10, 25, 3, False),
                                             (2000, 64, 100, 4, True), (1200, 32, 80, 5, False),
                                             (1000, 96, 130, 6, True), (1500, 128, 200, 10, True),
                                             (1200, 160, 100, 11, False), (800, 200, 330, 12, False)])
def test_enkf_update_vs_oracle(oracle, n, M, m, seed, diag):
    """Ensemble update == da.py:112-126 applied to the sample covariance (oracle.enkf_update).  Covers the
    direct m x m solve (M >= m) and the ensemble-space solve (M < m) with diagonal and dense R."""
    import torch
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.muskingum import Muskingum
    from tx_fast_hydrology_b200.da import EnsembleKalmanFilter
    net_d = S.make_network(n, seed)
    prm = S.make_params(n, seed, well_posed=True)
    rng = np.random.default_rng(seed)
    o0 = prm["o_t"][:, None] * rng.uniform(0.5, 1.5, size=(n, M))
    d = S.model_dict(net_d, prm, dt_s=300.0)
    d["o_t"] = o0
    mdl = Muskingum(d, members=M)
    gidx = S.make_gauges(net_d["endnodes"], m, seed=seed)
    t0 = mdl.datetime.value
    mt = t0 + np.arange(3, dtype=np.int64) * int(3600e9)
    meas = rng.uniform(0.5, 8.0, size=(3, m))
    cols = rng.permutation(m)
    mdf = frame(mt, meas[:, cols], [d["reach_ids"][j] for j in gidx[cols]])
    Rm = rng.standard_normal((m, m)); R = 1e-2 * np.eye(m) + (0.0 if diag else 1e-3) * (Rm @ Rm.T)
    Rc = R[np.ix_(cols, cols)]
    noise = 0.1 * rng.standard_normal((3, m, M))
    q = rng.uniform(0.5, 2.0, size=n)
    enkf = EnsembleKalmanFilter(mdl, mdf, q, Rc, obs_noise=noise[:, cols, :])
    O_f = mdl.o_t_next.copy(); I_f = mdl.i_t_next.copy()
    enkf.filter()
    ref_net = {"startnodes": net_d["startnodes"], "endnodes": net_d["endnodes"],
               "indegree": oracle.compute_indegree(net_d["startnodes"], net_d["endnodes"])}
    Zp = meas[0][:, None] + noise[0]
    O_ref, I_ref, _ = oracle.enkf_update(ref_net, O_f, I_f, gidx, Zp, q, R)
    assert relerr(mdl.o_t_next, O_ref) < RTOL
    assert relerr(mdl.i_t_next, I_ref) < RTOL


def _run_assimilating_case(oracle, n, M, m, seed, in_library, every=6, nwin=3, rest=0, gidx=None, dense_R=False):
    """`nwin` windows of `every` routing steps + one EnKF update each, then `rest` more routing steps, on the device
    (through the Python API) and on the CPU oracle; returns what the assertions need."""
    import torch
    c = make_case(n, M, m, seed, every, nwin, rest, gauges="synthetic" if gidx is None else gidx, dense_R=dense_R,
                  extra_reaches=None)
    mdl, enkf, f = model(c)
    nsteps, t0, Zp, gidx, q, R = c["nsteps"], c["t0"], c["Zp"], c["gidx"], c["q"], c["R"]
    # the observations travel on a side stream; the first update waits for the event, the first window does not
    Zh = torch.from_numpy(np.ascontiguousarray(Zp)).pin_memory()
    Zd = torch.empty(Zh.shape, dtype=torch.float64, device="cuda")
    side, ready = torch.cuda.Stream(), torch.cuda.Event()
    with torch.cuda.stream(side):
        Zd.copy_(Zh, non_blocking=True)
        ready.record(side)
    mdl.run_assimilating(f, nsteps, enkf, every, Zd if in_library else list(Zd), observations_ready=ready)
    mdl.network.check()
    assert enkf.n_updates == nwin and mdl.datetime.value == t0 + int(nsteps * 300e9)
    onet, o, i = oracle_start(oracle, c)
    times, table, mul = c["times"], c["table"], c["mul"]
    t = float(t0)
    tol = RTOL
    so, si = np.zeros((n, M)), np.zeros((n, M))                   # magnitudes of the forecasts the updates started from
    for k in range(nwin):
        oracle.run_members(onet, o, i, every, times.astype(np.float64), table, t, 300e9, wmul=mul)
        t += every * 300e9
        tol = max(tol, enkf_tolerance(o.T, gidx, q, R))          # eps * cond(S) of this update (tests/parity.py)
        so = np.maximum(so, np.abs(o.T)); si = np.maximum(si, np.abs(i.T))
        Op, Ip, _ = oracle.enkf_update(onet, o.T, i.T, gidx, Zp[k], q, R)
        o = np.ascontiguousarray(Op.T); i = np.ascontiguousarray(Ip.T)
    if rest:
        oracle.run_members(onet, o, i, rest, times.astype(np.float64), table, t, 300e9, wmul=mul)
    return mdl, o.T, i.T, so, si, tol


@pytest.mark.parametrize("n,M,m,seed", [(2000, 64, 50, 7), (1200, 20, 30, 8), (900, 70, 40, 9)])
@pytest.mark.parametrize("in_library", [True, False])
def test_run_assimilating_vs_oracle(oracle, n, M, m, seed, in_library):
    """The device-resident loop of the headline benchmark -- `every` routing steps in one window launch, the
    ensemble row sums riding on its last step, then one EnKF update, repeated -- equals the CPU oracle's
    routing (nutils.py:64-89 per member) + ensemble update (da.py:112-126) loop.  `in_library`: the loop runs
    inside libtxh (txh_run_assimilating, observations as one CUDA tensor: the small system in one cluster launch, the
    update applied by the next window launch while it loads its tasks) or in Python (a list of tensors: one launch per
    stage, the posterior written to memory by the transform kernel)."""
    mdl, o, i, so, si, tol = _run_assimilating_case(oracle, n, M, m, seed, in_library)
    # element-wise, relative to max(|posterior|, |forecast|): o + gain cancels on some reaches (tests/parity.py)
    assert relerr(mdl.o_t_next, o, scale=so) < tol
    assert relerr(mdl.i_t_next, i, scale=si) < tol


@pytest.mark.parametrize("M", [64, 10])
def test_run_assimilating_remainder_steps(oracle, M):
    """nsteps is not a multiple of `every`: the last update is applied by the launch that routes the remaining steps
    (txh_run_assimilating), nothing is left owed to the state."""
    mdl, o, i, so, si, tol = _run_assimilating_case(oracle, 1500, M, 25, 11, True, every=5, nwin=2, rest=3)
    assert relerr(mdl.o_t_next, o, scale=so) < tol
    assert relerr(mdl.i_t_next, i, scale=si) < tol


@pytest.mark.parametrize("M", [48, 70])
def test_run_assimilating_dense_R(oracle, M):
    """Correlated observation errors (dense R): the ensemble-space system takes the general launches (D^-1 dense), the
    update is still applied by the next window launch for M <= 64."""
    mdl, o, i, so, si, tol = _run_assimilating_case(oracle, 1400, M, 90, 17, True, every=5, nwin=3, dense_R=True)
    assert relerr(mdl.o_t_next, o, scale=so) < tol
    assert relerr(mdl.i_t_next, i, scale=si) < tol


def test_run_assimilating_gauges_at_confluences_and_outlets(oracle):
    """The gauge terms of the update applied at task load (route_window_kernel): a gauged reach adds qs W to its own
    outflow and to the inflow of the reach it drains into (nutils.py:127-134).  Gauges are put where that matters: on
    BOTH tributaries of confluences and on the confluence itself (three terms meet in one row), on reaches next to an
    outlet and on outlets (self-loop: no inflow term), on headwaters."""
    from tx_fast_hydrology_b200 import synthetic as S
    n, seed = 1800, 13
    end = S.make_network(n, seed)["endnodes"]
    start = np.arange(n)
    indeg = np.bincount(end[end != start], minlength=n)
    conf = np.flatnonzero(indeg >= 2)[:6]
    g = set()
    for c in conf:
        ups = np.flatnonzero((end == c) & (start != c))
        g.update(int(u) for u in ups[:2]); g.add(int(c))
    outlets = np.flatnonzero(end == start)
    g.update(int(x) for x in outlets[:2])
    for x in outlets[:2]:
        ups = np.flatnonzero((end == x) & (start != x))
        g.update(int(u) for u in ups[:1])
    g.update(int(x) for x in np.flatnonzero(indeg == 0)[:4])
    gidx = np.array(sorted(g), dtype=np.int64)
    assert gidx.size >= 20
    for in_library in (True, False):
        mdl, o, i, so, si, tol = _run_assimilating_case(oracle, n, 64, gidx.size, seed, in_library, every=4, nwin=3, gidx=gidx)
        assert relerr(mdl.o_t_next, o, scale=so) < tol
        assert relerr(mdl.i_t_next, i, scale=si) < tol


def test_run_assimilating_variants_agree():
    """Every fused stage of the in-library loop has a switch (TXH_ENKF_FUSED: the small system in one cluster launch;
    TXH_ENKF_FUSE_LOAD: the update applied at task load; TXH_PDL: programmatic dependent launch).  The switches are
    read once per process: a child process runs the same case with all of them off (one launch per stage, the
    posterior written by the transform kernel) and must agree with the default path to 1e-10 of the state."""
    import subprocess
    import sys
    import tempfile
    code = (
        "import sys, numpy as np, torch\n"
        "sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "from assim_case import make_case, model\n"
        "c = make_case(2500, 64, 40, 21, 6, 4, 0, gauges='synthetic', extra_reaches=None)\n"
        "mdl, enkf, f = model(c)\n"
        "Zp = torch.as_tensor(c['Zp'], device='cuda')\n"
        "mdl.run_assimilating(f, c['nsteps'], enkf, 6, Zp)\n"
        "mdl.network.check()\n"
        "np.savez(sys.argv[1], o=mdl.o_t_next, i=mdl.i_t_next)\n") % (os.path.dirname(HERE), HERE)
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        for name, env in (("fused", {}), ("plain", {"TXH_ENKF_FUSED": "0", "TXH_ENKF_FUSE_LOAD": "0", "TXH_PDL": "0"})):
            path = os.path.join(tmp, name + ".npz")
            e = dict(os.environ); e.update(env)
            subprocess.run([sys.executable, "-c", code, path], check=True, env=e, timeout=600)
            z = np.load(path)
            out[name] = (z["o"], z["i"])
    assert normerr(out["fused"][0], out["plain"][0]) < 1e-10
    assert normerr(out["fused"][1], out["plain"][1]) < 1e-10


def test_headline_window_full_size(oracle):
    """BASELINE.json configs[2] at FULL size -- 100,000 reaches, 64 members, 500 gauges: one hourly window
    (12 routing steps in one window launch) and one EnKF update against the CPU oracle, plus two
    size-independent properties of the update: observations equal to the forecast leave the ensemble
    unchanged, and the update commutes with a permutation of the members."""
    import torch
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.muskingum import Muskingum
    from tx_fast_hydrology_b200.da import EnsembleKalmanFilter
    n, M, m, seed, every = 100_000, 64, 500, 2, 12
    net_d = S.make_network(n, seed)
    prm = S.make_params(n, seed)
    rng = np.random.default_rng(seed + 7)
    o0 = prm["o_t"][:, None] * rng.uniform(0.5, 1.5, size=(n, M))
    d = S.model_dict(net_d, prm, dt_s=300.0)
    d["o_t"] = o0
    mdl = Muskingum(d, members=M)
    t0 = int(mdl.datetime.value)
    times, table = S.make_forcing(n, every, 300.0, seed, t0_ns=t0)
    mul = S.make_member_multipliers(times.size, M, seed)
    gidx = S.make_gauges(net_d["endnodes"], m, seed=4)
    mdf = frame(np.array([t0 + int(every * 300e9)], dtype=np.int64), rng.uniform(0.5, 8.0, size=(1, m)),
                [d["reach_ids"][j] for j in gidx])
    R = 1e-2 * np.eye(m)
    enkf = EnsembleKalmanFilter(mdl, mdf, 2.0, R)
    f = mdl.make_forcing(times_ns=times, table=table, member_mul=mul)
    # forecast on both sides
    mdl.run(f, every)
    mdl.network.check()
    ind = oracle.compute_indegree(net_d["startnodes"], net_d["endnodes"])
    al, be, ch, ga = oracle.compute_coeffs(prm["K"], prm["X"], 300.0)
    onet = {"startnodes": net_d["startnodes"], "endnodes": net_d["endnodes"], "indegree": ind,
            "alpha": al, "beta": be, "chi": ch, "gamma": ga}
    o = np.ascontiguousarray(o0.T)
    i = np.stack([oracle.init_states(net_d["startnodes"], net_d["endnodes"], x) for x in o])
    oracle.run_members(onet, o, i, every, times.astype(np.float64), table, float(t0), 300e9, wmul=mul)
    assert relerr(mdl.o_t_next, o.T) < RTOL and relerr(mdl.i_t_next, i.T) < RTOL
    O_d, I_d = mdl.device_state
    Of, If = O_d.clone(), I_d.clone()
    # (a) zero innovation: Zp == H x  ->  nothing moves
    HX = torch.as_tensor(np.ascontiguousarray(o.T[gidx]), device="cuda")
    enkf.filter(HX)
    mdl.network.check()
    assert (O_d - Of).abs().max().item() <= 1e-12 * Of.abs().max().item()
    assert (I_d - If).abs().max().item() <= 1e-12 * If.abs().max().item()
    # (b) the real update vs the oracle
    mdl.upload_state(np.ascontiguousarray(o.T), np.ascontiguousarray(i.T))
    Zp = np.ascontiguousarray(mdf.values[0][:, None] + 0.1 * rng.standard_normal((m, M)))
    enkf.filter(torch.as_tensor(Zp, device="cuda"))
    mdl.network.check()
    Op, Ip, _ = oracle.enkf_update(onet, o.T, i.T, gidx, Zp, np.full(n, 2.0), R)
    o_gpu, i_gpu = mdl.o_t_next.copy(), mdl.i_t_next.copy()
    tol = enkf_tolerance(o.T, gidx, 2.0, R)                      # max(1e-9, 64 eps cond(S)), tests/parity.py
    # element-wise, relative to max(|posterior|, |forecast|): o + gain cancels on some reaches (tests/parity.py)
    assert relerr(o_gpu, Op, scale=o.T) < tol and relerr(i_gpu, Ip, scale=i.T) < tol
    assert normerr(o_gpu, Op) < RTOL and normerr(i_gpu, Ip) < RTOL
    # (c) member permutation: update(P x, P z) == P update(x, z)
    perm = rng.permutation(M)
    mdl.upload_state(np.ascontiguousarray(o.T[:, perm]), np.ascontiguousarray(i.T[:, perm]))
    enkf.filter(torch.as_tensor(np.ascontiguousarray(Zp[:, perm]), device="cuda"))
    mdl.network.check()
    assert relerr(mdl.o_t_next, o_gpu[:, perm], scale=o.T[:, perm]) < tol and normerr(mdl.o_t_next, o_gpu[:, perm]) < 1e-10

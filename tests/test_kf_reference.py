"""The extended-precision reference of the dense Kalman filter, the RTS smoother and the pivoting inverse
(tests/kf_reference.py) on the CPU: it reproduces the oracle's filter and the reference's goldens, and the bounds
tests/test_gpu_dense_kf.py applies are sharp enough to catch a kernel that is subtly wrong.  Also the shape checks
that keep bad matrices away from the raw pointers of the C ABI (they run before any device work)."""
import os

import numpy as np
import pandas as pd
import pytest

import kf_reference as R
from parity import relerr, normerr


def _f64(x):
    return np.asarray(x, dtype=np.float64)


class _RefFilter:
    """OracleKalmanFilter with the update of kf_update_ref, the state kept FP64 for the routing in between."""

    def __init__(self, oracle, model, meas_times, meas, cols, Q, Rc, P0, exact_time=False):
        self.O = oracle
        self.base = oracle.OracleKalmanFilter(model, meas_times, meas, cols, Q, Rc, P0)
        self.exact_time = exact_time
        self.log = []

    def on_simulation_start(self):
        if self.base._due():
            self.filter()

    def on_step_start(self):
        pass

    def on_step_end(self):
        if self.base._due():
            self.filter()

    def on_simulation_end(self):
        pass

    def filter(self):
        b, mdl = self.base, self.base.model
        if self.exact_time:
            Z = b.meas[int(np.flatnonzero(b.meas_times == float(mdl.time_ns))[0])]
        else:
            Z = self.O.interpolate_sample(float(mdl.time_ns), b.meas_times, b.meas)
        prior = (mdl.i_t_next.copy(), mdl.o_t_next.copy())
        r = R.kf_update_ref(b.P_t_next, b.Q_cov, b.R_cov, b.reach_indices, Z, mdl.o_t_next, mdl.i_t_next,
                            mdl.endnodes, mdl.alpha, mdl.beta, mdl.chi)
        mdl.o_t_next, mdl.i_t_next = _f64(r["o"]), _f64(r["i"])
        b.P_t_next = r["P"]
        self.log.append((mdl.time_ns, r, prior))


def _golden_model(oracle, g):
    n = g["endnodes"].size
    return oracle.OracleModel(np.arange(n), g["endnodes"], g["K"], g["X"], g["o_init"], float(g["dt"]),
                              int(g["t0_ns"]))


def test_reference_reproduces_the_kalman_golden(oracle, golden_dir):
    """kalman_n120.npz (the unmodified reference: unsorted gauge columns, dense R, 24 steps) to 1e-13."""
    g = np.load(os.path.join(golden_dir, "kalman_n120.npz"))
    mdl = _golden_model(oracle, g)
    kf = _RefFilter(oracle, mdl, g["meas_times"], g["meas"], g["gauge_cols"], g["Q"], g["R"], g["P0"])
    mdl.callbacks["kf"] = kf
    O, I, Pd, gains = [], [], [], []
    for _ in mdl.simulate(g["times"], g["table"]):
        O.append(mdl.o_t_next.copy()); I.append(mdl.i_t_next.copy())
        Pd.append(np.diag(_f64(kf.base.P_t_next))); gains.append(_f64(kf.log[-1][1]["gain"]))
    assert relerr(np.stack(O), g["O"]) < 1e-13 and relerr(np.stack(I), g["I"]) < 1e-13
    assert normerr(np.stack(Pd), g["P_diag"]) < 1e-13 and normerr(np.stack(gains), g["gains"]) < 1e-13
    assert normerr(_f64(kf.base.P_t_next), g["P_final"]) < 1e-13
    assert normerr(_f64(kf.log[-1][1]["K"]), g["K_final"]) < 1e-13


def test_reference_reproduces_the_smoother_golden(oracle, golden_dir):
    """smoother_n60.npz: the forward filter at exact measurement times (kf_update_ref), the dicts KalmanSmoother keeps
    (da.py:170-219: the entries of the start time are overwritten by its first update), then rts_ref, to 1e-13."""
    g = np.load(os.path.join(golden_dir, "smoother_n60.npz"))
    mdl = _golden_model(oracle, g)
    kf = _RefFilter(oracle, mdl, g["meas_times"], g["meas"], g["gauge_idx"], g["Q"], g["R"], g["P0"],
                    exact_time=True)
    mdl.callbacks["ks"] = kf
    t0 = mdl.time_ns
    ts = [t0]
    P_f, P_p = {t0: g["P0"]}, {t0: g["P0"]}
    x0 = np.stack([mdl.i_t_next, mdl.o_t_next], axis=1)
    x_f, x_p = {t0: x0}, {t0: x0}
    for _ in mdl.simulate(g["times"], g["table"]):
        pass
    for t, r, (i_pr, o_pr) in kf.log:
        ts.append(t)
        P_f[t], P_p[t] = r["P"], r["Pm"]
        x_f[t] = np.stack([_f64(r["i"]), _f64(r["o"])], axis=1)
        x_p[t] = np.stack([i_pr, o_pr], axis=1)
    assert len(ts) == int(g["n_times"])
    x_s, P_s = R.rts_ref(ts, P_f, P_p, x_f, x_p, g["endnodes"], mdl.alpha, mdl.beta, mdl.chi)
    times = sorted(x_s)
    assert [int(t) for t in times] == [int(t) for t in g["smooth_times"]]
    assert relerr(mdl.o_t_next, g["o_final"]) < 1e-13 and relerr(mdl.i_t_next, g["i_final"]) < 1e-13
    assert normerr(np.stack([_f64(x_s[t][:, 1]) for t in times]), g["o_hat_s"]) < 1e-13
    assert normerr(np.stack([_f64(x_s[t][:, 0]) for t in times]), g["i_hat_s"]) < 1e-13
    assert normerr(_f64(P_f[times[-1]]), g["P_f_last"]) < 1e-13
    assert normerr(_f64(P_s[times[0]]), g["P_s_first"]) < 1e-13


def test_reference_reproduces_the_oracle_filter(oracle):
    """One update of oracle.OracleKalmanFilter (FP64, np.linalg.inv) on a 3-basin synthetic network, gauges at
    heads, confluences and outlets, dense Q and R: kf_update_ref agrees to 1e-13."""
    from tx_fast_hydrology_b200 import synthetic as S
    n, seed = 90, 5
    net = S.make_network(n, seed, n_basins=3)
    prm = S.make_params(n, seed)
    end = net["endnodes"]
    g = R.special_gauges(end, 14, seed)
    mdl = oracle.OracleModel(np.arange(n), end, prm["K"], prm["X"], prm["o_t"], 300.0, 0)
    Q, Rm, P0 = R.dense_covariances(n, g.size, seed, rank=n, r_scale=1e-2)
    z = prm["o_t"][g] * 1.1
    kf = oracle.OracleKalmanFilter(mdl, np.array([0]), z[None], g, Q, Rm, P0)
    o, i = mdl.o_t_next.copy(), mdl.i_t_next.copy()
    kf.filter()
    r = R.kf_update_ref(P0, Q, Rm, g, z, o, i, end, mdl.alpha, mdl.beta, mdl.chi)
    assert normerr(_f64(r["K"]), kf.K) < 1e-13 and normerr(_f64(r["P"]), kf.P_t_next) < 1e-13
    assert normerr(_f64(r["gain"]), kf.gain) < 1e-13 and normerr(_f64(r["dz"]), kf.dz) < 1e-13
    assert relerr(_f64(r["o"]), mdl.o_t_next) < 1e-13 and relerr(_f64(r["i"]), mdl.i_t_next) < 1e-13


@pytest.mark.parametrize("m", [1, 2, 7, 31, 64, 200])
def test_inverse_ref_against_numpy(m):
    rng = np.random.default_rng(m)
    A = rng.standard_normal((m, m)) + m * np.eye(m)[rng.permutation(m)]
    X, piv = R.inverse_ref(A)
    assert normerr(_f64(X), np.linalg.inv(A)) < 1e-14
    assert np.abs(_f64(X @ np.asarray(A, dtype=R.LD)) - np.eye(m)).max() < 1e-15
    with pytest.raises(np.linalg.LinAlgError):
        R.inverse_ref(np.zeros((m, m)))


def _inverse_error(A, X):
    """What the GPU test measures: against the longdouble inverse up to LD_INVERSE_MAX, else the FP64 residuals."""
    m = A.shape[0]
    if m <= R.LD_INVERSE_MAX:
        return normerr(_f64(X), _f64(R.inverse_ref(A)[0]))
    return max(np.abs(A @ _f64(X) - np.eye(m)).max(), np.abs(_f64(X) @ A - np.eye(m)).max())


MUTANTS = {"column un-swap left out": dict(unswap="none"), "un-swap in forward order": dict(unswap="forward"),
           "pivot row's factor from the wrong row": dict(pivot_factor="pivot row")}


@pytest.mark.parametrize("m", [m for m in R.INVERSE_SIZES if m > 1])
def test_inverse_tolerance_is_sharp(m):
    """Each planted defect of the Gauss-Jordan inverse misses the GPU bound by 10^3 at every size the GPU file uses
    (m = 1 cannot pivot; with two rows there is only one swap, so its order cannot matter).  Past LD_INVERSE_MAX the
    defective inverse is formed in FP64 and judged by its residual, as the GPU test judges the kernel."""
    kinds = ("spd_1e8", "permuted_dominant") if m <= R.LD_INVERSE_MAX else ("permuted_dominant",)
    for kind in kinds:
        A = R.inverse_input(kind, m)
        tol = R.inverse_tolerance(m, np.linalg.cond(A))
        dtype = R.LD if m <= R.LD_INVERSE_MAX else np.float64
        for name, kw in MUTANTS.items():
            if m == 2 and name == "un-swap in forward order":
                continue
            err = _inverse_error(A, R.inverse_ref(A, dtype=dtype, **kw)[0])
            assert err > 1e3 * tol, f"{kind} m={m}: {name} moves the inverse by {err:.2e}, the bar is {1e3 * tol:.2e}"


@pytest.mark.parametrize("case", R.FILTER_CASES, ids=[c["id"] for c in R.FILTER_CASES])
def test_filter_tolerance_is_sharp(oracle, case):
    """R left out of S moves K, gain or P+ of the first update of every dense-filter case of the GPU file by more
    than 10^3 x its bound; the cases also span cond(S) from ~1 to ~1e8, as they claim."""
    inp = R.filter_case_inputs(oracle, case)
    r = R.kf_update_ref(*inp)
    condS = np.linalg.cond(_f64(r["S"]))
    lo, hi = case["cond"]
    assert lo <= condS <= hi, f"cond(S) = {condS:.2e}, the case is meant for [{lo:.0e}, {hi:.0e}]"
    tol = R.kf_tolerance(condS)
    P, Q, Rm = inp[0], inp[1], inp[2]
    bad = R.kf_update_ref(P, Q, np.zeros_like(Rm), *inp[3:])
    moved = max(normerr(_f64(bad[k]), _f64(r[k])) for k in ("K", "gain", "P"))
    assert moved > 1e3 * tol, f"R left out moves the update by {moved:.2e}, the bar is {1e3 * tol:.2e}"


def test_stopped_filter_prior_covariance_is_sharp(oracle):
    """The batched case of the GPU file: for every filter that stops before the run ends, P before its last update
    differs from P after it by more than 10^3 x the bound the GPU test applies to P_t_prev."""
    for k, blk in enumerate(R.BATCH_BLOCKS):
        if blk["stop"] >= R.BATCH_STEPS:
            continue
        P_prev, P_next, condS = R.batch_block_last_update(oracle, k)
        tol = R.kf_tolerance(condS)
        assert normerr(P_prev, P_next) > 1e3 * tol, f"block {k}: P_t_prev := P_t_next would pass"


def test_bad_matrices_are_refused_before_the_c_abi():
    """dgemm, spd_solve and inverse hand raw device pointers to libtxh: shapes, strides, dtype and device are
    checked first (here with CPU tensors, which never reach the library)."""
    import torch
    from tx_fast_hydrology_b200.network import dgemm, inverse, spd_solve
    f = dict(dtype=torch.float64)
    A, B, C = torch.zeros(4, 3, **f), torch.zeros(3, 5, **f), torch.zeros(4, 5, **f)
    bad = [lambda: inverse(torch.zeros(4, 3, **f)),                     # not square
           lambda: inverse(torch.zeros(4, 4, **f).t()),                   # a transposed view
           lambda: inverse(torch.zeros(6, 6, **f)[:4, :4]),            # rows 6 apart
           lambda: inverse(torch.zeros(4, 4, dtype=torch.float32)),
           lambda: inverse(torch.zeros(4, 4, **f)),                     # not on the device
           lambda: inverse(torch.zeros(4, **f)),
           lambda: spd_solve(torch.zeros(4, 4, **f), torch.zeros(3, 2, **f)),
           lambda: spd_solve(torch.zeros(4, 3, **f), torch.zeros(4, 2, **f)),
           lambda: spd_solve(torch.zeros(4, 4, **f), torch.zeros(2, 4, **f).t()),
           lambda: spd_solve(torch.zeros(4, 4, **f), torch.zeros(4, 2, **f)),
           lambda: dgemm(A, B, torch.zeros(4, 4, **f)),                 # N
           lambda: dgemm(A, torch.zeros(2, 5, **f), C),                  # K
           lambda: dgemm(torch.zeros(5, 3, **f), B, C),                  # M
           lambda: dgemm(A, B, C, transA=True),
           lambda: dgemm(A, B, C, transB=True),
           lambda: dgemm(torch.zeros(3, 4, **f).t(), B, C),              # a transposed view
           lambda: dgemm(A, torch.zeros(5, 3, **f).t(), C),
           lambda: dgemm(A, B, torch.zeros(5, 4, **f).t()),
           lambda: dgemm(A.float(), B, C),
           lambda: dgemm(A, B, C)]                                      # not on the device
    for k, call in enumerate(bad):
        with pytest.raises(ValueError):
            call()

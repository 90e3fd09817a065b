"""The square-root (ETKF) and relaxed (RTPP) ensemble updates on the CPU: the extended-precision reference the GPU
tests use (tests/etkf_reference.py) against the Kalman filter it stands for, its identities, and the sharpness of the
GPU tolerance against planted defects."""
import numpy as np
import pytest

import enkf_reference as E
import etkf_reference as K
from parity import normerr

LD = E.LD


def _ensemble(n, M, m, seed, qs_zero=False):
    """A small state ensemble X [n][M], its gauges (the first m rows), one observation z [m], qs and a diagonal R."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, M)) @ np.diag(rng.uniform(0.5, 1.5, M)) + rng.uniform(2, 4, (n, 1))
    X[:m] += 0.3 * X[m:2 * m] if 2 * m <= n else 0.0          # correlated rows
    z = X[:m].mean(axis=1) + rng.uniform(-0.5, 0.5, m)
    qs = np.zeros(m) if qs_zero else rng.uniform(0.01, 0.1, m)
    R = np.diag(rng.uniform(0.05, 0.2, m))
    return X, np.arange(m), z, qs, R


def _solve(X, g, Zp, qs, R):
    mean = X.mean(axis=1)
    T, W, _ = E.solve_ref(X[g], Zp, mean[g], qs, R)
    return T, W


def _posterior(X, g, T, W, qs):
    Xl = np.asarray(X, dtype=LD)
    P = Xl + (Xl - Xl.mean(axis=1)[:, None]) @ T
    P[g] += np.asarray(qs, dtype=LD)[:, None] * W
    return P


@pytest.mark.parametrize("n,M,m", [(40, 9, 12), (30, 33, 10), (70, 64, 50), (12, 2, 3)])
def test_etkf_posterior_is_the_kalman_posterior(n, M, m):
    """Q = 0: the ETKF posterior ensemble has mean xbar + K dzbar and sample covariance (I - K H) P_e exactly, K the
    Kalman gain of the ensemble covariance P_e."""
    X, g, z, qs, R = _ensemble(n, M, m, 5 + M, qs_zero=True)
    Zp = np.repeat(z[:, None], M, axis=1)
    T, W = _solve(X, g, Zp, qs, R)
    Tp, Wp = K.etkf_post(T, W)
    P = _posterior(X, g, Tp, Wp, qs)
    Xl = np.asarray(X, dtype=LD)
    A = Xl - Xl.mean(axis=1)[:, None]
    Pe = A @ A.T / (M - 1)
    S = Pe[np.ix_(g, g)] + np.asarray(R, dtype=LD)
    Kg = Pe[:, g] @ K.inv_spd(S)
    mean_want = Xl.mean(axis=1) + Kg @ (np.asarray(z, dtype=LD) - Xl[g].mean(axis=1))
    H = np.zeros((m, n), dtype=LD); H[np.arange(m), g] = 1
    cov_want = (np.eye(n, dtype=LD) - Kg @ H) @ Pe
    Ap = P - P.mean(axis=1)[:, None]
    assert normerr(P.mean(axis=1), mean_want) < 1e-15
    assert normerr(Ap @ Ap.T / (M - 1), cov_want) < 1e-14
    # the stochastic update without perturbations does not: it keeps too little spread
    Pn = _posterior(X, g, T, W, qs)
    An = Pn - Pn.mean(axis=1)[:, None]
    assert np.trace(An @ An.T / (M - 1)) < 0.99 * np.trace(cov_want)


@pytest.mark.parametrize("M,m", [(5, 20), (33, 10), (64, 200)])
def test_square_root_is_symmetric_and_keeps_the_mean(M, m):
    """G^1/2 is symmetric, squares to G, and S 1 = 1 (so T' keeps the row means wbar and the posterior mean)."""
    inp = E.solve_inputs(M, m, E.case_seed(M, m))
    T, W, _ = E.solve_ref(inp["HX"], K.identical_columns(inp["Zp"]), inp["mean"], inp["qs"], inp["R"])
    wbar, G = K.split(T)
    ev = np.linalg.eigvalsh(np.asarray(G, dtype=np.float64))
    assert ev[0] > 0 and ev[-1] <= 1 + 1e-12
    S = K.sqrtm_spd(G)
    assert normerr(S, S.T) == 0.0
    assert normerr(S @ S, G) < 1e-15                      # 1e3 below the GPU tolerance
    # G 1 = 1 holds to the rounding of the FP64 ensemble mean the anomalies are formed from
    one = np.ones(M, dtype=LD)
    assert normerr(G @ one, one) < 1e-14
    assert normerr(S @ one, one) < 1e-14
    Tp, _ = K.etkf_post(T, W)
    assert normerr(Tp.mean(axis=1), wbar) < 1e-14


@pytest.mark.parametrize("rho", [0.25, 0.5, 0.9])
def test_rtpp_anomaly_identity(rho):
    """RTPP of the stochastic update: on every row (gauged or not) the posterior anomalies are (1 - rho) x those of the
    stochastic posterior plus rho x the prior's, and the mean is the stochastic posterior's."""
    n, M, m = 50, 17, 12
    X, g, z, qs, R = _ensemble(n, M, m, 31)
    rng = np.random.default_rng(3)
    Zp = z[:, None] + rng.standard_normal((m, M)) * np.sqrt(np.diagonal(R))[:, None]
    T, W = _solve(X, g, Zp, qs, R)
    Tr, Wr = K.rtpp_post(T, W, rho)
    P, Pr = _posterior(X, g, T, W, qs), _posterior(X, g, Tr, Wr, qs)
    anom = lambda Y: Y - Y.mean(axis=1)[:, None]                 # noqa: E731
    Xl = np.asarray(X, dtype=LD)
    assert normerr(Pr.mean(axis=1), P.mean(axis=1)) < 1e-17
    assert normerr(anom(Pr), (1 - LD(rho)) * anom(P) + LD(rho) * anom(Xl)) < 1e-15


def test_every_gauge_missing_gives_a_zero_transform():
    Tp, Wp, *_ = K.case(33, 40, False, "cluster", mask="all")[2:]
    assert not np.abs(Tp).any() and not np.abs(Wp).any()
    Tp, Wp, *_ = K.case(33, 40, False, "cluster", rho=0.5, mask="all")[2:]
    assert not np.abs(Tp).any() and not np.abs(Wp).any()


def test_stochastic_without_relaxation_is_the_solve_itself():
    inp = E.solve_inputs(9, 30, E.case_seed(9, 30))
    T, W, _ = E.solve_ref(inp["HX"], inp["Zp"], inp["mean"], inp["qs"], inp["R"])
    Tr, Wr = K.rtpp_post(T, W, 0.0)
    assert np.array_equal(Tr, T) and np.array_equal(Wr, W)


# ---- planted defects -----------------------------------------------------------------------------------------------
def _cholesky_root(G):
    return E.cholesky(G)


def _no_root(G):
    return np.asarray(G, dtype=LD)


def _column_means(T, W, rho):
    T = np.asarray(T, dtype=LD)
    wbar = T.mean(axis=0)
    G = T - wbar[None, :] + np.eye(T.shape[0], dtype=LD)
    G = (G + G.T) / 2
    Tp = wbar[:, None] + (1 - LD(rho)) * (K.sqrtm_spd(G) - np.eye(T.shape[0], dtype=LD))
    return Tp, K.etkf_post(T, W, rho)[1]


def _rtpp_on_the_mean(T, W, rho):
    Tp, Wp = K.etkf_post(T, W, 0.0)
    return (1 - LD(rho)) * Tp, (1 - LD(rho)) * Wp


DEFECTS = {
    "cholesky_root": lambda T, W, rho: K.etkf_post(T, W, rho, root=_cholesky_root),
    "G_not_root": lambda T, W, rho: K.etkf_post(T, W, rho, root=_no_root),
    "column_means": _column_means,
    "rtpp_on_mean": _rtpp_on_the_mean,
    "W_not_averaged": lambda T, W, rho: (K.etkf_post(T, W, rho)[0], np.asarray(W, dtype=LD)),
}


@pytest.mark.parametrize("defect", sorted(DEFECTS))
@pytest.mark.parametrize("M,m,path", [(5, 40, "cluster"), (33, 100, "cluster"), (64, 40, "direct")])
def test_planted_defects_miss_the_gpu_tolerance(defect, M, m, path):
    """Each defect's (T', W') misses the tolerance test_gpu_etkf.py applies by a factor of at least 1e3."""
    rho = 0.5 if defect == "rtpp_on_mean" else 0.0
    inp, _, Tp, Wp, tolT, tolW = K.case(M, m, False, path, rho=rho)
    Tz = np.repeat(inp["Zp"][:, :1], M, axis=1)
    T, W, _ = E.solve_ref(inp["HX"], Tz, inp["mean"], inp["qs"], inp["R"])
    Td, Wd = DEFECTS[defect](T, W, rho)
    ratio = max(normerr(Td, Tp) / tolT, normerr(Wd, Wp) / tolW)
    assert ratio > 1e3, f"{defect}: only {ratio:.1e} x the tolerance"
    assert normerr(Tp, K.etkf_post(T, W, rho)[0]) == 0.0

"""Extended-precision reference of the square-root ensemble update (ETKF) and of relaxation to prior perturbations
(RTPP) (test infrastructure, CPU, numpy longdouble, on top of tests/enkf_reference.py).

A solve run with identical observation columns, Zp[g][c] = z[g], leaves

    T = wbar 1^T - I + G,   G = (M-1) (C0 + (M-1) I)^-1   (SPD, spectrum in (0, 1], G 1 = 1),
    row means of W:  Wbar = D^-1 (dzbar - HA wbar)

and the ETKF update is T' = wbar 1^T + (1 - rho) (G^1/2 - I), W'[g][c] = Wbar[g].  RTPP of the stochastic update is
T' = wbar 1^T + (1 - rho) (T - wbar 1^T), W' = Wbar 1^T + (1 - rho) (W - Wbar 1^T).
G^1/2 comes from cyclic Jacobi in longdouble.
"""
import numpy as np

import enkf_reference as E
import enkf_missing_reference as X

LD = E.LD


def inv_spd(A):
    A = np.asarray(A, dtype=LD)
    return E.chol_solve(E.cholesky((A + A.T) / 2), np.eye(A.shape[0], dtype=LD))


def sqrtm_spd(G, sweeps=30):
    """The symmetric square root of a symmetric positive semi-definite matrix, longdouble: cyclic Jacobi (one
    rotation at a time) to off(G) <= 1e-19 ||G||_F, then V diag(sqrt(max(lambda, 0))) V^T."""
    A = np.array(G, dtype=LD)
    A = (A + A.T) / 2
    n = A.shape[0]
    V = np.eye(n, dtype=LD)
    fro = np.sqrt((A * A).sum())
    for _ in range(sweeps):
        if np.sqrt(((A - np.diag(np.diagonal(A))) ** 2).sum()) <= 1e-19 * fro:
            break
        for p in range(n - 1):
            for q in range(p + 1, n):
                if A[p, q] == 0:
                    continue
                tau = (A[q, q] - A[p, p]) / (2 * A[p, q])
                t = (1 if tau >= 0 else -1) / (abs(tau) + np.sqrt(1 + tau * tau))
                c = 1 / np.sqrt(1 + t * t)
                s = t * c
                ap, aq = A[p].copy(), A[q].copy()
                A[p], A[q] = c * ap - s * aq, s * ap + c * aq
                ap, aq = A[:, p].copy(), A[:, q].copy()
                A[:, p], A[:, q] = c * ap - s * aq, s * ap + c * aq
                A[p, q] = A[q, p] = 0
                vp, vq = V[:, p].copy(), V[:, q].copy()
                V[:, p], V[:, q] = c * vp - s * vq, s * vp + c * vq
    lam = np.sqrt(np.maximum(np.diagonal(A), 0))
    S = (V * lam) @ V.T
    return (S + S.T) / 2


def split(T):
    """(wbar, G) of a solved transform: the row means and T - wbar 1^T + I (symmetrised)."""
    T = np.asarray(T, dtype=LD)
    wbar = T.mean(axis=1)
    G = T - wbar[:, None] + np.eye(T.shape[0], dtype=LD)
    return wbar, (G + G.T) / 2


def etkf_post(T, W, rho=0.0, root=sqrtm_spd):
    """The ETKF form (T', W') of a transform solved with identical observation columns; `root` the square root."""
    wbar, G = split(T)
    W = np.asarray(W, dtype=LD)
    M = G.shape[0]
    Tp = wbar[:, None] + (1 - LD(rho)) * (root(G) - np.eye(M, dtype=LD))
    return Tp, np.repeat(W.mean(axis=1)[:, None], M, axis=1)


def rtpp_post(T, W, rho):
    T = np.asarray(T, dtype=LD)
    W = np.asarray(W, dtype=LD)
    if rho == 0:
        return T, W
    k = 1 - LD(rho)
    wb, Wb = T.mean(axis=1)[:, None], W.mean(axis=1)[:, None]
    return wb + k * (T - wb), Wb + k * (W - Wb)


def identical_columns(Zp):
    """Zp with every member column equal to member 0 (NaN rows stay NaN: the gauge is missing)."""
    Zp = np.asarray(Zp, dtype=np.float64)
    return np.ascontiguousarray(np.repeat(Zp[:, :1], Zp.shape[1], axis=1))


def lambda_min(T):
    """The smallest eigenvalue of G (the conditioning of the square root: d G^1/2 <= d G / (2 sqrt(lambda_min)))."""
    _, G = split(T)
    return float(np.linalg.eigvalsh(np.asarray(G, dtype=np.float64))[0])


def etkf_tolerance(tol_solve, T, Tp, lam_min):
    """Max-norm relative bound on the device's T' (against etkf_post of the reference T): the solve's error
    tol_solve * max|T| in any entry of G is at most M times that in the 2-norm, the square root amplifies a 2-norm
    error by 1 / (2 sqrt(lambda_min(G))), and the Jacobi eigensolve (stopped at off(G) <= 1e-14 ||G||_F) and the
    product V diag(sqrt(lambda)) V^T add a few hundred eps per entry; relative to max|T'|, at least 1e-12."""
    M = np.shape(T)[0]
    tmax = float(np.abs(np.asarray(T, dtype=np.float64)).max())
    abs_err = tol_solve * tmax * M / (2.0 * np.sqrt(lam_min)) + 1e-14 * M / np.sqrt(lam_min) + 256 * M * E.EPS64
    return max(1e-12, abs_err / max(1e-300, float(np.abs(np.asarray(Tp, dtype=np.float64)).max())))


def _scaled(tol, A, Ap):
    """tol relative to max|A| as a bound relative to max|Ap|."""
    a, ap = float(np.abs(np.asarray(A, dtype=np.float64)).max()), float(np.abs(np.asarray(Ap, dtype=np.float64)).max())
    return max(1e-12, tol * a / max(1e-300, ap))


def case(M, m, dense_R, path, rho=0.0, mask="none", method="etkf"):
    """Inputs of one ETKF (or RTPP) solve case of tests/test_gpu_etkf.py and their reference: the solve inputs of
    enkf_reference.solve_inputs (observation columns made identical for the ETKF), the NaN mask `mask` of
    enkf_missing_reference, then (T', W') and the max-norm relative tolerances of T' and W' (the solve tolerance of
    enkf_reference.solve_tolerance carried through the post-processing)."""
    inp = E.solve_inputs(M, m, E.case_seed(M, m), dense_R)
    Zp = identical_columns(inp["Zp"]) if method == "etkf" else inp["Zp"]
    Zp, miss = X.plant(Zp, mask) if mask != "none" else (Zp, np.zeros(m, dtype=bool))
    T, W, condS, ce = X.solve_masked(inp["HX"], Zp, inp["mean"], inp["qs"], inp["R"])
    tol = X.masked_tolerance(condS, ce, path)
    if method == "etkf":
        Tp, Wp = etkf_post(T, W, rho)
        tolT = etkf_tolerance(tol, T, Tp, lambda_min(T))
    else:
        Tp, Wp = rtpp_post(T, W, rho)
        tolT = _scaled(tol, T, Tp)
    return dict(inp, Zp=Zp), miss, Tp, Wp, tolT, _scaled(tol, W, Wp)

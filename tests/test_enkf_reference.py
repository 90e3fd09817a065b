"""The extended-precision reference of the ensemble update (tests/enkf_reference.py) on the CPU: it reproduces the
oracle's update, its two solve forms agree, and the tolerance tests/test_gpu_enkf_paths.py applies at each of its
solve cases is sharp enough to catch a kernel that is subtly wrong."""
import numpy as np
import pytest

import enkf_reference as E
from parity import relerr, normerr


def _move(a, b):
    return normerr(np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64))


def test_longdouble_is_wider_than_fp64():
    assert np.finfo(E.LD).eps < 1e-18
    x = E.LD(1) + E.LD(2.0) ** -60
    assert x != E.LD(1)


def test_cholesky_and_solve():
    rng = np.random.default_rng(3)
    A = rng.standard_normal((30, 30))
    S = A @ A.T + 30 * np.eye(30)
    L = E.cholesky(S)
    assert np.abs(np.asarray(L @ L.T - S, dtype=np.float64)).max() < 1e-15 * np.abs(S).max()
    B = rng.standard_normal((30, 5))
    X = E.chol_solve(L, B)
    assert normerr(np.asarray(X, dtype=np.float64), np.linalg.solve(S, B)) < 1e-13
    with pytest.raises(np.linalg.LinAlgError):
        E.cholesky(-S)


@pytest.mark.parametrize("M,m", [(16, 20), (40, 12), (7, 30)])
def test_reference_reproduces_oracle_update(oracle, M, m):
    """solve_ref + apply_ref = oracle.enkf_update (explicit inverse in FP64, the reference's algebra) to 1e-13,
    element-wise relative to max(|posterior|, |forecast|)."""
    fc = E.forecast()
    n = fc["O"].shape[0]
    inp = E.solve_inputs(M, m, E.case_seed(M, m))
    O, I = fc["O"][:, :M], fc["I"][:, :M]
    g = inp["gauges"]
    q = np.ones(n)
    q[g] = inp["qs"]
    T, W, _ = E.solve_ref(inp["HX"], inp["Zp"], inp["mean"], inp["qs"], inp["R"])
    Op, Ip = E.apply_ref(O, I, inp["mean_all"], T, W, g, inp["qs"], fc["endnodes"])
    net = {"startnodes": fc["startnodes"], "endnodes": fc["endnodes"],
           "indegree": oracle.compute_indegree(fc["startnodes"], fc["endnodes"])}
    Oo, Io, _ = oracle.enkf_update(net, O, I, g, inp["Zp"], q, inp["R"])
    assert relerr(np.asarray(Op, dtype=np.float64), Oo, scale=np.abs(O)) < 1e-13
    assert relerr(np.asarray(Ip, dtype=np.float64), Io, scale=np.abs(I)) < 1e-13


@pytest.mark.parametrize("M,m", [(2, 30), (8, 60), (33, 120), (64, 401)])
def test_solve_forms_agree(M, m):
    """The m x m form and the M x M push-through form give the same T and W (both in longdouble)."""
    inp = E.solve_inputs(M, m, E.case_seed(M, m))
    a = E.solve_direct(inp["HX"], inp["Zp"], inp["mean"], inp["qs"], inp["R"])
    b = E.solve_pushthrough(inp["HX"], inp["Zp"], inp["mean"], inp["qs"], inp["R"])
    assert _move(b[0], a[0]) < 1e-15
    assert _move(b[1], a[1]) < 1e-15


def test_cond_bound_bounds_cond():
    for M, m in ((3, 300), (64, 350)):
        inp = E.solve_inputs(M, m, E.case_seed(M, m))
        _, _, S = E.solve_direct(inp["HX"], inp["Zp"], inp["mean"], inp["qs"], inp["R"])
        c = E.cond_spd(np.asarray(S, dtype=np.float64))
        b = E.cond_bound_lowrank(inp["HX"], inp["mean"], inp["qs"], inp["R"])
        assert c <= b * (1 + 1e-9)
        d = inp["qs"] + np.diagonal(inp["R"])
        assert b <= c * d.max() / d.min() * (1 + 1e-9)


def _mutants(inp, m):
    """T and W of five subtly wrong updates: M for M - 1, the last gauge dropped, the mean over M + 1 columns
    (a zero pad column counted as a member), T transposed, Q[s, s] left out."""
    HX, Zp, mean, qs, R = inp["HX"], inp["Zp"], inp["mean"], inp["qs"], inp["R"]
    M = HX.shape[1]
    form = E.solve_direct if m <= E.DIRECT_MAX_M else E.solve_pushthrough
    out = {"M for M-1": form(HX, Zp, mean, qs, R, denom=M)[:2]}
    if m > 1:
        out["last gauge dropped"] = form(HX[:-1], Zp[:-1], mean[:-1], qs[:-1], R[:-1, :-1])[:2]
    else:
        out["last gauge dropped"] = (np.zeros((M, M)), np.zeros((0, M)))
    out["mean over M+1 columns"] = form(HX, Zp, mean * M / (M + 1), qs, R)[:2]
    out["qs left out"] = form(HX, Zp, mean, np.zeros_like(qs), R)[:2]
    return out


@pytest.mark.parametrize("M,m,dense_R,dinv_kind,path", E.SOLVE_CASES)
def test_solve_tolerance_is_sharp(M, m, dense_R, dinv_kind, path):
    inp, T, W, tol = E.case_reference(M, m, dense_R, dinv_kind, path)
    bar = 1e3 * tol
    assert _move(T.T, T) > bar, "T transposed"
    for name, (Tm, Wm) in _mutants(inp, m).items():
        k = min(Wm.shape[0], W.shape[0])
        moved = max(_move(Tm, T), _move(Wm[:k], W[:k]) if k else 0.0)
        assert moved > bar, f"{name}: moves T / W by {moved:.2e}, the bar is {bar:.2e}"

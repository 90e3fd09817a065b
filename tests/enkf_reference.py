"""Extended-precision reference of the ensemble Kalman update (test infrastructure, CPU, numpy).

The solve, for M members and m gauges (HX [m][M] the gauge rows of the forecast, Zp [m][M] the perturbed
observations, mean [m] the ensemble mean at the gauges, qs [m] the diagonal of Q at the gauges, R [m][m]):

    HA = HX - mean,   dz = Zp - HX,   S = HA HA^T / (M - 1) + diag(qs) + R
    W  = S^-1 dz      [m][M]
    T  = HA^T W / (M - 1)   [M][M]

so that the gain of every state row is (O - mean) T + Q[:, s] W.  Both solve forms of the library (the m x m system
and the M x M ensemble-space one) must meet this contract.  Everything here runs in np.longdouble (x87 80-bit on
x86-64: 64-bit mantissa, eps = 1.1e-19), so the reference is about 2,000 times more precise than FP64 and its own
rounding is invisible at the FP64 tolerances the GPU tests apply.  numpy's linalg has no longdouble support: the
Cholesky factorisation and the triangular solves are written out here.
"""
import functools

import numpy as np

LD = np.longdouble
assert np.finfo(LD).eps < 1e-18, "np.longdouble is no wider than FP64 on this platform: the reference would be FP64"

EPS64 = float(np.finfo(np.float64).eps)
DIRECT_MAX_M = 400                 # solve_ref: m x m Cholesky up to here, the M x M push-through form beyond


def cholesky(A):
    """Lower-triangular L with L L^T = A (right-looking, in longdouble).  Raises on a non-positive pivot."""
    A = np.array(A, dtype=LD)
    n = A.shape[0]
    L = np.zeros_like(A)
    for j in range(n):
        d = A[j, j]
        if not d > 0:
            raise np.linalg.LinAlgError(f"matrix is not positive definite (pivot {j})")
        L[j, j] = np.sqrt(d)
        col = A[j + 1:, j] / L[j, j]
        L[j + 1:, j] = col
        A[j + 1:, j + 1:] -= np.outer(col, col)
    return L


def chol_solve(L, B):
    """X = (L L^T)^-1 B for lower-triangular L, B [n][k], in longdouble."""
    B = np.array(B, dtype=LD)
    n = L.shape[0]
    Y = np.empty_like(B)
    for i in range(n):
        Y[i] = (B[i] - L[i, :i] @ Y[:i]) / L[i, i]
    X = np.empty_like(B)
    for i in range(n - 1, -1, -1):
        X[i] = (Y[i] - L[i + 1:, i] @ X[i + 1:]) / L[i, i]
    return X


def _innovation(HX, Zp, mean):
    HX = np.asarray(HX, dtype=LD)
    HA = HX - np.asarray(mean, dtype=LD).reshape(-1, 1)
    dz = np.asarray(Zp, dtype=LD) - HX
    return HA, dz


def solve_direct(HX, Zp, mean, qs, R, denom=None):
    """The m x m form: (T, W, S) with S the innovation covariance, all longdouble.  `denom` replaces M - 1."""
    HA, dz = _innovation(HX, Zp, mean)
    M = HA.shape[1]
    dn = LD(M - 1) if denom is None else LD(denom)
    S = HA @ HA.T / dn + np.diag(np.asarray(qs, dtype=LD)) + np.asarray(R, dtype=LD)
    W = chol_solve(cholesky(S), dz)
    T = HA.T @ W / dn
    return T, W, S


def solve_pushthrough(HX, Zp, mean, qs, R, denom=None):
    """The M x M form for a diagonal D = diag(qs) + R: with C = (M-1) I + HA^T D^-1 HA (push-through identity /
    Woodbury), T = C^-1 HA^T D^-1 dz and W = D^-1 (dz - HA T).  Returns (T, W, C), longdouble."""
    R = np.asarray(R, dtype=LD)
    if np.count_nonzero(R - np.diag(np.diagonal(R))):
        raise ValueError("the push-through form here needs a diagonal R")
    HA, dz = _innovation(HX, Zp, mean)
    M = HA.shape[1]
    dn = LD(M - 1) if denom is None else LD(denom)
    dinv = LD(1) / (np.asarray(qs, dtype=LD) + np.diagonal(R))
    DA = HA * dinv[:, None]
    C = HA.T @ DA + dn * np.eye(M, dtype=LD)
    T = chol_solve(cholesky(C), DA.T @ dz)
    W = (dz - HA @ T) * dinv[:, None]
    return T, W, C


def solve_ref(HX, Zp, mean, qs, R):
    """(T, W, condS): the extended-precision T and W (longdouble) and cond(S).  `mean` is the ensemble mean at the
    gauges ([m], the state mean restricted to the gauged rows).  Up to DIRECT_MAX_M gauges the m x m system is
    solved and cond(S) computed; beyond, the M x M push-through form (R must then be diagonal) and condS is the
    upper bound of cond_bound_lowrank."""
    m = np.shape(HX)[0]
    if m <= DIRECT_MAX_M:
        T, W, S = solve_direct(HX, Zp, mean, qs, R)
        return T, W, cond_spd(np.asarray(S, dtype=np.float64))
    T, W, _ = solve_pushthrough(HX, Zp, mean, qs, R)
    return T, W, cond_bound_lowrank(HX, mean, qs, R)


def cond_bound_lowrank(HX, mean, qs, R):
    """An upper bound of cond(S) for S = D + HA HA^T / (M-1), D diagonal, from M x M quantities only (an m x m
    eigensolve at thousands of gauges costs seconds): HA HA^T is positive semi-definite, so
    lambda_min(S) >= min(D), and lambda_max(S) <= max(D) + ||HA||_2^2 / (M-1).  With more gauges than members
    HA HA^T is singular and lambda_min(S) <= max(D): the bound is within a factor max(D) / min(D) of cond(S)."""
    HA = np.asarray(HX, dtype=np.float64) - np.asarray(mean, dtype=np.float64).reshape(-1, 1)
    d = np.asarray(qs, dtype=np.float64) + np.diagonal(np.asarray(R, dtype=np.float64))
    top = float(np.linalg.eigvalsh(HA.T @ HA)[-1]) / (HA.shape[1] - 1)
    return (float(d.max()) + top) / float(d.min())


def cond_spd(S):
    """2-norm condition number of a symmetric positive definite matrix."""
    ev = np.linalg.eigvalsh(np.asarray(S, dtype=np.float64))
    return float(ev[-1] / ev[0])


def ensemble_space_cond(HX, mean, qs, R):
    """cond((M-1) I + HA^T D^-1 HA), D = diag(qs) + R: the matrix the ensemble-space solve factors."""
    HA = np.asarray(HX, dtype=np.float64) - np.asarray(mean, dtype=np.float64).reshape(-1, 1)
    R = np.asarray(R, dtype=np.float64)
    if np.count_nonzero(R - np.diag(np.diagonal(R))):
        DA = np.linalg.solve(np.diag(np.asarray(qs, dtype=np.float64)) + R, HA)
    else:
        DA = HA / (np.asarray(qs, dtype=np.float64) + np.diagonal(R))[:, None]
    C = HA.T @ DA + (HA.shape[1] - 1) * np.eye(HA.shape[1])
    return cond_spd((C + C.T) / 2)


def solve_tolerance(condS, cond_ens=None):
    """Max-norm relative bound on the FP64 T and W of the device: max(1e-12, 64 eps cond), cond the larger of
    cond(S) and, on the ensemble-space paths, that of the M x M system.  A backward-stable Cholesky solve has a
    forward error of a small multiple of eps * cond relative to the solution; 64 covers the accumulation
    orders of the split-K products."""
    c = max(condS, cond_ens or 0.0)
    return max(1e-12, 64.0 * EPS64 * c)


def apply_ref(O, I, mean, T, W, gauges, qs, endnodes):
    """The posterior (O', I') in longdouble, in reach order: O' = O + (O - mean) T + Q[:, s] W, and every reach's
    inflow takes the gains of the reaches draining into it (nutils.py:116-134; an outlet drains into itself and
    adds nothing).  O, I [n][M], mean [n], T [M][M], W [m][M], gauges [m], qs [m]."""
    O = np.asarray(O, dtype=LD)
    gain = (O - np.asarray(mean, dtype=LD)[:, None]) @ np.asarray(T, dtype=LD)
    g = np.asarray(gauges, dtype=np.int64)
    gain[g] += np.asarray(qs, dtype=LD)[:, None] * np.asarray(W, dtype=LD)
    return gain_to_state(gain, O, I, endnodes)


def gain_to_state(gain, O_cols, I_cols, endnodes):
    end = np.asarray(endnodes, dtype=np.int64)
    n = end.size
    O_post = np.asarray(O_cols, dtype=LD) + gain
    I_post = np.array(I_cols, dtype=LD)
    up = end != np.arange(n)
    np.add.at(I_post, end[up], gain[up])
    return O_post, I_post


def apply_ref_shard(O_full, I_shard, mean, T, W, gauges, qs, endnodes, col0, Mloc):
    """apply_ref of the whole ensemble O_full [n][Mtot], restricted to the columns col0 .. col0 + Mloc (a shard)."""
    cols = slice(col0, col0 + Mloc)
    O = np.asarray(O_full, dtype=LD)
    gain = (O - np.asarray(mean, dtype=LD)[:, None]) @ np.asarray(T, dtype=LD)[:, cols]
    g = np.asarray(gauges, dtype=np.int64)
    gain[g] += np.asarray(qs, dtype=LD)[:, None] * np.asarray(W, dtype=LD)[:, cols]
    return gain_to_state(gain, O[:, cols], I_shard, endnodes)


# ---- inputs shared by the CPU and GPU tests ---------------------------------------------------------------------
FORECAST_N, FORECAST_M, FORECAST_SEED = 4000, 257, 71


@functools.lru_cache(maxsize=None)
def forecast(n=FORECAST_N, M=FORECAST_M, seed=FORECAST_SEED, steps=6):
    """A real ensemble forecast (synthetic network, members started from perturbed outflows, routed `steps` steps
    by the CPU oracle with per-member forcing multipliers).  Returns a dict with the network, the outflows and
    inflows [n][M] in reach order.  Member k of a smaller ensemble is column k."""
    from oracle import oracle as Orc
    from tx_fast_hydrology_b200 import synthetic as Syn
    net = Syn.make_network(n, seed)
    prm = Syn.make_params(n, seed, well_posed=True)
    rng = np.random.default_rng(seed)
    o = np.ascontiguousarray((prm["o_t"][:, None] * rng.uniform(0.5, 1.5, size=(n, M))).T)
    i = np.stack([Orc.init_states(net["startnodes"], net["endnodes"], x) for x in o])
    al, be, ch, ga = Orc.compute_coeffs(prm["K"], prm["X"], 300.0)
    onet = {"startnodes": net["startnodes"], "endnodes": net["endnodes"],
            "indegree": Orc.compute_indegree(net["startnodes"], net["endnodes"]),
            "alpha": al, "beta": be, "chi": ch, "gamma": ga}
    t0 = 1_700_000_000 * 10**9
    times, table = Syn.make_forcing(n, steps, 300.0, seed, t0_ns=t0, rows_every=2)
    mul = Syn.make_member_multipliers(times.size, M, seed)
    Orc.run_members(onet, o, i, steps, times.astype(np.float64), table, float(t0), 300e9, wmul=mul)
    return {"endnodes": net["endnodes"], "startnodes": net["startnodes"], "O": np.ascontiguousarray(o.T),
            "I": np.ascontiguousarray(i.T)}


def gauge_set(endnodes, m, seed):
    """m distinct gauged reaches, ascending: outlets and confluences first, then random reaches."""
    end = np.asarray(endnodes, dtype=np.int64)
    n = end.size
    rng = np.random.default_rng(seed)
    indeg = np.bincount(end[end != np.arange(n)], minlength=n)
    special = np.concatenate([np.flatnonzero(end == np.arange(n))[:3], np.flatnonzero(indeg >= 2)[:4]])
    special = np.unique(special)[:max(0, m // 2)]
    rest = rng.choice(np.setdiff1d(np.arange(n), special), size=m - special.size, replace=False)
    return np.sort(np.concatenate([special, rest])).astype(np.int64)


def solve_inputs(M, m, seed, dense_R=False):
    """Inputs of one solve case, all FP64 (the device and the reference see the same numbers): gauges, HX (the gauge
    rows of the forecast, M members), the ensemble mean at every reach (reach order) and at the gauges, Zp
    (measurements near the ensemble mean plus noise of the observation error's size), qs and R."""
    fc = forecast()
    O = fc["O"][:, :M]
    g = gauge_set(fc["endnodes"], m, seed)
    rng = np.random.default_rng(1000 + seed)
    mean = O.sum(axis=1) / M
    HX = np.ascontiguousarray(O[g])
    qs = rng.uniform(0.05, 0.5, size=m) * mean[g] ** 2 * 1e-2
    if dense_R:
        B = rng.standard_normal((m, m))
        R = 1e-2 * (np.eye(m) + 0.5 * (B @ B.T) / m)
    else:
        R = np.diag(rng.uniform(0.5e-2, 2e-2, size=m))
    z = mean[g] * rng.uniform(0.8, 1.2, size=m)
    Zp = np.ascontiguousarray(z[:, None] + 0.1 * rng.standard_normal((m, M)))
    return {"gauges": g, "HX": HX, "mean_all": mean, "mean": mean[g].copy(), "Zp": Zp, "qs": qs, "R": R}


# The solve cases of tests/test_gpu_enkf_paths.py: (M, m, dense_R, dinv_kind, path).  dinv_kind is what the solve
# is given: 1 the diagonal of D^-1 (what the filter passes for a diagonal D = diag(qs) + R), 2 the full matrix D^-1
# (what it passes for a dense R; here also for a diagonal D), 0 none.  `path` names the dispatch row of
# txh_capi.cu:enkf_solve_impl the case takes: "cluster" (M < m, M <= 64, dinv_kind 1), "woodbury" (M < m, M <= 128,
# dinv_kind 2 or M > 64), "woodbury_big" (M < m, M > 128), "direct" (M >= m, or dinv_kind 0).
def _solve_cases():
    cases = []
    for M in (2, 3, 7, 8, 9, 31, 33, 57, 63, 64):
        for m in sorted({M + 1, 17, 65, 500, 1025, 2100}):
            if M < m:
                cases.append((M, m, False, 1, "cluster"))
    for M in (33, 64, 65, 95, 97, 127, 128):
        cases.append((M, 160, True, 2, "woodbury"))
        cases.append((M, 150, False, 2, "woodbury"))
    cases += [(65, 300, False, 1, "woodbury"), (97, 300, False, 1, "woodbury")]
    cases += [(129, 450, False, 1, "woodbury_big"), (200, 520, False, 1, "woodbury_big"),
              (129, 170, True, 2, "woodbury_big")]
    cases += [(64, m, False, 1, "direct") for m in (1, 2, 63, 64)]
    cases += [(33, 33, False, 1, "direct"), (64, 64, True, 2, "direct"), (16, 40, False, 0, "direct")]
    return cases


SOLVE_CASES = _solve_cases()


def case_seed(M, m):
    return 7919 * M + m


ENSEMBLE_SPACE_PATHS = ("cluster", "woodbury", "woodbury_big")


def case_reference(M, m, dense_R, dinv_kind, path):
    """The inputs of a solve case, its reference (T, W) and the tolerance the GPU test applies to them."""
    inp = solve_inputs(M, m, case_seed(M, m), dense_R)
    T, W, condS = solve_ref(inp["HX"], inp["Zp"], inp["mean"], inp["qs"], inp["R"])
    ce = ensemble_space_cond(inp["HX"], inp["mean"], inp["qs"], inp["R"]) if path in ENSEMBLE_SPACE_PATHS else None
    return inp, T, W, solve_tolerance(condS, ce)

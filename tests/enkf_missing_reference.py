"""Reference of the ensemble Kalman update with missing gauge observations (test infrastructure, CPU, numpy).

A gauge is missing at an update when its row of the perturbed observations Zp holds a NaN in any member.  With a
diagonal R the update must then equal the update of a filter without that gauge: T is the transform of the reduced
system and W is its W with zero rows at the missing gauges (tests/enkf_reference.py:solve_ref on the kept gauges).
With every gauge missing, T = 0 and W = 0.

Also the masks the GPU tests plant per solve case, and the planted defects the CPU tests show the GPU tolerance to
catch.
"""
import numpy as np

import enkf_reference as E


def missing_rows(Zp):
    """The rule: a row is missing when it holds a NaN in any member."""
    return np.isnan(np.asarray(Zp, dtype=np.float64)).any(axis=1)


def solve_masked(HX, Zp, mean, qs, R, miss=None):
    """(T, W, condS, cond_ens) of the update without the gauges `miss` ([m] bool; None: the rule on Zp): solve_ref of
    the kept gauges, W zero-filled back to m rows; T and W longdouble.  cond_ens: that of the reduced ensemble-space
    system (None when nothing is kept, or never asked for by the caller).  An empty mask is solve_ref itself."""
    HX = np.asarray(HX, dtype=np.float64)
    m, M = HX.shape
    miss = missing_rows(Zp) if miss is None else np.asarray(miss, dtype=bool)
    if not miss.any():
        T, W, condS = E.solve_ref(HX, Zp, mean, qs, R)
        return T, W, condS, E.ensemble_space_cond(HX, mean, qs, R)
    keep = ~miss
    W = np.zeros((m, M), dtype=E.LD)
    if not keep.any():
        return np.zeros((M, M), dtype=E.LD), W, 1.0, None
    R = np.asarray(R, dtype=np.float64)
    sub = (HX[keep], np.asarray(Zp)[keep], np.asarray(mean)[keep], np.asarray(qs)[keep], R[np.ix_(keep, keep)])
    T, Wk, condS = E.solve_ref(*sub)
    W[keep] = Wk
    return T, W, condS, E.ensemble_space_cond(sub[0], sub[2], sub[3], sub[4])


def masked_tolerance(condS, cond_ens, path):
    """The solve tolerance of tests/enkf_reference.py for the reduced system."""
    return E.solve_tolerance(condS, cond_ens if path in E.ENSEMBLE_SPACE_PATHS else None)


# ---- the masks of the GPU solve tests ----------------------------------------------------------------------------
MASKS = ("none", "one", "edges", "cta", "all_but_one", "all", "one_member")


def cta_share(m, nc=16):
    """Gauges per CTA of enkf_small_system_kernel with nc CTAs (txh_da.cu: mc)."""
    return ((-(-m // nc)) + 3) & ~3


def plant(Zp, kind):
    """Zp with the NaNs of mask `kind`: whole rows (a gap in the gauge's feed) except `one_member`, which puts a NaN in
    the last member of one row only (a NaN in that member's observation noise).  Returns (Zp', missing rows)."""
    Zp = np.array(Zp, dtype=np.float64, copy=True)
    m, M = Zp.shape
    rows = set()
    if kind == "one":
        rows = {m // 2}
    elif kind == "edges":
        # first and last gauge of a 64-gauge tile and of a cluster CTA's share (16 or 8 CTAs)
        rows = {0, 63, 64, m - 1}
        for nc in (16, 8):
            mc = cta_share(m, nc)
            rows |= {mc - 1, mc, 2 * mc - 1, mc + 63, mc + 64}
    elif kind == "cta":
        mc = cta_share(m)
        rows = set(range(mc, min(m, 2 * mc))) if mc < m else set(range((m + 1) // 2))
    elif kind == "all_but_one":
        rows = set(range(m)) - {m // 3}
    elif kind == "all":
        rows = set(range(m))
    elif kind == "one_member":
        Zp[(m - 1) // 2, M - 1] = np.nan
        return Zp, missing_rows(Zp)
    elif kind != "none":
        raise ValueError(kind)
    rows = sorted(r for r in rows if 0 <= r < m)
    Zp[rows] = np.nan
    return Zp, missing_rows(Zp)


# ---- planted defects ---------------------------------------------------------------------------------------------
def filled(HX, Zp):
    """The NaN entries of Zp replaced by the forecast, i.e. dz = 0 there."""
    Zp = np.asarray(Zp, dtype=np.float64)
    return np.where(np.isnan(Zp), np.asarray(HX, dtype=np.float64), Zp)


def defect_dz_zero(HX, Zp, mean, qs, R):
    """A missing gauge treated as observed to equal the forecast: dz = 0, the gauge kept with its weight."""
    T, W, _ = E.solve_ref(HX, filled(HX, Zp), mean, qs, R)
    return T, W


def defect_dz_only_direct(HX, Zp, mean, qs, R):
    """The direct form with only the dz row of a missing gauge zeroed, its HA row kept (so S still couples it)."""
    miss = missing_rows(Zp)
    HA = np.asarray(HX, dtype=E.LD) - np.asarray(mean, dtype=E.LD).reshape(-1, 1)
    dz = np.asarray(Zp, dtype=E.LD) - np.asarray(HX, dtype=E.LD)
    dz[miss] = 0
    M = HA.shape[1]
    S = HA @ HA.T / E.LD(M - 1) + np.diag(np.asarray(qs, dtype=E.LD)) + np.asarray(R, dtype=E.LD)
    W = E.chol_solve(E.cholesky(S), dz)
    return HA.T @ W / E.LD(M - 1), W


def defect_shifted(HX, Zp, mean, qs, R):
    """The mask shifted by one gauge (NaN entries zeroed so the defect is finite)."""
    miss = np.roll(missing_rows(Zp), 1)
    T, W, _, _ = solve_masked(HX, filled(HX, Zp), mean, qs, R, miss)
    return T, W


def defect_member0(HX, Zp, mean, qs, R):
    """The mask read from member 0 only; NaN entries elsewhere zeroed."""
    miss = np.isnan(np.asarray(Zp)[:, 0])
    T, W, _, _ = solve_masked(HX, filled(HX, Zp), mean, qs, R, miss)
    return T, W


def defect_late(HX, Zp, mean, qs, R, miss_before):
    """The mask of the previous update applied to this one (NaN entries zeroed)."""
    T, W, _, _ = solve_masked(HX, filled(HX, Zp), mean, qs, R, miss_before)
    return T, W

"""Missing gauge observations (NaN) in the ensemble Kalman filter, on the CPU: the masked reference the GPU tests use
(tests/enkf_missing_reference.py), the host interpolation rule of EnsembleKalmanFilter.perturbed_observations
(da.interpolate_gappy), and the sharpness of the GPU tolerance against planted defects."""
import os

import numpy as np
import pytest

import enkf_reference as E
import enkf_missing_reference as X
from parity import normerr
from tx_fast_hydrology_b200 import nutils
from tx_fast_hydrology_b200.da import interpolate_gappy


# ---- the masked reference ------------------------------------------------------------------------------------------
def test_masked_reference_empty_mask_is_solve_ref():
    inp = E.solve_inputs(33, 120, E.case_seed(33, 120))
    args = (inp["HX"], inp["Zp"], inp["mean"], inp["qs"], inp["R"])
    T0, W0, c0 = E.solve_ref(*args)
    T, W, c, _ = X.solve_masked(*args)
    assert np.array_equal(T, T0) and np.array_equal(W, W0) and c == c0


def test_masked_reference_full_mask_is_zero():
    inp = E.solve_inputs(33, 120, E.case_seed(33, 120))
    Zp, miss = X.plant(inp["Zp"], "all")
    assert miss.all()
    T, W, _, _ = X.solve_masked(inp["HX"], Zp, inp["mean"], inp["qs"], inp["R"])
    assert not np.abs(T).any() and not np.abs(W).any()


def test_masked_reference_is_the_reduced_filter():
    """Kept gauges: the reduced system's W; missing gauges: zero rows; a NaN in one member masks the whole row."""
    inp = E.solve_inputs(31, 90, E.case_seed(31, 90))
    Zp, miss = X.plant(inp["Zp"], "one_member")
    assert miss.sum() == 1 and np.isnan(Zp).sum() == 1
    T, W, _, _ = X.solve_masked(inp["HX"], Zp, inp["mean"], inp["qs"], inp["R"])
    k = ~miss
    Tr, Wr, _ = E.solve_ref(inp["HX"][k], inp["Zp"][k], inp["mean"][k], inp["qs"][k], inp["R"][np.ix_(k, k)])
    assert np.array_equal(T, Tr) and np.array_equal(W[k], Wr) and not W[miss].any()


# ---- the host interpolation rule -----------------------------------------------------------------------------------
@pytest.mark.parametrize("fname", ["kernels_n60.npz", "kernels_n160.npz"])
def test_gappy_interpolation_of_a_finite_table_is_interpolate_sample(golden_dir, fname):
    g = np.load(os.path.join(golden_dir, fname))
    for x in g["xs"]:
        a = interpolate_gappy(float(x), g["xp"], g["fp"])
        assert np.array_equal(a, nutils.interpolate_sample(float(x), g["xp"], g["fp"]))


def _gappy_table():
    xp = np.array([0.0, 10.0, 20.0, 30.0, 40.0])
    rng = np.random.default_rng(3)
    fp = rng.uniform(1.0, 5.0, size=(5, 4))
    return xp, fp


def _probe_times(xp):
    mids = (xp[:-1] + xp[1:]) / 2
    return np.unique(np.concatenate([xp, mids, xp[:-1] + 1e-3, xp[1:] - 1e-3, [xp[0] - 5, xp[-1] + 5]]))


@pytest.mark.parametrize("j", [0, 2, 4])
def test_gappy_interpolation_masks_exactly_where_the_nan_row_has_weight(j):
    xp, fp = _gappy_table()
    gap = fp.copy()
    gap[j, 1] = np.nan
    n = xp.size
    for x in _probe_times(xp):
        a = interpolate_gappy(float(x), xp, gap)
        lo = xp[j - 1] if j > 0 else -np.inf
        hi = xp[j + 1] if j + 1 < n else np.inf
        weighted = lo < x < hi                      # row j's weight: frac on (xp[j-1], xp[j]], 1 - frac on [xp[j], xp[j+1])
        assert np.isnan(a[1]) == weighted, (x, a)
        ref = nutils.interpolate_sample(float(x), xp, fp)
        others = [0, 2, 3]
        assert np.array_equal(a[others], ref[others])
        if not weighted:
            assert a[1] == ref[1]


def test_gappy_interpolation_exact_row_time_after_a_nan_row():
    """interpolate_sample gives NaN at the exact time of the row after a NaN row (0 * NaN); the rule does not."""
    xp, fp = _gappy_table()
    gap = fp.copy()
    gap[1, :] = np.nan
    with np.errstate(invalid="ignore"):
        assert np.isnan(nutils.interpolate_sample(20.0, xp, gap)).all()
    assert np.array_equal(interpolate_gappy(20.0, xp, gap), fp[2])
    assert np.isnan(interpolate_gappy(19.0, xp, gap)).all()
    assert np.isnan(interpolate_gappy(10.0, xp, gap)).all()


def test_gappy_interpolation_clamped_ends():
    xp, fp = _gappy_table()
    gap = fp.copy()
    gap[0, 0] = np.nan
    gap[-1, 3] = np.nan
    a, b = interpolate_gappy(-3.0, xp, gap), interpolate_gappy(99.0, xp, gap)
    assert np.isnan(a[0]) and np.array_equal(a[1:], fp[0, 1:])
    assert np.isnan(b[3]) and np.array_equal(b[:3], fp[-1, :3])


# ---- sharpness: every planted defect misses the GPU tolerance by more than 10^3 ------------------------------------
SHARP_CASES = [c for c in E.SOLVE_CASES if c[3] == 1] + [(64, 1100, False, 1, "cluster")]


def _miss_ratio(T, W, ref, tol):
    e = max(normerr(np.asarray(T, dtype=np.float64), np.asarray(ref[0], dtype=np.float64)),
            normerr(np.asarray(W, dtype=np.float64), np.asarray(ref[1], dtype=np.float64)))
    return (np.inf if np.isnan(e) else e) / tol


@pytest.mark.parametrize("M,m,dense_R,dinv_kind,path", SHARP_CASES)
def test_planted_defects_miss_the_tolerance(M, m, dense_R, dinv_kind, path):
    inp = E.solve_inputs(M, m, E.case_seed(M, m), dense_R)
    base = (inp["HX"], inp["mean"], inp["qs"], inp["R"])

    def ref_of(Zp):
        T, W, condS, ce = X.solve_masked(inp["HX"], Zp, inp["mean"], inp["qs"], inp["R"])
        return (T, W), X.masked_tolerance(condS, ce, path)

    def args(Zp):
        return (base[0], Zp) + base[1:]

    Zp1, miss1 = X.plant(inp["Zp"], "one")
    ref1, tol1 = ref_of(Zp1)
    ratios = {}
    Zpm, _ = X.plant(inp["Zp"], "one_member")
    refm, tolm = ref_of(Zpm)
    ratios["member0"] = _miss_ratio(*X.defect_member0(*args(Zpm)), refm, tolm)
    if m >= 2:
        # (with a single gauge, missing means every gauge missing, and dz = 0 everywhere is then the same update:
        # W = S^-1 0 = 0; likewise a shifted or late mask needs a second gauge to differ)
        ratios["dz_zero"] = _miss_ratio(*X.defect_dz_zero(*args(Zp1)), ref1, tol1)
        if path == "direct":
            ratios["dz_only_direct"] = _miss_ratio(*X.defect_dz_only_direct(*args(Zp1)), ref1, tol1)
        ratios["shifted"] = _miss_ratio(*X.defect_shifted(*args(Zp1)), ref1, tol1)
        before = np.zeros(m, dtype=bool)
        before[(m // 2 + 1) % m] = True                 # the previous update missed another gauge
        ratios["late"] = _miss_ratio(*X.defect_late(*args(Zp1), before), ref1, tol1)
    bad = {k: v for k, v in ratios.items() if not v > 1e3}
    assert not bad, f"defects within 10^3 of the tolerance: {bad}"

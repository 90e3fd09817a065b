"""Extended-precision reference of a routing run driven by a forcing table (test infrastructure, CPU, numpy).

Every routing kernel interpolates the lateral inflow of step s from the resident table at the step's end,
x = t0 + (s + 1) dt, as nutils.interpolate_sample does (nutils.py:5-39).  Two layers:

* `step_records` resolves each step to (r0, r1, w0, w1) in FP64, exactly as nutils does: the integer time
  converted to float64 once, np.searchsorted side 'left', clamped ends, frac = dx0 / (dx0 + dx1) and w0 = 1 - frac
  for the linear method, the nearer row (ties to the earlier one) for the nearest method.  These records DEFINE the
  semantics; the kernels must reproduce them bit for bit.
* `route_ref` runs the member-batched recurrence of nutils._ax_bu (o' = alpha i' + beta i + chi o + gamma q,
  i' = sum of the o' draining in) in np.longdouble with the FP64 coefficients and those records, the forcing of
  member m being q = w0 mul[r0, m] F[r0] + w1 mul[r1, m] F[r1].  The same sweep on |coefficients|, |weights|, |F|,
  |mul| and |initial state| (the magnitude run) gives every element a scale, and the running-error bound
  `C_BOUND * u * (nsteps + depth + 4) * scale` (u the FP64 unit roundoff, depth the longest upstream path).  chi and
  alpha can be negative, so a bound relative to the element itself would not be sound; the magnitude run is.

`DEFECTS` are switches that plant one plausible kernel defect each in the reference; a test that cannot tell a
planted defect from the truth by more than 10^3 times the bound could not catch that defect in a kernel either.

The case lists the GPU tests run (tests/test_gpu_forcing.py) live here too, so the CPU tests can show that they
separate every planted defect from the truth.
"""
import functools
import zlib

import numpy as np

from enkf_reference import LD, EPS64

U64 = EPS64 / 2                    # FP64 unit roundoff
# The constant of the bound.  A correct FP64 evaluation (the C oracle, fed the same per-step forcing) stays below
# 0.02 of the bound with C_BOUND = 4, 0.08 with 1 (tests/test_forcing_reference.py reports it); 4 leaves the kernels
# room for their re-associated confluence sums, FMA contraction and the affine hops of spine segments.
C_BOUND = 4.0

DEFECTS = (
    "start_of_step",     # 1: forcing sampled at the start of the step, t0 + s dt
    "ties_later",        # 2: nearest-method ties go to the later row
    "method_ignored",    # 3: the nearest method computed as linear
    "always_shift",      # 4: every bracket change taken as a one-row shift (a cached bracket that only shifts)
    "mul_r0",            # 5: the member multiplier of r0 applied to both rows
    "clamp_r2",          # 6: steps past the last row clamped to row R-2
    "held_bracket",      # 7: the first step of a call uses the previous call's last record
)


# ---------------------------------------------------------------------------------------------------------------
# Step records (FP64, nutils semantics)
# ---------------------------------------------------------------------------------------------------------------
def record_at(xp, x, method, defect=None):
    """(r0, r1, w0, w1) of float64 `x` in the float64 row times `xp` (nutils.py:21-34)."""
    R = len(xp)
    ix = int(np.searchsorted(xp, x, side="left"))
    if ix == 0:
        return 0, 0, 1.0, 0.0
    if ix >= R:
        r = max(R - 2, 0) if defect == "clamp_r2" else R - 1
        return r, r, 1.0, 0.0
    dx0 = float(x - xp[ix - 1])
    dx1 = float(xp[ix] - x)
    if method == 1 or defect == "method_ignored":
        frac = dx0 / (dx0 + dx1)
        return ix - 1, ix, 1.0 - frac, frac
    if defect == "ties_later":
        r = ix - 1 if abs(dx0) < abs(dx1) else ix
    else:
        r = ix - 1 if abs(dx0) <= abs(dx1) else ix
    return r, r, 1.0, 0.0


def step_times(t0_ns, dt_ns, nsteps, defect=None):
    """float64 x of every step: the integer t0 + (s + 1) dt converted once (start of the step for 'start_of_step')."""
    k = 0 if defect == "start_of_step" else 1
    return np.array([float(int(t0_ns) + (s + k) * int(dt_ns)) for s in range(int(nsteps))], dtype=np.float64)


def step_records(times_ns, t0_ns, dt_ns, nsteps, method, defect=None):
    """(r0, r1, w0, w1) per step as int64 / float64 arrays."""
    xp = np.asarray(times_ns).astype(np.float64)
    recs = [record_at(xp, x, method, defect) for x in step_times(t0_ns, dt_ns, nsteps, defect)]
    if not recs:
        return (np.zeros(0, np.int64),) * 2 + (np.zeros(0),) * 2
    r0, r1, w0, w1 = zip(*recs)
    return (np.array(r0, dtype=np.int64), np.array(r1, dtype=np.int64), np.array(w0, dtype=np.float64),
            np.array(w1, dtype=np.float64))


def apply_records(recs, fp):
    """The FP64 rows w0 fp[r0] + w1 fp[r1], term order of nutils (equal to its result bit for bit)."""
    r0, r1, w0, w1 = recs
    fp = np.asarray(fp, dtype=np.float64)
    return w0[:, None] * fp[r0] + w1[:, None] * fp[r1]


# ---------------------------------------------------------------------------------------------------------------
# Topology, vectorised per level
# ---------------------------------------------------------------------------------------------------------------
class Topo:
    """Topological levels of the in-forest `endnodes` (self-loops = outlets) and, per level, the reaches in it and
    how their outflows reduce onto their downstream reaches."""

    def __init__(self, endnodes):
        end = np.asarray(endnodes, dtype=np.int64)
        n = end.size
        ids = np.arange(n, dtype=np.int64)
        flows = end != ids
        indeg = np.bincount(end[flows], minlength=n)
        frontier = ids[indeg == 0]
        pending = indeg.copy()
        lev = 0
        self.levels = []
        while frontier.size:
            self.levels.append(frontier)
            f = frontier[flows[frontier]]
            tgt = end[f]
            np.subtract.at(pending, tgt, 1)
            u = np.unique(tgt)
            frontier = u[pending[u] == 0]
            lev += 1
        assert sum(x.size for x in self.levels) == n, "not a forest of in-trees"
        self.n, self.depth = n, lev
        self.reduce = []
        for idx in self.levels:
            f = idx[flows[idx]]
            order = np.argsort(end[f], kind="stable")
            src = f[order]
            tg = end[src]
            starts = np.flatnonzero(np.r_[True, tg[1:] != tg[:-1]]) if tg.size else np.zeros(0, np.int64)
            self.reduce.append((src, tg[starts], starts))


@functools.lru_cache(maxsize=16)
def _topo_cached(key, end_bytes):
    return Topo(np.frombuffer(end_bytes, dtype=np.int64))


def topo_of(endnodes):
    end = np.ascontiguousarray(endnodes, dtype=np.int64)
    return _topo_cached((end.size, hash(end.tobytes())), end.tobytes())


# ---------------------------------------------------------------------------------------------------------------
# The routing run
# ---------------------------------------------------------------------------------------------------------------
def _pair(x):
    """[n] FP64 -> [n][2] longdouble: the value and its magnitude."""
    x = np.asarray(x, dtype=np.float64)
    return np.stack([x.astype(LD), np.abs(x).astype(LD)], axis=1)


def route_ref(endnodes, alpha, beta, chi, gamma, o0, i0, times, table, mul, t0, dt, nsteps, method,
              defect=None, rec_reach=None, rec_every=1):
    """Routing run of `nsteps` steps (an int, or a list of the step counts of consecutive calls, call k starting
    where call k-1 ended) from the state o0, i0 ([n][M], FP64) with the forcing table `times` [R] (int ns),
    `table` [R][n], `mul` [R][M] or None.  Returns a dict: O, I ([n][M] longdouble), their bounds bO, bI (FP64),
    and with `rec_reach` (a single call only) rec [slots][k][M] and brec, the outflows of those reaches after every
    `rec_every`-th step, as route_run records them."""
    tp = topo_of(endnodes)
    n = tp.n
    calls = [int(nsteps)] if np.isscalar(nsteps) else [int(c) for c in nsteps]
    total = sum(calls)
    o0 = np.asarray(o0, dtype=np.float64).reshape(n, -1)
    i0 = np.asarray(i0, dtype=np.float64).reshape(n, -1)
    M = o0.shape[1]
    A, B, C, G = (_pair(c)[:, :, None] for c in (alpha, beta, chi, gamma))       # [n][2][1]
    O = np.stack([o0.astype(LD), np.abs(o0).astype(LD)], axis=1)                # [n][2][M]
    I = np.stack([i0.astype(LD), np.abs(i0).astype(LD)], axis=1)
    F = np.asarray(table, dtype=np.float64)
    R = F.shape[0]
    FL = np.stack([F.astype(LD), np.abs(F).astype(LD)], axis=1)                  # [R][2][n]
    if mul is None:
        WL = np.ones((R, 2, 1), dtype=LD)
    else:
        mu = np.asarray(mul, dtype=np.float64)
        assert mu.shape == (R, M)
        WL = np.stack([mu.astype(LD), np.abs(mu).astype(LD)], axis=1)           # [R][2][M]
    rec = None
    if rec_reach is not None:
        assert len(calls) == 1, "recording is compared on single calls"
        rec_reach = np.asarray(rec_reach, dtype=np.int64)
        rec = np.zeros((total // rec_every, rec_reach.size, 2, M), dtype=LD)
    base = 0
    prev_last = None
    for ci, ns in enumerate(calls):
        t0c = int(t0) + base * int(dt)
        r0, r1, w0, w1 = step_records(times, t0c, dt, ns, method, defect)
        if defect == "held_bracket" and prev_last is not None and ns > 0:
            r0[0], r1[0], w0[0], w1[0] = prev_last
        if ns > 0:
            prev_last = (r0[-1], r1[-1], w0[-1], w1[-1])
        c0 = c1 = None
        for s in range(ns):
            f0, f1 = r0[s], r1[s]
            if defect == "always_shift":
                # a bracket cache that only knows the one-row shift: (c0, c1) -> (c1, the row after them)
                if s == 0:
                    c0, c1 = r0[s], r1[s]
                elif (r0[s], r1[s]) != (r0[s - 1], r1[s - 1]):
                    c0, c1 = c1, min(max(c0, c1) + 1, R - 1)
                f0, f1 = c0, c1
            m1 = r0[s] if defect == "mul_r0" else r1[s]
            ww0 = np.array([LD(w0[s]), abs(LD(w0[s]))], dtype=LD)[:, None, None]
            ww1 = np.array([LD(w1[s]), abs(LD(w1[s]))], dtype=LD)[:, None, None]
            # q [2][n][M]: w0 mul[r0] F[r0] + w1 mul[r1] F[r1] (value and magnitude)
            q = (ww0 * WL[r0[s]][:, None, :] * FL[f0][:, :, None] + ww1 * WL[m1][:, None, :] * FL[f1][:, :, None])
            q = np.transpose(q, (1, 0, 2))                                       # [n][2][M]
            On = np.empty_like(O)
            In = np.zeros_like(I)
            for idx, (src, tg, starts) in zip(tp.levels, tp.reduce):
                On[idx] = A[idx] * In[idx] + B[idx] * I[idx] + C[idx] * O[idx] + G[idx] * q[idx]
                if src.size:
                    In[tg] += np.add.reduceat(On[src], starts, axis=0)
            O, I = On, In
            gs = s + 1
            if rec is not None and gs % rec_every == 0:
                rec[gs // rec_every - 1] = O[rec_reach]
        base += ns
    k = C_BOUND * U64 * (total + tp.depth + 4)
    out = {"O": O[:, 0], "I": I[:, 0], "bO": k * O[:, 1].astype(np.float64), "bI": k * I[:, 1].astype(np.float64),
           "depth": tp.depth, "steps": total}
    if rec is not None:
        out["rec"] = rec[:, :, 0]
        out["brec"] = k * rec[:, :, 1].astype(np.float64)
    return out


def bound_ratio(got, ref, bound):
    """max |got - ref| / bound over the elements (an element with a zero bound must match exactly)."""
    d = np.abs(np.asarray(got).astype(LD) - np.asarray(ref, dtype=LD)).astype(np.float64)
    b = np.asarray(bound, dtype=np.float64)
    if not np.isfinite(d).all() or np.any((b == 0) & (d != 0)):
        return float("inf")
    with np.errstate(invalid="ignore", divide="ignore"):
        r = np.where(b > 0, d / np.where(b > 0, b, 1.0), 0.0)
    return float(r.max()) if r.size else 0.0


def miss_ratio(ref, other):
    """How far a defective reference run lands outside the bound of the correct one (max over O, I, records)."""
    r = max(bound_ratio(other["O"], ref["O"], ref["bO"]), bound_ratio(other["I"], ref["I"], ref["bI"]))
    if "rec" in ref:
        r = max(r, bound_ratio(other["rec"], ref["rec"], ref["brec"]))
    return r


# ---------------------------------------------------------------------------------------------------------------
# The cases of tests/test_gpu_forcing.py
# ---------------------------------------------------------------------------------------------------------------
T0_NS = 1_700_000_000 * 10 ** 9
DT_NS = 300 * 10 ** 9
_S = 10 ** 9                        # one second in ns

NETWORKS = {
    "n300": (300, 5, 2),
    "n1000": (1000, 1, 3),
    "n3000": (3000, 4, 3),
    "chain": None,                  # make_longchain_network(2000, 2000): a 2,000-reach main stem
}


def make_times(kind, nsteps):
    """Row times (int64 ns) of a table kind for a run of `nsteps` 300 s steps from T0_NS."""
    end = T0_NS + nsteps * DT_NS
    if kind == "aligned":                          # a row every 4 steps from t0 (synthetic.make_forcing's grid)
        return T0_NS + np.arange(nsteps // 4 + 2, dtype=np.int64) * 4 * DT_NS
    if kind == "every_step":                       # a row at every step end
        return T0_NS + np.arange(nsteps + 1, dtype=np.int64) * DT_NS
    if kind == "sub150":                           # two rows per step: the bracket moves 2 rows a step
        return T0_NS - 2 * 150 * _S + np.arange(2 * nsteps + 5, dtype=np.int64) * 150 * _S
    if kind == "sub100":                           # three rows per step
        return T0_NS + np.arange(3 * nsteps + 4, dtype=np.int64) * 100 * _S
    if kind == "irregular":                        # gaps of 1 s to 6 h, off the step grid, one of 5 h 21 min
        gaps = [1, 7, 299, 301, 1033, 3600, 19260, 43, 2, 21600, 611, 150, 899, 5, 7200, 1799, 301, 59]
        t = [T0_NS - 787 * _S]
        i = 0
        while t[-1] <= end + DT_NS:
            t.append(t[-1] + gaps[i % len(gaps)] * _S)
            i += 1
        return np.array(t, dtype=np.int64)
    if kind == "late_start":                       # the first row half way through step 7
        return T0_NS + 15 * DT_NS // 2 + np.arange(nsteps // 3 + 2, dtype=np.int64) * (3 * DT_NS + 41 * _S)
    if kind == "early_end":                        # the last row before the run ends, mid-launch
        last = (3 * nsteps // 5) * DT_NS + 97 * _S
        return T0_NS + np.linspace(0, last, 9).astype(np.int64) // _S * _S
    if kind == "R1":
        return np.array([T0_NS + 11 * DT_NS // 2], dtype=np.int64)
    if kind == "R2":
        return np.array([T0_NS + 13 * DT_NS // 4, T0_NS + 47 * DT_NS // 4], dtype=np.int64)
    if kind == "ties":                             # a row every 2 steps: odd steps end on exact midpoints
        return T0_NS + np.arange(nsteps // 2 + 2, dtype=np.int64) * 2 * DT_NS
    if kind == "offgrid_t0":                       # hourly rows, t0 17 min 13 s past a row
        return T0_NS - 1033 * _S + np.arange(nsteps // 12 + 3, dtype=np.int64) * 3600 * _S
    raise ValueError(kind)


class Case:
    """One routing run: network, table kind, method (1 linear, 0 nearest), members, multipliers, the step counts of
    its calls, and which kernels run it.  `env`: extra environment of the run; `rec`: (reaches, every);
    `lane_in_place`: route_lane_kernel reads the step records of its launch in place, not from shared memory."""

    def __init__(self, name, net, kind, method, M, mul, calls, kernels, env=None, rec=None, lane_in_place=False):
        self.name, self.net, self.kind, self.method, self.M, self.mul = name, net, kind, method, M, mul
        self.calls = [calls] if np.isscalar(calls) else list(calls)
        self.kernels, self.env, self.rec, self.lane_in_place = kernels, dict(env or {}), rec, lane_in_place

    @property
    def nsteps(self):
        return sum(self.calls)

    def __repr__(self):
        return self.name


ALL = ("lane", "window", "dataflow")
WD = ("window", "dataflow")
LIN, NEAR = 1, 0

CASES = [
    # tables x both methods, M in {1, 3}, on every kernel; the step counts cover the window kernel's launch shapes
    # (1, 16: records resolved in the kernel; 17, 64: by the init kernel; 65, 150: several launches)
    Case("aligned-lin", "n1000", "aligned", LIN, 1, False, 17, ALL),
    Case("aligned-near", "n1000", "aligned", NEAR, 3, True, 17, ALL),
    Case("every_step-lin", "n1000", "every_step", LIN, 3, True, 65, ALL),
    Case("every_step-near", "n300", "every_step", NEAR, 1, False, 16, ALL),
    Case("sub150-lin", "n1000", "sub150", LIN, 1, False, 64, ALL),
    Case("sub150-near", "n300", "sub150", NEAR, 3, True, 30, ALL),
    Case("sub100-lin", "n300", "sub100", LIN, 3, True, 65, ALL),
    Case("sub100-near", "n1000", "sub100", NEAR, 1, False, 16, ALL),
    Case("irregular-lin", "n1000", "irregular", LIN, 3, True, 150, ALL),
    Case("irregular-near", "n1000", "irregular", NEAR, 1, False, 150, ALL),
    Case("late_start-lin", "n300", "late_start", LIN, 3, True, 16, ALL),
    Case("late_start-near", "n1000", "late_start", NEAR, 1, False, 30, ALL),
    Case("early_end-lin", "n1000", "early_end", LIN, 1, False, 65, ALL),
    Case("early_end-near", "n300", "early_end", NEAR, 3, True, 40, ALL),
    Case("R1-lin", "n300", "R1", LIN, 3, True, 17, ALL),
    Case("R1-near", "n1000", "R1", NEAR, 1, False, 1, ALL),
    Case("R2-lin", "n1000", "R2", LIN, 1, False, 17, ALL),
    Case("R2-near", "n300", "R2", NEAR, 3, True, 20, ALL),
    Case("ties-near", "n1000", "ties", NEAR, 3, True, 30, ALL),
    Case("ties-lin", "n300", "ties", LIN, 1, False, 30, ALL),
    Case("offgrid_t0-lin", "n1000", "offgrid_t0", LIN, 1, False, 64, ALL),
    Case("offgrid_t0-near", "n300", "offgrid_t0", NEAR, 3, True, 40, ALL),
    # a run split over calls, brackets spanning every call boundary
    Case("calls-lin", "n1000", "irregular", LIN, 3, True, [1, 7, 30, 17, 65], ALL),
    Case("calls-near", "n300", "aligned", NEAR, 1, False, [1, 7, 30, 17, 5], ALL),
    Case("calls-ties", "n300", "ties", NEAR, 3, True, [3, 1, 7, 9], ALL),
    # recorded hydrographs, every 3rd step
    Case("rec-irregular", "n1000", "irregular", LIN, 3, True, 31, ALL, rec=(40, 3)),
    # the lane kernel: 16 members; a launch split (TXH_LANE_SPL) at a step that is not a multiple of the row spacing
    Case("lane16-irregular-near", "n3000", "irregular", NEAR, 16, True, 40, ("lane",)),
    Case("lane16-every_step-lin", "n1000", "every_step", LIN, 16, False, 30, ("lane",)),
    Case("lane-split-aligned", "n1000", "aligned", LIN, 3, True, 30, ("lane",), env={"TXH_LANE_SPL": "7"}),
    Case("lane-split-sub150-near", "n300", "sub150", NEAR, 1, False, 30, ("lane",), env={"TXH_LANE_SPL": "5"}),
    # 16 members on n3000: the largest region leaves shared memory for 432 step records, so these launches read
    # their records in place (the rotate_bracket path, and the shift with the dense-table wait)
    Case("lane16-inplace-irregular-near", "n3000", "irregular", NEAR, 16, True, 450, ("lane",), lane_in_place=True),
    Case("lane16-inplace-every_step-lin", "n3000", "every_step", LIN, 16, False, 440, ("lane",), lane_in_place=True),
    # window and dataflow: 64 members (one member block) and 70 (two)
    Case("m70-irregular-lin", "n3000", "irregular", LIN, 70, True, 65, WD),
    Case("m64-sub100-near", "n1000", "sub100", NEAR, 64, True, 17, WD),
    Case("m70-every_step-lin", "n3000", "every_step", LIN, 70, False, 16, WD),
    Case("m64-ties-near", "n300", "ties", NEAR, 64, False, 30, WD),
    # the long chain: spine segments take the forcing through the affine hop
    Case("chain-irregular-lin", "chain", "irregular", LIN, 1, False, 17, WD),
    Case("chain-ties-near", "chain", "ties", NEAR, 3, True, 12, WD),
]

CASE_BY_NAME = {c.name: c for c in CASES}


def lane_records_in_place(net, M, spl):
    """Whether route_lane_kernel reads the step records of a `spl`-step launch in place: run_lane stages them in
    shared memory only while the largest region (LaneSchedule::region_bytes) and 32 bytes a step fit 200 KiB."""
    s = net.lane_schedule(M)
    mt, rg = s["member_tile"], s["regions"]

    def up16(x):
        return (int(x) + 15) & ~15
    region = max(16 * mt * (r + v + 1) + 256 * mt * v + 16 * v + up16(2 * c) + (up16(8 * mt * r) if mt > 4 else 0)
                 + up16(8 * r) for r, v, c in zip(rg[:, 1], rg[:, 2], rg[:, 4]))
    return ((region + 31) & ~15) + 32 * spl > 200 * 1024


@functools.lru_cache(maxsize=8)
def network(key):
    from tx_fast_hydrology_b200 import synthetic as S
    if key == "chain":
        d = S.make_longchain_network(2000, 2000)
        seed = 5
    else:
        n, seed, nb = NETWORKS[key]
        d = S.make_network(n, seed, n_basins=nb)
    n = d["endnodes"].size
    return d["endnodes"], make_params(n, seed, neg=0.02 if key == "chain" else 0.1)


def make_params(n, seed, neg=0.1):
    """K, X and initial outflows of the cases.  synthetic.make_params draws K up to 7,200 s, so against 300 s steps
    alpha is negative on most reaches; the magnitude run then grows by about 2 K X / dt per reach along every path
    and over the steps, and its bound would sit orders of magnitude above any real error.  Here most reaches have
    all three coefficients non-negative (2 K X <= dt <= 2 K (1 - X)), and a fraction `neg` each has a negative chi
    (dt > 2 K (1 - X)) or a negative alpha (2 K X > dt), so the bound is sharp and still has signs to handle."""
    rng = np.random.default_rng(seed + 7000003)
    dt = DT_NS / 1e9
    X = rng.uniform(0.05, 0.3, size=n)
    lo, hi = dt / (2 * (1 - X)), dt / (2 * X)
    K = lo + rng.uniform(0.02, 0.98, size=n) * (hi - lo)
    kind = rng.uniform(size=n)
    nchi, nal = kind < neg, (kind >= neg) & (kind < 2 * neg)
    K[nchi] = lo[nchi] * rng.uniform(0.6, 0.95, size=int(nchi.sum()))
    K[nal] = hi[nal] * rng.uniform(1.05, 1.5, size=int(nal.sum()))
    o_t = rng.uniform(0.1, 10.0, size=n)
    return {"K": K, "X": X, "o_t": o_t}


def coefficients(K, X, dt_s):
    """muskingum.py:332-360 (the C oracle's arithmetic; the library's is bit-identical to it)."""
    from oracle import oracle as O
    return O.compute_coeffs(K, X, dt_s)


def case_inputs(case):
    """Deterministic inputs of a case: endnodes, coefficients, o0, i0 ([n][M]), times, table, mul, rec reaches."""
    end, prm = network(case.net)
    n = end.size
    seed = zlib.crc32(case.name.encode())
    rng = np.random.default_rng(seed)
    coef = coefficients(prm["K"], prm["X"], DT_NS / 1e9)
    o0 = prm["o_t"][:, None] * rng.uniform(0.5, 1.5, size=(n, case.M))
    i0 = np.zeros_like(o0)
    flows = end != np.arange(n)
    np.add.at(i0, end[flows], o0[flows])
    times = make_times(case.kind, case.nsteps)
    R = times.size
    base = rng.gamma(0.5, 2.0, size=n) + 0.05
    table = np.ascontiguousarray(base[None, :] * rng.uniform(0.2, 1.8, size=(R, n)))
    mul = np.ascontiguousarray(np.exp(0.3 * rng.standard_normal((R, case.M)))) if case.mul else None
    rec = None
    if case.rec is not None:
        rec = (np.sort(rng.choice(n, size=case.rec[0], replace=False)).astype(np.int64), case.rec[1])
    return dict(endnodes=end, coef=coef, o0=o0, i0=i0, times=times, table=table, mul=mul, rec=rec)


def case_ref(case, defect=None, inputs=None):
    x = inputs or case_inputs(case)
    al, be, ch, ga = x["coef"]
    kw = {}
    if x["rec"] is not None:
        kw = dict(rec_reach=x["rec"][0], rec_every=x["rec"][1])
    return route_ref(x["endnodes"], al, be, ch, ga, x["o0"], x["i0"], x["times"], x["table"], x["mul"], T0_NS, DT_NS,
                     case.calls, case.method, defect=defect, **kw)

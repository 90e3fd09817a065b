"""Extended-precision reference of the dense Kalman filter and the RTS smoother (test infrastructure, CPU, numpy).

The update of `KalmanFilter.filter` (da.py:112-126, oracle.OracleKalmanFilter.filter), for the gauged reaches s:

    P-  = A (A P)^T + Q          the routing operator applied to the columns, twice (_aqat_par, nutils.py:194-214)
    S   = P-[s][:, s] + R,   K = P-[:, s] S^-1,   dz = z - o[s],   gain = K dz,   P+ = P- - K P-[s]
    o  += gain,   i[j] += sum of the gains of the reaches draining into j   (_apply_gain, nutils.py:116-134)

and the backward pass of `KalmanSmoother.smooth` (da.py:221-264) as it is written, quirks included: no trailing J^T
on the covariance recursion, J = (P_p[t+1]^-1 A P_f[t])^T.  Everything runs in np.longdouble (tests/enkf_reference.py
checks at import that it is wider than FP64).  `inverse_ref` is the Gauss-Jordan inverse with partial pivoting in the
in-place form the device runs (txh_kf.cu:inverse_in_cta), with switches that plant the defects a test of that kernel
must be able to see.
"""
import numpy as np

from enkf_reference import LD, EPS64

__all__ = ["LD", "EPS64", "topo_order", "ap_ref", "aqat_ref", "apply_gain_ref", "inverse_ref", "kf_update_ref",
           "rts_ref", "inverse_tolerance", "kf_tolerance"]


def topo_order(endnodes):
    """Every reach after all the reaches that drain into it."""
    end = np.asarray(endnodes, dtype=np.int64)
    n = end.size
    up = end != np.arange(n)
    pending = np.bincount(end[up], minlength=n)
    order, frontier = [], list(np.flatnonzero(pending == 0))
    while frontier:
        j = frontier.pop()
        order.append(j)
        e = end[j]
        if e != j:
            pending[e] -= 1
            if pending[e] == 0:
                frontier.append(e)
    assert len(order) == n, "not a forest of in-trees"
    return np.asarray(order, dtype=np.int64)


def ap_ref(P, endnodes, alpha, beta, chi, order=None):
    """A P, column by column as _ap_par does (nutils.py:157-169): a column is o_prev, its inflows i_prev come from
    numba_init_inflows (no self-loop guard: an outlet adds its own outflow to its inflow), then one homogeneous
    routing step o[s] = alpha i_next[s] + beta i_prev[s] + chi o_prev[s] in topological order."""
    P = np.asarray(P, dtype=LD)
    end = np.asarray(endnodes, dtype=np.int64)
    n = end.size
    order = topo_order(end) if order is None else order
    a, b, c = (np.asarray(x, dtype=LD) for x in (alpha, beta, chi))
    i_prev = np.zeros_like(P)
    np.add.at(i_prev, end, P)
    i_next = np.zeros_like(P)
    out = np.zeros_like(P)
    for s in order:
        out[s] = a[s] * i_next[s] + b[s] * i_prev[s] + c[s] * P[s]
        if end[s] != s:
            i_next[end[s]] += out[s]
    return out


def aqat_ref(P, endnodes, alpha, beta, chi):
    """A (A P)^T, the matrix _aqat_par returns (nutils.py:194-214)."""
    order = topo_order(endnodes)
    return ap_ref(ap_ref(P, endnodes, alpha, beta, chi, order).T, endnodes, alpha, beta, chi, order)


def apply_gain_ref(gain, endnodes):
    """(i_gain, o_gain) of _apply_gain (nutils.py:116-134): o takes the gain, the inflow of every reach the gains of
    the reaches draining into it; an outlet drains into itself and adds nothing."""
    g = np.asarray(gain, dtype=LD)
    end = np.asarray(endnodes, dtype=np.int64)
    up = end != np.arange(end.size)
    i_g = np.zeros_like(g)
    np.add.at(i_g, end[up], g[up])
    return i_g, g.copy()


def inverse_ref(A, dtype=LD, unswap="reverse", pivot_factor="moved row"):
    """In-place Gauss-Jordan inverse with partial pivoting, step for step as txh_kf.cu:inverse_in_cta: at column j
    the first row of largest |a[i][j]|, i >= j, is the pivot row pr; rows j and pr are swapped, the pivot row scaled
    (its a[j][j] taken as 1), column j eliminated from every other row, the columns swapped back at the end.
    Returns (inverse, pivot rows).  Raises LinAlgError on a zero pivot.

    The switches plant defects: unswap "none" / "forward" (the column swaps left out / undone first to last), and
    pivot_factor "pivot row" (row pr, which now holds what row j held, eliminated with the factor of the row it
    held before the swap)."""
    a = np.array(A, dtype=dtype)
    m = a.shape[0]
    pivots = []
    for j in range(m):
        col = a[:, j].copy()                       # column j before the swap
        pr = j + int(np.argmax(np.abs(col[j:])))   # argmax: the first of equal maxima
        if col[pr] == 0:
            raise np.linalg.LinAlgError(f"singular matrix (pivot {j})")
        row = a[pr].copy()
        row[j] = 1
        prow = row / col[pr]                       # the scaled pivot row
        a[pr] = a[j]
        f = col.copy()                             # elimination factors: column j as each row holds it now
        if pivot_factor == "moved row":
            f[pr] = col[j]
        f[j] = 0
        a[:, j] = 0
        a -= f[:, None] * prow[None, :]
        a[j] = prow
        pivots.append(pr)
    seq = range(m - 1, -1, -1) if unswap == "reverse" else (range(m) if unswap == "forward" else ())
    for j in seq:
        pr = pivots[j]
        if pr != j:
            a[:, [j, pr]] = a[:, [pr, j]]
    return a, np.asarray(pivots, dtype=np.int64)


def kf_update_ref(P, Q, R, gauges, z, o, i, endnodes, alpha, beta, chi):
    """One KalmanFilter.filter update in longdouble.  gauges ascending; returns a dict with Pm (P-), S, K, dz, gain,
    P (P+), o, i (corrected), all longdouble.  S^-1 by inverse_ref, as the reference takes np.linalg.inv."""
    s = np.asarray(gauges, dtype=np.int64)
    Pm = aqat_ref(P, endnodes, alpha, beta, chi) + np.asarray(Q, dtype=LD)
    S = Pm[np.ix_(s, s)] + np.asarray(R, dtype=LD)
    K = Pm[:, s] @ inverse_ref(S)[0]
    dz = np.asarray(z, dtype=LD) - np.asarray(o, dtype=LD)[s]
    gain = K @ dz
    Pp = Pm - K @ Pm[s]
    i_g, o_g = apply_gain_ref(gain, endnodes)
    return {"Pm": Pm, "S": S, "K": K, "dz": dz, "gain": gain, "P": Pp,
            "o": np.asarray(o, dtype=LD) + o_g, "i": np.asarray(i, dtype=LD) + i_g}


def rts_ref(ts, P_f, P_p, x_f, x_p, endnodes, alpha, beta, chi):
    """KalmanSmoother.smooth (da.py:221-264) on the forward quantities it stored: `ts` the list of update times
    (datetimes), P_f / P_p / x_f / x_p dicts keyed by time (x an [n][2] array of (i, o)).  Returns (x_s, P_s) dicts:
    J = (P_p[t+1]^-1 A P_f[t])^T, x_s[t] = x_f[t] + J (x_s[t+1] - x_p[t+1]), P_s[t] = P_f[t] + J (P_s[t+1] - P_p[t+1])."""
    order = topo_order(endnodes)
    last = ts[-1]
    P_s = {last: np.asarray(P_f[last], dtype=LD)}
    x_s = {last: np.asarray(x_f[last], dtype=LD)}
    for k in reversed(range(len(ts) - 1)):
        t, tp1 = ts[k], ts[k + 1]
        APf = ap_ref(P_f[t], endnodes, alpha, beta, chi, order)
        Pp = np.asarray(P_p[tp1], dtype=LD)
        J = (inverse_ref(Pp)[0] @ APf).T
        x_s[t] = np.asarray(x_f[t], dtype=LD) + J @ (x_s[tp1] - np.asarray(x_p[tp1], dtype=LD))
        P_s[t] = np.asarray(P_f[t], dtype=LD) + J @ (P_s[tp1] - Pp)
    return x_s, P_s


def inverse_tolerance(m, cond):
    """Max-norm relative bound on a computed inverse (or its residual): Gauss-Jordan with partial pivoting has a
    forward error of a small multiple of m eps cond(A) in the 2-norm; the max-norm costs at most another factor m
    between the two sides, which the floor and the constant 1 (not m) leave out, since growth is modest here."""
    return max(1e-12, m * EPS64 * cond)


def kf_tolerance(condS):
    """Max-norm relative bound on K, gain and P+ of one update: the gain is P-[:, s] S^-1, whose forward error is a
    small multiple of eps cond(S) relative to the gain (64 covers the accumulation orders of the products)."""
    return max(1e-12, 64.0 * EPS64 * condS)


# ---- inputs shared by the CPU and GPU tests ---------------------------------------------------------------------
INVERSE_SIZES = (1, 2, 31, 32, 33, 158, 159, 500, 1025)     # 158 | 159: the shared / global memory switch
INVERSE_KINDS = ("permutation", "permuted_dominant", "zero_leading_diagonal", "spd_1e8", "ties")
LD_INVERSE_MAX = 400                                         # beyond: FP64 residuals instead of a longdouble inverse


def inverse_input(kind, m, seed=0):
    """A FP64 test matrix of size m: a permutation (exact inverse: its transpose), a permuted diagonally dominant
    matrix (every column pivots off the diagonal), a well-conditioned matrix with a zero at [0][0], an SPD matrix of
    condition ~1e8 whose pivot sequence has swaps, or a matrix of small integers whose columns tie in |pivot|."""
    rng = np.random.default_rng(1000 * m + INVERSE_KINDS.index(kind) + 17 * seed)
    perm = rng.permutation(m)
    if kind == "permutation":
        return np.eye(m)[perm]
    if kind == "permuted_dominant":
        D = rng.uniform(-1, 1, (m, m)) + np.diag(rng.choice([-1.0, 1.0], m) * (m + rng.uniform(1, 2, m)))
        return D[perm]
    if kind == "zero_leading_diagonal":
        A = rng.standard_normal((m, m)) / np.sqrt(m) + 2.0 * np.eye(m)
        A[0, 0] = 0.0
        return A
    if kind == "spd_1e8":
        U, _ = np.linalg.qr(rng.standard_normal((m, m)))
        A = (U * np.logspace(0, -8, m)) @ U.T
        return (A + A.T) / 2
    if kind == "ties":
        # entries from {-2, -1, 1, 2} with column 0 all +-2: at least the first pivot is a tie between every row
        A = rng.choice([-2.0, -1.0, 1.0, 2.0], size=(m, m)) + 2 * m * np.diag(rng.choice([-1.0, 1.0], m))[perm]
        A[:, 0] = rng.choice([-2.0, 2.0], m)
        return A
    raise ValueError(kind)


DT_S, T0_NS = 300.0, 1_704_067_200 * 10**9            # 2024-01-01T00:00:00Z, the start of synthetic.model_dict


def special_gauges(endnodes, m, seed):
    """m gauged reaches, ascending: heads, confluences and outlets first (where the gain terms of _apply_gain meet
    or stop), then random reaches."""
    end = np.asarray(endnodes, dtype=np.int64)
    n = end.size
    up = end != np.arange(n)
    indeg = np.bincount(end[up], minlength=n)
    special = np.unique(np.concatenate([np.flatnonzero(~up)[:3], np.flatnonzero(indeg >= 2)[:4],
                                        np.flatnonzero(indeg == 0)[:3]]))[:m]
    rng = np.random.default_rng(seed)
    rest = rng.choice(np.setdiff1d(np.arange(n), special), size=m - special.size, replace=False)
    return np.sort(np.concatenate([special, rest])).astype(np.int64)


def neighbour_gauges(endnodes, m):
    """m reaches along downstream paths (each next to the one before it): strongly correlated rows of P."""
    end = np.asarray(endnodes, dtype=np.int64)
    n = end.size
    indeg = np.bincount(end[end != np.arange(n)], minlength=n)
    out = []
    for h in np.flatnonzero(indeg == 0):
        j = int(h)
        while len(out) < m and j not in out:
            out.append(j)
            if end[j] == j:
                break
            j = int(end[j])
        if len(out) >= m:
            break
    return np.sort(np.asarray(out, dtype=np.int64))


def dense_covariances(n, m, seed, rank, r_scale, floor=0.0):
    """Dense SPD Q (rank `rank` plus floor I), P0 = 1.5 Q, dense SPD R = r_scale (I + 0.5 B B^T / m)."""
    rng = np.random.default_rng(seed + 77)
    C = rng.standard_normal((n, rank))
    Q = C @ C.T / rank + floor * np.eye(n)
    B = rng.standard_normal((m, m))
    Rm = r_scale * (np.eye(m) + 0.5 * B @ B.T / m)
    return (Q + Q.T) / 2, (Rm + Rm.T) / 2, 1.5 * (Q + Q.T) / 2


# Dense-filter cases of tests/test_gpu_dense_kf.py: n reaches (3 basins), m gauges chosen by `gauges`, covariances of
# dense_covariances, `cond` the range cond(S) of the first update lies in (tests/test_kf_reference.py checks it).
FILTER_CASES = [
    dict(id="n1_m1", n=1, m=1, gauges="special", rank=1, floor=0.0, r_scale=1e-2, cond=(1, 1)),
    dict(id="n40_every_reach", n=40, m=40, gauges="special", rank=40, floor=0.0, r_scale=1e-2, cond=(1, 1e5)),
    dict(id="n200_m158", n=200, m=158, gauges="special", rank=200, floor=0.0, r_scale=1e-2, cond=(1, 1e6)),
    dict(id="n200_m159", n=200, m=159, gauges="special", rank=200, floor=0.0, r_scale=1e-2, cond=(1, 1e6)),
    dict(id="n400_special_cond1", n=400, m=12, gauges="special", rank=400, floor=0.0, r_scale=1e3, cond=(1, 3)),
    dict(id="n300_neighbours_cond1e9", n=300, m=30, gauges="neighbours", rank=4, floor=1e-9, r_scale=2e-8,
         cond=(1e7, 3e9)),
]
FILTER_STEPS = 3


def filter_case(case):
    """Network, parameters, gauges (ascending), Q, R (ascending gauge order), P0, the forcing of every step and the
    measurement of every update time (step k: row k, k = 0 the start)."""
    from tx_fast_hydrology_b200 import synthetic as S
    n, m, seed = case["n"], case["m"], 1000 + case["n"] + case["m"]
    net = S.make_network(n, seed, n_basins=min(3, n))
    prm = S.make_params(n, seed, well_posed=True)
    end = net["endnodes"]
    g = special_gauges(end, m, seed) if case["gauges"] == "special" else neighbour_gauges(end, m)
    assert g.size == m
    Q, Rm, P0 = dense_covariances(n, m, seed, case["rank"], case["r_scale"], case["floor"])
    rng = np.random.default_rng(seed + 5)
    q = rng.uniform(0.0, 2.0, size=(FILTER_STEPS + 1, n))
    z = prm["o_t"][g][None, :] * rng.uniform(0.9, 1.3, size=(FILTER_STEPS + 1, m))
    return dict(net=net, prm=prm, gauges=g, Q=Q, R=Rm, P0=P0, q=q, z=z)


def filter_case_inputs(oracle, case):
    """The arguments of kf_update_ref for the first update after one routing step (oracle, FP64)."""
    c = filter_case(case)
    n, end = c["net"]["endnodes"].size, c["net"]["endnodes"]
    mdl = oracle.OracleModel(np.arange(n), end, c["prm"]["K"], c["prm"]["X"], c["prm"]["o_t"], DT_S, T0_NS)
    mdl.step(c["q"][0])
    return (c["P0"], c["Q"], c["R"], c["gauges"], c["z"][1], mdl.o_t_next, mdl.i_t_next, end, mdl.alpha, mdl.beta,
            mdl.chi)


# Batched case: independent sub-models run BATCH_STEPS steps; block k's measurement table ends after step "stop",
# so its filter updates at the start and after steps 1 .. stop, then is not due any more (da.py:49-61).
BATCH_BLOCKS = [dict(n=1, m=1, stop=2), dict(n=30, m=30, stop=4), dict(n=200, m=158, stop=8), dict(n=80, m=5, stop=6),
                dict(n=120, m=40, stop=8)]
BATCH_STEPS = 8


def batch_block(k, m=None):
    """Block k (with m gauges in place of its own if given): network, parameters, gauges, Q, R, P0, lateral inflow q [n] (constant) and measurements z
    [stop + 1][m] at the start and after every step up to `stop`."""
    blk = BATCH_BLOCKS[k]
    n, m, seed = blk["n"], blk["m"] if m is None else m, 500 + 31 * k
    from tx_fast_hydrology_b200 import synthetic as S
    net = S.make_network(n, seed, n_basins=min(2, n))
    prm = S.make_params(n, seed, well_posed=True)
    g = special_gauges(net["endnodes"], m, seed)
    Q, Rm, P0 = dense_covariances(n, m, seed, n, 1e-2)
    rng = np.random.default_rng(seed + 9)
    q = rng.uniform(0.0, 1.0, size=n)
    z = prm["o_t"][g][None, :] * rng.uniform(0.8, 1.2, size=(blk["stop"] + 1, m))
    return dict(net=net, prm=prm, gauges=g, Q=Q, R=Rm, P0=P0, q=q, z=z)


def batch_block_last_update(oracle, k):
    """(P before, P after, cond(S)) of block k's last update, the filter chained in longdouble on the oracle's
    routing (FP64)."""
    c = batch_block(k)
    n, end = c["net"]["endnodes"].size, c["net"]["endnodes"]
    mdl = oracle.OracleModel(np.arange(n), end, c["prm"]["K"], c["prm"]["X"], c["prm"]["o_t"], DT_S, T0_NS)
    P = c["P0"]
    for t in range(BATCH_BLOCKS[k]["stop"] + 1):
        if t:
            mdl.step(c["q"])
        r = kf_update_ref(P, c["Q"], c["R"], c["gauges"], c["z"][t], mdl.o_t_next, mdl.i_t_next, end, mdl.alpha,
                          mdl.beta, mdl.chi)
        P_before, P = P, r["P"]
        mdl.o_t_next, mdl.i_t_next = (np.asarray(x, dtype=np.float64) for x in (r["o"], r["i"]))
    return (np.asarray(P_before, dtype=np.float64), np.asarray(P, dtype=np.float64),
            float(np.linalg.cond(np.asarray(r["S"], dtype=np.float64))))

"""The extended-precision reference of forcing-driven routing (tests/forcing_reference.py) on the CPU: its step
records are nutils' interpolation bit for bit, its runs reproduce the reference's golden run and the FP64 oracle, a
correct FP64 evaluation sits well under its bound, and every planted defect misses that bound by more than 10^3 on
the cases tests/test_gpu_forcing.py runs.  Also the `method` checks of Muskingum.run and RiverNetwork.route_run,
which refuse a bad method before any device work."""
import functools
import os

import numpy as np
import pytest

import forcing_reference as F
from parity import relerr

MISS = 1e3                        # a planted defect must land this far outside the bound


@functools.lru_cache(maxsize=None)
def _ref(name, defect=None):
    return F.case_ref(F.CASE_BY_NAME[name], defect)


def _dense(recs, R):
    """The records as the rows of weights nutils would apply to the identity table."""
    r0, r1, w0, w1 = recs
    out = np.zeros((r0.size, R))
    k = np.arange(r0.size)
    out[k, r0] += w0
    out[k, r1] += w1
    return out


@pytest.mark.parametrize("fname", ["kernels_n60.npz", "kernels_n160.npz"])
def test_records_reproduce_golden_interpolation(golden_dir, oracle, fname):
    """At the golden points (before the table, on knots, inside, after it) both methods give the reference's own
    interpolation, nutils' and the C oracle's, bit for bit."""
    from tx_fast_hydrology_b200 import nutils
    g = np.load(os.path.join(golden_dir, fname))
    xp, fp, xs = g["xp"], g["fp"], g["xs"]
    for method, key in ((1, "interp_lin"), (0, "interp_near")):
        recs = tuple(np.array(v) for v in zip(*[F.record_at(xp, float(x), method) for x in xs]))
        got = F.apply_records(recs, fp)
        assert np.array_equal(got, g[key])
        for x, row in zip(xs, got):
            assert np.array_equal(row, nutils.interpolate_sample(float(x), xp, fp, method))
            assert np.array_equal(row, oracle.interpolate_sample(float(x), xp, fp, method))


def _table_cases():
    seen = {}
    for c in F.CASES:
        seen.setdefault((c.kind, c.nsteps, c.method), c)
    return list(seen.values())


@pytest.mark.parametrize("case", _table_cases(), ids=repr)
def test_records_match_nutils_on_every_case_table(oracle, case):
    """Every step of every GPU case table: the records weight the rows exactly as nutils.interpolate_sample and the
    oracle do (the identity table makes the weights the result), and the records of a run split over calls are those
    of the same steps in one call."""
    from tx_fast_hydrology_b200 import nutils
    times = F.make_times(case.kind, case.nsteps)
    xp = times.astype(np.float64)
    R = xp.size
    eye = np.eye(R)
    recs = F.step_records(times, F.T0_NS, F.DT_NS, case.nsteps, case.method)
    dense = _dense(recs, R)
    for s, x in enumerate(F.step_times(F.T0_NS, F.DT_NS, case.nsteps)):
        assert x == float(F.T0_NS + (s + 1) * F.DT_NS)
        assert np.array_equal(dense[s], nutils.interpolate_sample(x, xp, eye, case.method)), s
        assert np.array_equal(dense[s], oracle.interpolate_sample(x, xp, eye, case.method)), s
    base, parts = 0, []
    for ns in case.calls:
        parts.append(F.step_records(times, F.T0_NS + base * F.DT_NS, F.DT_NS, ns, case.method))
        base += ns
    for a, b in zip(recs, (np.concatenate(p) for p in zip(*parts))):
        assert np.array_equal(a, b)


def test_case_tables_reach_the_edges():
    """The tables do what their names say: brackets that jump 2 and 3 rows, a row every step, gaps from 1 s to over a
    64-step launch, clamping before the first and after the last row, exact nearest-method ties."""
    def recs(kind, n, method=1):
        return F.step_records(F.make_times(kind, n), F.T0_NS, F.DT_NS, n, method)
    r0 = recs("sub150", 64)[0]
    assert set(np.diff(r0)) == {2}
    assert set(np.diff(recs("sub100", 65)[0])) == {3}
    assert set(np.diff(recs("every_step", 65)[0])) == {1}
    gaps = np.diff(F.make_times("irregular", 150))
    assert gaps.min() == F._S and gaps.max() >= 6 * 3600 * F._S and (gaps > 64 * F.DT_NS).sum() >= 2
    assert (gaps % F.DT_NS != 0).any()
    r0, r1, w0, w1 = recs("late_start", 30)
    assert (r0[:7] == 0).all() and (w1[:7] == 0).all() and w1[7] > 0
    t = F.make_times("early_end", 65)
    r0, r1, w0, w1 = recs("early_end", 65)
    last = int(np.searchsorted(F.step_times(F.T0_NS, F.DT_NS, 65), float(t[-1])))
    assert 16 < last < 64 and (r0[last + 1:] == t.size - 1).all() and (w1[last + 1:] == 0).all()
    r0, r1, w0, w1 = recs("ties", 30, 0)
    x = F.step_times(F.T0_NS, F.DT_NS, 30)
    xp = F.make_times("ties", 30).astype(np.float64)
    mid = np.abs(x - xp[r0]) == np.abs(x - xp[np.minimum(r0 + 1, xp.size - 1)])
    assert mid.sum() >= 10
    assert (recs("R1", 17)[0] == 0).all()
    r0, r1, w0, w1 = recs("R2", 17)
    assert (r0[:3] == 0).all() and (w1[3:11] > 0).all() and (r0[11:] == 1).all()


def test_reference_reproduces_golden_model_c1(golden_dir, oracle):
    """1,000 reaches x 288 steps of the reference's Muskingum.simulate (golden), every kept step, within the bound
    (and within 1e-12 element-wise: the golden was computed in FP64)."""
    g = np.load(os.path.join(golden_dir, "model_c1.npz"))
    n = g["endnodes"].size
    al, be, ch, ga = oracle.compute_coeffs(g["K"], g["X"], float(g["dt"]))
    i0 = oracle.init_states(np.arange(n), g["endnodes"], g["o_init"])
    T = 288
    r = F.route_ref(g["endnodes"], al, be, ch, ga, g["o_init"], i0, g["times"], g["table"], None, int(g["t0_ns"]),
                    int(300e9), T, 1, rec_reach=np.arange(n), rec_every=1)
    keep = g["keep"]
    rec = r["rec"][keep, :, 0]
    ratio = F.bound_ratio(g["O"], rec, r["brec"][keep, :, 0])
    ratio = max(ratio, F.bound_ratio(g["I"][-1], r["I"][:, 0], r["bI"][:, 0]))
    print(f"model_c1 golden: error/bound {ratio:.3g}")
    assert ratio <= 1.0
    assert relerr(rec.astype(np.float64), g["O"]) < 1e-12
    assert relerr(r["I"][:, 0].astype(np.float64), g["I"][-1]) < 1e-12


@pytest.mark.parametrize("M,mul", [(1, False), (3, True)])
def test_reference_matches_oracle_on_aligned_tables(oracle, M, mul):
    """The member-batched C oracle (linear, multipliers applied per row) on an aligned table."""
    c = F.Case("aligned", "n1000", "aligned", F.LIN, M, mul, 40, F.ALL)
    x = F.case_inputs(c)
    r = F.case_ref(c, inputs=x)
    al, be, ch, ga = x["coef"]
    end = x["endnodes"]
    n = end.size
    net = {"startnodes": np.arange(n), "endnodes": end, "indegree": oracle.compute_indegree(np.arange(n), end),
           "alpha": al, "beta": be, "chi": ch, "gamma": ga}
    o = np.ascontiguousarray(x["o0"].T); i = np.ascontiguousarray(x["i0"].T)
    oracle.run_members(net, o, i, c.nsteps, x["times"].astype(np.float64), x["table"], float(F.T0_NS), float(F.DT_NS),
                       wmul=x["mul"])
    ratio = max(F.bound_ratio(o.T, r["O"], r["bO"]), F.bound_ratio(i.T, r["I"], r["bI"]))
    print(f"oracle.run_members M={M}: error/bound {ratio:.3g}")
    assert ratio <= 1.0


def _oracle_run(oracle, case, x):
    """The FP64 oracle fed each member's per-step forcing through a table with one row per step end (the identity
    interpolation): a correct FP64 evaluation of the same run."""
    al, be, ch, ga = x["coef"]
    end = x["endnodes"]
    n = end.size
    net = {"startnodes": np.arange(n), "endnodes": end, "indegree": oracle.compute_indegree(np.arange(n), end),
           "alpha": al, "beta": be, "chi": ch, "gamma": ga}
    base, parts = 0, []
    for ns in case.calls:
        parts.append(F.step_records(x["times"], F.T0_NS + base * F.DT_NS, F.DT_NS, ns, case.method))
        base += ns
    r0, r1, w0, w1 = (np.concatenate(p) for p in zip(*parts))
    T = case.nsteps
    rows = (np.arange(1, T + 1) * float(F.DT_NS))             # t0 = 0: every row time exact
    O = np.empty((n, case.M)); I = np.empty((n, case.M))
    for m in range(case.M):
        mu = x["mul"][:, m] if x["mul"] is not None else np.ones(x["table"].shape[0])
        q = (w0 * mu[r0])[:, None] * x["table"][r0] + (w1 * mu[r1])[:, None] * x["table"][r1]
        o = np.ascontiguousarray(x["o0"][:, m][None]); i = np.ascontiguousarray(x["i0"][:, m][None])
        oracle.run_members(net, o, i, T, rows, np.ascontiguousarray(q), 0.0, float(F.DT_NS))
        O[:, m], I[:, m] = o[0], i[0]
    return O, I


CALIBRATION = ["aligned-lin", "every_step-lin", "sub100-near", "irregular-lin", "irregular-near", "early_end-lin",
               "calls-lin", "lane16-irregular-near", "m70-irregular-lin", "chain-irregular-lin", "chain-ties-near"]


def test_fp64_oracle_sits_well_under_the_bound(oracle):
    """Calibrates C_BOUND: a correct FP64 implementation must pass with margin.  The worst ratio is reported."""
    worst = 0.0
    for name in CALIBRATION:
        c = F.CASE_BY_NAME[name]
        x = F.case_inputs(c)
        O, I = _oracle_run(oracle, c, x)
        r = _ref(name)
        ratio = max(F.bound_ratio(O, r["O"], r["bO"]), F.bound_ratio(I, r["I"], r["bI"]))
        print(f"FP64 oracle {name}: error/bound {ratio:.3g}")
        worst = max(worst, ratio)
    print(f"FP64 oracle: worst error/bound {worst:.3g} (C_BOUND = {F.C_BOUND})")
    assert worst < 0.1


# the case each defect is looked for first; any case of a kernel's list will do
WITNESS = {"start_of_step": "aligned-lin", "ties_later": "ties-near", "method_ignored": "aligned-near",
           "always_shift": "sub150-lin", "mul_r0": "every_step-lin", "clamp_r2": "early_end-lin",
           "held_bracket": "calls-lin"}


@pytest.mark.parametrize("defect", F.DEFECTS)
def test_planted_defects_miss_the_bound(defect):
    """For every kernel, some case of its GPU list lands more than 10^3 bounds away from the truth when the defect is
    planted (a run split over calls for the held bracket)."""
    for kernel in F.ALL:
        cands = [c for c in F.CASES if kernel in c.kernels and (defect != "held_bracket" or len(c.calls) > 1)]
        cands.sort(key=lambda c: (c.name != WITNESS[defect], c.M * c.nsteps))
        found = None
        for c in cands:
            miss = F.miss_ratio(_ref(c.name), _ref(c.name, defect))
            if miss > MISS:
                found = (c.name, miss)
                break
        assert found is not None, f"no case of the {kernel} list separates defect {defect!r}"
        print(f"defect {defect} on the {kernel} list: {found[0]} misses by {found[1]:.3g}")


def test_defects_leave_unaffected_cases_alone():
    """A defect that cannot show in a case changes nothing there (the switches do only what they say)."""
    assert F.miss_ratio(_ref("aligned-lin"), _ref("aligned-lin", "ties_later")) == 0.0
    assert F.miss_ratio(_ref("aligned-lin"), _ref("aligned-lin", "method_ignored")) == 0.0
    assert F.miss_ratio(_ref("aligned-lin"), _ref("aligned-lin", "mul_r0")) == 0.0
    assert F.miss_ratio(_ref("aligned-lin"), _ref("aligned-lin", "held_bracket")) == 0.0


def test_lane_cases_read_their_step_records_where_they_say(libtxh):
    """The lane cases marked `lane_in_place` launch more steps than the shared memory beside their largest region
    holds records for (the kernel then reads them in place); every other lane case stages them (host-side schedule
    of a 148-SM B200)."""
    from tx_fast_hydrology_b200.network import RiverNetwork
    lane = [c for c in F.CASES if "lane" in c.kernels]
    assert any(c.lane_in_place for c in lane)
    for c in lane:
        net = RiverNetwork(F.network(c.net)[0])
        spl = min(max(c.calls), int(c.env.get("TXH_LANE_SPL", 4096)))
        assert F.lane_records_in_place(net, c.M, spl) == c.lane_in_place, c.name


@pytest.mark.parametrize("method", ["Linear", "nearset", "", None, 1])
def test_muskingum_run_refuses_unknown_method(libtxh, method):
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.muskingum import Muskingum
    nd = S.make_network(10, 1)
    m = Muskingum(S.model_dict(nd, S.make_params(10, 1)))
    with pytest.raises(ValueError, match="method"):
        m.run(None, 4, method=method)


@pytest.mark.parametrize("method", [2, -1, "linear", True, 0.5])
def test_route_run_refuses_unknown_method(libtxh, method):
    from tx_fast_hydrology_b200.network import RiverNetwork
    net = RiverNetwork(np.array([1, 2, 2], dtype=np.int64))
    with pytest.raises(ValueError, match="method"):
        net.route_run(None, None, 1, None, 0, 1, 1, method=method)

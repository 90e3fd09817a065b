"""The forcing interpolation of every routing kernel against the extended-precision reference (tests/forcing_reference.py):
nearest rows and linear weights, tables with a row every step or several rows per step, irregular and off-grid row
times, tables that start after or end before the run, one- and two-row tables, nearest-method ties, runs split over
launches and calls, recorded hydrographs.  Every element of O, I and the records must sit within the running-error
bound of the reference, C_BOUND * u * (nsteps + depth + 4) * (magnitude run).

Every case also checks that the kernel it names is the one that routed it (a kernel that declines a schedule hands
the run to the next one quietly), and, on the lane kernel, whether the launch's step records were staged in shared
memory or read in place.

What the cases reach in route_lane_kernel: every nearest-method case with more than one row, and the linear cases
on the sub-step, irregular, early-end and two-row tables, change the bracket by something other than a one-row shift
(rotate_bracket); a table with a row every step ('every_step', linear) shifts the bracket one iteration after the
previous request, the cp.async wait of dense tables.  The two 'lane16-inplace' cases (16 members on n3000, over 432
steps) read their step records in place, on both of those paths; all other lane cases stage them.
"""
import numpy as np
import pytest

import forcing_reference as F

pytestmark = pytest.mark.gpu

_REFS = {}
_WORST = {}


@pytest.fixture(scope="module", autouse=True)
def _report_worst_ratios():
    """Prints the worst error/bound of every kernel and method once the module's cases have run (with -s)."""
    yield
    for (kernel, method), r in sorted(_WORST.items()):
        print(f"worst error/bound {kernel:9s} {method:8s} {r:.3g}")


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (no CPU fallback exists)"
    return torch


def _case(case):
    """Inputs and reference of a case, computed once and compared against every kernel that runs it."""
    if case.name not in _REFS:
        x = F.case_inputs(case)
        _REFS[case.name] = (x, F.case_ref(case, inputs=x))
    return _REFS[case.name]


def _upload(net, a, M):
    X = net.alloc_state(M)
    net.pack_host(np.ascontiguousarray(a, dtype=np.float64).reshape(net.n, M), M, X)
    return X


def _check(label, kernel, method, got, ref):
    """|gpu - ref| <= bound element-wise for O, I (and the records); the ratio is reported per kernel and method."""
    ratio = max(F.bound_ratio(got["O"], ref["O"], ref["bO"]), F.bound_ratio(got["I"], ref["I"], ref["bI"]))
    if "rec" in ref:
        ratio = max(ratio, F.bound_ratio(got["rec"], ref["rec"], ref["brec"]))
    key = (kernel, "linear" if method == F.LIN else "nearest")
    _WORST[key] = max(_WORST.get(key, 0.0), ratio)
    print(f"{label} [{kernel}]: error/bound {ratio:.3g}")
    assert ratio <= 1.0, f"{label} on the {kernel} kernel: error/bound {ratio:.3g}"


def _kernel_that_routes(net, M, f, tmp_path, monkeypatch):
    """The kernel the handle's routing calls run on, from one more step with the launch timelines on: route_lane_kernel
    writes TXH_LANE_TRACE; the window and dataflow kernels write TXH_TRACE_FILE, whose header word 3 is minus the
    member blocks for the window kernel and plus them for the dataflow kernel (txh_capi.cu, run_window / run_dataflow)."""
    lane, route = tmp_path / "lane.bin", tmp_path / "route.bin"
    monkeypatch.setenv("TXH_LANE_TRACE", str(lane))
    monkeypatch.setenv("TXH_TRACE_FILE", str(route))
    try:
        O, I = net.alloc_state(M), net.alloc_state(M)
        net.route_run(O, I, M, f, F.T0_NS, F.DT_NS, 1)
        net.check()
    finally:
        monkeypatch.delenv("TXH_LANE_TRACE")
        monkeypatch.delenv("TXH_TRACE_FILE")
    if lane.exists():
        assert not route.exists()
        return "lane"
    return "window" if np.fromfile(route, dtype=np.int64, count=4)[3] < 0 else "dataflow"


def _cases():
    return [pytest.param(c, k, id=f"{c.name}-{k}") for c in F.CASES for k in c.kernels]


@pytest.mark.parametrize("case,kernel", _cases())
def test_forcing_case(torch_cuda, libtxh, monkeypatch, tmp_path, case, kernel):
    torch = torch_cuda
    from tx_fast_hydrology_b200.network import Forcing, RiverNetwork
    monkeypatch.setenv("TXH_ROUTE_KERNEL", kernel)
    for k, v in case.env.items():
        monkeypatch.setenv(k, v)
    x, ref = _case(case)
    M = case.M
    net = RiverNetwork(x["endnodes"])
    net.set_coeffs(*x["coef"])
    f = Forcing(net, x["times"], x["table"], x["mul"])
    try:
        O, I = _upload(net, x["o0"], M), _upload(net, x["i0"], M)
        kw = {}
        if x["rec"] is not None:
            reaches, every = x["rec"]
            rec = torch.full((case.nsteps // every, reaches.size, M), float("nan"), dtype=torch.float64, device="cuda")
            kw = dict(rec_reach=reaches, rec_every=every, rec_out=rec)
        base = 0
        for ns in case.calls:
            net.route_run(O, I, M, f, F.T0_NS + base * F.DT_NS, F.DT_NS, ns, method=case.method, **kw)
            base += ns
        net.check()
        got = {"O": net.unpack_host(O, M), "I": net.unpack_host(I, M)}
        if kw:
            got["rec"] = kw["rec_out"].cpu().numpy()
        _check(case.name, kernel, case.method, got, ref)
        assert _kernel_that_routes(net, M, f, tmp_path, monkeypatch) == kernel
        if kernel == "lane":
            spl = min(max(case.calls), int(case.env.get("TXH_LANE_SPL", 4096)))
            assert F.lane_records_in_place(net, M, spl) == case.lane_in_place
    finally:
        f.close()


def test_public_api_nearest(torch_cuda, libtxh):
    """Muskingum.run(..., method='nearest') on the nearest-tie table, from the model's own initial state."""
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.muskingum import Muskingum
    c = F.Case("api-ties-near", "n300", "ties", F.NEAR, 1, False, 20, ())
    x = F.case_inputs(c)
    end, prm = F.network(c.net)
    n = end.size
    mdl = Muskingum(S.model_dict({"startnodes": np.arange(n), "endnodes": end}, prm, dt_s=300.0,
                                 t0="2023-11-14T22:13:20Z"))
    assert int(mdl.datetime.value) == F.T0_NS
    for a, b in zip((mdl.alpha, mdl.beta, mdl.chi, mdl.gamma), x["coef"]):
        assert np.array_equal(a, b)
    O, I = mdl.device_state
    o0, i0 = mdl.network.unpack_host(O, 1), mdl.network.unpack_host(I, 1)
    f = mdl.make_forcing(times_ns=x["times"], table=x["table"])
    mdl.run(f, c.nsteps, method="nearest")
    mdl.network.check()
    ref = F.route_ref(end, *x["coef"], o0, i0, x["times"], x["table"], None, F.T0_NS, F.DT_NS, c.nsteps, F.NEAR)
    O, I = mdl.device_state
    got = {"O": mdl.network.unpack_host(O, 1), "I": mdl.network.unpack_host(I, 1)}
    _check(c.name, "api", F.NEAR, got, ref)

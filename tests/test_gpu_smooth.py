"""Ensemble Kalman smoother of recorded hydrographs (Muskingum.run_assimilating(smooth_lag=...), txh_enks_smooth,
txh_set_transform_history) against the gain-form reference (tests/enks_oracle.py) on top of the CPU oracle's filter.

Tolerance: after the updates, relative to max(|smoothed|, |filtered|, |forecast at update steps|) and the sum of the
eps * cond(S) bounds of every update of the run (parity.enkf_tolerance): each update's solve carries its own forward
error, and a smoothed slot has been through several of them."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from assim_case import make_case, model, run_device, reference_loop, update_fp64  # noqa: E402
from parity import relerr, normerr                        # noqa: E402
from enks_oracle import enks_gain, smooth_transforms      # noqa: E402


def _case(n, M, m, seed, every, nwin, rest, dense_R=False):
    """The assimilation case of test_gpu_record.py."""
    return make_case(n, M, m, seed, every, nwin, rest, gauges="synthetic", dense_R=dense_R, extra_reaches=60)


def _smoothed_oracle(slots, upd, every, record_every, lag):
    out = slots.copy()
    for j in range(out.shape[0]):
        s = (j + 1) * record_every
        for u, (HA, dz, S) in enumerate(upd):
            if s < (u + 1) * every <= s + lag:
                out[j] += enks_gain(out[j] - out[j].mean(axis=1, keepdims=True), HA, dz, S)
    return out


def _scale(filt, smooth, pri, every, record_every):
    sc = np.maximum(np.abs(filt), np.abs(smooth))
    for j in range(sc.shape[0]):
        s = (j + 1) * record_every
        if s % every == 0 and s // every <= pri.shape[0]:
            sc[j] = np.maximum(sc[j], np.abs(pri[s // every - 1]))
    return sc


CASES = [(2000, 64, 50, 51, 6, 3, 0, 1, False),
         (1200, 20, 30, 52, 6, 3, 4, 4, False),       # 4 does not divide 6; remainder steps
         (900, 70, 40, 53, 5, 3, 2, 1, False),        # two member blocks: the transform kernel applies the update
         (1400, 48, 90, 54, 5, 3, 0, 5, True),        # dense R: the general launches of the ensemble-space system
         (1500, 64, 25, 55, 5, 2, 3, 3, False)]


@pytest.mark.parametrize("n,M,m,seed,every,nwin,rest,record_every,dense_R", CASES)
@pytest.mark.parametrize("in_library", [True, False])
def test_smoothed_hydrographs_vs_oracle(oracle, n, M, m, seed, every, nwin, rest, record_every, dense_R, in_library):
    """For lags 0, 3 (below `every`), every + 2, 2 every and beyond the run (fixed interval): the smoothed slots equal
    the gain-form smoother applied to the oracle's filtered slots; lag 0 and the slots after the last update are the
    filtered ones bit for bit; `rec` and `prior` stay the filtered hydrographs."""
    nsteps = every * nwin + rest
    ref = None
    for lag in (0, 3, every + 2, 2 * every, nsteps + 5):
        c = _case(n, M, m, seed, every, nwin, rest, dense_R)
        rec, prior, sm = run_device(c, in_library, record_every=record_every, lag=lag)["res"]
        if ref is None:
            # the oracle's filter with the recorded slots (posterior at update steps) and, per update, what the
            # smoother needs
            ref = reference_loop(oracle, c, update_fp64, record_every=record_every)
        slots, upd, tols, pri = ref["hyd"], ref["kept"], ref["tols"], ref["pri"]
        want = _smoothed_oracle(slots, upd, every, record_every, lag)
        tol = sum(tols)
        assert sm.shape == rec.shape == want.shape
        assert relerr(prior, pri) < max(tols)
        assert relerr(sm, want, scale=_scale(rec, want, pri, every, record_every)) < tol, f"lag {lag}"
        if lag == 0:
            assert (sm == rec).all()
        after = [j for j in range(rec.shape[0]) if (j + 1) * record_every >= nwin * every]
        assert (sm[after] == rec[after]).all()


def test_smoothing_leaves_the_filter_alone():
    """rec, prior and the final state are bit-identical with and without smooth_lag (in-library and Python loop): the
    transform history does not change the filter."""
    for in_library in (True, False):
        out = []
        for lag in (None, 7):
            d = run_device(_case(1500, 64, 40, 61, 6, 3, 2), in_library, lag=lag)
            r = d["res"]
            assert len(r) == (2 if lag is None else 3)
            out.append((r[0], r[1], d["mdl"].o_t_next, d["mdl"].i_t_next, d["enkf"]._T.cpu().numpy()))
        for a, b in zip(*out):
            assert (a == b).all()


@pytest.mark.parametrize("lag", [4, 100])
def test_in_library_and_python_loop_agree(lag):
    a = run_device(_case(1500, 64, 40, 62, 6, 3, 2), True, record_every=2, lag=lag)["res"]
    b = run_device(_case(1500, 64, 40, 62, 6, 3, 2), False, record_every=2, lag=lag)["res"]
    assert normerr(a[2], b[2]) < 1e-10
    assert normerr(a[0], b[0]) < 1e-10


def test_transform_history_adds_no_launch():
    """The loop issues the same launches with the transform history set (the pointers move on the host)."""
    import torch
    from tx_fast_hydrology_b200 import _lib
    lib = _lib.load()
    counts, T_last = [], None
    for hist in (False, True):
        c = _case(1500, 64, 40, 63, 6, 4, 3)
        mdl, enkf, f = model(c)
        Zd = torch.as_tensor(np.ascontiguousarray(c["Zp"]), device="cuda")
        mdl._ensure_device()
        T_hist = torch.empty((4, 64, 64), dtype=torch.float64, device="cuda")
        if hist:
            mdl.network.set_transform_history(T_hist)
        n0 = lib.txh_launch_count()
        mdl.run_assimilating(f, c["nsteps"], enkf, 6, Zd, record_reaches=c["reaches"], record_prior=True)
        counts.append(lib.txh_launch_count() - n0)
        mdl.network.set_transform_history(None)
        mdl.network.check()
        if hist:                                   # the last update's transform went to the history
            assert (T_hist[3] == T_last).all()
        else:
            T_last = enkf._T.clone()
    assert counts[0] == counts[1]


def test_transform_history_capacity_is_checked():
    import torch
    from tx_fast_hydrology_b200._lib import TxhError
    c = _case(800, 16, 20, 64, 5, 3, 0)
    mdl, enkf, f = model(c)
    mdl._ensure_device()
    mdl.network.set_transform_history(torch.empty((2, 16, 16), dtype=torch.float64, device="cuda"))
    Zd = torch.as_tensor(np.ascontiguousarray(c["Zp"]), device="cuda")
    O0 = mdl.o_t_next.copy()
    with pytest.raises(TxhError, match="transform history"):
        mdl.run_assimilating(f, c["nsteps"], enkf, 5, Zd)
    mdl.network.set_transform_history(None)
    assert (mdl.o_t_next == O0).all()                     # refused before any device work


def test_fused_and_plain_paths_agree():
    """With the fused stages switched off (TXH_ENKF_FUSED=0 TXH_ENKF_FUSE_LOAD=0 TXH_PDL=0, read once per process: a
    child process), the smoothed hydrographs agree with the default path to 1e-10."""
    import subprocess
    import sys
    import tempfile
    here = os.path.dirname(os.path.abspath(__file__))
    code = (
        "import sys, numpy as np\n"
        "sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "from assim_case import make_case, run_device\n"
        "c = make_case(2500, 64, 40, 65, 6, 4, 3, gauges='synthetic', extra_reaches=60)\n"
        "rec, pri, sm = run_device(c, True, record_every=2, lag=13)['res']\n"
        "np.savez(sys.argv[1], rec=rec, sm=sm)\n"
    ) % (os.path.dirname(here), here)
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        for name, env in (("fused", {}), ("plain", {"TXH_ENKF_FUSED": "0", "TXH_ENKF_FUSE_LOAD": "0", "TXH_PDL": "0"})):
            path = os.path.join(tmp, name + ".npz")
            e = dict(os.environ); e.update(env)
            subprocess.run([sys.executable, "-c", code, path], check=True, env=e, timeout=600)
            z = np.load(path)
            out[name] = (z["rec"], z["sm"])
    assert normerr(out["fused"][0], out["plain"][0]) < 1e-10
    assert normerr(out["fused"][1], out["plain"][1]) < 1e-10


@pytest.mark.parametrize("M", [2, 5, 64, 70, 128])
@pytest.mark.parametrize("nupd,every,rec_every,lag", [
    (30, 3, 1, 7),            # ranges inside a block of ceil(sqrt(30)) = 6 updates: the in-block chain
    (30, 3, 2, 20),           # ranges over two and three blocks
    (30, 3, 1, 1000),         # fixed interval: suffixes
    (17, 4, 3, 2),            # lag below `every`: one update or none
    (9, 1, 1, 4)])
def test_enks_smooth_vs_definition(M, nupd, every, rec_every, lag):
    """txh_enks_smooth on random slots and transforms against a loop of the definition."""
    import torch
    from tx_fast_hydrology_b200.network import RiverNetwork
    rng = np.random.default_rng(M * 1000 + nupd + lag)
    nsteps = nupd * every + 2
    nslots, k = nsteps // rec_every, 37
    T = rng.standard_normal((nupd, M, M)) * (0.3 / np.sqrt(M))
    rec = 3.0 + rng.standard_normal((nslots, k, M))
    want = smooth_transforms(rec, T, nupd, every, rec_every, lag)
    net = RiverNetwork(np.array([1, 1], dtype=np.int64))
    Td = torch.as_tensor(T, device="cuda")
    rd = torch.as_tensor(rec, device="cuda")
    got = net.enks_smooth(M, nupd, every, Td, rd, rec_every, lag, torch.full_like(rd, np.nan)).cpu().numpy()
    assert normerr(got, want) < 1e-12
    assert (rd.cpu().numpy() == rec).all()

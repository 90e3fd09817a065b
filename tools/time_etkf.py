"""Cost and effect of the square-root ensemble update (ETKF) at the C3 shape (100,000 reaches, 64 members, 7 days of
5-minute steps, an hourly update over 500 gauges, the in-library loop Muskingum.run_assimilating).

Three arms, alternated in one process, CUDA events around whole runs ending in a device synchronise, the L2 cache
overwritten before every run: the stochastic filter with perturbed observations (what bench.py runs), the ETKF, and
the ETKF with relaxation to prior perturbations rtpp = 0.5.  Reports ms per run, the kernel launches of a run (the
ETKF adds one per update), the time of enkf_transform_post_kernel from a separate torch.profiler run, and the card with
its power limit.  Then a seeded twin experiment (a one-member truth run on the unperturbed forcing and initial state,
the gauges observed from it with noise of standard deviation 0.1, R = 0.01 I): RMSE of the ensemble mean against the
truth at the gauges over every step, and the mean ensemble spread there, for the stochastic filter with perturbed
observations, the stochastic filter without (every member sees the same observation), and the ETKF.

    python tools/time_etkf.py [--reps 5] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N, M, M_GAUGES, EVERY, NSTEPS, SEED, DT_S, SIGMA = 100000, 64, 500, 12, 2016, 2, 300.0, 0.1
ARMS = ("stochastic_noise", "etkf", "etkf_rtpp0.5")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:                          # noqa: BLE001 -- informational only
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import pandas as pd
    from torch.profiler import profile, ProfilerActivity
    from tx_fast_hydrology_b200 import synthetic as S, _lib
    from tx_fast_hydrology_b200.muskingum import Muskingum
    from tx_fast_hydrology_b200.da import EnsembleKalmanFilter
    assert torch.cuda.is_available(), "time_etkf.py measures on the GPU"
    lib = _lib.load()
    net = S.make_network(N, SEED); prm = S.make_params(N, SEED)
    rng = np.random.default_rng(SEED)
    d = S.model_dict(net, prm, dt_s=DT_S)
    dm = dict(d); dm["o_t"] = prm["o_t"][:, None] * rng.uniform(0.5, 1.5, size=(N, M))
    mdl = Muskingum(dm, members=M)
    t0 = int(mdl.datetime.value)
    times, table = S.make_forcing(N, NSTEPS, DT_S, SEED, t0_ns=t0, rows_every=12)
    f = mdl.make_forcing(times_ns=times, table=table, member_mul=S.make_member_multipliers(times.size, M, SEED))
    gauges = S.make_gauges(net["endnodes"], M_GAUGES, seed=4)
    m, nwin = gauges.size, NSTEPS // EVERY
    # the truth of the twin experiment: one member, the unperturbed forcing, the unperturbed initial state
    dt = dict(d); dt["o_t"] = prm["o_t"]
    truth_mdl = Muskingum(dt, members=1)
    truth = truth_mdl.run(truth_mdl.make_forcing(times_ns=times, table=table), NSTEPS,
                          record_reaches=gauges).cpu().numpy()[:, :, 0]             # [steps][m], gauges' order
    obs = truth[EVERY - 1::EVERY][:nwin]
    order = np.argsort(gauges)                                  # the filter takes its gauges in ascending order
    idx = pd.DatetimeIndex(pd.to_datetime(t0 + (np.arange(nwin, dtype=np.int64) + 1) * int(EVERY * DT_S * 1e9),
                                          unit="ns", utc=True)).as_unit("ns")
    meas = pd.DataFrame(obs, index=idx, columns=[d["reach_ids"][j] for j in gauges])
    every = pd.Timedelta(seconds=EVERY * DT_S)
    R = SIGMA ** 2 * np.eye(m)
    filters = {
        "stochastic_noise": EnsembleKalmanFilter(mdl, meas, 2.0, R, every=every, group=False),
        "stochastic_no_noise": EnsembleKalmanFilter(mdl, meas, 2.0, R, every=every, group=False),
        "etkf": EnsembleKalmanFilter(mdl, meas, 2.0, R, every=every, group=False, method="etkf"),
        "etkf_rtpp0.5": EnsembleKalmanFilter(mdl, meas, 2.0, R, every=every, group=False, method="etkf", rtpp=0.5),
    }
    z = obs[:, order]
    clean = torch.as_tensor(np.ascontiguousarray(np.repeat(z[:, :, None], M, axis=2)), device="cuda")
    noisy = torch.as_tensor(z[:, :, None] + SIGMA * rng.standard_normal((nwin, m, M)), device="cuda").contiguous()
    obs_of = {"stochastic_noise": noisy, "stochastic_no_noise": clean, "etkf": clean, "etkf_rtpp0.5": clean}
    O, I = mdl.device_state
    O0, I0 = O.clone(), I.clone()
    t_start = mdl.datetime
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def run(arm, record=False):
        flush.fill_(1)
        Oc, Ic = mdl.device_state
        Oc.copy_(O0); Ic.copy_(I0)
        mdl._datetime = t_start
        torch.cuda.synchronize()
        n0 = int(lib.txh_launch_count())
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rec = mdl.run_assimilating(f, NSTEPS, filters[arm], EVERY, obs_of[arm],
                                   record_reaches=gauges if record else None)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), int(lib.txh_launch_count()) - n0, rec

    for arm in ARMS:
        run(arm)                                            # warm-up of every arm
    mdl.network.check()
    ms = {s: [] for s in ARMS}
    launches = {s: set() for s in ARMS}
    for _ in range(a.reps):
        for arm in ARMS:
            t, n, _ = run(arm)
            ms[arm].append(t)
            launches[arm].add(n)
    mdl.network.check()

    # the post kernel's time, in a run of its own under the profiler
    post = {}
    for arm in ("etkf", "etkf_rtpp0.5"):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run(arm)
        ev = [e for e in prof.events() if "enkf_transform_post_kernel(" in e.name]
        us = [e.device_time if hasattr(e, "device_time") else e.cuda_time for e in ev]
        post[arm] = {"launches": len(ev), "mean_us": round(float(np.mean(us)), 2) if us else None,
                     "max_us": round(float(np.max(us)), 2) if us else None}
    mdl.network.check()

    # the twin experiment
    twin = {}
    for arm in ("stochastic_noise", "stochastic_no_noise", "etkf"):
        _, _, rec = run(arm, record=True)
        x = rec.cpu().numpy()                                                    # [steps][m][M]
        twin[arm] = {"rmse_mean_vs_truth_gauged": round(float(np.sqrt(np.mean((x.mean(axis=2) - truth) ** 2))), 6),
                     "mean_spread_gauged": round(float(np.mean(x.std(axis=2, ddof=1))), 6)}
    mdl.network.check()
    base = float(np.median(ms["stochastic_noise"]))
    res = {
        "card": card(),
        "shape": {"reaches": N, "members": M, "gauges": m, "steps": NSTEPS, "every": EVERY, "updates": nwin},
        "arms": {arm: {"ms_per_run": [round(x, 3) for x in ms[arm]],
                       "median_ms_per_run": round(float(np.median(ms[arm])), 3),
                       "median_ms_over_stochastic": round(float(np.median(ms[arm])) - base, 3),
                       "launches_per_run": sorted(launches[arm])} for arm in ARMS},
        "post_kernel_profiled": post,
        "twin_experiment": twin,
    }
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()

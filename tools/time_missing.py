"""Cost of missing gauge observations, at the C3 shape (100,000 reaches, 64 members, 7 days of 5-minute steps, an hourly
EnKF over 500 gauges, the in-library loop Muskingum.run_assimilating).  Per update a seeded share of the gauges -- 0 %,
10 %, 50 % -- has a NaN observation row and is left out of the update.  One process, CUDA events around whole runs
ending in a device synchronise, the arms alternated, the L2 cache overwritten before every run.  Reports ms per run,
the kernel launches of a run (equal across the arms: the masking adds none) and the card with its power limit.

    python tools/time_missing.py [--reps 5] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N, M, M_GAUGES, EVERY, NSTEPS, SEED, DT_S = 100000, 64, 500, 12, 2016, 2, 300.0
SHARES = (0.0, 0.1, 0.5)


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
    from tx_fast_hydrology_b200 import synthetic as S, _lib
    from tx_fast_hydrology_b200.muskingum import Muskingum
    from tx_fast_hydrology_b200.da import EnsembleKalmanFilter
    lib = _lib.load()
    net = S.make_network(N, SEED); prm = S.make_params(N, SEED)
    rng = np.random.default_rng(SEED)
    d = S.model_dict(net, prm, dt_s=DT_S)
    d["o_t"] = prm["o_t"][:, None] * rng.uniform(0.5, 1.5, size=(N, M))
    mdl = Muskingum(d, members=M)
    t0 = int(mdl.datetime.value)
    times, table = S.make_forcing(N, NSTEPS, DT_S, SEED, t0_ns=t0, rows_every=12)
    f = mdl.make_forcing(times_ns=times, table=table, member_mul=S.make_member_multipliers(times.size, M, SEED))
    gauges = S.make_gauges(net["endnodes"], M_GAUGES, seed=4)
    m, nwin = gauges.size, NSTEPS // EVERY
    idx = pd.DatetimeIndex(pd.to_datetime(t0 + (np.arange(nwin, dtype=np.int64) + 1) * int(EVERY * DT_S * 1e9),
                                          unit="ns", utc=True)).as_unit("ns")
    truth = prm["o_t"][gauges]
    meas = pd.DataFrame(np.repeat(truth[None], nwin, 0), index=idx, columns=[d["reach_ids"][j] for j in gauges])
    enkf = EnsembleKalmanFilter(mdl, meas, 2.0, 1e-2 * np.eye(m), every=pd.Timedelta(seconds=EVERY * DT_S), group=False)
    base = truth[None, :, None] + 0.1 * rng.standard_normal((nwin, m, M))
    obs = {}
    for share in SHARES:
        z = base.copy()
        z[np.random.default_rng(SEED + int(1000 * share)).random((nwin, m)) < share] = np.nan
        obs[share] = torch.as_tensor(z, device="cuda")
    O, I = mdl.device_state
    O0, I0 = O.clone(), I.clone()
    t_start = mdl.datetime
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def run(share):
        flush.fill_(1)
        Oc, Ic = mdl.device_state
        Oc.copy_(O0); Ic.copy_(I0)
        mdl._datetime = t_start
        torch.cuda.synchronize()
        n0 = int(lib.txh_launch_count())
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        mdl.run_assimilating(f, NSTEPS, enkf, EVERY, obs[share])
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), int(lib.txh_launch_count()) - n0

    for share in SHARES:
        run(share)                                          # warm-up of every arm
    mdl.network.check()
    ms = {s: [] for s in SHARES}
    launches = {s: set() for s in SHARES}
    for _ in range(a.reps):
        for share in SHARES:
            t, n = run(share)
            ms[share].append(t)
            launches[share].add(n)
    mdl.network.check()
    O, _ = mdl.device_state
    res = {
        "card": card(),
        "shape": {"reaches": N, "members": M, "gauges": m, "steps": NSTEPS, "every": EVERY, "updates": nwin},
        "arms": {f"{int(100 * s)}%": {"ms_per_run": [round(x, 3) for x in ms[s]],
                                     "median_ms_per_run": round(float(np.median(ms[s])), 3),
                                     "launches_per_run": sorted(launches[s]),
                                     "missing_rows": int(torch.isnan(obs[s]).any(dim=2).sum())} for s in SHARES},
        "finite_state_after_50%": bool(torch.isfinite(O[:, :M]).all()),
    }
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()

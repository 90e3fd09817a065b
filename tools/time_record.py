"""Cost of recording ensemble hydrographs, at the C3 shape (100,000 reaches, 64 members, 7 days of 5-minute steps, an
hourly EnKF over 500 gauges).  One process, CUDA events around whole runs ending in a device synchronise, the arms
alternated, the L2 cache overwritten before every run:

  * Muskingum.run_assimilating without recording vs recording 1,000 reaches (the 500 gauges + 500 others) after every
    step with record_prior=True: ms per run, the difference per window, the time of the posterior-record kernel
    (torch.profiler, a run of its own), bytes recorded;
  * Muskingum.run(forcing, 2016, record_reaches=<the same 1,000>) at 64 members on the window kernel vs the dataflow
    kernel (TXH_ROUTE_KERNEL, read once per process: one child process per arm, alternated).

    python tools/time_record.py [--reps 5] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N, M, M_GAUGES, EVERY, NSTEPS, SEED, DT_S = 100000, 64, 500, 12, 2016, 2, 300.0


def setup():
    import torch
    import pandas as pd
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.muskingum import Muskingum
    from tx_fast_hydrology_b200.da import EnsembleKalmanFilter
    net = S.make_network(N, SEED); prm = S.make_params(N, SEED)
    rng = np.random.default_rng(SEED)
    d = S.model_dict(net, prm, dt_s=DT_S)
    d["o_t"] = prm["o_t"][:, None] * rng.uniform(0.5, 1.5, size=(N, M))
    mdl = Muskingum(d, members=M)
    t0 = int(mdl.datetime.value)
    times, table = S.make_forcing(N, NSTEPS, DT_S, SEED, t0_ns=t0, rows_every=12)
    f = mdl.make_forcing(times_ns=times, table=table, member_mul=S.make_member_multipliers(times.size, M, SEED))
    gauges = S.make_gauges(net["endnodes"], M_GAUGES, seed=4)
    nwin = NSTEPS // EVERY
    others = rng.choice(np.setdiff1d(np.arange(N), gauges), size=500, replace=False)
    reaches = np.concatenate([gauges, others]).astype(np.int64)
    return dict(torch=torch, pd=pd, S=S, Muskingum=Muskingum, EnKF=EnsembleKalmanFilter, net=net, prm=prm, mdl=mdl,
                t0=t0, f=f, gauges=gauges, nwin=nwin, reaches=reaches, rng=rng, d=d)


def assim(out):
    c = setup()
    torch, pd, mdl = c["torch"], c["pd"], c["mdl"]
    gauges, nwin, rng = c["gauges"], c["nwin"], c["rng"]
    m = gauges.size
    idx = pd.DatetimeIndex(pd.to_datetime(c["t0"] + (np.arange(nwin, dtype=np.int64) + 1) * int(EVERY * DT_S * 1e9),
                                          unit="ns", utc=True)).as_unit("ns")
    truth = c["prm"]["o_t"][gauges]
    meas = pd.DataFrame(np.repeat(truth[None], nwin, 0), index=idx, columns=[c["d"]["reach_ids"][j] for j in gauges])
    enkf = c["EnKF"](mdl, meas, 2.0, 1e-2 * np.eye(m), every=pd.Timedelta(seconds=EVERY * DT_S), group=False)
    Zp = torch.as_tensor(truth[None, :, None] + 0.1 * rng.standard_normal((nwin, m, M)), device="cuda")
    O, I = mdl.device_state
    O0, I0 = O.clone(), I.clone()
    t_start = mdl.datetime
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def run(record):
        flush.fill_(1)
        Oc, Ic = mdl.device_state
        Oc.copy_(O0); Ic.copy_(I0)
        mdl._datetime = t_start
        if record:
            return mdl.run_assimilating(c["f"], NSTEPS, enkf, EVERY, Zp, record_reaches=c["reaches"], record_every=1,
                                        record_prior=True)
        return mdl.run_assimilating(c["f"], NSTEPS, enkf, EVERY, Zp)

    def timed(record):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        r = run(record)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), r

    for rec in (False, True):
        run(rec)                                          # warm-up of every shape
    torch.cuda.synchronize()
    ms = {False: [], True: []}
    for _ in range(out["reps"]):
        for rec in (False, True):
            ms[rec].append(timed(rec)[0])
    mdl.network.check()
    _, (r, p) = timed(True)
    # kernel times of one run of each arm (torch.profiler, runs of their own)
    from torch.profiler import profile, ProfilerActivity
    kern = {}
    for rec in (False, True):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run(rec)
            torch.cuda.synchronize()
        tot = {}
        for e in prof.events():
            if "CUDA" not in str(getattr(e, "device_type", "")):
                continue
            name = e.name
            for key in ("enkf_record_kernel", "route_window_kernel", "enkf_small_system_kernel"):
                if key in name:
                    t = tot.setdefault(key, [0.0, 0])
                    t[0] += getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
                    t[1] += 1
        kern["record" if rec else "plain"] = {k: {"us_total": round(v[0], 1), "launches": v[1],
                                                  "us_per_launch": round(v[0] / max(1, v[1]), 2)}
                                              for k, v in tot.items()}
    a, b = np.median(ms[False]), np.median(ms[True])
    out["assimilating"] = {
        "shape": {"reaches": N, "members": M, "gauges": m, "steps": NSTEPS, "every": EVERY, "windows": nwin,
                  "recorded_reaches": int(c["reaches"].size)},
        "ms_plain": [round(x, 3) for x in ms[False]], "ms_record": [round(x, 3) for x in ms[True]],
        "median_ms_plain": round(float(a), 3), "median_ms_record": round(float(b), 3),
        "overhead_pct": round(100.0 * (b - a) / a, 2),
        "overhead_us_per_window": round(1e3 * (b - a) / nwin, 2),
        "bytes_recorded": int(r.numel() * 8 + p.numel() * 8),
        "kernels": kern,
    }


CHILD = r"""
import json, os, sys, numpy as np, torch
sys.path.insert(0, %r)
sys.argv = ['x']
import importlib.util
spec = importlib.util.spec_from_file_location('tr', %r); tr = importlib.util.module_from_spec(spec); spec.loader.exec_module(tr)
c = tr.setup(); mdl = c['mdl']
O, I = mdl.device_state; O0, I0 = O.clone(), I.clone(); t_start = mdl.datetime
flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
res = []
for it in range(1 + %d):
    flush.fill_(1); O.copy_(O0); I.copy_(I0); mdl._datetime = t_start
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    rec = mdl.run(c['f'], tr.NSTEPS, record_reaches=c['reaches'])
    e1.record(); torch.cuda.synchronize()
    if it: res.append(e0.elapsed_time(e1))
mdl.network.check()
np.save(sys.argv[1] if len(sys.argv) > 1 else os.environ['TR_OUT'], rec.cpu().numpy()[::97])
print(json.dumps(res))
"""


def run_kernels(out):
    import tempfile
    res = {"window": [], "dataflow": []}
    samples = {}
    with tempfile.TemporaryDirectory() as tmp:
        for rnd in range(2):
            for k in ("window", "dataflow"):
                env = dict(os.environ, TXH_ROUTE_KERNEL=k, TR_OUT=os.path.join(tmp, k + ".npy"))
                code = CHILD % (ROOT, os.path.abspath(__file__), out["reps"])
                p = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=1800)
                if p.returncode != 0:
                    raise RuntimeError(p.stderr[-2000:])
                res[k] += json.loads(p.stdout.strip().splitlines()[-1])
                samples[k] = np.load(os.path.join(tmp, k + ".npy"))
    from parity import relerr  # noqa: E402  (tests/)
    out["run_record"] = {
        "shape": {"reaches": N, "members": M, "steps": NSTEPS, "recorded_reaches": 1000, "record_every": 1},
        "ms_window": [round(x, 3) for x in res["window"]], "ms_dataflow": [round(x, 3) for x in res["dataflow"]],
        "median_ms_window": round(float(np.median(res["window"])), 3),
        "median_ms_dataflow": round(float(np.median(res["dataflow"])), 3),
        "relerr_window_vs_dataflow_sampled": relerr(samples["window"], samples["dataflow"]),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--skip-run", action="store_true")
    args = ap.parse_args()
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch
    assert torch.cuda.is_available(), "time_record.py measures on the GPU"
    out = {"reps": args.reps, "gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        out["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except Exception as e:  # noqa: BLE001
        out["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    t = time.time()
    assim(out)
    if not args.skip_run:
        run_kernels(out)
    out["wall_s"] = round(time.time() - t, 1)
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fp:
            fp.write(s + "\n")


if __name__ == "__main__":
    main()

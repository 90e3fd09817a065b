"""Cost and effect of the ensemble Kalman smoother of recorded hydrographs, at the C3 shape of tools/time_record.py
(100,000 reaches, 64 members, 2,016 5-minute steps, an hourly EnKF over 500 gauges, 1,000 reaches recorded after every
step).  One process; CUDA events around work that ends in a device synchronise; the L2 cache overwritten before every
timed run:

  * the recorded in-library loop without and with the transform history set (txh_set_transform_history), alternated:
    ms per run and launches per run (txh_launch_count);
  * the smoothing pass (txh_enks_smooth) for lags of 288 steps (24 h) and 2,016 steps (the whole run): ms per pass, its
    kernels (torch.profiler, a run of its own), the FLOPs and bytes of the pass over the recorded rows computed from
    the shapes, and their share of the FP64 tensor-core rate and HBM bandwidth measured on this card class
    (tools/ubench/fp64.cu: 37 TFLOP/s; 6.53 TB/s);
  * a seeded twin experiment: a one-member truth run with the unperturbed forcing, gauges observed from it with noise
    of standard deviation 0.1; RMSE of the ensemble mean against the truth at the gauged recorded reaches, filtered
    and smoothed (reported, not asserted).

    python tools/time_smooth.py [--reps 5] [--out result.json]
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

DMMA_PEAK = 37e12            # FP64 tensor-core FLOP/s measured by tools/ubench/fp64.cu on a B200
HBM_PEAK = 6.53e12           # bytes/s measured on a B200
LAGS = (288, 2016)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "time_smooth.py measures on the GPU"
    spec = importlib.util.spec_from_file_location("time_record", os.path.join(ROOT, "tools", "time_record.py"))
    tr = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tr)
    from tx_fast_hydrology_b200 import _lib
    lib = _lib.load()
    out = {"reps": args.reps, "gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        out["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except Exception as e:  # noqa: BLE001
        out["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    t_wall = time.time()
    c = tr.setup()
    pd, mdl, net_d, prm, d = c["pd"], c["mdl"], c["net"], c["prm"], c["d"]
    N, M, EVERY, NSTEPS, DT_S = tr.N, tr.M, tr.EVERY, tr.NSTEPS, tr.DT_S
    gauges, nwin, reaches, rng = c["gauges"], c["nwin"], c["reaches"], c["rng"]
    m = gauges.size

    # the truth of the twin experiment: one member, the unperturbed forcing, the unperturbed initial state
    from tx_fast_hydrology_b200.muskingum import Muskingum
    dt = dict(d); dt["o_t"] = prm["o_t"]
    truth_mdl = Muskingum(dt, members=1)
    times, table = c["S"].make_forcing(N, NSTEPS, DT_S, tr.SEED, t0_ns=c["t0"], rows_every=12)
    truth = truth_mdl.run(truth_mdl.make_forcing(times_ns=times, table=table), NSTEPS,
                          record_reaches=reaches).cpu().numpy()[:, :, 0]          # [steps][k]
    obs = truth[EVERY - 1::EVERY][:nwin, :m]                                      # gauges are reaches[:m]
    order = np.argsort(gauges)                                  # the filter takes its gauges in ascending order
    Zp = torch.as_tensor(obs[:, order, None] + 0.1 * rng.standard_normal((nwin, m, M)), device="cuda").contiguous()
    idx = pd.DatetimeIndex(pd.to_datetime(c["t0"] + (np.arange(nwin, dtype=np.int64) + 1) * int(EVERY * DT_S * 1e9),
                                          unit="ns", utc=True)).as_unit("ns")
    meas = pd.DataFrame(obs, index=idx, columns=[d["reach_ids"][j] for j in gauges])
    enkf = c["EnKF"](mdl, meas, 2.0, 1e-2 * np.eye(m), every=pd.Timedelta(seconds=EVERY * DT_S), group=False)
    net = mdl.network
    O, I = mdl.device_state
    O0, I0, t_start = O.clone(), I.clone(), mdl.datetime
    T_hist = torch.empty((nwin, M, M), dtype=torch.float64, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def run(hist):
        flush.fill_(1)
        Oc, Ic = mdl.device_state
        Oc.copy_(O0); Ic.copy_(I0)
        mdl._datetime = t_start
        net.set_transform_history(T_hist if hist else None)
        try:
            torch.cuda.synchronize()
            n0 = lib.txh_launch_count()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rec, prior = mdl.run_assimilating(c["f"], NSTEPS, enkf, EVERY, Zp, record_reaches=reaches, record_every=1,
                                              record_prior=True)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1), lib.txh_launch_count() - n0, rec
        finally:
            net.set_transform_history(None)

    for hist in (False, True):
        run(hist)
    ms = {False: [], True: []}
    launches = {}
    for _ in range(args.reps):
        for hist in (False, True):
            t, nl, _ = run(hist)
            ms[hist].append(t)
            launches[hist] = nl
    _, _, rec_plain = run(False)
    _, _, rec = run(True)
    net.check()
    a, b = float(np.median(ms[False])), float(np.median(ms[True]))
    out["loop"] = {
        "shape": {"reaches": N, "members": M, "gauges": m, "steps": NSTEPS, "every": EVERY, "updates": nwin,
                  "recorded_reaches": int(reaches.size), "record_every": 1},
        "ms_record": [round(x, 3) for x in ms[False]], "ms_record_with_history": [round(x, 3) for x in ms[True]],
        "median_ms_record": round(a, 3), "median_ms_record_with_history": round(b, 3),
        "launches_record": int(launches[False]), "launches_record_with_history": int(launches[True]),
        "rec_bitwise_equal_with_history": bool(torch.equal(rec, rec_plain)),
    }

    # the smoothing pass
    nslots, k = rec.shape[0], rec.shape[1]
    rows = nslots * k
    work = torch.empty(net.enks_work_size(M, nwin), dtype=torch.float64, device="cuda")
    sm = torch.empty_like(rec)
    passes = {}
    mean_truth = truth[:, :m]
    filt_rmse = float(np.sqrt(np.mean((rec[:, :m].mean(dim=2).cpu().numpy() - mean_truth) ** 2)))
    from torch.profiler import profile, ProfilerActivity
    for lag in LAGS:
        net.enks_smooth(M, nwin, EVERY, T_hist, rec, 1, lag, sm, work)
        tl = []
        for _ in range(args.reps):
            flush.fill_(1)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            net.enks_smooth(M, nwin, EVERY, T_hist, rec, 1, lag, sm, work)
            e1.record()
            torch.cuda.synchronize()
            tl.append(e0.elapsed_time(e1))
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            net.enks_smooth(M, nwin, EVERY, T_hist, rec, 1, lag, sm, work)
            torch.cuda.synchronize()
        kern = {}
        for e in prof.events():
            if "enks_" in e.name:
                key = e.name.split("enks_")[1].split("_kernel")[0]
                kern[key] = round(kern.get(key, 0.0) + (getattr(e, "device_time_total", None)
                                                        or getattr(e, "cuda_time_total", 0.0)), 1)
        # stage (b) over the rows some update reaches (the rest are copied): 2 M^2 flops per row, rec read, out written
        smoothed_slots = sum(1 for j in range(nslots) if (j + 1) // EVERY < nwin and lag > 0)
        flops = 2.0 * M * M * smoothed_slots * k
        nbytes = 2.0 * rows * M * 8
        t_ms = float(np.median(tl))
        t_flop, t_mem = flops / DMMA_PEAK, nbytes / HBM_PEAK
        sm_rmse = float(np.sqrt(np.mean((sm[:, :m].mean(dim=2).cpu().numpy() - mean_truth) ** 2)))
        passes[str(lag)] = {
            "ms": [round(x, 4) for x in tl], "median_ms": round(t_ms, 4), "kernels_us": kern,
            "flops_stage_b": flops, "bytes_stage_b": nbytes,
            "dmma_share": round(t_flop / (t_ms * 1e-3), 3), "hbm_share": round(t_mem / (t_ms * 1e-3), 3),
            "bound": "fp64 tensor" if t_flop > t_mem else "hbm",
            "pct_of_recorded_run": round(100.0 * t_ms / a, 2),
            "rmse_mean_vs_truth_gauged_filtered": round(filt_rmse, 6),
            "rmse_mean_vs_truth_gauged_smoothed": round(sm_rmse, 6),
        }
    out["smooth"] = {"rec_bytes": rows * M * 8, "passes": passes}
    net.check()
    out["wall_s"] = round(time.time() - t_wall, 1)
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fp:
            fp.write(s + "\n")


if __name__ == "__main__":
    main()

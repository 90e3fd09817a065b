#!/usr/bin/env python
"""bench.py -- headline benchmark of the routing + assimilation hot path (driver contract).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

Workload = BASELINE.json configs[2] ("C3"): the synthetic Texas-scale network (100,000 reaches,
1,000 topological levels, seed 2), a 64-member ensemble PER GPU, a 7-day run at a 5-minute step
(2,016 routing steps) with an EnKF assimilation of 500 synthetic gauges every hour (168 updates).
One bench "step" is one whole 7-day run.  The metric is reach*timestep*member updates per second.

  value : device-resident run (inputs already in HBM), CUDA events, max over ranks
  e2e   : the same run through the public Python API from PINNED HOST buffers: initial ensemble,
          forcing table, member multipliers and observations copied host->device and the final
          ensemble copied device->host inside the timed region
  roofline : route_window_kernel (the window-resident routing kernel, one launch per hourly window),
          algorithmic bytes per launch / its mean CUDA-event duration / measured HBM copy bandwidth
  cpu_baseline : the reference's own numba kernels (oracle/_ref: `_ax_bu` + `interpolate_sample`, nutils.py,
          members fanned out over one process per host core) + the numpy ensemble update, on a bounded
          sample of the same workload; `port_value` = the C/OpenMP restatement (oracle/txh_oracle.c) beside
          it; rank 0 at N=1 only.  Without oracle/_ref the port alone is timed (kind "port").
  parity_max_rel_err : element-wise relative error (floor 1e-12 of the largest element) of the GPU ensemble
          against that CPU sample after its windows (routing + EnKF updates), same inputs
  members / c4_basins (N > 1): the member-sharded form of the same C3 run (one 64-member ensemble over the
          ranks, EnKF statistics combined over NVLink) and BASELINE.json configs[3] (2.7M reaches partitioned
          by independent basins over the ranks, no collective), each timed like `value`

--impl reference times the CPU arm alone: the reference's kernels from oracle/_ref when present, else the
port, on all the host cores of the box, on the same workload configuration the GPU arm reports at --gpus N.

--dump-outputs DIR writes, after the timed steps of the GPU arm, the state the last timed step left (what
`Muskingum.o_t_next` / `i_t_next` would hand a caller), float64, on rank 0, as DIR/<name>.npy:
  c3_outflow, c3_inflow : [32,768 reaches][members] of the C3 ensemble (`value`)
  c4_outflow, c4_inflow : [262,144 reaches] of the C4 forest (`c4_basins`, rank 0's shard), unless --no-extras
The reaches are a fixed sorted sample (numpy default_rng(0), independent of --seed), in ascending reach order; all
inputs derive from --seed, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "reach*timestep*member updates/sec"
UNIT = "updates/s"
DT_S = 300.0
T0 = "2024-01-01T00:00:00Z"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    # workload knobs (defaults = the configuration the metric is quoted on)
    ap.add_argument("--reaches", type=int, default=100000)
    ap.add_argument("--members", type=int, default=64, help="ensemble members per GPU")
    ap.add_argument("--days", type=float, default=7.0)
    ap.add_argument("--gauges", type=int, default=500)
    ap.add_argument("--assim-every", type=int, default=12, help="routing steps between EnKF updates")
    ap.add_argument("--seed", type=int, default=2)
    ap.add_argument("--cpu-windows", type=int, default=3, help="hourly windows in the CPU sample")
    ap.add_argument("--sharding", default="basins", choices=["basins", "members"],
                    help="N > 1: one independent basin (network + ensemble + gauges) per GPU, no collective; or the "
                         "members of ONE network's ensemble over the GPUs, EnKF statistics combined with NCCL")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the C4 (basin-partitioned) and member-sharded arms")
    ap.add_argument("--c4-reaches", type=int, default=2_700_000)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the state of the last timed step as DIR/<name>.npy (see the module docstring)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return a


def algorithmic_bytes_per_update(M):
    """SURVEY.md section 8d: read o_prev, i_prev, write o_next, i_next (32 B) + per reach*step terms
    shared by the members: 4 coefficients (32 B), forcing (8 B), one index (4 B)."""
    return 32.0 + 44.0 / M


DUMP_C3_REACHES = 32768           # x 64 members x 8 B x 2 arrays = 33.6 MB
DUMP_C4_REACHES = 262144          # x 8 B x 2 arrays = 4.2 MB
DUMP_LIMIT_BYTES = 64 << 20


def sample_reaches(n, k):
    """A fixed sorted sample of k of n reach indices (all of them when k >= n): the same in every run and build."""
    if k >= n:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))


def write_outputs(out_dir, arrays):
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes (limit {DUMP_LIMIT_BYTES})")
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


# ------------------------------------------------------------------------------------------------
# workload (identical numbers for the GPU arm and the CPU arm)
# ------------------------------------------------------------------------------------------------
class Workload:
    def __init__(self, a, rank=0, world=1):
        from tx_fast_hydrology_b200 import synthetic as S
        self.a = a
        self.n = n = a.reaches
        self.M = M = a.members
        self.Mtot = M * world
        self.rank, self.world = rank, world
        self.by_basin = a.sharding == "basins" and world > 1
        if self.by_basin:
            # basin sharding: every rank owns an independent basin of the same size with its own ensemble
            # and gauges (the reference's app runs one Kalman filter per sub-basin model, app.py:130-141)
            self.Mtot = M
        seed = a.seed + (1000 * rank if self.by_basin else 0)
        self.seed = seed
        self.nsteps = int(round(a.days * 86400.0 / DT_S))
        self.every = a.assim_every
        self.nwin = self.nsteps // self.every
        self.net = S.make_network(n, seed)
        self.params = S.make_params(n, seed)
        import pandas as pd
        self.t0_ns = int(pd.Timestamp(T0).value)
        self.times, self.table = S.make_forcing(n, self.nsteps, DT_S, seed, t0_ns=self.t0_ns, rows_every=12)
        mul_all = S.make_member_multipliers(self.times.size, self.Mtot, seed)
        c0 = 0 if self.by_basin else rank * M
        self.mul = np.ascontiguousarray(mul_all[:, c0:c0 + M])
        rng = np.random.default_rng(seed + 7)
        spread = rng.uniform(0.5, 1.5, size=(n, self.Mtot))
        self.o0 = np.ascontiguousarray(self.params["o_t"][:, None] * spread[:, c0:c0 + M])
        self.gauges = S.make_gauges(self.net["endnodes"], a.gauges, seed=4)
        self.m = self.gauges.size
        self.R = 1e-2 * np.eye(self.m)             # app.py:137-138 values
        self.Q = 2.0
        self.model_dict = S.model_dict(self.net, self.params, dt_s=DT_S, t0=T0)
        self.Zp = None

    def make_observations(self, truth):
        """truth [nwin][m] -> per-member perturbed observations [nwin][m][Mtot] (all ranks identical)."""
        rng = np.random.default_rng(self.seed + 11)
        obs = truth + 0.1 * rng.standard_normal(truth.shape)                 # N(0, R), R = 1e-2 I
        noise = 0.1 * rng.standard_normal((truth.shape[0], self.m, self.Mtot))
        self.obs = obs
        self.Zp = np.ascontiguousarray(obs[:, :, None] + noise)
        return self.Zp

    def updates_per_run(self):
        """whole job: all ranks"""
        return float(self.n) * self.M * self.world * self.nsteps


# ------------------------------------------------------------------------------------------------
# clocks (pynvml sampling thread; nvidia-smi is the fallback)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}
    NOTE = {"sw_power_cap": 0x4}

    def __init__(self, device_index):
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._h = None
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            self._nv = pynvml
            h = None
            try:
                uuid = str(torch.cuda.get_device_properties(device_index).uuid)
                h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self._h = h
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._h = None
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h))
                for k, bit in {**self.BAD, **self.NOTE}.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        if self._h is not None:
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._h is not None and self._t.is_alive():
            self._t.join(timeout=2)
        med = int(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port on a bounded sample of the workload
# ------------------------------------------------------------------------------------------------
class CpuSample:
    """`windows` hourly windows of the workload on the host: members routed over OpenMP threads
    (oracle.run_members, nutils.py:64-89 per member), then the ensemble update (oracle.enkf_update,
    da.py:112-126 on the sample covariance) in numpy/LAPACK."""

    def __init__(self, wl, windows):
        from oracle import oracle as O
        O.build()
        self.O, self.wl, self.windows = O, wl, windows
        net = wl.net
        ind = O.compute_indegree(net["startnodes"], net["endnodes"])
        al, be, ch, ga = O.compute_coeffs(wl.params["K"], wl.params["X"], DT_S)
        self.net = {"startnodes": net["startnodes"], "endnodes": net["endnodes"], "indegree": ind,
                    "alpha": al, "beta": be, "chi": ch, "gamma": ga}
        self.threads = O.max_threads()
        self.o_init = np.ascontiguousarray(wl.o0.T)                      # [M][n]
        self.i_init = np.stack([O.init_states(net["startnodes"], net["endnodes"], o) for o in self.o_init])
        self.q_diag = np.full(wl.n, wl.Q)
        if wl.Zp is None:
            # the CPU arm alone: observations around the initial state (timing does not depend on values)
            rng = np.random.default_rng(5)
            self.Zp = wl.params["o_t"][wl.gauges][None, :, None] + 0.1 * rng.standard_normal(
                (windows, wl.m, wl.M))
        else:
            self.Zp = wl.Zp[:windows, :, :wl.M]
        self.updates = float(wl.n) * wl.M * wl.every * windows

    def run(self):
        O, wl = self.O, self.wl
        o = self.o_init.copy(); i = self.i_init.copy()
        xp = wl.times.astype(np.float64)
        step_ns = DT_S * 1e9
        t = float(wl.t0_ns)
        t0 = time.perf_counter()
        for k in range(self.windows):
            O.run_members(self.net, o, i, wl.every, xp, wl.table, t, step_ns, wmul=wl.mul, threads=self.threads)
            t += wl.every * step_ns
            Op, Ip, _ = O.enkf_update(self.net, o.T, i.T, wl.gauges, self.Zp[k], self.q_diag, wl.R)
            o = np.ascontiguousarray(Op.T); i = np.ascontiguousarray(Ip.T)
        return time.perf_counter() - t0, o

    def describe(self):
        wl = self.wl
        return (f"{self.windows} hourly windows of the workload: {wl.every * self.windows} routing steps x "
                f"{wl.M} members x {wl.n} reaches + {self.windows} EnKF updates of {wl.m} gauges; "
                f"oracle/txh_oracle.c over {self.threads} OpenMP threads + numpy")


# state shared with the forked workers of RefSample (set before the pool is created)
_REF = {}


def _ref_worker(job):
    """One worker = a slice of the members: `every` steps of the reference's simulate loop (muskingum.py:527-533:
    interpolate the forcing at t + dt, then `_ax_bu`, nutils.py:64-89) on the shared state arrays."""
    lo, hi, t_ns = job
    R = _REF
    nu, xp, table, mul = R["nutils"], R["xp"], R["table"], R["mul"]
    o, i = R["o"], R["i"]
    for m in range(lo, hi):
        t = t_ns
        om, im = o[m].copy(), i[m].copy()
        for _ in range(R["every"]):
            t += R["step_ns"]
            # member m sees table[r] * mul[r][m]; the bracket weights come from the reference's own
            # interpolate_sample (nutils.py:5-39) applied to a table whose row r is the unit vector e_(r mod 2)
            ix = int(np.searchsorted(xp, t))
            if ix == 0:
                q = table[0] * mul[0, m]
            elif ix >= xp.size:
                q = table[-1] * mul[-1, m]
            else:
                w = nu.interpolate_sample(t, xp, R["unit"])
                q = (w[(ix - 1) % 2] * mul[ix - 1, m]) * table[ix - 1] + (w[ix % 2] * mul[ix, m]) * table[ix]
            im, om = nu._ax_bu(R["heads"], R["end"], R["alpha"], R["beta"], R["chi"], R["gamma"], im, om, q, R["indegree"])
        o[m] = om; i[m] = im
    return hi - lo


class RefSample:
    """The same bounded sample on the UNMODIFIED reference kernels (oracle/_ref, numba): one process per host core,
    each routing a slice of the members with `_ax_bu`; the ensemble update (which the reference does not have) is
    the oracle's numpy restatement of da.py:112-126 in the parent."""

    def __init__(self, wl, windows, nutils):
        import multiprocessing as mp
        from oracle import oracle as O
        self.O, self.wl, self.windows = O, wl, windows
        net = wl.net
        ind = O.compute_indegree(net["startnodes"], net["endnodes"])
        al, be, ch, ga = O.compute_coeffs(wl.params["K"], wl.params["X"], DT_S)
        self.net = {"startnodes": net["startnodes"], "endnodes": net["endnodes"], "indegree": ind,
                    "alpha": al, "beta": be, "chi": ch, "gamma": ga}
        M, n = wl.M, wl.n
        self.cores = min(O.max_threads(), M)
        shm_o = np.frombuffer(mp.RawArray("d", M * n), dtype=np.float64).reshape(M, n)
        shm_i = np.frombuffer(mp.RawArray("d", M * n), dtype=np.float64).reshape(M, n)
        self.o, self.i = shm_o, shm_i
        self.o_init = np.ascontiguousarray(wl.o0.T)
        self.i_init = np.stack([O.init_states(net["startnodes"], net["endnodes"], o) for o in self.o_init])
        R = wl.times.size
        unit = np.zeros((R, 2)); unit[0::2, 0] = 1.0; unit[1::2, 1] = 1.0     # row r -> e_(r mod 2): weights of a bracket
        _REF.update(nutils=nutils, xp=wl.times.astype(np.float64), table=wl.table, mul=wl.mul, o=shm_o, i=shm_i,
                    every=wl.every, step_ns=DT_S * 1e9, heads=net["startnodes"][ind == 0], end=net["endnodes"],
                    alpha=al, beta=be, chi=ch, gamma=ga, indegree=ind, unit=unit)
        # JIT in the parent, so the forked workers inherit the compiled kernels
        nutils._ax_bu(_REF["heads"], _REF["end"], al, be, ch, ga, self.i_init[0], self.o_init[0], wl.table[0], ind)
        nutils.interpolate_sample(float(wl.times[0]) + 1.0, _REF["xp"], unit)
        self.pool = mp.get_context("fork").Pool(self.cores)
        self.q_diag = np.full(n, wl.Q)
        if wl.Zp is None:
            rng = np.random.default_rng(5)
            self.Zp = wl.params["o_t"][wl.gauges][None, :, None] + 0.1 * rng.standard_normal((windows, wl.m, M))
        else:
            self.Zp = wl.Zp[:windows, :, :M]
        self.updates = float(n) * M * wl.every * windows
        bounds = np.linspace(0, M, self.cores + 1).astype(int)
        self.slices = [(int(bounds[k]), int(bounds[k + 1])) for k in range(self.cores) if bounds[k + 1] > bounds[k]]

    def run(self):
        O, wl = self.O, self.wl
        self.o[:] = self.o_init; self.i[:] = self.i_init
        t = float(wl.t0_ns)
        t0 = time.perf_counter()
        for k in range(self.windows):
            self.pool.map(_ref_worker, [(lo, hi, t) for lo, hi in self.slices])
            t += wl.every * DT_S * 1e9
            Op, Ip, _ = O.enkf_update(self.net, self.o.T, self.i.T, wl.gauges, self.Zp[k], self.q_diag, wl.R)
            self.o[:] = Op.T; self.i[:] = Ip.T
        return time.perf_counter() - t0, np.array(self.o)

    def close(self):
        self.pool.close(); self.pool.join()

    def describe(self):
        wl = self.wl
        return (f"{self.windows} hourly windows of the workload: {wl.every * self.windows} routing steps x {wl.M} members x "
                f"{wl.n} reaches on the reference's numba _ax_bu + interpolate_sample (oracle/_ref/tx_fast_hydrology/"
                f"nutils.py), members over {self.cores} processes, + {self.windows} EnKF updates of {wl.m} gauges (numpy "
                f"restatement of da.py:112-126; the reference has no ensemble filter)")


def cpu_samples(wl, windows):
    """(reference sample or None, port sample)"""
    from oracle import oracle as O
    nu = O.reference_nutils()
    ref = None
    if nu is not None:
        try:
            ref = RefSample(wl, windows, nu)
        except Exception as e:                       # numba missing or fork refused: the port still runs
            print(f"bench.py: reference kernels unavailable ({e}); timing the port", file=sys.stderr)
    return ref, CpuSample(wl, windows)


def reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return 0
    # the same workload description the GPU arm prints at --gpus N: with basin sharding every GPU owns one basin of
    # this size; the CPU routes them one after another, so its throughput is that of one basin (rank 0's)
    a_cfg = argparse.Namespace(**vars(a))
    wl = Workload(a, 0, 1)
    try:
        from threadpoolctl import threadpool_limits
        from oracle import oracle as O
        threadpool_limits(limits=O.max_threads())    # numpy's BLAS too (torchrun exports OMP_NUM_THREADS=1)
    except Exception:
        pass
    ref, port = cpu_samples(wl, a.cpu_windows)
    cs = ref if ref is not None else port
    for _ in range(max(1, a.warmup)):
        cs.run()
    tot = 0.0
    for _ in range(a.steps):
        dt, _ = cs.run()
        tot += dt
    val = cs.updates * a.steps / tot
    cores = cs.cores if ref is not None else cs.threads
    cpu = {"value": val, "unit": UNIT, "cores": cores, "kind": "reference" if ref is not None else "port",
           "sample": cs.describe()}
    if ref is not None:
        port.run()
        cpu["port_value"] = port.updates / min(port.run()[0] for _ in range(2))
        cpu["port_cores"] = port.threads
        ref.close()
    n_gpus = max(a.gpus, world)
    cfg_wl = wl
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": n_gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * tot / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(cfg_wl, a_cfg, n_gpus, by_basin=(n_gpus > 1 and a.sharding == "basins")),
        "cpu_baseline": cpu,
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def workload_config(wl, a, world, by_basin=None):
    by_basin = wl.by_basin if by_basin is None else by_basin
    return {
        "workload": (f"C3: synthetic Texas-scale network, ONE {wl.Mtot}-member ensemble with its members sharded over "
                     f"{world} GPUs ({wl.M} per GPU), 7-day run at a 5-min step, hourly EnKF of 500 gauges "
                     "(BASELINE.json configs[2])" if (world > 1 and not by_basin) else
                     "C3: synthetic Texas-scale network, 64-member ensemble per GPU, 7-day run at a 5-min step, "
                     "hourly EnKF of 500 gauges (BASELINE.json configs[2])"),
        "reaches": wl.n * (world if by_basin else 1), "reaches_per_gpu": wl.n, "levels": 1000,
        "members_per_gpu": wl.M, "members_per_ensemble": wl.Mtot,
        "routing_steps": wl.nsteps, "dt_s": DT_S, "gauges": wl.m, "enkf_updates": wl.nwin,
        "assimilate_every_steps": wl.every, "seed": a.seed,
        "sharding": ("single GPU" if world == 1 else
                     "independent basins, one per GPU, each with its own ensemble, gauges and EnKF; no collective"
                     if by_basin else
                     "ensemble members of one network over ranks (network replicated); EnKF statistics combined with NCCL"),
        "l2": "256 MiB buffer written between bench steps (inside the timed region); per-run inputs "
              "(forcing 135 MB + observations + 102 MB state) exceed the 126 MB L2",
    }


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def gpu_arm(a):
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback); "
                         "use --impl reference for the CPU arm")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    numa = pin_to_gpu_numa_node(local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from tx_fast_hydrology_b200 import build
    build.build_lib()
    dump = {} if (a.dump_outputs and rank == 0) else None
    # the headline line: C3 on one GPU, or one independent C3 basin per GPU (weak scaling, no collective)
    line = c3_arm(a, rank, world, local, full=True, dump=dump)
    if world > 1 and not a.no_extras and a.sharding == "basins":
        # BASELINE.json configs[2] as written: ONE 64-member ensemble with its members sharded over the ranks
        # (strong scaling: 64 / N members per GPU), EnKF statistics combined over NVLink
        if a.members % world == 0:
            am = argparse.Namespace(**vars(a))
            am.sharding, am.members = "members", a.members // world
            sub = c3_arm(am, rank, world, local, full=False)
            if rank == 0:
                line["members"] = {k: sub[k] for k in ("value", "unit", "ms_per_step", "scaling", "config", "gpu_launches",
                                                       "roofline", "update_path")}
    if not a.no_extras:
        c4 = c4_arm(a, rank, world, local, dump=dump)
        if rank == 0:
            line["c4_basins"] = c4
    if rank == 0:
        line["host_affinity"] = numa
        if dump is not None:
            write_outputs(a.dump_outputs, dump)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def pin_to_gpu_numa_node(local):
    """N ranks share the host: run this rank (and first-touch its pinned buffers) on the CPUs next to its GPU
    (/sys/bus/pci/devices/<bus id>/local_cpulist), so the end-to-end uploads do not cross the socket interconnect.
    Best effort; returns what was done."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local).pci_bus_id
        dom = getattr(torch.cuda.get_device_properties(local), "pci_domain_id", 0)
        dev = getattr(torch.cuda.get_device_properties(local), "pci_device_id", 0)
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/local_cpulist"
        with open(path) as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            if "-" in part:
                lo, hi = part.split("-"); cpus.update(range(int(lo), int(hi) + 1))
            elif part:
                cpus.add(int(part))
        allowed = cpus & set(os.sched_getaffinity(0))
        if not allowed:
            return {"pinned": False, "why": "no overlap with the allowed CPUs", "local_cpulist": spec}
        os.sched_setaffinity(0, allowed)
        return {"pinned": True, "cpus": len(allowed), "local_cpulist": spec}
    except Exception as e:                           # noqa: BLE001
        return {"pinned": False, "why": str(e)[:120]}


def c4_arm(a, rank, world, local, dump=None):
    """BASELINE.json configs[3]: the CONUS-scale forest (2.7M reaches, 64 independent basins, seed 3), deterministic,
    24 hours at a 5-min step (288 steps), whole basins bin-packed over the ranks (sharding.shard_basins) and routed
    with no collective: strong scaling of a fixed forest.  Device-resident timing like `value`."""
    import torch
    import torch.distributed as dist
    import pandas as pd
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.muskingum import Muskingum
    from tx_fast_hydrology_b200.sharding import shard_basins, extract_shard
    dev = torch.device("cuda", local)
    n_total, nsteps, seed = a.c4_reaches, 288, 3
    net = S.make_network(n_total, seed, n_basins=64)
    parts = shard_basins(net["basin"], world)
    sub_end, idx = extract_shard(net["endnodes"], net["basin"], parts[rank])
    prm = S.make_params(n_total, seed)
    t0_ns = int(pd.Timestamp(T0).value)
    times, table = S.make_forcing(n_total, nsteps, DT_S, seed, t0_ns=t0_ns, rows_every=12)
    n = idx.size
    sub_net = {"startnodes": np.arange(n, dtype=np.int64), "endnodes": sub_end}
    sub_prm = {k: np.ascontiguousarray(v[idx]) for k, v in prm.items()}
    t_topo = time.perf_counter()
    mdl = Muskingum(S.model_dict(sub_net, sub_prm, dt_s=DT_S, t0=T0), members=1)
    t_topo = time.perf_counter() - t_topo
    f = mdl.make_forcing(times_ns=times, table=np.ascontiguousarray(table[:, idx]))
    del table
    O, I = mdl.device_state
    O0, I0 = O.clone(), I.clone()
    t_start = pd.Timestamp(T0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def run():
        flush.fill_(1)
        O.copy_(O0); I.copy_(I0)
        mdl._datetime = t_start
        mdl.run(f, nsteps)

    for _ in range(max(3, a.warmup)):
        run()
    mdl.network.check()
    ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(a.steps):
        run()
    ev1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    mdl.network.check()
    ms = ev0.elapsed_time(ev1) / a.steps
    counts = [n]
    if world > 1:
        t = torch.tensor([ms, float(n)], dtype=torch.float64, device=dev)
        allv = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(allv, t)
        ms = max(float(x[0]) for x in allv)
        counts = [int(x[1]) for x in allv]
    o_fin = mdl.download_state()[0]
    ok = bool(np.isfinite(o_fin).all())
    if dump is not None:
        keep = sample_reaches(n, DUMP_C4_REACHES)
        dump["c4_outflow"] = o_fin[keep, 0]
        dump["c4_inflow"] = mdl.network.unpack_host(I, 1)[keep, 0]
    f.close()
    del mdl, O0, I0, flush
    torch.cuda.empty_cache()
    upd = float(n_total) * nsteps
    ab = algorithmic_bytes_per_update(1)
    return {"workload": "C4: CONUS-scale synthetic forest, 64 independent basins, deterministic, 24-hour run at a 5-min "
                        "step (BASELINE.json configs[3]); whole basins bin-packed over the ranks, no collective",
            "value": upd / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "scaling": "strong", "reaches": n_total,
            "routing_steps": nsteps, "members": 1, "reaches_per_rank": counts,
            "load_imbalance": max(counts) / (sum(counts) / len(counts)), "topology_pass_s_rank0": round(t_topo, 3),
            "algorithmic_GBps": upd * ab / (ms * 1e-3) / 1e9, "finite": ok,
            "l2": "256 MiB buffer written between bench steps (inside the timed region)"}


def c3_arm(a, rank, world, local, full, dump=None):
    """One C3 measurement (see the module docstring).  `full`: also the end-to-end arm, the CPU baseline and the
    in-run parity number (rank 0, single GPU).  `dump`: a dict that receives samples of the final state of the timed
    steps.  Returns the JSON line as a dict (meaningful on rank 0)."""
    import torch
    import torch.distributed as dist
    from tx_fast_hydrology_b200 import _lib
    lib = _lib.load()
    import pandas as pd
    from tx_fast_hydrology_b200.muskingum import Muskingum
    from tx_fast_hydrology_b200.da import EnsembleKalmanFilter

    wl = Workload(a, rank, world)
    n, M, m, nsteps, every, nwin = wl.n, wl.M, wl.m, wl.nsteps, wl.every, wl.nwin
    dev = torch.device("cuda", local)

    # ---- truth run (setup, untimed): one deterministic member, gauge outflows every hour -------
    truth_mdl = Muskingum(dict(wl.model_dict), members=1)
    f1 = truth_mdl.make_forcing(times_ns=wl.times, table=wl.table)
    rec = truth_mdl.run(f1, nwin * every, record_reaches=wl.gauges, record_every=every)
    truth_mdl.network.check()
    truth = rec.cpu().numpy()[:, :, 0]
    f1.close()
    del truth_mdl
    Zp_host = wl.make_observations(truth)

    # ---- the ensemble model + filter ---------------------------------------------------------------
    d = dict(wl.model_dict)
    d["o_t"] = wl.o0
    mdl = Muskingum(d, members=M)
    idx = pd.DatetimeIndex(pd.to_datetime(wl.t0_ns + (np.arange(nwin, dtype=np.int64) + 1) * int(every * DT_S * 1e9),
                                          unit="ns", utc=True)).as_unit("ns")
    meas = pd.DataFrame(wl.obs, index=idx, columns=[d["reach_ids"][j] for j in wl.gauges])
    enkf = EnsembleKalmanFilter(mdl, meas, wl.Q, wl.R, every=pd.Timedelta(seconds=every * DT_S),
                                group=False if (wl.by_basin or world == 1) else None)
    assert enkf.Mtot == wl.Mtot

    # pinned host inputs / outputs of the end-to-end arm
    def pinned(x):
        t = torch.from_numpy(np.ascontiguousarray(x)).pin_memory()
        return t
    o0_pin = pinned(wl.o0)
    table_pin = pinned(wl.table)
    mul_pin = pinned(wl.mul)
    Zp_pin = pinned(Zp_host)
    out_pin = torch.empty((n, M), dtype=torch.float64).pin_memory()
    Zp_dev = torch.empty((nwin, m, wl.Mtot), dtype=torch.float64, device=dev)

    # device-resident inputs of the `value` arm
    forcing = mdl.make_forcing(times_ns=wl.times, table=table_pin, member_mul=mul_pin)
    mdl.upload_state(o0_pin)
    O, I = mdl.device_state
    O0, I0 = O.clone(), I.clone()
    Zp_dev.copy_(Zp_pin)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    t_start = pd.Timestamp(T0)

    def resident_run(timers=None):
        flush.fill_(1)                                   # L2 flush between bench steps
        Oc, Ic = mdl.device_state                        # (a member-sharded filter alternates two state buffers)
        Oc.copy_(O0); Ic.copy_(I0)
        mdl._datetime = t_start
        mdl.run_assimilating(forcing, nsteps, enkf, every, Zp_dev, timers=timers)

    e2e_parts = {}
    copy_stream = torch.cuda.Stream()
    obs_ready = torch.cuda.Event()

    def e2e_run():
        def lap(key, t0, sync=True):
            if sync:
                torch.cuda.synchronize()
            t1 = time.perf_counter()
            e2e_parts[key] = e2e_parts.get(key, 0.0) + (t1 - t0)
            return t1
        t = time.perf_counter()
        mdl.upload_state(o0_pin)                                                     # H2D
        t = lap("upload_state_ms", t)
        # H2D into the resident table, in row chunks on the forcing's copy stream: the routing launches wait only for
        # the hours they read, so the upload overlaps the first windows (its time shows up inside run_ms)
        forcing.update(wl.times, table_pin, mul_pin, overlap=True)
        f = forcing
        t = lap("forcing_enqueue_ms", t, sync=False)
        with torch.cuda.stream(copy_stream):                                         # H2D beside the first window
            Zp_dev.copy_(Zp_pin, non_blocking=True)
            obs_ready.record(copy_stream)
        t = lap("observations_enqueue_ms", t, sync=False)
        mdl._datetime = t_start
        mdl.run_assimilating(f, nsteps, enkf, every, Zp_dev, observations_ready=obs_ready)
        t = lap("run_ms", t)
        mdl.download_state(out_o=out_pin)                                            # D2H (synchronises)
        lap("download_ms", t)

    h2d = o0_pin.numel() * 8 + table_pin.numel() * 8 + mul_pin.numel() * 8 + Zp_pin.numel() * 8
    d2h = out_pin.numel() * 8

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return float(x)
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- warm-up ---------------------------------------------------------------------------------------
    for _ in range(a.warmup):
        resident_run()
    mdl.network.check()

    # ---- timed: K device-resident runs ---------------------------------------------------------------
    clocks = ClockSampler(local)
    timers = []
    ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
    launches0 = int(lib.txh_launch_count())
    barrier()
    clocks.start()
    wall0 = time.perf_counter()
    ev0.record()
    for _ in range(a.steps):
        resident_run(timers)
    ev1.record()
    barrier()
    wall = time.perf_counter() - wall0
    clk = clocks.stop()
    launches = int(lib.txh_launch_count()) - launches0
    mdl.network.check()
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    ms_step = ms_total / a.steps
    value = wl.updates_per_run() / (ms_step * 1e-3)
    final_o = mdl.download_state()[0]
    if not np.isfinite(final_o).all():
        raise SystemExit("bench.py: non-finite ensemble state after the run")
    if dump is not None:
        keep = sample_reaches(n, DUMP_C3_REACHES)
        dump["c3_outflow"] = final_o[keep]
        dump["c3_inflow"] = mdl.network.unpack_host(mdl.device_state[1], M)[keep]

    # routing kernel roofline: mean CUDA-event duration of one launch (one hourly window)
    # (an unsharded ensemble runs inside the library, which keeps the event pairs; the member-sharded loop hands
    # back torch events)
    k_list = [e0.elapsed_time(e1) for e0, e1 in timers] if timers else list(mdl.network.route_timings())
    k_ms = float(np.mean(k_list)) if k_list else float("nan")
    ab = algorithmic_bytes_per_update(M)
    bytes_per_launch = float(n) * M * every * ab
    achieved = bytes_per_launch / (k_ms * 1e-3) / 1e9
    peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fpk:
            peak = float(json.load(fpk)["hbm_gbs"]); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        pass
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as ft:
            traffic = json.load(ft).get("route_window_kernel_dram_bytes_per_launch")
    except Exception:
        pass
    kernel = "route_lane_kernel" if M <= 8 else "route_window_kernel"
    if kernel != "route_window_kernel":
        traffic = None
    roofline = {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": bytes_per_launch, "kernel_ms_per_launch": k_ms,
                "launches_timed": len(k_list), "bytes_per_update": ab,
                "note": ("from the second window on the launch also applies the previous EnKF update while it loads its "
                         "tasks (DESIGN.md 4.4); the algorithmic bytes count the routing only"),
                "routing_share_of_step": k_ms * nwin / ms_step if ms_step > 0 else None}
    if traffic:
        # The state stays in shared memory for the 12 steps of a window, so the kernel moves ~10x fewer bytes than
        # the algorithmic figure: what it physically does to HBM, and the floor that traffic sets for a launch
        roofline["physical"] = {"dram_bytes_per_launch": traffic, "achieved": traffic / (k_ms * 1e-3) / 1e9, "unit": "GB/s",
                                "frac": traffic / (k_ms * 1e-3) / 1e9 / peak, "floor_ms_per_launch": traffic / (peak * 1e9) * 1e3}

    # ---- end to end through the public API, host buffers in and out --------------------------------
    e2e = None
    if full and not a.no_e2e:
        e2e_run()                                         # warm-up (allocations)
        e2e_parts.clear()
        barrier()
        t0 = time.perf_counter()
        reps = a.steps
        for _ in range(reps):
            e2e_run()
        barrier()
        s_e2e = max_over_ranks((time.perf_counter() - t0) / reps)
        e2e = {"value": wl.updates_per_run() / s_e2e, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * s_e2e, "runs": reps,
               "breakdown_ms": {k: round(1e3 * v / reps, 3) for k, v in e2e_parts.items()}}

    # ---- CPU baseline (rank 0, single GPU only) -------------------------------------------------------
    cpu, parity = None, None
    if full and rank == 0 and world == 1 and not a.no_cpu_baseline:
        ref, port = cpu_samples(wl, a.cpu_windows)
        port.run()                                        # warm-up (page faults, OpenMP pool)
        runs = [port.run() for _ in range(2)]
        best = min(r[0] for r in runs)
        o_cpu = runs[-1][1]                               # [M][n] after the sample's windows
        cpu = {"value": port.updates / best, "unit": UNIT, "cores": port.threads, "kind": "port",
               "sample": port.describe()}
        if ref is not None:
            ref.run()
            rruns = [ref.run() for _ in range(2)]
            cpu = {"value": ref.updates / min(r[0] for r in rruns), "unit": UNIT, "cores": ref.cores, "kind": "reference",
                   "sample": ref.describe(), "port_value": port.updates / best, "port_cores": port.threads}
            o_cpu = rruns[-1][1]
            ref.close()
        # the same on ONE core, one window (SURVEY.md section 8d asks for both)
        c1 = CpuSample(wl, 1)
        c1.threads = 1
        cpu["port_value_1core"] = c1.updates / c1.run()[0]
        # ---- parity of THIS run: the GPU ensemble after the sample's windows against the CPU sample --------
        Oc, Ic = mdl.device_state
        Oc.copy_(O0); Ic.copy_(I0)
        mdl._datetime = t_start
        mdl.run_assimilating(forcing, a.cpu_windows * every, enkf, every, Zp_dev)
        mdl.network.check()
        o_gpu = mdl.download_state()[0]
        ref_o = o_cpu.T
        scale = float(np.abs(ref_o).max())
        parity = {"max_rel_err": float((np.abs(o_gpu - ref_o) / np.maximum(np.abs(ref_o), 1e-12 * scale)).max()),
                  "metric": "element-wise |gpu - cpu| / max(|cpu|, 1e-12 max|cpu|) over the ensemble outflows",
                  "after": f"{a.cpu_windows} windows ({a.cpu_windows * every} routing steps + {a.cpu_windows} EnKF updates)",
                  "against": cpu["kind"], "tolerance": 1e-9}
        parity["ok"] = parity["max_rel_err"] <= 1e-9

    sharded = world > 1 and not wl.by_basin
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong" if sharded else "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": workload_config(wl, a, world),
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches,
        "parity_max_rel_err": None if parity is None else parity["max_rel_err"], "parity": parity,
        "clocks": clk, "wall_s_timed_region": wall,
        "roofline_whole_step": {"achieved": value * ab / 1e9, "unit": "GB/s", "frac": value * ab / 1e9 / peak / world},
        "update_path": getattr(enkf, "update_path", None),
    }
    forcing.close()
    path = getattr(enkf, "update_path", None)
    line["update_path"] = path
    if hasattr(enkf, "release_peers"):
        enkf.release_peers()                              # collective: peers may still read this rank's state buffers
    del mdl, enkf, O0, I0, flush, Zp_dev
    torch.cuda.empty_cache()
    return line


def main():
    a = parse_args()
    if a.impl == "reference":
        return reference_arm(a)
    return gpu_arm(a)


if __name__ == "__main__":
    sys.exit(main())

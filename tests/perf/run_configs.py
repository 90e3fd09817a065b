"""BASELINE.json configs[0..4] on one GPU: device time of the routing path and parity against the CPU oracle
(FP64 max relative error; the oracle runs the reference's algorithm, nutils.py:64-89, per member).
Development / documentation aid; bench.py is the contract benchmark."""
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))


def run(name, net_d, M, nsteps, seed, parity_steps, parity_members, chunk=None):
    import torch
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.network import RiverNetwork, Forcing
    from oracle import oracle as O
    n = net_d["endnodes"].size
    chunk = chunk or nsteps                  # one call for the whole run: the library sizes its launches
    prm = S.make_params(n, seed)
    t0 = 1_700_000_000 * 10**9
    times, table = S.make_forcing(n, nsteps, 300.0, seed, t0_ns=t0)
    mul = S.make_member_multipliers(times.size, M, seed) if M > 1 else None
    tb = time.time()
    net = RiverNetwork(net_d["endnodes"])
    tb = time.time() - tb
    al, be, ch, ga = net.compute_coeffs(prm["K"], prm["X"], 300.0)
    _, nlev = net.levels()
    rng = np.random.default_rng(seed)
    o0 = prm["o_t"][:, None] * (rng.uniform(0.5, 1.5, size=(n, M)) if M > 1 else np.ones((n, 1)))
    f = Forcing(net, times, table, mul)
    Od = net.alloc_state(M); Id = net.alloc_state(M)

    def reset():
        net.pack_host(o0, M, Od); net.init_inflows(Od, Id, M)

    def go(steps):
        t = t0
        for s0 in range(0, steps, chunk):
            ns = min(chunk, steps - s0)
            net.route_run(Od, Id, M, f, t, int(300e9), ns)
            t += ns * int(300e9)
    reset(); go(nsteps); net.check()          # warm-up of the same shape: rings and step tables are sized on first use
    reset()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(); go(nsteps); e1.record(); torch.cuda.synchronize(); net.check()
    ms = e0.elapsed_time(e1)
    # parity on the first `parity_steps` steps and `parity_members` members
    reset(); go(parity_steps); net.check()
    og = net.unpack_host(Od, M)[:, :parity_members]; ig = net.unpack_host(Id, M)[:, :parity_members]
    ind = O.compute_indegree(net_d["startnodes"], net_d["endnodes"])
    ref = {"startnodes": net_d["startnodes"], "endnodes": net_d["endnodes"], "indegree": ind,
           "alpha": al, "beta": be, "chi": ch, "gamma": ga}
    o_ref = np.ascontiguousarray(o0[:, :parity_members].T)
    i_ref = np.stack([O.init_states(net_d["startnodes"], net_d["endnodes"], x) for x in o_ref])
    tc = time.time()
    O.run_members(ref, o_ref, i_ref, parity_steps, times.astype(np.float64), table, float(t0), 300e9,
                  wmul=None if mul is None else np.ascontiguousarray(mul[:, :parity_members]))
    tc = time.time() - tc
    eo = float(np.abs(og - o_ref.T).max() / np.abs(o_ref).max()); ei = float(np.abs(ig - i_ref.T).max() / np.abs(i_ref).max())
    upd = float(n) * M * nsteps
    extra = {k: os.environ[k] for k in ("TXH_ROUTE_KERNEL",) if k in os.environ}
    out = {"config": name, "env": extra, "reaches": n, "levels": nlev, "members": M, "steps": nsteps, "topology_pass_s": round(tb, 3),
           "gpu_ms": round(ms, 3), "updates_per_s": upd / (ms * 1e-3),
           "algorithmic_GBps": upd * (32 + 44.0 / M) / (ms * 1e-3) / 1e9,
           "parity": {"steps": parity_steps, "members": parity_members, "max_rel_err_o": eo, "max_rel_err_i": ei,
                      "ok": eo <= 1e-9 and ei <= 1e-9},
           "cpu_oracle_updates_per_s": float(n) * parity_members * parity_steps / tc, "cpu_threads": O.max_threads()}
    print(json.dumps(out), flush=True)
    f.close(); net.close()


def main():
    from tx_fast_hydrology_b200 import synthetic as S
    which = sys.argv[1:] or ["c1", "c2", "c4", "c5"]
    if "c1" in which:
        run("C1: 1,000-reach dendritic network, 288 steps, deterministic", S.make_network(1000, 1), 1, 288, 1, 288, 1)
    if "c2" in which:
        run("C2: Texas-scale network, 7-day run, deterministic", S.make_network(100000, 2), 1, 2016, 2, 2016, 1)
    if "c4" in which:
        run("C4: CONUS-scale forest of 64 independent basins (2.7M reaches) on ONE GPU, 24-hour run",
            S.make_network(2_700_000, 3, n_basins=64), 1, 288, 3, 48, 1)
    if "c2w" in which:      # hourly windows (12 steps per call) on the Texas-scale network, small ensembles
        for M in (1, 2, 4, 8, 16):
            run(f"C2-net, {M} members, 168 windows of 12 steps", S.make_network(100000, 2), M, 2016, 2, 24, min(M, 2), chunk=12)
    if "c5" in which:
        run("C5: long-chain stress (10k-reach main stem + tributaries), 1024 members, 288 steps",
            S.make_longchain_network(), 1024, 288, 5, 12, 32)


if __name__ == "__main__":
    main()

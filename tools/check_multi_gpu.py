"""Member-sharded run on N GPUs == the same ensemble on one GPU (launch with torchrun, one rank per GPU).

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29531 \
        tools/check_multi_gpu.py

Every rank routes its M members of a synthetic network for a few hourly windows with an EnKF update after each
(row sums all-reduced and gauge rows all-gathered over NCCL; the transform reads the other shards' state rows in
place over NVLink -- TXH_MEMBER_UPDATE=peers, the default -- or after an NCCL all-gather -- =allgather); rank 0
also runs all N*M members unsharded and compares the gathered shards with it (FP64, element-wise relative error
<= 1e-9 with the forecast-scale floor of tests/parity.py).  Both update paths are run, with the stochastic filter
and, from two GPUs on, with the square-root filter (method='etkf', rtpp 0.3, the same observation in every member):
every rank post-processes the same Mtot x Mtot system."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import pandas as pd
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    singles = [dist.new_group(ranks=[r]) for r in range(world)]
    from tx_fast_hydrology_b200 import synthetic as S
    from tx_fast_hydrology_b200.muskingum import Muskingum
    from tx_fast_hydrology_b200.da import EnsembleKalmanFilter
    n, M, m, every, nwin, seed = 20000, 16, 60, 12, 3, 3
    Mt = M * world
    net_d = S.make_network(n, seed)
    prm = S.make_params(n, seed, well_posed=True)
    rng = np.random.default_rng(seed)
    o_all = prm["o_t"][:, None] * rng.uniform(0.5, 1.5, size=(n, Mt))
    d0 = S.model_dict(net_d, prm, dt_s=300.0)
    t0 = int(pd.Timestamp(d0["datetime"]).value)
    times, table = S.make_forcing(n, every * nwin, 300.0, seed, t0_ns=t0)
    mul_all = S.make_member_multipliers(times.size, Mt, seed)
    gidx = S.make_gauges(net_d["endnodes"], m, seed=seed)
    mt = t0 + (np.arange(nwin, dtype=np.int64) + 1) * int(every * 300e9)
    meas = rng.uniform(0.5, 8.0, size=(nwin, m))
    idx = pd.DatetimeIndex(pd.to_datetime(mt, unit="ns", utc=True)).as_unit("ns")
    mdf = pd.DataFrame(meas, index=idx, columns=[d0["reach_ids"][j] for j in gidx])
    R = 1e-2 * np.eye(m)
    q = rng.uniform(0.5, 2.0, size=n)
    Zp = {"stochastic": np.ascontiguousarray(meas[:, :, None] + 0.1 * rng.standard_normal((nwin, m, Mt))),
          "etkf": np.ascontiguousarray(np.repeat(meas[:, :, None], Mt, axis=2))}

    from parity import relerr

    def run(cols, group, method):
        d = dict(d0); d["o_t"] = np.ascontiguousarray(o_all[:, cols])
        mdl = Muskingum(d, members=len(cols))
        enkf = EnsembleKalmanFilter(mdl, mdf, q, R, group=group, method=method, rtpp=0.3 if method == "etkf" else 0.0)
        path = enkf.update_path
        f = mdl.make_forcing(times_ns=times, table=table, member_mul=np.ascontiguousarray(mul_all[:, cols]))
        mdl.run_assimilating(f, every * nwin, enkf, every, torch.as_tensor(Zp[method][:, :, :enkf.Mtot], device="cuda"))
        mdl.network.check()
        enkf.release_peers()                                         # collective on the peer-read path
        return mdl.o_t_next.reshape(n, -1), mdl.i_t_next.reshape(n, -1), path

    ok = True
    cols = list(range(rank * M, (rank + 1) * M))
    methods = ["stochastic"] + (["etkf"] if world >= 2 else [])
    if world < 2 and rank == 0:
        print("multi-GPU check: the ETKF case needs two GPUs: skipped", flush=True)
    for method, want in [(a, b) for a in methods for b in ("peers", "allgather")]:
        o_ref = i_ref = None
        if rank == 0:
            o_ref, i_ref, _ = run(list(range(Mt)), singles[0], method)   # the whole ensemble on one GPU
        os.environ["TXH_MEMBER_UPDATE"] = want
        o_loc, i_loc, path = run(cols, None, method)                 # sharded: default group = all ranks
        parts = [torch.empty((n, 2 * M), dtype=torch.float64, device="cuda") for _ in range(world)] if rank == 0 else None
        mine = torch.as_tensor(np.concatenate([o_loc, i_loc], axis=1), device="cuda")
        dist.gather(mine, parts, dst=0)
        if rank == 0:
            o_sh = np.concatenate([p.cpu().numpy()[:, :M] for p in parts], axis=1)
            i_sh = np.concatenate([p.cpu().numpy()[:, M:] for p in parts], axis=1)
            # posterior elements are sums o + gain that may cancel: relative to max(|element|, ensemble scale of the row)
            so = np.abs(o_ref).max(axis=1, keepdims=True) * np.ones_like(o_ref)
            si = np.abs(i_ref).max(axis=1, keepdims=True) * np.ones_like(i_ref)
            eo, ei = relerr(o_sh, o_ref, scale=so), relerr(i_sh, i_ref, scale=si)
            good = eo <= 1e-9 and ei <= 1e-9 and path == want
            ok = ok and good
            print(f"multi-GPU check: {method} world={world} members={Mt} n={n} update_path={path} (asked {want})  "
                  f"max rel err o={eo:.2e} i={ei:.2e}  {'OK' if good else 'FAIL'}", flush=True)
        dist.barrier()
    flag = torch.tensor([1.0 if ok else 0.0], device="cuda")
    dist.broadcast(flag, src=0)
    dist.destroy_process_group()
    return 0 if float(flag.item()) == 1.0 else 1


if __name__ == "__main__":
    sys.exit(main())

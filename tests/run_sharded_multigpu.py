"""Launched with torchrun (one rank per GPU): one cluster split by houses across the ranks, stepped
with (a) the NCCL all-gather exchange and (b) the peer-memory exchange, against an unsharded run of
the same cluster on rank 0.  Exits non-zero on any mismatch."""
import copy
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from marl_demandresponse_b200 import BatchedEnv  # noqa: E402
from marl_demandresponse_b200.batched import synthetic_state  # noqa: E402
from marl_demandresponse_b200.sharded import ShardedClusterEnv  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n, R, T = 20000, 2, 40
    prop = {"start_datetime": "2021-06-15T11:58:20", "start_datetime_mode": "fixed", "time_step": 4.0,
            "cluster_prop": {"nb_agents": n, "house_prop": {"target_temp": 19.0}},
            "power_grid_prop": {"signal_properties": {"mode": "sinusoidals"}}}
    st = synthetic_state(prop, R, seed=3)
    acts = (np.random.default_rng(2).random((T, R, n)) < 0.5).astype(np.uint8)
    for layout in ("tarmac", "hand_engineered"):   # the second exchanges a halo of ring-neighbour messages as well
        results = {}
        for exchange in ("nccl", "peer"):
            env = ShardedClusterEnv(prop, R, rank=rank, world=world, device=local, noise="philox", seed=9, exchange=exchange,
                                    obs_layout=layout)
            env.reset(copy.deepcopy(st))
            for t in range(T):
                a = torch.as_tensor(acts[t][:, env.lo:env.hi], device="cuda")
                env.state["actions"].copy_(a)
                env.step(None)
            torch.cuda.synchronize()
            if exchange == "peer":
                env.sim.peer_status()
            results[exchange] = {k: env.state[k].clone()
                                 for k in ("dt_air", "sso", "flags", "reward", "power", "signal", "obs", "metrics")}
            # timing of the exchange variants (device events, max over ranks)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            dist.barrier(); torch.cuda.synchronize()
            e0.record()
            for t in range(200):
                env.step(None)
            e1.record(); torch.cuda.synchronize()
            ms = torch.tensor([e0.elapsed_time(e1) / 200], device="cuda")
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            if rank == 0:
                print(f"layout={layout} exchange={exchange}: {ms.item() * 1e3:.1f} us/step for {n} houses x {R} replicas "
                      f"on {world} GPUs", flush=True)
            lo, hi = env.lo, env.hi
            del env
        for k in results["nccl"]:
            assert torch.equal(results["nccl"][k], results["peer"][k]), f"{layout}: peer vs nccl exchange differ in {k}"
        # unsharded reference on every rank (cheap), compared with this rank's shard
        whole = BatchedEnv(prop, R, device=local, obs_layout=layout, noise="philox", seed=9, path="split")
        whole.set_state(copy.deepcopy(st))
        for t in range(T):
            whole.step(torch.as_tensor(acts[t], device="cuda"))
        torch.cuda.synchronize()
        ws = whole.state
        assert torch.equal(ws["sso"][:, lo:hi], results["peer"]["sso"]) and torch.equal(ws["flags"][:, lo:hi], results["peer"]["flags"])
        assert torch.equal(ws["dt_air"][:, lo:hi], results["peer"]["dt_air"])
        torch.testing.assert_close(ws["power"], results["peer"]["power"], rtol=1e-12, atol=0)
        torch.testing.assert_close(ws["signal"], results["peer"]["signal"], rtol=1e-12, atol=0)
        torch.testing.assert_close(ws["reward"][:, lo:hi], results["peer"]["reward"], rtol=1e-6, atol=1e-7)
        # observation rows, including the neighbour messages that cross the shard edges
        torch.testing.assert_close(ws["obs"][:, lo:hi], results["peer"]["obs"], rtol=1e-6, atol=1e-7)
        # running metrics: whole-cluster sums on every rank (partials folded in another order)
        wm, pm = ws["metrics"], results["peer"]["metrics"]
        assert torch.equal(wm[:, 0], pm[:, 0]) and bool((wm[:, 0] == T).all()), f"{layout}: metric step counts"
        mtol = 1e-5 * wm.abs()
        mtol[:, 1] += 1e-5 * T
        assert bool(((pm - wm).abs() <= mtol).all()), f"{layout}: running metrics differ from the unsharded cluster"
    dist.barrier()
    if rank == 0:
        print("sharded multi-GPU check OK", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()

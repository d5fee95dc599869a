"""One very large cluster split by houses across the GPUs of a box (BASELINE config 5).

Each rank owns houses ``[rank * N / W, (rank + 1) * N / W)`` of every replica.  Per step:
``drsim_step_begin`` (local house update + partial sums) -> one tiny all-gather of the per-rank
partials over NCCL / NVLink (48 bytes per rank and replica) -> ``drsim_step_finish`` (identical
combination on every rank, env epilogue, rewards, observations).  This is the only data-path
collective in the package; replica-sharded runs (``BatchedEnv``) have none.

With the hand-engineered observation layout the rows carry the messages of ring neighbours
(cluster.py:91-111), so the shards also exchange a *halo*: the message records of each shard's first
``ceil(c/2)`` and last ``floor(c/2)`` houses (64 bytes per house).  ``exchange="peer"`` pushes them
into the adjacent ranks' inboxes with the same NVLink stores as the partial sums; ``exchange="nccl"``
all-gathers the ``halo_out`` blocks next to the partials.
"""
from __future__ import annotations

from typing import Any, Dict, Optional

import numpy as np

from .batched import reset_counter, synthetic_state
from .core import DrSim, flatten_config
from .properties import as_props


def house_shard(n_houses: int, rank: int, world: int):
    """Contiguous, 4-aligned house ranges (the planes are accessed with 128-bit vectors)."""
    per = (n_houses + world - 1) // world
    per = (per + 3) // 4 * 4
    lo = min(n_houses, rank * per)
    hi = min(n_houses, lo + per)
    return lo, hi


def halo_edge_houses(n_global: int, rank: int, world: int, nb_comm: int):
    """Global ids of the houses whose message records ``drsim_ptrs.halo_out`` of ``rank`` carries after a
    step: its FIRST ``H = ceil(c/2)`` houses (entries ``[0, H)``) and its LAST ``L = floor(c/2)`` houses
    (entries ``[H, H + L)``) -- the ring neighbours of agent_communication_builder.py:74-84 that the two
    adjacent shards cannot find at home."""
    lo, hi = house_shard(n_global, rank, world)
    L = nb_comm // 2
    H = nb_comm - L
    return list(range(lo, lo + H)) + list(range(hi - L, hi))


def halo_lookup(gathered, n_global: int, rank: int, world: int, nb_comm: int, house: int, k: int):
    """Host restatement of how ``k_obs`` resolves ring neighbour ``k`` of global ``house`` on ``rank``
    from the all-gathered halo blocks ``gathered[world][nb_comm]`` (``drsim_step_finish_gathered``):
    returns ``("local", global_id)`` or ``("halo", entry)`` with the entry taken from the previous
    rank's LAST-houses part or the next rank's FIRST-houses part."""
    lo, hi = house_shard(n_global, rank, world)
    L = nb_comm // 2
    H = nb_comm - L
    nb = (house - L + k) % n_global if k < L else (house + 1 + (k - L)) % n_global
    if lo <= nb < hi:
        return "local", nb
    d = (nb - lo) % n_global
    if d >= n_global - L:                                  # one of the L houses before the shard
        return "halo", gathered[(rank - 1) % world][H + (d - (n_global - L))]
    return "halo", gathered[(rank + 1) % world][d - (hi - lo)]


class ShardedClusterEnv:
    def __init__(self, env_props: Any, n_replicas: int = 1, rank: int = 0, world: int = 1, device: int = 0,
                 precision: str = "f32", obs_layout: str = "tarmac", policy: str = "external", noise: str = "philox",
                 seed: int = 0, group=None, exchange: str = "nccl", obs_dtype: str = "float32"):
        self.props = as_props(env_props)
        self.rank, self.world, self.group = int(rank), int(world), group
        self.n_global = int(self.props.cluster_prop.nb_agents)
        self.lo, self.hi = house_shard(self.n_global, rank, world)
        if self.hi <= self.lo:
            raise ValueError("more ranks than 4-house blocks")
        mode = self.props.cluster_prop.agents_comm_prop.mode
        if mode == "random_sample" and obs_layout == "hand_engineered":
            raise ValueError("`random_sample` neighbour messages are drawn from the whole cluster every step: they are "
                             "available on replicas (BatchedEnv), not on a cluster split across GPUs")
        cfg = flatten_config(self.props, n_replicas, precision, obs_layout, policy, noise, seed, "split",
                             comm_table=mode != "neighbours", house_offset=self.lo, n_house_local=self.hi - self.lo,
                             obs_dtype=obs_dtype)
        self.sim = DrSim(cfg, device)
        self.device = device
        self._v = self.sim.views()
        self._gathered = None
        self._halo_gathered = None
        self.exchange = exchange if world > 1 else "none"
        if self.exchange == "peer":
            # one-off: swap CUDA IPC handles of the slabs so the kernels can store into peer inboxes
            import torch.distributed as dist

            handles = [None] * world
            dist.all_gather_object(handles, self.sim.ipc_export(), group=group)
            self.sim.ipc_attach(rank, world, handles)
            dist.barrier(group=group)

    def reset(self, state: Optional[Dict[str, np.ndarray]] = None, seed: int = 1234):
        """``state``: full-cluster state dict (every rank passes the same one) or None = synthetic.  A new episode
        begins: the running metrics (``state["metrics"]``) start again from zero, and the interpolator's counter at
        ``interp_update_period + 1`` unless ``state`` carries ``t_since_interp`` (its first step fires it, as the
        reference's reset would: a house-sharded handle has no refresh)."""
        if state is None:
            state = synthetic_state(self.props, self.sim.R, seed)
        local = {}
        for k, v in state.items():
            v = np.asarray(v)
            local[k] = v[:, self.lo:self.hi] if v.ndim == 2 else v
        self.sim.set_state(reset_counter(self.props, local, self.sim.R))
        self._v["metrics"].zero_()   # on the current stream, like drsim_reset
        return self

    def step(self, actions=None):
        import torch

        sim = self.sim
        a = None
        if actions is not None:
            if sim.N == sim.Ns and actions.is_contiguous():
                a = actions
            else:
                self._v["actions"].copy_(actions)
        if self.exchange == "peer" or self.world == 1:
            # the exchange (if any) happens inside the kernels (NVLink peer stores): one call for both halves
            sim.step_sharded(a)
            return self._v["obs"], self._v["reward"]
        sim.step_begin(a)
        acc = self._v["acc"]
        if self.world > 1:
            import torch.distributed as dist

            if self._gathered is None:
                # concatenation along dim 0 == [world][R][N_ACC] in rank order
                self._gathered = torch.empty((self.world * acc.shape[0], acc.shape[1]), dtype=acc.dtype, device=acc.device)
            dist.all_gather_into_tensor(self._gathered, acc, group=self.group)
            halo = self._v.get("halo_out")
            if halo is None:
                sim.step_finish(self._gathered, self.world)
            else:
                if self._halo_gathered is None:
                    self._halo_gathered = torch.empty((self.world,) + tuple(halo.shape), dtype=halo.dtype, device=halo.device)
                dist.all_gather_into_tensor(self._halo_gathered, halo, group=self.group)
                sim.step_finish_gathered(self._gathered, self._halo_gathered, self.world, self.rank)
        return self._v["obs"], self._v["reward"]

    def run(self, n_steps: int, action_tape=None, rotate: bool = False):
        """``n_steps`` sharded steps enqueued by ONE C call (``drsim_run_tape``): peer exchange or a single rank
        only (the NCCL exchange needs the host between the two halves of every step).  ``action_tape``: u8 CUDA
        ``[T, R, n_local]`` (``rotate``: step k replays plane ``k % T``) / ``[R, n_local]`` / None; every rank must
        run the same number of steps."""
        if not (self.exchange == "peer" or self.world == 1):
            raise ValueError("ShardedClusterEnv.run needs the peer exchange (or one rank)")
        sim = self.sim
        if action_tape is not None and sim.N != sim.Ns:
            raise ValueError("run(): shard sizes are multiples of 4 except on the last rank; pad the tape to the plane stride")
        sim.run(n_steps, action_tape, rotate=rotate)
        return self._v["obs"], self._v["reward"]

    @property
    def state(self):
        return self._v

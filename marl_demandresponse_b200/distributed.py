"""Multi-GPU plumbing: replica sharding (no per-step collective) and the end-of-rollout metric
reduction (one all-reduce of a handful of fp64 sums; NCCL over NVLink on the GPU box, gloo in the
CPU tests)."""
from __future__ import annotations

from typing import Dict

from . import _lib

# the running sums of BatchedEnv.metrics; each step adds 1, mean_i reward_i, |sum_i (Ta_i - target_i)| / N,
# sum_i (Ta_i - target_i)^2 / N, |P - S_old| and (P - S_old)^2 (Ta and cluster power P after the step, S_old the
# regulation signal before it)
METRIC_NAMES = ("steps", "sum_mean_reward", "sum_abs_mean_temp_offset", "sum_mean_sq_temp_error",
                "sum_abs_signal_error", "sum_sq_signal_error")


def replica_shard(n_replicas_total: int, rank: int, world: int):
    """Contiguous replica range of ``rank``: ``(rep_offset, n_local)``; sizes differ by at most 1."""
    base, extra = divmod(n_replicas_total, world)
    n_local = base + (1 if rank < extra else 0)
    offset = rank * base + min(rank, extra)
    return offset, n_local


def reduce_rollout_metrics(metrics, group=None) -> Dict[str, float]:
    """``metrics``: this rank's ``[R_local, N_METRICS]`` running sums (``BatchedEnv.metrics``).
    Returns the job-wide per-replica-step averages (identical on every rank).

    Made for replica-sharded runs, where each rank holds different replicas.  On a house-sharded cluster
    (``ShardedClusterEnv``) every rank holds the same whole-cluster rows: the averages still come out right, but
    ``replicas`` and ``replica_steps`` are ``world`` times too large."""
    import torch
    import torch.distributed as dist

    tot = metrics.double().sum(dim=0)
    tot = torch.cat([tot, torch.tensor([float(metrics.shape[0])], dtype=torch.float64, device=tot.device)])
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.SUM, group=group)
    tot = tot.cpu().tolist()
    steps = max(tot[0], 1.0)
    out = {"replicas": tot[_lib.N_METRICS], "replica_steps": tot[0]}
    out["mean_reward"] = tot[1] / steps
    out["mean_abs_temp_offset"] = tot[2] / steps
    out["rms_temp_error"] = (tot[3] / steps) ** 0.5
    out["mean_abs_signal_error"] = tot[4] / steps
    out["rms_signal_error"] = (tot[5] / steps) ** 0.5
    return out

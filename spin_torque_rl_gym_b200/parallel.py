"""Multi-GPU plumbing: the env batch shards by contiguous global env-id ranges (one process per GPU, no data-path
collective); one all-reduce(SUM) of the STG_NSTATS-element episode-statistics vector per rollout (SURVEY.md §8e — the
reference analogue is the per-env EnvironmentMonitor, utils/monitoring.py:89-116), and, under a synchronised VecNormalize, one
all-gather of the 27-double moment vector per env step (all_gather_moments), and, for data-parallel PPO, two all-gathers per
minibatch (K12: the advantage moments and the gradient sums)."""
from __future__ import annotations

from typing import Dict, Tuple

from . import _lib


def shard_range(total_envs: int, rank: int, world_size: int) -> Tuple[int, int]:
    """[start, stop) of the global env ids owned by `rank`. Philox counters use the GLOBAL id (env_offset=start), so results
    do not depend on the number of GPUs."""
    if not (0 <= rank < world_size):
        raise ValueError("rank out of range")
    base, rem = divmod(int(total_envs), int(world_size))
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def reduce_step_stats(stats, reward=None, step_energy=None, terminated=None, truncated=None, n_sub=None, status=None,
                      step_count=None):
    """Add the statistics of stored env-step results (any shape, e.g. a rollout buffer [T, N]) to the CUDA vector `stats`
    [STG_NSTATS] f64 with the standalone K5 kernel (stg_stats_reduce_f64) and return `stats`. The step kernels already
    accumulate the same vector when the env was built with collect_stats=True; this serves arrays produced without it."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    if not (isinstance(stats, torch.Tensor) and stats.is_cuda and stats.dtype == torch.float64 and stats.numel() == _lib.NSTATS
            and stats.is_contiguous()):
        raise ValueError(f"stats must be a contiguous CUDA float64 tensor of {_lib.NSTATS} elements")
    dev, n, keep = stats.device, None, []

    def prep(x, dtype):
        nonlocal n
        if x is None:
            return None
        t = x.to(device=dev, dtype=dtype).reshape(-1).contiguous()
        if n is not None and t.numel() != n:
            raise ValueError("all step-result arrays must have the same number of elements")
        n = t.numel()
        keep.append(t)
        return t.data_ptr()

    ptrs = [prep(reward, torch.float64), prep(step_energy, torch.float64), prep(terminated, torch.uint8),
            prep(truncated, torch.uint8), prep(n_sub, torch.int32), prep(status, torch.int32), prep(step_count, torch.int32)]
    if n is None:
        raise ValueError("at least one step-result array is required")
    with torch.cuda.device(dev):
        _lib.check(lib.stg_stats_reduce_f64(*ptrs, n, stats.data_ptr(), torch.cuda.current_stream(dev).cuda_stream),
                   "stg_stats_reduce_f64")
    return stats


def all_reduce_stats(stats, group=None) -> Dict[str, float]:
    """SUM-reduce the per-rank statistics vector (NCCL for CUDA tensors, gloo for CPU tensors) and return it as a dict with
    the derived episode metrics. Without an initialised process group the local vector is returned."""
    import torch
    import torch.distributed as dist
    t = stats.clone()
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return episode_metrics(dict(zip(_lib.STAT_NAMES, t.detach().to("cpu", torch.float64).tolist())))


def episode_metrics(totals: Dict[str, float]) -> Dict[str, float]:
    """The statistics `totals` (one value per STAT_NAMES entry, e.g. the difference of two readings) with the derived episode
    metrics added: episodes, success_rate, mean_episode_length, mean_step_energy and mean_reward (per step)."""
    out = dict(totals)
    episodes = out["terminated"] + out["truncated"]
    out["episodes"] = episodes
    out["success_rate"] = out["terminated"] / episodes if episodes else 0.0
    out["mean_episode_length"] = out["episode_length"] / episodes if episodes else 0.0
    out["mean_step_energy"] = out["energy"] / out["steps"] if out["steps"] else 0.0
    out["mean_reward"] = out["reward"] / out["steps"] if out["steps"] else 0.0
    return out


def world_size(group=None) -> int:
    """The world size of the initialised process group, or 1 without one."""
    import torch.distributed as dist
    return dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1


def all_gather_moments(local, group=None):
    """[G, 27] stack of every rank's moment vector `local` [27] (float64, VecNormalize / K8), in rank order; any other 1-D
    vector of the same size on every rank works too (the K12 advantage moments and PPO sums). The list form of
    all_gather, so it serves gloo (CPU tensors) and NCCL (CUDA tensors) alike; with NCCL it is enqueued on the current stream
    and nothing waits on the host. Without an initialised process group, or with world size 1, it returns `local[None]` and
    issues no collective."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return local[None]
    outs = [torch.empty_like(local) for _ in range(dist.get_world_size(group))]
    dist.all_gather(outs, local.contiguous(), group=group)
    return torch.stack(outs)

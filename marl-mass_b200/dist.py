"""Multi-GPU plumbing: env instances shard across ranks with no step-path traffic (SURVEY.md §8e).

One process per GPU (torch.distributed, NCCL on GPUs / gloo in the CPU tests).  The only collectives are the
all-reduce of the episode-statistics vector (SUM for the counters, MIN for min_headway) and, with update statistics
on, of the learner's PPO statistics vectors (SUM, MIN for the smallest ratio, MAX for the largest).
"""
import os

SUM_KEYS = ("agent_steps", "env_steps", "episodes", "crashed_episodes", "reward_sum", "speed_sum",
            "merge_percent_sum", "shield_solves", "shield_active", "lane_change_vetoes")
MIN_KEYS = ("min_headway",)


def rank_world():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def shard_range(total_envs, rank, world):
    """Contiguous block [begin, end) of a global env index space for `rank` (sizes differ by at most 1)."""
    base, rem = divmod(int(total_envs), int(world))
    begin = rank * base + min(rank, rem)
    return begin, begin + base + (1 if rank < rem else 0)


def rank_seed(seed, rank):
    """Distinct spawn stream per rank: the device RNG is keyed by (seed, local env index, episode)."""
    return (int(seed) * 0x9E3779B97F4A7C15 + int(rank) * 0xD1B54A32D192ED03) & (2 ** 64 - 1)


def bind_to_gpu(device_index):
    """Pin the calling process to the CPU cores nearest to its GPU (NVML's ideal affinity), so that the pinned host
    buffers of the host path are first-touched on that GPU's NUMA node and eight ranks do not push their
    device-to-host traffic across the socket interconnect.  Returns the number of cores, or 0 if NVML is unavailable."""
    try:
        import pynvml
        pynvml.nvmlInit()
        idx = device_index
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if device_index < len(ids) and ids[device_index].isdigit():
                idx = int(ids[device_index])
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        n_words = (os.cpu_count() + 63) // 64
        words = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cores = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        allowed = cores & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
        return len(allowed)
    except Exception:
        return 0


def all_reduce_stats(stats, device=None):
    """Fold per-rank stats dicts (MergeEnvBatched.stats()) into job totals; no-op without a process group."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return dict(stats)
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
    s = torch.tensor([stats[k] for k in SUM_KEYS], dtype=torch.float64, device=device)
    m = torch.tensor([stats[k] for k in MIN_KEYS], dtype=torch.float64, device=device)
    dist.all_reduce(s, op=dist.ReduceOp.SUM)
    dist.all_reduce(m, op=dist.ReduceOp.MIN)
    out = {k: float(v) for k, v in zip(SUM_KEYS, s.tolist())}
    out.update({k: float(v) for k, v in zip(MIN_KEYS, m.tolist())})
    return out


def all_reduce_ppo_stats(v):
    """Fold per-rank PPO statistics vectors (`rollout.ppo_stats`: f64 [..., PPO_STATS_LEN] on the device) into job totals:
    SUM for the sums and counts, MIN for ratio_min, MAX for ratio_max (as a MIN of its negation).  Returns a new tensor;
    no-op (the same tensor) without a process group."""
    import torch
    import torch.distributed as dist
    from ._lib import PPO_STAT
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return v
    lo, hi = PPO_STAT["ratio_min"], PPO_STAT["ratio_max"]
    s = v.clone()
    s[..., lo] = 0.0
    s[..., hi] = 0.0
    m = torch.stack([v[..., lo], -v[..., hi]], -1).contiguous()
    dist.all_reduce(s, op=dist.ReduceOp.SUM)
    dist.all_reduce(m, op=dist.ReduceOp.MIN)
    s[..., lo] = m[..., 0]
    s[..., hi] = -m[..., 1]
    return s


def summarize(stats):
    """Derived episode metrics the reference logs to wandb (run_mappo.py:317-332)."""
    ep = max(stats["episodes"], 1.0)
    es = max(stats["env_steps"], 1.0)
    return {
        "agent_steps": stats["agent_steps"], "episodes": stats["episodes"],
        "crash_rate": stats["crashed_episodes"] / ep, "mean_step_reward": stats["reward_sum"] / es,
        "average_speed": stats["speed_sum"] / es, "merge_percent": stats["merge_percent_sum"] / ep,
        "min_headway": stats["min_headway"],
        "shield_active_frac": stats["shield_active"] / max(stats["shield_solves"], 1.0),
        "lane_change_veto_frac": stats["lane_change_vetoes"] / max(stats["shield_solves"], 1.0),
    }

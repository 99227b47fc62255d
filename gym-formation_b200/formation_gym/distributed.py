"""Multi-GPU plumbing: one process per GPU, envs sharded by contiguous global index ranges.

Envs never interact (all state is per env; the reference itself runs one env per process --
train/maddpg-v2/utils/env_wrappers.py:48-55), so there is NO collective on the step path.  The only
exchange is a ``torch.distributed`` all-reduce (NCCL over NVLink/NVSwitch on GPUs, gloo in the CPU
tests) of the 4-double episode-statistics vector at logging cadence.  Philox streams are keyed by
the GLOBAL env id (``env_offset``), so a job gives identical per-env results at 1, 2, 4 or 8 ranks.
"""
import os

import torch
import torch.distributed as dist


def bind_to_gpu(device_index):
    """Pin this process to the host cores (hence the NUMA node) closest to GPU ``device_index`` -- NVML's ideal CPU
    affinity for the device -- BEFORE any pinned host memory is allocated.  One process per GPU otherwise runs wherever
    the OS puts it: its pinned staging buffers are first-touched on an arbitrary node and every D2H / H2D copy of the
    VecEnv adapter may cross the socket interconnect (round 1: the e2e rate of 8 ranks collapsed to 11.7 GB/s per GPU).
    Returns the CPU set that was applied, or None when NVML / the affinity call is unavailable (containers with a
    restricted cpuset keep their set)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        # CUDA_VISIBLE_DEVICES remaps indices: resolve through the PCI bus id of the torch device
        bus = torch.cuda.get_device_properties(device_index).pci_bus_id if hasattr(
            torch.cuda.get_device_properties(device_index), "pci_bus_id") else None
        h = None
        if bus is not None:
            for i in range(pynvml.nvmlDeviceGetCount()):
                hi = pynvml.nvmlDeviceGetHandleByIndex(i)
                if int(pynvml.nvmlDeviceGetPciInfo(hi).bus) == int(bus):
                    h = hi
                    break
        if h is None:
            h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return sorted(cpus)
    except Exception:
        return None


def shard_range(num_envs_total, rank, world_size):
    """Contiguous range [lo, hi) of global env ids owned by ``rank``; sizes differ by at most 1."""
    if not (0 <= rank < world_size):
        raise ValueError("rank %d out of range for world size %d" % (rank, world_size))
    base, rem = divmod(int(num_envs_total), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def all_reduce_stats(stats):
    """Sum the per-rank statistics vector [n_episodes, sum R, sum R^2, sum collisions] over ranks
    (no-op when torch.distributed is not initialised).  Returns the tensor."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
    return stats


def summarize(stats):
    """mean / std of the episode return and collisions per episode from a (reduced) stats vector."""
    n, s, s2, c = [float(x) for x in stats.tolist()]
    if n <= 0:
        return {"episodes": 0.0, "return_mean": float("nan"), "return_std": float("nan"),
                "collisions_per_episode": float("nan")}
    mean = s / n
    var = max(s2 / n - mean * mean, 0.0)
    return {"episodes": n, "return_mean": mean, "return_std": var ** 0.5, "collisions_per_episode": c / n}


def make_sharded_env(scenario, num_envs_total, num_agents, episode_length=None, **kwargs):
    """This rank's shard of a ``num_envs_total``-env job (rank/world from torch.distributed).  A ``target_index`` of
    the whole job ([num_envs_total]) is sliced to the shard; target banks are shared by all ranks."""
    from .batched import BatchedFormationEnv
    rank = dist.get_rank() if dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_initialized() else 1
    lo, hi = shard_range(num_envs_total, rank, world)
    if kwargs.get("target_index") is not None:
        ti = torch.as_tensor(kwargs["target_index"])
        if tuple(ti.shape) != (int(num_envs_total),):
            raise ValueError("target_index must have shape (%d,) (one task per env of the job)" % int(num_envs_total))
        kwargs["target_index"] = ti[lo:hi]
    return BatchedFormationEnv(scenario, hi - lo, num_agents, episode_length, env_offset=lo, **kwargs)

"""Multi-GPU sharding: envs are independent units, so the env index range is split contiguously over
the ranks with NO per-step communication (SURVEY.md 8e). Every rank keeps GLOBAL env ids
(`env_id_base`), so per-env random streams -- and therefore every result -- do not depend on the
number of GPUs. The only collective is the optional all-reduce (sum) of the 8 episode-statistics
doubles."""
from __future__ import annotations

import os


def shard(num_envs: int, rank: int | None = None, world_size: int | None = None) -> tuple[int, int]:
    """-> (env_id_base, local_num_envs) of this rank for `num_envs` global envs."""
    rank = int(os.environ.get("RANK", "0")) if rank is None else rank
    world_size = int(os.environ.get("WORLD_SIZE", "1")) if world_size is None else world_size
    if not 0 <= rank < world_size:
        raise ValueError("rank out of range")
    base = num_envs * rank // world_size
    end = num_envs * (rank + 1) // world_size
    if end <= base:
        raise ValueError("more ranks than envs")
    return base, end - base


def all_reduce_stats(stats):
    """Sum the 8 episode-statistics doubles over all ranks (NCCL for CUDA tensors, gloo for CPU)."""
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(stats)
    return stats


def _parse_cpulist(text: str) -> set[int]:
    cpus: set[int] = set()
    for part in text.strip().split(","):
        if not part:
            continue
        lo, _, hi = part.partition("-")
        cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def bind_to_gpu_numa_node(device_index: int, sysfs: str = "/sys/bus/pci/devices") -> dict | None:
    """Pin this process to the CPUs next to its GPU (the PCI device's `local_cpulist`), so that the pinned host buffers it
    allocates afterwards -- and the threads that read them -- live on the GPU's own NUMA node: the host-buffer entry
    points (`pgtg_step_host*`) are bounded by device->host copies, and on a two-socket node a buffer on the far socket
    sends every copy across the socket interconnect. Call it before allocating pinned memory. Returns what it did
    ({"numa_node", "cpus"}), or None when the topology is not exposed (single node, container without sysfs)."""
    import torch

    try:
        prop = torch.cuda.get_device_properties(device_index)
        addr = f"{prop.pci_domain_id:04x}:{prop.pci_bus_id:02x}:{prop.pci_device_id:02x}.0"
        with open(os.path.join(sysfs, addr, "local_cpulist")) as fh:
            cpus = _parse_cpulist(fh.read())
        with open(os.path.join(sysfs, addr, "numa_node")) as fh:
            node = int(fh.read().strip())
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if not cpus or cpus == allowed:
            return {"numa_node": node, "cpus": len(allowed), "bound": False}
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus), "bound": True}
    except (OSError, AttributeError, ValueError, RuntimeError, AssertionError):
        return None


def make_sharded(total_envs: int, device=None, bind_numa: bool = True, **kwargs):
    """A `PGTGVectorEnv` over this rank's shard of `total_envs` global envs (one process per GPU,
    launched with torchrun). Level sets (num_levels, start_level, level_sampling) pass through: the pool depends only on
    the map keyword arguments and start_level, so every rank builds the same one."""
    import torch

    from .vector_env import PGTGVectorEnv

    base, n = shard(total_envs)
    if device is None:
        device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    if bind_numa and torch.device(device).type == "cuda":
        bind_to_gpu_numa_node(torch.device(device).index or 0)
    return PGTGVectorEnv(n, device=device, env_id_base=base, **kwargs)

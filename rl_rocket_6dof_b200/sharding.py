"""Index-range sharding of the environments over the GPUs of one box (SURVEY.md §8e).

Environments are independent, so there is no data-path collective: rank g owns the contiguous
global env ids `[offset_g, offset_g + count_g)`; the Philox counters of reset / action streams are
keyed by the *global* env id, so trajectories do not depend on the shard count.  The only exchange
is one `all_reduce(SUM)` over the 8-double episode-statistics vector (`R6_S_*` in include/r6dof.h)
per report — NCCL over NVLink on the GPUs, gloo in the CPU tests.
"""
from __future__ import annotations

import os
from typing import Optional, Tuple

import torch
import torch.distributed as dist


def shard_range(n_global: int, world: int, rank: int) -> Tuple[int, int]:
    """(offset, count) of rank's contiguous slice; the first `n_global % world` ranks get one more."""
    if world <= 0 or not (0 <= rank < world) or n_global < 0:
        raise ValueError("bad shard request")
    base, rem = divmod(n_global, world)
    count = base + (1 if rank < rem else 0)
    offset = rank * base + min(rank, rem)
    return offset, count


def shard_batch_kwargs(n_local: int, rank: int, world: int) -> dict:
    """`Rocket6DOFBatch` keyword arguments of rank's shard when every one of `world` ranks holds n_local envs (what the
    data-parallel `ppo.PPOTrainer` expects): env_offset = rank n_local, num_envs_global = world n_local."""
    if n_local < 1 or world < 1 or not (0 <= rank < world):
        raise ValueError("bad shard request")
    return dict(env_offset=rank * n_local, num_envs_global=world * n_local)


def env_world() -> Tuple[int, int, int]:
    """(rank, local_rank, world_size) from the torchrun environment (1 process = 1 GPU)."""
    return (int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")),
            int(os.environ.get("WORLD_SIZE", "1")))


def init_process_group(device: Optional[torch.device] = None) -> bool:
    """Joins the torchrun rendezvous (nccl for CUDA devices, gloo otherwise). False when world == 1."""
    _, _, world = env_world()
    if world <= 1:
        return False
    if not dist.is_initialized():
        if device is not None and device.type == "cuda":
            dist.init_process_group("nccl", device_id=device)
        else:
            dist.init_process_group("gloo")
    return True


def reduce_stats(stats: torch.Tensor, group=None) -> torch.Tensor:
    """Sum of the per-rank `[8]` float64 statistics vector over all ranks (a copy; input untouched)."""
    out = stats.detach().clone()
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(out, op=dist.ReduceOp.SUM, group=group)
    return out


def max_over_ranks(x: float, device: torch.device, group=None) -> float:
    """Timing rule: a multi-GPU duration is the max over ranks."""
    t = torch.tensor([x], dtype=torch.float64, device=device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return float(t[0])


def bind_to_gpu_numa_node(device_index: int) -> Optional[int]:
    """Pins this process to the CPUs of the NUMA node its GPU hangs off, BEFORE any pinned host memory is allocated.
    The host-facing path streams ~58 B per env-step per GPU into pinned memory; with one process per GPU and default
    placement those buffers can land on the other socket and every PCIe write then crosses the inter-socket link.
    Returns the node id, or None when the topology cannot be read (nothing is changed then)."""
    try:
        pr = torch.cuda.get_device_properties(device_index)              # integer PCI ids in recent torch
        bus = f"{int(pr.pci_domain_id):04x}:{int(pr.pci_bus_id):02x}:{int(pr.pci_device_id):02x}.0"
    except Exception:
        bus = None
    try:
        if bus is None:
            import subprocess
            bus = subprocess.check_output(["nvidia-smi", "-i", str(device_index), "--query-gpu=pci.bus_id",
                                           "--format=csv,noheader"], text=True).strip()
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:              # nvidia-smi prints an 8-digit domain, sysfs uses 4
            bus = bus[4:]
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return node
    except Exception:
        return None

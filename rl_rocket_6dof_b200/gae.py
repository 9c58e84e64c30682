"""On-device generalised advantage estimation for rollouts recorded by `Rocket6DOFBatch.rollout(record=True)`.

The consumer of the env step in the reference is SB3's PPO (`model.learn`, main_6DOF.py:136), whose
`RolloutBuffer.compute_returns_and_advantage` runs on the host.  `compute_gae` is the same recurrence as one CUDA
kernel over the `[T, N]` trajectory tensors the rollout kernel already wrote, so a training loop never has to
leave the GPU.  Bootstrapping of time-limit truncations with the critic, which SB3 does while collecting, happens
before this scan: `Rocket6DOFBatch.collect_rollout(..., bootstrap_truncated=True)` files each truncation's terminal
observation as it is stepped and adds gamma * V to its reward (`r6_trunc_record` / `r6_trunc_bootstrap`).  The fused
`rollout(k, record=True)` keeps the env state in registers for all k steps and does not file them: there the
bootstrapping is left to the caller.
"""
from __future__ import annotations

from typing import Tuple

import torch

from . import _lib


def compute_gae(rewards: torch.Tensor, values: torch.Tensor, dones: torch.Tensor, last_values: torch.Tensor,
                gamma: float = 0.99, gae_lambda: float = 0.95) -> Tuple[torch.Tensor, torch.Tensor]:
    """rewards, values: float32 CUDA [T, N]; dones: uint8/bool CUDA [T, N] (episode ended at step t);
    last_values: float32 CUDA [N] (critic on the observation after the last step).  Returns (advantages, returns)."""
    if rewards.dim() != 2 or values.shape != rewards.shape or dones.shape != rewards.shape:
        raise ValueError("rewards, values and dones must all be [T, N]")
    T, n = rewards.shape
    if last_values.shape != (n,):
        raise ValueError("last_values must be [N]")
    for x in (rewards, values, last_values):
        if x.dtype != torch.float32 or not x.is_cuda:
            raise ValueError("rewards / values / last_values must be float32 CUDA tensors")
    if not dones.is_cuda:
        raise ValueError("dones must be a CUDA tensor")
    L = _lib.load()
    rewards, values, last_values = rewards.contiguous(), values.contiguous(), last_values.contiguous()
    d8 = (dones if dones.dtype == torch.uint8 else dones.to(torch.uint8)).contiguous()
    adv, ret = torch.empty_like(rewards), torch.empty_like(rewards)
    with torch.cuda.device(rewards.device):
        _lib.check(L.r6_gae(rewards.data_ptr(), values.data_ptr(), d8.data_ptr(), last_values.data_ptr(), int(T), int(n),
                            float(gamma), float(gae_lambda), adv.data_ptr(), ret.data_ptr(),
                            torch.cuda.current_stream(rewards.device).cuda_stream), L)
    return adv, ret

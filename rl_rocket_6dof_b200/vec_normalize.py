"""Observation and reward normalization on the device: SB3 1.6's `VecNormalize` for a `Rocket6DOFBatch`.

    vn = VecNormalize(batch, gamma=0.99)                   # VecNormalize(make_vec_env(...), gamma=0.99)
    trainer = PPOTrainer(batch, params, PPOConfig(), vec_normalize=vn)
    trainer.learn(10_000_000)
    vn.save("vecnormalize.npz")

The object holds SB3's running statistics as float64 CUDA tensors, `obs_rms` [13 means, 13 variances, count] and
`ret_rms` [mean, var, count], and the per-env discounted return `returns` [n].  `Rocket6DOFBatch.collect_rollout(...,
vec_normalize=vn)` updates them step by step with the r6_vn_* kernels and returns the normalized observations and
rewards; `step_policy(..., vec_normalize=vn)` and `montecarlo.run_montecarlo(..., vec_normalize=...)` apply frozen
statistics.  The batch's own `obs` and the episode statistics stay raw, as the env inside SB3's wrapper sees them.

SB3 semantics [memory] (SB3 is not a dependency; tests/vecnorm_ref.py restates them in numpy):
  - RunningMeanStd(epsilon=1e-4) starts at mean 0, var 1, count 1e-4; `update_from_moments` as include/r6dof.h states.
  - reset(): returns = 0; when training and norm_obs, obs_rms.update(reset observations).
  - each step: obs_rms.update(obs) (training and norm_obs); obs' = fl32(clip((obs - mean) / sqrt(var + eps), +-clip_obs));
    when training, returns = returns gamma + r (float64) and ret_rms.update(returns); r' = clip(r / sqrt(ret_var + eps),
    +-clip_reward) when norm_reward; terminal observations normalized with the statistics just updated; returns = 0
    where done.  ret_rms is updated whenever training, with or without norm_reward, as SB3 does.
Deliberate deviation: SB3 takes the observation batch's mean and variance of the float32 array, so numpy reduces in
float32; here the batch moments are float64 (at 2^20 envs a float32 sum over 2^20 rows loses most of its digits).
Everything after the batch moments (the update order, the divisions, sqrt, the clip, the one rounding to float32) is
SB3's arithmetic.

With a process group (data-parallel training, one env shard per rank), every rank's per-step observation moments and
per-rollout return moments are all_gathered and combined in rank order with `ppo.combine_moments`, so every rank holds
bit-identical statistics; `returns` stays per rank (its shard's envs).
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional

import numpy as np
import torch

from . import _lib

OBS_DIM = 13
# the construction-time consistency row of a data-parallel VecNormalize (what must agree across the ranks)
GROUP_FIELDS = ("training", "norm_obs", "norm_reward", "clip_obs", "clip_reward", "gamma", "epsilon", "num_envs")


def group_errors(rows: np.ndarray) -> list:
    """What is inconsistent in the gathered GROUP_FIELDS rows [W, F]: a function of the rows only, so every rank finds
    the same list."""
    return [f"{k} differs across ranks ({rows[:, i].tolist()})" for i, k in enumerate(GROUP_FIELDS)
            if not np.all(rows[:, i] == rows[0, i])]


def _rms(dim: int, device) -> torch.Tensor:
    """RunningMeanStd(epsilon=1e-4, shape): mean 0, var 1, count 1e-4, as [mean[dim], var[dim], count] float64."""
    t = torch.zeros(2 * dim + 1, dtype=torch.float64, device=device)
    t[dim:2 * dim] = 1.0
    t[2 * dim] = 1e-4
    return t


class VecNormalize:
    """SB3 1.6's `VecNormalize(venv, training, norm_obs, norm_reward, clip_obs, clip_reward, gamma, epsilon)` for
    `batch` (a Rocket6DOFBatch), with device-resident statistics (module docstring).  `group`: the data-parallel process
    group (the PPOTrainer's); construction then checks the settings across ranks (the same ValueError on every rank)
    and broadcasts the group's first rank's statistics."""

    def __init__(self, batch, *, training: bool = True, norm_obs: bool = True, norm_reward: bool = True,
                 clip_obs: float = 10.0, clip_reward: float = 10.0, gamma: float = 0.99, epsilon: float = 1e-8,
                 group=None):
        if not float(clip_obs) > 0 or not float(clip_reward) > 0:
            raise ValueError("clip_obs and clip_reward must be > 0")
        if not float(epsilon) >= 0 or not math.isfinite(float(epsilon)):
            raise ValueError("epsilon must be finite and >= 0")
        if not math.isfinite(float(gamma)) or not float(gamma) >= 0:
            raise ValueError("gamma must be finite and >= 0")
        self.batch, self.group = batch, group
        self.training, self.norm_obs, self.norm_reward = bool(training), bool(norm_obs), bool(norm_reward)
        self.clip_obs, self.clip_reward = float(clip_obs), float(clip_reward)
        self.gamma, self.epsilon = float(gamma), float(epsilon)
        self.lib = _lib.load()
        self.device = batch.device
        n = batch.num_envs
        self.obs_rms = _rms(OBS_DIM, self.device)
        self.ret_rms = _rms(1, self.device)
        self.returns = torch.zeros(n, dtype=torch.float64, device=self.device)
        self._mom = torch.empty(OBS_DIM, 3, dtype=torch.float64, device=self.device)
        self._work = torch.empty(max(int(self.lib.r6_vn_moments_work_bytes(n, OBS_DIM)), 8), dtype=torch.uint8,
                                 device=self.device)
        self.world = 1
        if group is not None:
            self._join_group(group)

    # ------------------------------------------------------------------ data-parallel plumbing
    def _join_group(self, group):
        import torch.distributed as dist
        self.world = dist.get_world_size(group)
        vals = dict(training=self.training, norm_obs=self.norm_obs, norm_reward=self.norm_reward, clip_obs=self.clip_obs,
                    clip_reward=self.clip_reward, gamma=self.gamma, epsilon=self.epsilon, num_envs=self.batch.num_envs)
        row = torch.tensor([float(vals[k]) for k in GROUP_FIELDS], dtype=torch.float64, device=self.device)
        rows = torch.empty(self.world, len(GROUP_FIELDS), dtype=torch.float64, device=self.device)
        dist.all_gather(list(rows.unbind(0)), row, group=group)
        errors = group_errors(rows.cpu().numpy())
        if errors:
            raise ValueError("data-parallel VecNormalize: " + "; ".join(errors))
        src = dist.get_global_rank(group, 0)
        dist.broadcast(self.obs_rms, src=src, group=group)
        dist.broadcast(self.ret_rms, src=src, group=group)

    def combine(self, mom: torch.Tensor) -> torch.Tensor:
        """The group's moments [R, 3] from this rank's (count, mean, M2) rows [R, 3]: every rank's rows all_gathered and
        combined row by row in rank order with `ppo.combine_moments`.  Without a group (or with one rank) `mom` itself."""
        if self.world == 1:
            return mom
        import torch.distributed as dist
        from .ppo import combine_moments
        rows = torch.empty((self.world,) + tuple(mom.shape), dtype=torch.float64, device=mom.device)
        dist.all_gather(list(rows.unbind(0)), mom.contiguous(), group=self.group)
        return combine_moments(rows.permute(0, 2, 1)).t().contiguous()

    # ------------------------------------------------------------------ kernels
    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def obs_moments(self, obs: torch.Tensor) -> torch.Tensor:
        """(count, mean, M2) [13, 3] float64 of rows 0..12 of the component-major obs [>= 13, n] (r6_vn_moments), this
        rank's only."""
        n = obs.shape[1]
        need = int(self.lib.r6_vn_moments_work_bytes(n, OBS_DIM))
        if self._work.numel() < need:
            self._work = torch.empty(need, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.r6_vn_moments(obs.data_ptr(), n, OBS_DIM, 0, n, self._mom.data_ptr(), self._work.data_ptr(),
                                              self._stream()), self.lib)
        return self._mom

    def update(self, rms: torch.Tensor, mom: torch.Tensor, steps: int, hist: Optional[torch.Tensor] = None):
        """`steps` update_from_moments of rms with mom [steps, dim, 3]; hist [steps + 1, 2, dim] receives
        (mean, sqrt(var + eps)) before and after each update (r6_vn_update)."""
        dim = (rms.numel() - 1) // 2
        with torch.cuda.device(self.device):
            _lib.check(self.lib.r6_vn_update(rms.data_ptr(), dim, mom.data_ptr() if steps else None, int(steps), self.epsilon,
                                             None if hist is None else hist.data_ptr(), self._stream()), self.lib)

    def obs_hist(self, rows: int = 1) -> torch.Tensor:
        """[rows, 2, 13] float64: every row the current obs statistics' (mean, sqrt(var + eps)), as the normalize pass
        reads them."""
        h = torch.empty(rows, 2, OBS_DIM, dtype=torch.float64, device=self.device)
        self.update(self.obs_rms, None, 0, h[:1])
        if rows > 1:
            h[1:] = h[:1]
        return h

    def normalize(self, src: torch.Tensor, dst: torch.Tensor, hist: torch.Tensor, row: int = 0, first: int = 0,
                  count: Optional[int] = None, step: Optional[torch.Tensor] = None,
                  stream: Optional[torch.cuda.Stream] = None):
        """Rows 0..12 of dst[:, first:first + count] = the normalized src (r6_vn_normalize), with history row `row` of
        hist [R, 2, 13], or row step[i] + 1 per env; src and dst are component-major with n columns and may be one."""
        n = src.shape[-1]
        count = n - first if count is None else count
        s = (stream or torch.cuda.current_stream(self.device)).cuda_stream
        with torch.cuda.device(self.device):
            _lib.check(self.lib.r6_vn_normalize(src.data_ptr(), dst.data_ptr(), n, first, count, hist.data_ptr(), int(row),
                                                None if step is None else step.data_ptr(), hist.shape[0], self.clip_obs, s),
                       self.lib)

    def normalize_obs(self, obs: torch.Tensor) -> torch.Tensor:
        """SB3's normalize_obs with the current statistics: a new [14, n] tensor (the mass row copied, raw), or a copy
        of obs when norm_obs is off."""
        out = obs.clone()
        if self.norm_obs:
            self.normalize(obs, out, self.obs_hist())
        return out

    def observe(self, obs: torch.Tensor, hist: Optional[torch.Tensor] = None):
        """obs_rms.update(rows 0..12 of obs), the group's moments when there is one; hist [2, 2, 13] (nullable) gets the
        statistics before and after."""
        self.update(self.obs_rms, self.combine(self.obs_moments(obs)), 1, hist)

    def reward_pass(self, rews: torch.Tensor, dones: torch.Tensor):
        """After a T-step collection (raw float32 rewards [T, n], dones [T, n]): the return scan and T ret_rms updates
        when training, then the rewards normalized in place when norm_reward."""
        T, n = rews.shape
        hist = torch.empty(T + 1, 2, 1, dtype=torch.float64, device=self.device)
        if self.training:
            mom = torch.empty(T, 3, dtype=torch.float64, device=self.device)
            work = torch.empty(max(int(self.lib.r6_vn_ret_work_bytes(T, n)), 8), dtype=torch.uint8, device=self.device)
            with torch.cuda.device(self.device):
                _lib.check(self.lib.r6_vn_ret_moments(rews.data_ptr(), dones.data_ptr(), T, n, self.returns.data_ptr(),
                                                      self.gamma, mom.data_ptr(), work.data_ptr(), self._stream()), self.lib)
            self.update(self.ret_rms, self.combine(mom).reshape(T, 1, 3), T, hist)
        elif self.norm_reward:
            self.update(self.ret_rms, None, 0, hist[:1])
            hist[1:] = hist[:1]
        if self.norm_reward:
            with torch.cuda.device(self.device):
                _lib.check(self.lib.r6_vn_scale_rewards(rews.data_ptr(), T, n, hist.data_ptr(), self.clip_reward,
                                                        self._stream()), self.lib)

    # ------------------------------------------------------------------ SB3's API
    def reset(self) -> torch.Tensor:
        """SB3's VecNormalize.reset after the batch's reset: returns = 0, obs_rms updated with the batch's observations
        when training and norm_obs; returns the normalized observations [14, n] (a new tensor)."""
        self.batch.join()
        self.returns.zero_()
        if self.training and self.norm_obs:
            self.observe(self.batch.obs)
        return self.normalize_obs(self.batch.obs)

    def save(self, path: str):
        """The statistics and settings as .npz with SB3's names (obs_rms.mean, obs_rms.var, obs_rms.count, ret_rms.*,
        clip_obs, ...).  As SB3's pickle, `returns` is not saved."""
        o, r = self.obs_rms.cpu().numpy(), self.ret_rms.cpu().numpy()
        np.savez(path, **{"obs_rms.mean": o[:OBS_DIM], "obs_rms.var": o[OBS_DIM:2 * OBS_DIM],
                          "obs_rms.count": o[2 * OBS_DIM], "ret_rms.mean": r[0], "ret_rms.var": r[1],
                          "ret_rms.count": r[2], "clip_obs": self.clip_obs, "clip_reward": self.clip_reward,
                          "norm_obs": self.norm_obs, "norm_reward": self.norm_reward, "gamma": self.gamma,
                          "epsilon": self.epsilon, "training": self.training})

    @classmethod
    def frozen(cls, batch, source, into: Optional["VecNormalize"] = None) -> "VecNormalize":
        """A `VecNormalize(batch, training=False)` holding frozen observation statistics for a deterministic evaluation:
        `source` is the path of a `save` .npz (everything `load` restores), or a VecNormalize whose obs_rms, norm_obs,
        clip_obs and epsilon are copied (SB3's sync_envs_normalization; rewards are not normalized by an evaluation).
        `into` (a VecNormalize of `batch`) is refreshed instead of building a new one."""
        vn = into if into is not None else cls(batch, training=False)
        if isinstance(source, VecNormalize):
            vn.obs_rms.copy_(source.obs_rms)
            vn.norm_obs, vn.clip_obs, vn.epsilon = source.norm_obs, source.clip_obs, source.epsilon
        else:
            vn.load(source)
        return vn

    def load(self, path: str) -> "VecNormalize":
        """Restores what `save` wrote (statistics and settings, as unpickling SB3's object does); `returns` is left as
        it is.  Returns self."""
        z = np.load(path)
        o = np.concatenate([np.asarray(z["obs_rms.mean"], np.float64).reshape(OBS_DIM),
                            np.asarray(z["obs_rms.var"], np.float64).reshape(OBS_DIM),
                            np.asarray(z["obs_rms.count"], np.float64).reshape(1)])
        r = np.array([float(z["ret_rms.mean"]), float(z["ret_rms.var"]), float(z["ret_rms.count"])], np.float64)
        self.obs_rms.copy_(torch.from_numpy(o))
        self.ret_rms.copy_(torch.from_numpy(r))
        self.clip_obs, self.clip_reward = float(z["clip_obs"]), float(z["clip_reward"])
        self.norm_obs, self.norm_reward = bool(z["norm_obs"]), bool(z["norm_reward"])
        self.gamma, self.epsilon, self.training = float(z["gamma"]), float(z["epsilon"]), bool(z["training"])
        return self

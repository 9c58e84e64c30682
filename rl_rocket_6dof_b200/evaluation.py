"""Deterministic evaluation during on-device PPO training: SB3 1.6's `EvalCallback` with `evaluate_policy(...,
deterministic=True)`, the callback of main_6DOF.py:116-133 that writes the `best_model` checkpoints
montecarlo_script.py loads.

    eval_batch = Rocket6DOFBatch(1024, seed=1042, auto_reset=False, time_limit=True, split_step=True)
    cb = EvalCallback(eval_batch, eval_freq=3200, log_path="run", best_model_save_path="run")
    trainer.learn(20_000_000, eval_callback=cb)           # logs gain eval/..., run/best_model.npz is the best iterate

Every env of the evaluation batch runs exactly one episode per evaluation (`montecarlo.run_episodes`: the policy kernel
and the env-step kernels, with the batch's one-episode semantics), so n_eval_episodes is the batch's global env count.
The batch persists between evaluations and r6_reset keys the initial conditions by (seed, global env id, episode id),
so each evaluation draws fresh ones, as SB3's eval env does.

SB3 1.6 semantics [memory] (SB3 is not a dependency; tests/evalcb_ref.py restates them):
  - `_on_step` evaluates when n_calls % eval_freq == 0, n_calls counting vec-env steps.  With VecNormalize it first runs
    sync_envs_normalization (the eval env gets a copy of the training statistics and never updates them).
  - `evaluate_policy` with n_envs == n_eval_episodes: episode_count_targets are all 1, so each env contributes its
    first episode; at every step the envs are visited in index order and a finished one appends its Monitor
    info["episode"]["r"] (the float64 sum of the rewards, rounded to 6 decimals by Python's round) and "l".  All
    episodes start together, so the result order is a stable sort by length.
  - mean / std are np.mean / np.std (ddof=0) of the results in that order; best_mean_reward starts at -inf and a
    strictly greater mean_reward saves `best_model`; `log_path` rewrites <log_path>/evaluations.npz (timesteps,
    results, ep_lengths) after every evaluation.
Deviations:
  - Evaluations run at rollout boundaries: after collection i (vec-env steps (i n_steps, (i + 1) n_steps]) when that
    range holds a multiple of eval_freq, once however many it holds, before that iteration's train() and with the
    parameters and VecNormalize statistics that collected it.  When eval_freq is a multiple of n_steps this is SB3's
    schedule exactly; otherwise an evaluation is late by less than n_steps vec-env steps, and `timesteps` records the
    end of the collection.
  - The best model is `ActorCriticParams.save_npz` (`best_model.npz`, read by `policy.load_npz` and the Monte-Carlo
    CLI), not an SB3 zip; with VecNormalize the training statistics of that evaluation are saved beside it
    (`best_model_vecnormalize.npz`), since the model cannot be evaluated without the statistics of its own moment.
  - eval/landing_rate is logged (the env has no is_success): the share of episodes with every landing bit set.

Data-parallel (`group=`, the trainer's process group): rank r holds the eval shard [r m, (r + 1) m) of W m episodes
(`sharding.shard_batch_kwargs(m, r, W)`).  Construction all_gathers every rank's shard, seed, eval_freq and
tensor_cores, and anything inconsistent makes every rank raise the same ValueError.  Each rank runs its shard; the
per-episode returns, lengths and flags are all_gathered (bytes only) into global env order, and every rank computes the
logs and the best-model decision from the same array.  Only the group's first rank writes files.  Philox streams are
keyed by global env id and the replicas are bit-identical, so the result is the one-process evaluation of W m envs.
"""
from __future__ import annotations

import math
import os
from typing import Optional

import numpy as np
import torch

from . import montecarlo

# the construction-time consistency row of a data-parallel EvalCallback (what must agree across the ranks)
GROUP_FIELDS = ("num_envs", "env_offset", "num_envs_global", "seed_hi", "seed_lo", "eval_freq", "tensor_cores",
                "local_error")
_PER_RANK = ("env_offset", "local_error")            # checked against the rank's index, not against rank 0
_LOCAL_ERRORS = {1: "the evaluation batch must have auto_reset=False (one episode per env and evaluation)",
                 2: "the evaluation batch must have time_limit=True (without it an episode need not end)",
                 3: "only deterministic evaluation is implemented (deterministic=True)",
                 4: "n_eval_episodes must be the evaluation batch's global env count (num_envs_global)",
                 5: "eval_freq must be >= 1"}


def evaluation_due(n_calls: int, n_steps: int, eval_freq: int) -> bool:
    """Whether the collection that took the vec-env step count from n_calls - n_steps to n_calls evaluates: its steps
    (n_calls - n_steps, n_calls] hold at least one multiple of eval_freq (SB3's n_calls % eval_freq == 0)."""
    return n_calls // eval_freq > (n_calls - n_steps) // eval_freq


def monitor_rewards(returns: np.ndarray) -> np.ndarray:
    """Monitor's info["episode"]["r"] of float64 episode returns: Python's round(r, 6), as Rocket6DOFVecEnv reports it
    (numpy's round scales by 10^6 and can differ in the last ulp)."""
    return np.array([round(r, 6) for r in np.asarray(returns, np.float64).tolist()], np.float64)


def result_order(lengths: np.ndarray) -> np.ndarray:
    """evaluate_policy's append order of one episode per env, all started together: by completion step (the length),
    then by env index."""
    return np.argsort(np.asarray(lengths), kind="stable")


def summarize(rewards: np.ndarray, lengths: np.ndarray, landed: np.ndarray) -> dict:
    """The eval/ logs of one evaluation (without best_mean_reward): np.mean / np.std (ddof=0) as SB3 computes them, over
    rewards and lengths in SB3's result order (`result_order`: the float64 sums depend on it in the last bits)."""
    return {"eval/mean_reward": float(np.mean(rewards)), "eval/std_reward": float(np.std(rewards)),
            "eval/mean_ep_length": float(np.mean(lengths)), "eval/std_ep_length": float(np.std(lengths)),
            "eval/landing_rate": float(np.mean(landed))}


def group_errors(rows: np.ndarray, world: int) -> list:
    """What is inconsistent in the gathered GROUP_FIELDS rows [W, F]: a function of the rows only, so every rank finds
    the same list."""
    col = {k: rows[:, i] for i, k in enumerate(GROUP_FIELDS)}
    n = int(col["num_envs"][0])
    errors = [f"rank {r}: {_LOCAL_ERRORS.get(int(e), 'local check failed')}"
              for r, e in enumerate(col["local_error"]) if e != 0]
    errors += [f"{k} differs across ranks ({col[k].tolist()})" for k in GROUP_FIELDS
               if k not in _PER_RANK and not np.all(col[k] == col[k][0])]
    errors += [f"rank {r} has env_offset {int(o)}, its eval shard starts at {r * n}"
               for r, o in enumerate(col["env_offset"]) if o != r * n]
    if col["num_envs_global"][0] != world * n:
        errors.append(f"num_envs_global {int(col['num_envs_global'][0])} is not world {world} x num_envs {n}")
    return errors


class EvaluationLog:
    """SB3's evaluations.npz: one row per evaluation of timesteps [k], results [k, n] float64 and ep_lengths [k, n]
    int64, the whole file rewritten after every evaluation."""

    def __init__(self, path: Optional[str]):
        self.path = path
        self.timesteps, self.results, self.ep_lengths = [], [], []

    def append(self, timesteps: int, results: np.ndarray, ep_lengths: np.ndarray):
        self.timesteps.append(int(timesteps))
        self.results.append(np.asarray(results, np.float64))
        self.ep_lengths.append(np.asarray(ep_lengths, np.int64))

    def save(self):
        np.savez(self.path, timesteps=np.array(self.timesteps, np.int64), results=np.array(self.results, np.float64),
                 ep_lengths=np.array(self.ep_lengths, np.int64))


class EvalCallback:
    """SB3 1.6's `EvalCallback(eval_env, eval_freq, n_eval_episodes, log_path, best_model_save_path, deterministic)` for
    `PPOTrainer.learn(..., eval_callback=...)` (module docstring).

    eval_batch: a Rocket6DOFBatch with auto_reset=False and time_limit=True (ValueError otherwise), on the trainer's
    device; n_eval_episodes (None: the batch's) must be its num_envs_global.  eval_freq is in vec-env steps (SB3's
    n_calls).  tensor_cores (None: the trainer's PPOConfig.tensor_cores) is the `step_policy` mode of the policy kernel.
    The evaluation touches nothing of the trainer (batch, generator, Adam state, VecNormalize), so training with it is
    bit-identical to training without it."""

    def __init__(self, eval_batch, *, eval_freq: int, n_eval_episodes: Optional[int] = None,
                 log_path: Optional[str] = None, best_model_save_path: Optional[str] = None, deterministic: bool = True,
                 tensor_cores: Optional[int] = None, group=None):
        b = eval_batch
        local_error = 0
        if b.auto_reset:
            local_error = 1
        elif not b.time_limit:
            local_error = 2
        elif not deterministic:
            local_error = 3
        elif n_eval_episodes is not None and int(n_eval_episodes) != b.num_envs_global:
            local_error = 4
        elif not int(eval_freq) >= 1:
            local_error = 5
        self.batch, self.group = b, group
        self.eval_freq, self.tensor_cores = int(eval_freq), tensor_cores
        self.n_eval_episodes = b.num_envs_global
        self.world, self.rank = 1, 0
        if group is None:
            if local_error:
                raise ValueError(_LOCAL_ERRORS[local_error] + (f" ({n_eval_episodes} != {b.num_envs_global})"
                                                               if local_error == 4 else ""))
        else:
            self._join_group(local_error)
        self.writer = self.rank == 0
        self.log_path = None if log_path is None else os.path.join(log_path, "evaluations.npz")
        self.best_model_save_path = best_model_save_path
        if self.writer:
            for d in (log_path, best_model_save_path):
                if d is not None:
                    os.makedirs(d, exist_ok=True)
        self.evaluations = EvaluationLog(self.log_path)
        self.best_mean_reward = -math.inf
        self.last_mean_reward = -math.inf
        self.n_calls = 0
        self.vec_normalize = None            # the frozen copy of the trainer's statistics, built at the first evaluation

    def _join_group(self, local_error: int):
        import torch.distributed as dist
        self.world, self.rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        b = self.batch
        seed = int(b.seed_value) % (1 << 64)
        vals = dict(num_envs=b.num_envs, env_offset=b.env_offset, num_envs_global=b.num_envs_global, seed_hi=seed >> 32,
                    seed_lo=seed & 0xFFFFFFFF, eval_freq=self.eval_freq,
                    tensor_cores=-1 if self.tensor_cores is None else int(self.tensor_cores), local_error=local_error)
        row = torch.tensor([float(vals[k]) for k in GROUP_FIELDS], dtype=torch.float64, device=b.device)
        rows = torch.empty(self.world, len(GROUP_FIELDS), dtype=torch.float64, device=b.device)
        dist.all_gather(list(rows.unbind(0)), row, group=self.group)
        errors = group_errors(rows.cpu().numpy(), self.world)
        if errors:
            raise ValueError("data-parallel EvalCallback: " + "; ".join(errors))

    def on_rollout_end(self, trainer) -> dict:
        """Called by `PPOTrainer.learn` after each collection, before train(): counts the collection's n_steps vec-env
        steps and, when an evaluation is due, runs it and returns its eval/ logs (otherwise {})."""
        if trainer.group is not self.group:
            raise ValueError("the EvalCallback must have the trainer's process group")
        self.n_calls += trainer.cfg.n_steps
        if not evaluation_due(self.n_calls, trainer.cfg.n_steps, self.eval_freq):
            return {}
        return self.evaluate(trainer)

    def run(self, trainer) -> dict:
        """One evaluation of trainer.params over every env of the (global) evaluation batch, with frozen copies of the
        trainer's VecNormalize statistics: {"episode_return" float64, "episode_length" int64, "flags" uint8} [W m] in
        global env order, on the host."""
        tc = trainer.cfg.tensor_cores if self.tensor_cores is None else self.tensor_cores
        vn = None
        if trainer.vec_normalize is not None:
            from .vec_normalize import VecNormalize
            vn = self.vec_normalize = VecNormalize.frozen(self.batch, trainer.vec_normalize, into=self.vec_normalize)
        ep = montecarlo.run_episodes(self.batch, trainer.params.mlp(), tensor_cores=tc, vec_normalize=vn)
        rows = torch.stack([ep["episode_return"], ep["episode_length"].double(), ep["flags"].double()])   # [3, m], exact
        if self.world > 1:
            import torch.distributed as dist
            out = torch.empty((self.world,) + tuple(rows.shape), dtype=rows.dtype, device=rows.device)
            dist.all_gather(list(out.unbind(0)), rows, group=self.group)
            rows = out.permute(1, 0, 2).reshape(3, -1)
        h = rows.cpu().numpy()
        return {"episode_return": h[0], "episode_length": h[1].astype(np.int64), "flags": h[2].astype(np.uint8)}

    def evaluate(self, trainer) -> dict:
        """One evaluation now (whether or not it is due): logs, evaluations.npz, best model."""
        ep = self.run(trainer)
        order = result_order(ep["episode_length"])         # SB3's order, in which it also sums for the mean
        rewards, lengths = monitor_rewards(ep["episode_return"])[order], ep["episode_length"][order]
        logs = summarize(rewards, lengths, (ep["flags"] & 0xF8) == 0xF8)
        self.evaluations.append(trainer.num_timesteps, rewards, lengths)
        if self.writer and self.log_path is not None:
            self.evaluations.save()
        mean = logs["eval/mean_reward"]
        self.last_mean_reward = mean
        if mean > self.best_mean_reward:
            if self.writer and self.best_model_save_path is not None:
                trainer.params.save_npz(os.path.join(self.best_model_save_path, "best_model.npz"))
                if trainer.vec_normalize is not None:
                    trainer.vec_normalize.save(os.path.join(self.best_model_save_path, "best_model_vecnormalize.npz"))
            self.best_mean_reward = mean
        logs["eval/best_mean_reward"] = float(self.best_mean_reward)
        return logs

"""PPO training on the device: the update of stable-baselines3 1.6's `PPO.train` (the `model.learn` of main_6DOF.py:136)
over rollouts collected by `Rocket6DOFBatch.collect_rollout`, with the loss gradient (`r6_ppo_grad`) and the Adam step
(`r6_adam_step`) as CUDA kernels.  Nothing leaves the GPU during an update unless `target_kl` is set.  As SB3's
`collect_rollouts` does, the collection bootstraps episodes cut by the TimeLimit with the critic
(`collect_rollout(..., bootstrap_truncated=True)`), so the batch must auto-reset.

    params = ActorCriticParams.sb3_init(seed=0, device="cuda:0")
    trainer = PPOTrainer(batch, params, PPOConfig(), seed=0)
    logs = trainer.learn(total_timesteps=10_000_000)

The network is SB3's default `MlpPolicy` of SB3 1.6: a shared tanh trunk 13 -> 128 -> 64, `action_net` 64 -> 3,
`value_net` 64 -> 1 and a state-independent `log_std` (no gSDE, no `clip_range_vf`).
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import Callable, Dict, Optional, Union

import numpy as np
import torch

from . import _lib

# flat parameter layout of include/r6dof.h: (name, shape), in order
LAYOUT = (("w0", (128, 13)), ("b0", (128,)), ("w1", (64, 128)), ("b1", (64,)), ("w2", (3, 64)), ("b2", (3,)),
          ("wv", (64,)), ("bv", (1,)), ("log_std", (3,)))
NPARAMS = _lib.PPO_NPARAMS
_LOG_SQRT_2PI = 0.5 * math.log(2.0 * math.pi)


class ActorCriticParams:
    """The actor-critic as one flat float32 CUDA tensor `flat` [R6_PPO_NPARAMS] with views w0 ... log_std into it."""

    def __init__(self, flat: torch.Tensor):
        if flat.dtype != torch.float32 or not flat.is_cuda or flat.shape != (NPARAMS,) or not flat.is_contiguous():
            raise ValueError(f"flat parameters must be a contiguous float32 CUDA tensor of {NPARAMS} elements")
        self.flat = flat
        o = 0
        for name, shape in LAYOUT:
            size = int(np.prod(shape))
            setattr(self, name, flat[o:o + size].view(shape))
            o += size
        assert o == NPARAMS

    @classmethod
    def sb3_init(cls, seed: int = 0, device="cuda") -> "ActorCriticParams":
        """SB3's construction-time weights (ortho_init): `torch.nn.init.orthogonal_` with gain sqrt(2) on the trunk,
        0.01 on action_net and 1 on value_net, zero biases, log_std 0.  Drawn on the CPU with a generator seeded by
        `seed`, so they do not depend on the device."""
        gen = torch.Generator().manual_seed(int(seed))
        w = {}
        for name, shape, gain in (("w0", (128, 13), math.sqrt(2)), ("w1", (64, 128), math.sqrt(2)), ("w2", (3, 64), 0.01),
                                  ("wv", (1, 64), 1.0)):
            t = torch.empty(shape, dtype=torch.float32)
            torch.nn.init.orthogonal_(t, gain=gain, generator=gen)
            w[name] = t.reshape(-1)
        return cls._from(w, device)

    @classmethod
    def from_weights(cls, w: Dict[str, np.ndarray], device="cuda") -> "ActorCriticParams":
        """From `policy.load_sb3_zip` / `policy.load_npz` output (the critic head and log_std must be present)."""
        missing = [k for k, _ in LAYOUT if w.get(k) is None]
        if missing:
            raise ValueError(f"weights lack {missing}: training needs the critic head and log_std")
        return cls._from(w, device)

    @classmethod
    def _from(cls, w, device) -> "ActorCriticParams":
        flat = torch.zeros(NPARAMS, dtype=torch.float32)
        o = 0
        for name, shape in LAYOUT:
            size = int(np.prod(shape))
            if name in w:
                flat[o:o + size] = torch.as_tensor(np.asarray(w[name], np.float32).reshape(-1))
            o += size
        return cls(flat.to(device))

    def mlp(self) -> Dict[str, torch.Tensor]:
        """The weight dict `collect_rollout`, `step_policy`, `policy_forward` and `montecarlo` accept."""
        return {name: getattr(self, name) for name, _ in LAYOUT}

    def save_npz(self, path: str):
        """Writes `mlp_w0` ... `mlp_log_std`: what `policy.load_npz` and the Monte-Carlo CLI read."""
        np.savez(path, **{"mlp_" + k: v.detach().cpu().numpy() for k, v in self.mlp().items()})


def _progress_lr(lr, progress_remaining: float) -> float:
    return float(lr(progress_remaining)) if callable(lr) else float(lr)


@dataclass
class PPOConfig:
    """SB3 1.6 PPO defaults, except n_steps and batch_size.

    SB3's n_steps = 2048 and batch_size = 64 are sized for a handful of CPU envs; at 2^16 and more envs on one GPU they
    would mean 2^27-sample rollouts in 2^21 minibatches of 64.  Here a rollout is `n_steps` (default 32) steps of every
    env, and `batch_size` defaults to a quarter of it (4 minibatches per epoch).  As in SB3 the last minibatch of an
    epoch may be short.  A minibatch of one sample is not normalised (its std is undefined: SB3 1.6 yields NaN there
    [memory]; later SB3 releases add the same guard).  A callable learning_rate is SB3's schedule: it is called once per
    update with progress_remaining (see `PPOTrainer.learn`)."""
    learning_rate: Union[float, Callable[[float], float]] = 3e-4
    n_steps: int = 32
    batch_size: Optional[int] = None
    n_epochs: int = 10
    gamma: float = 0.99
    gae_lambda: float = 0.95
    clip_range: float = 0.2
    normalize_advantage: bool = True
    ent_coef: float = 0.0
    vf_coef: float = 0.5
    max_grad_norm: float = 0.5
    target_kl: Optional[float] = None
    tensor_cores: int = 3          # policy kernel of the collection (r6_policy: 3 = tcgen05 3xTF32, float32-faithful)


def _check_cuda(name, t, dtype, dev):
    if not isinstance(t, torch.Tensor) or t.dtype != dtype or t.device != dev:
        raise ValueError(f"{name} must be a {dtype} tensor on {dev}")


def loss_and_grad(params: ActorCriticParams, rollout: dict, idx: torch.Tensor, *, clip_range: float = 0.2,
                  vf_coef: float = 0.5, ent_coef: float = 0.0, normalize_advantage: bool = True,
                  grad_sum: Optional[torch.Tensor] = None, terms: Optional[torch.Tensor] = None,
                  work: Optional[torch.Tensor] = None):
    """SUM over the minibatch `idx` (int64 sample indices t * N + i into the [T, N] rollout) of the per-sample PPO loss
    gradient, and the float64 term sums (policy-gradient loss, (R - V)^2, clipped count, approx-kl, bad indices).
    `rollout` is `collect_rollout`'s dict (obs [T, N, 13] with any strides, actions [T, N, 3], log_probs, advantages,
    returns [T, N]).  Indices outside [0, T N) are skipped and counted in terms[4] (checking them here would
    synchronise).  The minibatch's advantage mean and 1 / (std + 1e-8) are computed on the device (no synchronise).
    Returns (grad_sum float32 [R6_PPO_NPARAMS], terms float64 [5])."""
    dev = params.flat.device
    obs, act = rollout["obs"], rollout["actions"]
    lp, adv, ret = rollout["log_probs"], rollout["advantages"], rollout["returns"]
    for name, t in (("obs", obs), ("actions", act), ("log_probs", lp), ("advantages", adv), ("returns", ret)):
        _check_cuda(name, t, torch.float32, dev)
    if adv.dim() != 2:
        raise ValueError("advantages must be [T, N]")
    T, n = adv.shape
    if obs.shape != (T, n, 13) or act.shape != (T, n, 3) or lp.shape != (T, n) or ret.shape != (T, n):
        raise ValueError("rollout shapes must be obs [T, N, 13], actions [T, N, 3], log_probs / advantages / returns [T, N]")
    if not (act.is_contiguous() and lp.is_contiguous() and adv.is_contiguous() and ret.is_contiguous()):
        raise ValueError("actions, log_probs, advantages and returns must be contiguous")
    _check_cuda("idx", idx, torch.int64, dev)
    if idx.dim() != 1 or not idx.is_contiguous():
        raise ValueError("idx must be a contiguous 1-D int64 tensor")
    B = idx.numel()
    if grad_sum is None:
        grad_sum = torch.empty(NPARAMS, dtype=torch.float32, device=dev)
    if terms is None:
        terms = torch.empty(_lib.PPO_NTERMS, dtype=torch.float64, device=dev)
    _check_cuda("grad_sum", grad_sum, torch.float32, dev)
    _check_cuda("terms", terms, torch.float64, dev)
    if grad_sum.shape != (NPARAMS,) or terms.shape != (_lib.PPO_NTERMS,) or not grad_sum.is_contiguous():
        raise ValueError("grad_sum / terms have the wrong shape")
    L = _lib.load()
    need = int(L.r6_ppo_work_bytes(B))
    if work is None or work.numel() < need:
        work = torch.empty(max(need, 1), dtype=torch.uint8, device=dev)
    stats = None
    if normalize_advantage and B > 1:
        # clamped: an index outside the rollout must not reach torch's gather (a device-side assert); the kernel skips
        # and counts such indices (terms[4]), and a caller that sees a non-zero count discards the result
        a = adv.reshape(-1)[idx.clamp(0, max(T * n - 1, 0))].double()
        stats = torch.stack([a.mean(), 1.0 / (a.std() + 1e-8)])
    ro = _lib.R6PpoRollout(obs.data_ptr(), obs.stride(0), obs.stride(2), obs.stride(1), act.data_ptr(), lp.data_ptr(),
                           adv.data_ptr(), ret.data_ptr(), T, n)
    coef = _lib.R6PpoCoef(float(clip_range), float(vf_coef), float(ent_coef), None if stats is None else stats.data_ptr())
    m = _lib.make_mlp(params.mlp())
    with torch.cuda.device(dev):
        _lib.check(L.r6_ppo_grad(C.byref(m), C.byref(ro), idx.data_ptr(), B, C.byref(coef), grad_sum.data_ptr(),
                                 terms.data_ptr(), work.data_ptr(), torch.cuda.current_stream(dev).cuda_stream), L)
    return grad_sum, terms


def adam_step(params: torch.Tensor, grad_sum: torch.Tensor, m: torch.Tensor, v: torch.Tensor, *, lr: float, step: int,
              scale: float = 1.0, max_grad_norm: float = 0.5, betas=(0.9, 0.999), eps: float = 1e-5,
              grad_norm: Optional[torch.Tensor] = None):
    """torch.optim.Adam(eps=1e-5, SB3's setting) after clip_grad_norm_(max_grad_norm) on g = scale * grad_sum, in place
    on the flat float32 tensors params, m, v.  `step` counts updates including this one.  grad_norm (optional float64
    [1] CUDA tensor) receives the norm before clipping."""
    dev = params.device
    for name, t in (("params", params), ("grad_sum", grad_sum), ("m", m), ("v", v)):
        _check_cuda(name, t, torch.float32, dev)
        if t.dim() != 1 or not t.is_contiguous() or t.numel() != params.numel():
            raise ValueError(f"{name} must be contiguous 1-D with params' size")
    if grad_norm is not None:
        _check_cuda("grad_norm", grad_norm, torch.float64, dev)
    coef = _lib.R6AdamCoef(float(lr), float(betas[0]), float(betas[1]), float(eps), float(max_grad_norm), float(scale))
    L = _lib.load()
    with torch.cuda.device(dev):
        _lib.check(L.r6_adam_step(params.data_ptr(), grad_sum.data_ptr(), m.data_ptr(), v.data_ptr(), params.numel(),
                                  C.byref(coef), int(step), None if grad_norm is None else grad_norm.data_ptr(),
                                  torch.cuda.current_stream(dev).cuda_stream), L)


class PPOTrainer:
    """SB3 1.6 `PPO.learn` over a `Rocket6DOFBatch`: collection by `collect_rollout`, update by `train`."""

    def __init__(self, batch, params: ActorCriticParams, cfg: Optional[PPOConfig] = None, seed: int = 0):
        self.batch, self.params, self.cfg = batch, params, cfg or PPOConfig()
        dev = params.flat.device
        self.m = torch.zeros_like(params.flat)
        self.v = torch.zeros_like(params.flat)
        self.gen = torch.Generator(device=dev)
        self.gen.manual_seed(int(seed))
        self.n_updates = 0            # SB3's _n_updates (epochs run)
        self.adam_steps = 0
        self.num_timesteps = 0
        self.progress_remaining = 1.0
        self._grad = torch.empty(NPARAMS, dtype=torch.float32, device=dev)
        self._work = None

    def batch_size(self, total: int) -> int:
        return int(self.cfg.batch_size) if self.cfg.batch_size else max(1, -(-total // 4))

    def train(self, rollout: dict) -> dict:
        """n_epochs passes over the rollout in minibatches of a seeded on-device permutation; returns SB3's train/ logs.

        As SB3 1.6 logs them [memory]: policy_gradient_loss, value_loss, clip_fraction and entropy_loss are means over
        every minibatch that ran (the one `target_kl` stops at included), approx_kl is the mean over the minibatches of
        the last epoch that ran, entropy_loss and loss use each minibatch's log_std before its Adam step, and loss is the
        last minibatch's.  The learning rate is `learning_rate(progress_remaining)`."""
        cfg, dev = self.cfg, self.params.flat.device
        T, n = rollout["advantages"].shape
        total = T * n
        bs = self.batch_size(total)
        lr = _progress_lr(cfg.learning_rate, self.progress_remaining)
        nmb = -(-total // bs)
        terms = torch.zeros(cfg.n_epochs * nmb, _lib.PPO_NTERMS, dtype=torch.float64, device=dev)
        log_std_sums = torch.zeros(cfg.n_epochs * nmb, dtype=torch.float64, device=dev)
        sizes = []
        L = _lib.load()
        need = int(L.r6_ppo_work_bytes(min(bs, total)))
        if self._work is None or self._work.numel() < need:
            self._work = torch.empty(need, dtype=torch.uint8, device=dev)
        done = False
        for epoch in range(cfg.n_epochs):
            perm = torch.randperm(total, generator=self.gen, device=dev)
            epoch_start = len(sizes)
            for start in range(0, total, bs):
                idx = perm[start:start + bs]
                k = len(sizes)
                loss_and_grad(self.params, rollout, idx, clip_range=cfg.clip_range, vf_coef=cfg.vf_coef,
                              ent_coef=cfg.ent_coef, normalize_advantage=cfg.normalize_advantage, grad_sum=self._grad,
                              terms=terms[k], work=self._work)
                log_std_sums[k] = self.params.log_std.sum(dtype=torch.float64)    # this minibatch's entropy (no sync)
                sizes.append(idx.numel())
                if cfg.target_kl is not None:
                    kl = float(terms[k, _lib.PPO_NTERMS - 2]) / idx.numel()      # the one host read per minibatch
                    if kl > 1.5 * cfg.target_kl:
                        done = True
                        break
                self.adam_steps += 1
                adam_step(self.params.flat, self._grad, self.m, self.v, lr=lr, step=self.adam_steps,
                          scale=1.0 / idx.numel(), max_grad_norm=cfg.max_grad_norm)
            if done:
                break
        self.n_updates += cfg.n_epochs
        t = terms[:len(sizes)].cpu().numpy()
        if t[:, 4].sum() != 0:
            raise ValueError("a minibatch index was outside the rollout")
        means = t[:, :4] / np.asarray(sizes, np.float64)[:, None]
        entropy = log_std_sums[:len(sizes)].cpu().numpy() + 3 * (0.5 + _LOG_SQRT_2PI)     # per minibatch
        log_std = self.params.log_std.detach().double().cpu().numpy()
        v, r = rollout["values"].reshape(-1).double(), rollout["returns"].reshape(-1).double()
        var_r = float(r.var())
        ev = float("nan") if var_r == 0 else 1.0 - float((r - v).var()) / var_r
        return {"train/policy_gradient_loss": float(means[:, 0].mean()), "train/value_loss": float(means[:, 1].mean()),
                "train/entropy_loss": float(-entropy.mean()), "train/approx_kl": float(means[epoch_start:, 3].mean()),
                "train/clip_fraction": float(means[:, 2].mean()),
                "train/loss": float(means[-1, 0] - cfg.ent_coef * entropy[-1] + cfg.vf_coef * means[-1, 1]),
                "train/explained_variance": ev, "train/std": float(np.exp(log_std).mean()),
                "train/n_updates": self.n_updates, "train/learning_rate": lr, "train/clip_range": cfg.clip_range}

    def learn(self, total_timesteps: int, callback: Optional[Callable[[dict], None]] = None) -> list:
        """Alternates collect_rollout (n_steps of every env) and train until total_timesteps env-steps; returns one log
        dict per iteration (train/ logs plus the env's episode statistics of that collection under rollout/).  As in
        SB3, progress_remaining is updated after the collection, so update i of a run from 0 uses
        1 - i n_steps N / total_timesteps (the last one 0 when total_timesteps is a multiple of n_steps N)."""
        b, cfg = self.batch, self.cfg
        if self.num_timesteps == 0:
            b.reset()
        logs = []
        while self.num_timesteps < total_timesteps:
            b.reset_stats()
            ro = b.collect_rollout(cfg.n_steps, self.params.mlp(), gamma=cfg.gamma, gae_lambda=cfg.gae_lambda,
                                   tensor_cores=cfg.tensor_cores, bootstrap_truncated=True)
            self.num_timesteps += cfg.n_steps * b.num_envs
            self.progress_remaining = 1.0 - self.num_timesteps / total_timesteps
            log = {"rollout/" + k: v for k, v in b.stats_dict().items()}
            log.update(self.train(ro))
            log["time/total_timesteps"] = self.num_timesteps
            logs.append(log)
            if callback is not None:
                callback(log)
        return logs

"""Cost of gSDE exploration at 2^20 envs on one GPU, in one run:
  - collection: `collect_rollout(16, ...)` with the diagonal Gaussian, with gSDE (sde_sample_freq -1) and with gSDE
    resampled every 4 steps; two stream lanes, tensor_cores = 3 (what `PPOTrainer.learn` collects with); alternated,
    CUDA events around each whole call (policy, env steps, GAE) after a device synchronise; env-steps/s from the median;
  - the noise draw alone (`reset_noise`, r6_sde_noise over all envs);
  - r6_ppo_grad and r6_ppo_grad_sde on one 2^20-sample minibatch of a gSDE rollout (the same observations).
The card name, power limit and max SM clock are read with nvidia-smi in the same run.

    python profiles/sde_collection.py --out profiles/r05_sde_collection.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def timed(fn):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from rl_rocket_6dof_b200 import Rocket6DOFBatch
    from rl_rocket_6dof_b200.ppo import ActorCriticParams, loss_and_grad

    dev = "cuda:0"
    b = Rocket6DOFBatch(a.envs, device=dev, seed=0, lanes=2)
    b.reset()
    diag = ActorCriticParams.sb3_init(seed=0, device=dev)
    sde = ActorCriticParams.sb3_init(seed=0, device=dev, use_sde=True)
    cases = {"diag": (diag, -1), "sde_freq_-1": (sde, -1), "sde_freq_4": (sde, 4)}
    times = {c: [] for c in cases}
    for c, (p, f) in cases.items():           # warm-up
        b.collect_rollout(a.steps, p.mlp(), tensor_cores=3, sde_sample_freq=f)
    for _ in range(a.reps):
        for c, (p, f) in cases.items():
            times[c].append(timed(lambda: b.collect_rollout(a.steps, p.mlp(), tensor_cores=3, sde_sample_freq=f)))
    noise = [timed(b.reset_noise) for _ in range(20)][2:]
    ro = b.collect_rollout(a.steps, sde.mlp(), tensor_cores=3)
    idx = torch.randperm(a.steps * a.envs, device=dev)[: 1 << 20]
    grad = {}
    for name, p in (("r6_ppo_grad", diag), ("r6_ppo_grad_sde", sde)):
        loss_and_grad(p, ro, idx)
        grad[name] = [timed(lambda: loss_and_grad(p, ro, idx)) for _ in range(10)]
    res = dict(gpu=gpu_info(), envs=a.envs, steps=a.steps, lanes=2, tensor_cores=3, reps=a.reps,
               collect_ms=times, collect_median_ms={c: float(np.median(t)) for c, t in times.items()},
               env_steps_per_s={c: a.steps * a.envs / (float(np.median(t)) * 1e-3) for c, t in times.items()},
               noise_draw_ms=noise, noise_draw_median_ms=float(np.median(noise)),
               grad_minibatch=1 << 20, grad_ms=grad, grad_median_ms={k: float(np.median(v)) for k, v in grad.items()})
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()

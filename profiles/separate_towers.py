"""Shared trunk (net_arch [128, 64]) against SB3 1.6's separate towers (net_arch [dict(pi=[64, 64], vf=[64, 64])]) at
2^20 envs on one GPU, the two alternated in one run:
  - the policy kernel alone (r6_policy_ex, deterministic, value and log-prob written) in tensor_cores 0, 2 and 3: CUDA
    events around 20 back-to-back launches, per launch;
  - r6_ppo_grad on one 2^20-sample minibatch of a collected rollout;
  - `collect_rollout(16, ...)` on two stream lanes in mode 3 (what `PPOTrainer.learn` collects with).
Medians over `--reps` alternated repetitions.  The card name, power limit and max SM clock are read with nvidia-smi in
the same run.

    python profiles/separate_towers.py --out profiles/r06_separate_towers.json
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


def timed(fn, reps=1):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from rl_rocket_6dof_b200 import Rocket6DOFBatch
    from rl_rocket_6dof_b200.ppo import ActorCriticParams, loss_and_grad

    dev = "cuda:0"
    b = Rocket6DOFBatch(a.envs, device=dev, seed=0, lanes=2)
    b.reset()
    nets = {"shared": ActorCriticParams.sb3_init(seed=0, device=dev),
            "separate": ActorCriticParams.sb3_init(seed=0, device=dev, net_arch=[dict(pi=[64, 64], vf=[64, 64])])}
    ro = {k: b.collect_rollout(a.steps, p.mlp(), tensor_cores=3) for k, p in nets.items()}      # warm-up, rollouts
    idx = torch.randperm(a.steps * a.envs, device=dev)[: 1 << 20]
    pol = {f"{k}_tc{tc}": [] for k in nets for tc in (0, 2, 3)}
    grad = {k: [] for k in nets}
    coll = {k: [] for k in nets}
    for _ in range(a.reps):
        for k, p in nets.items():
            m = p.mlp()
            for tc in (0, 2, 3):
                b.policy_forward(m, tensor_cores=tc)
                pol[f"{k}_tc{tc}"].append(timed(lambda: b.policy_forward(m, tensor_cores=tc), 20))
            loss_and_grad(p, ro[k], idx)
            grad[k].append(timed(lambda: loss_and_grad(p, ro[k], idx)))
            coll[k].append(timed(lambda: b.collect_rollout(a.steps, m, tensor_cores=3)))
    med = lambda d: {k: float(np.median(v)) for k, v in d.items()}
    res = dict(gpu=gpu_info(), envs=a.envs, reps=a.reps,
               policy_forward_ms=pol, policy_forward_median_ms=med(pol),
               grad_minibatch=1 << 20, grad_ms=grad, grad_median_ms=med(grad),
               collect_steps=a.steps, collect_lanes=2, collect_tensor_cores=3, collect_ms=coll, collect_median_ms=med(coll),
               ratio_separate_over_shared={**{f"policy_tc{tc}": med(pol)[f"separate_tc{tc}"] / med(pol)[f"shared_tc{tc}"]
                                              for tc in (0, 2, 3)},
                                           "grad": med(grad)["separate"] / med(grad)["shared"],
                                           "collect": med(coll)["separate"] / med(coll)["shared"]})
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()

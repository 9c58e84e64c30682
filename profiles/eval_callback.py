"""Cost of one EvalCallback evaluation (montecarlo.run_episodes on a persistent one-episode batch, the gather to the
host, Monitor's rounding, the logs) beside the cost of one PPO iteration (32-step collection + update) in the same run.

Evaluations: 2^14, 2^16 and 2^20 eval episodes for the shared trunk and the separate towers, and 2^16 for the shared
trunk under VecNormalize; the policy kernel in mode 3 (tcgen05 3xTF32, the trainer's default), sb3_init parameters
(an untrained policy: the mean episode length is recorded beside each time, since the closed loop runs until the last
episode ends).  One warm-up evaluation, then the wall time of each of `--reps` evaluations between device
synchronizations; the env-steps the loop ran (it stops at the first chunk of 64 steps after which every env is
done) and, in a separate profiled evaluation, the kernels it launched.  Training: PPOTrainer.learn of 2^12, 2^16 and
2^20 envs x 32 steps, one warm-up iteration, then the wall time per iteration over `--reps` iterations.  Card name,
power limit and max SM clock from nvidia-smi in the same run.

    python profiles/eval_callback.py --out profiles/r11_eval.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

SEP = [dict(pi=[64, 64], vf=[64, 64])]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def _trainer(n, net_arch, vecnorm, dev, lanes):
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    from rl_rocket_6dof_b200.ppo import ActorCriticParams, PPOConfig, PPOTrainer
    from rl_rocket_6dof_b200.vec_normalize import VecNormalize
    env = Rocket6DOFBatch(n, device=dev, seed=42, lanes=lanes)
    params = ActorCriticParams.sb3_init(seed=42, device=dev, net_arch=net_arch)
    return PPOTrainer(env, params, PPOConfig(n_steps=32), seed=42, vec_normalize=VecNormalize(env) if vecnorm else None)


def time_eval(n, arch, vecnorm, reps, dev):
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    from rl_rocket_6dof_b200.evaluation import EvalCallback
    lanes = 2 if n >= 1 << 16 else 1
    tr = _trainer(1024, SEP if arch == "separate" else None, vecnorm, dev, 1)
    if vecnorm:
        tr.vec_normalize.reset()
    eb = Rocket6DOFBatch(n, device=dev, seed=1042, auto_reset=False, time_limit=True, split_step=True, lanes=lanes)
    cb = EvalCallback(eb, eval_freq=32)
    logs = cb.evaluate(tr)                      # warm-up
    times, lengths = [], [logs["eval/mean_ep_length"]]
    steps0 = eb.steps_done
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        logs = cb.evaluate(tr)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
        lengths.append(logs["eval/mean_ep_length"])
    steps = (eb.steps_done - steps0) / reps
    # kernel launches of one evaluation (CUDA activities of torch.profiler, a run of its own)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        cb.evaluate(tr)
        torch.cuda.synchronize()
    kernels = sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                  and "memcpy" not in e.name.lower() and "memset" not in e.name.lower())
    # the host part alone: Monitor's rounding, the order and the statistics of n episodes
    from rl_rocket_6dof_b200.evaluation import monitor_rewards, result_order, summarize
    r, l = np.random.default_rng(0).standard_normal(n), np.full(n, 700, np.int64)
    t0 = time.perf_counter()
    o = result_order(l)
    summarize(monitor_rewards(r)[o], l[o], np.zeros(n, bool))
    host = time.perf_counter() - t0
    return dict(episodes=n, net=arch, vecnormalize=vecnorm, lanes=lanes, eval_s=times, eval_s_median=float(np.median(times)),
                mean_ep_length=lengths, env_steps_run=steps, kernels_per_evaluation=kernels,
                kernels_per_step=kernels / steps, host_round_sort_stats_s=host)


def time_train(n, reps, dev):
    lanes = 2 if n >= 1 << 16 else 1
    tr = _trainer(n, None, False, dev, lanes)
    per = n * 32
    tr.learn(per)                               # warm-up iteration
    times = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        tr.learn(tr.num_timesteps + per)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    return dict(envs=n, n_steps=32, lanes=lanes, iteration_s=times, iteration_s_median=float(np.median(times)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="the JSON file to write")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    dev = "cuda:0"
    res = dict(gpu=gpu_info(), evaluations=[], training=[])
    for arch in ("shared", "separate"):
        for n in (1 << 14, 1 << 16, 1 << 20):
            res["evaluations"].append(time_eval(n, arch, False, a.reps, dev))
            print(json.dumps(res["evaluations"][-1]), flush=True)
    res["evaluations"].append(time_eval(1 << 16, "shared", True, a.reps, dev))
    print(json.dumps(res["evaluations"][-1]), flush=True)
    for n in (1 << 12, 1 << 16, 1 << 20):
        res["training"].append(time_train(n, a.reps, dev))
        print(json.dumps(res["training"][-1]), flush=True)
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

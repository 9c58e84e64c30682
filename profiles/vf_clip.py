"""The cost of SB3's value clipping (`clip_range_vf`) in the PPO gradient: r6_ppo_grad (shared trunk, separate towers)
and r6_ppo_grad_sde per 2^20-sample minibatch of a rollout collected from 2^20 envs x 16 steps (the obs trajectory
alone is 1.1 GB, far beyond the 126 MB L2), with clipping off and on alternated in one run after a warm-up of every
shape.  CUDA events around `--launches` back-to-back calls, per call; medians over `--reps` alternated repetitions.
The card name, power limit and max SM clock are read with nvidia-smi in the same run, and the ptxas registers / stack /
spills of the PPO gradient kernels are taken from the library's build log.

    python profiles/vf_clip.py --out profiles/r07_vf_clip.json
"""
import argparse
import json
import os
import re
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


def ptxas_info():
    """{kernel<flag>: 'R registers, S stack, L spill loads'} of the PPO gradient kernels from lib/build.log."""
    path = os.path.join(ROOT, "rl_rocket_6dof_b200", "lib", "build.log")
    if not os.path.exists(path):
        return "build.log not found"
    out, cur, stack = {}, None, None
    for line in open(path):
        m = re.search(r"Compiling entry function '\S*?(ppo_grad_(?:sep_|sde_)?kernel)ILb([01])E", line)
        if m:
            cur = f"{m.group(1)}<{'true' if m.group(2) == '1' else 'false'}>"
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            stack = m.groups()
        m = re.search(r"Used (\d+) registers", line)
        if m and cur:
            out[cur] = f"{m.group(1)} registers, {stack[0]} B stack, {stack[1]} B spill stores, {stack[2]} B spill loads"
            cur = None
    return out


def timed(fn, reps):
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
    ap.add_argument("--minibatch", type=int, default=1 << 20)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--launches", type=int, default=10)
    ap.add_argument("--clip-range-vf", type=float, default=0.2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    from rl_rocket_6dof_b200 import Rocket6DOFBatch
    from rl_rocket_6dof_b200.ppo import ActorCriticParams, loss_and_grad

    dev = "cuda:0"
    info = gpu_info()
    b = Rocket6DOFBatch(a.envs, device=dev, seed=0, lanes=2)
    nets = {"shared": ActorCriticParams.sb3_init(seed=0, device=dev),
            "separate": ActorCriticParams.sb3_init(seed=0, device=dev, net_arch=[dict(pi=[64, 64], vf=[64, 64])]),
            "gsde": ActorCriticParams.sb3_init(seed=0, device=dev, use_sde=True)}
    ro = {}
    for k, p in nets.items():
        b.reset()
        ro[k] = b.collect_rollout(a.steps, p.mlp(), tensor_cores=3)
        # old values spread around the critic's so that part of every minibatch is clipped
        g = torch.Generator(device=dev).manual_seed(1)
        ro[k]["values"] = (ro[k]["values"] + (torch.rand(ro[k]["values"].shape, generator=g, device=dev) - 0.5)
                           * (4 * a.clip_range_vf)).contiguous()
    idx = torch.randperm(a.steps * a.envs, device=dev, generator=torch.Generator(device=dev).manual_seed(0))[:a.minibatch]
    settings = {"off": {}, "on": dict(clip_range_vf=a.clip_range_vf)}
    call = {}
    for k, p in nets.items():
        for s, kw in settings.items():
            gs = torch.empty(p.flat.numel(), device=dev)
            call[(k, s)] = (lambda p=p, r=ro[k], kw=kw, gs=gs: loss_and_grad(p, r, idx, grad_sum=gs, **kw))
            call[(k, s)]()                                                         # warm-up
    times = {f"{k}_{s}": [] for k in nets for s in settings}
    for _ in range(a.reps):
        for k in nets:
            for s in settings:
                times[f"{k}_{s}"].append(timed(call[(k, s)], a.launches))
    med = {k: float(np.median(v)) for k, v in times.items()}
    res = dict(gpu=info, envs=a.envs, steps=a.steps, minibatch=a.minibatch, clip_range_vf=a.clip_range_vf,
               reps=a.reps, launches_per_rep=a.launches, ms_per_call=times, median_ms_per_call=med,
               ratio_on_over_off={k: med[f"{k}_on"] / med[f"{k}_off"] for k in nets},
               ptxas=ptxas_info())
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()

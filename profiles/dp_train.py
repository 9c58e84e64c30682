"""Weak scaling of data-parallel PPO training (PPOTrainer(..., group=...)): 2^20 envs per GPU, n_steps = 32, 4 global
minibatches, 5 epochs, the shared trunk and the separate towers.  Per iteration: collection time, update time and,
inside the update, the time of the two exchanges (advantage moments; gradient + terms gather and r6_rank_sum), split
out with CUDA events around them.  A duration is the max over ranks.  Rank 0 merges its result under the world size
into --out, so runs at 1, 2, 4 and 8 GPUs fill one file:

    torchrun --nproc-per-node {1,2,4,8} profiles/dp_train.py --out profiles/r09_dp_train.json
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
import torch.distributed as dist  # noqa: E402

SEP = [dict(pi=[64, 64], vf=[64, 64])]


def gpu_info(index):
    q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def timed(fn, spans):
    """fn wrapped so that every call records a pair of CUDA events into spans."""
    def wrapper(*a, **kw):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        out = fn(*a, **kw)
        e.record()
        spans.append((s, e))
        return out
    return wrapper


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1 << 20, help="envs per GPU")
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from rl_rocket_6dof_b200 import sharding
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    from rl_rocket_6dof_b200.ppo import ActorCriticParams, PPOConfig, PPOTrainer
    rank, local, world = sharding.env_world()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD
    try:
        gpu = gpu_info(local)
        res = {"world": world, "envs_per_gpu": args.envs, "n_steps": 32, "n_epochs": 5, "minibatches": 4, "gpu": gpu,
               "layouts": {}}
        n = args.envs
        for name, kw in (("shared", {}), ("separate", dict(net_arch=SEP))):
            env = Rocket6DOFBatch(n, device=dev, seed=1, lanes=2, **sharding.shard_batch_kwargs(n, rank, world))
            params = ActorCriticParams.sb3_init(seed=0, device=dev, **kw)
            cfg = PPOConfig(n_steps=32, n_epochs=5)
            tr = PPOTrainer(env, params, cfg, seed=0, group=group)
            spans = []
            if world > 1:
                tr._exchange_moments = timed(tr._exchange_moments, spans)
                tr._exchange_grad = timed(tr._exchange_grad, spans)
            env.reset()
            rows = []
            for it in range(args.warmup + args.iters):
                env.reset_stats()
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                spans.clear()
                ev[0].record()
                ro = env.collect_rollout(cfg.n_steps, params.mlp(), tensor_cores=cfg.tensor_cores, bootstrap_truncated=True)
                ev[1].record()
                tr.train(ro)
                ev[2].record()
                torch.cuda.synchronize()
                t = [ev[0].elapsed_time(ev[1]) * 1e-3, ev[1].elapsed_time(ev[2]) * 1e-3,
                     sum(s.elapsed_time(e) for s, e in spans) * 1e-3]
                t = [sharding.max_over_ranks(x, dev) for x in t]
                if it >= args.warmup:
                    rows.append(dict(collect_s=t[0], update_s=t[1], exchange_s=t[2], exchanges=len(spans)))
            med = {k: float(np.median([r[k] for r in rows])) for k in ("collect_s", "update_s", "exchange_s")}
            res["layouts"][name] = dict(iterations=rows, median=med)
            if rank == 0:
                print(name, json.dumps(med), flush=True)
            del env, tr, params, ro
            torch.cuda.empty_cache()
        if rank == 0 and args.out:
            data = {}
            if os.path.exists(args.out):
                with open(args.out) as f:
                    data = json.load(f)
            data.setdefault("runs", {})[str(world)] = res
            base = data["runs"].get("1")
            if base:
                data["weak_scaling_update_efficiency"] = {
                    w: {name: base["layouts"][name]["median"]["update_s"] / r["layouts"][name]["median"]["update_s"]
                        for name in r["layouts"]} for w, r in sorted(data["runs"].items())}
            with open(args.out, "w") as f:
                json.dump(data, f, indent=1)
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()

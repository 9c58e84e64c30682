"""Cost of bootstrapping TimeLimit truncations during PPO collection: `collect_rollout(k, ..., bootstrap_truncated=False)`
against `True`, alternated in one run, at 2^20 envs x 32 steps, two stream lanes, tensor_cores = 3 (what
`PPOTrainer.learn` collects with).  Three cases:
  (a) the default 1500-step TimeLimit on a pre-rolled batch whose step counts are spread over [0, 1500) before every
      rollout (scattered truncations, one slot layer);
  (b) a 16-step TimeLimit from reset(): every env truncates at steps 15 and 31 (two slot layers, the full mask);
  (c) time_limit=False (no slots: the flag must cost nothing).
Each call is timed with CUDA events around the whole collect_rollout (collection, value pass, bootstrap, GAE), after a
device synchronise.

    python profiles/bootstrap_overhead.py --out profiles/r04_bootstrap_overhead.json
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


def run_case(name, n, k, lanes, reps, mlp):
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    from rl_rocket_6dof_b200.params import derive_params, load_config
    sb3, cfg = load_config()
    ep = derive_params(cfg, sb3)
    if name == "b_full_mask":
        ep.max_episode_steps = 16
    env = Rocket6DOFBatch(n, params=ep, device="cuda", seed=3, lanes=lanes, time_limit=name != "c_no_time_limit")
    env.reset()
    if name == "a_scattered":
        env.step_policy(150, mlp)                   # a mid-training mix of episodes
        counts = torch.from_numpy(np.random.default_rng(0).integers(0, ep.max_episode_steps, n).astype(np.int32)).cuda()

    def prep():
        if name == "a_scattered":
            env.step_count.copy_(counts)           # ~k / 1500 of the envs truncate inside the rollout, anywhere in it
        else:
            env.reset()
        env.reset_stats()

    times = {False: [], True: []}
    truncs = {False: [], True: []}
    for r in range(reps + 1):                     # round 0 warms up both variants (allocator, modules)
        for boot in ((False, True) if r % 2 == 0 else (True, False)):
            prep()
            ms = timed(lambda: env.collect_rollout(k, mlp, tensor_cores=3, bootstrap_truncated=boot))
            if r > 0:
                times[boot].append(ms)
                truncs[boot].append(env.stats_dict()["truncated"])
    off, on = np.array(times[False]), np.array(times[True])
    limit = int(env._p.max_episode_steps)
    return {"max_episode_steps": limit, "slots": -(-k // limit) if limit else 0,
            "truncations_per_rollout": float(np.mean(truncs[True])),
            "off_ms": off.tolist(), "on_ms": on.tolist(),
            "off_median_ms": float(np.median(off)), "on_median_ms": float(np.median(on)),
            "overhead_median_ms": float(np.median(on) - np.median(off)),
            "overhead_median_pct": float(100 * (np.median(on) / np.median(off) - 1)),
            "off_spread_ms": float(off.max() - off.min()), "on_spread_ms": float(on.max() - on.min())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--lanes", type=int, default=2)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    from rl_rocket_6dof_b200.ppo import ActorCriticParams
    mlp = ActorCriticParams.sb3_init(0, "cuda").mlp()
    res = {"gpu": gpu_info(), "device": torch.cuda.get_device_name(), "envs": a.envs, "steps": a.steps, "lanes": a.lanes,
           "tensor_cores": 3, "reps": a.reps, "cases": {}}
    for name in ("a_scattered", "b_full_mask", "c_no_time_limit"):
        res["cases"][name] = c = run_case(name, a.envs, a.steps, a.lanes, a.reps, mlp)
        print(f"{name}: off {c['off_median_ms']:.3f} ms, on {c['on_median_ms']:.3f} ms, overhead "
              f"{c['overhead_median_ms']:.3f} ms ({c['overhead_median_pct']:+.2f} %), {c['truncations_per_rollout']:.0f} "
              f"truncations per rollout, spread off {c['off_spread_ms']:.3f} / on {c['on_spread_ms']:.3f} ms", flush=True)
    print(json.dumps({k: v for k, v in res.items() if k != "cases"}))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

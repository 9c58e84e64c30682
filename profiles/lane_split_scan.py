"""Joined step time of the 2-lane multi-pass step against the share of the envs given to lane 0 (launched first):
    python profiles/lane_split_scan.py [--envs N]        -> one JSON line"""
import argparse, json, os, sys
import torch

sys.path.insert(0, os.getcwd())
from rl_rocket_6dof_b200.batch import Rocket6DOFBatch

ap = argparse.ArgumentParser()
ap.add_argument("--envs", type=int, default=1 << 20)
ap.add_argument("--steps", type=int, default=200)
a = ap.parse_args()
n = a.envs
env = Rocket6DOFBatch(n, device="cuda:0", seed=42, lanes=2)
env.reset()
env.step_random(1024)
torch.cuda.synchronize()
res = {"envs": n}
for rep in range(2):
    for frac in (0.5, 0.52, 0.54, 0.56, 0.58, 0.62, 0.46):
        n0 = int(n * frac) // 1024 * 1024
        env.join()
        env._lane_ranges = [(0, n0), (n0, n - n0)]
        for _ in range(20):
            env.step_random(1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.steps):
            env.step_random(1)          # joins every step
        e1.record()
        torch.cuda.synchronize()
        res[f"{frac:.2f}_{rep}"] = round(e0.elapsed_time(e1) / a.steps * 1e3, 1)
print(json.dumps(res))

"""gSDE on SB3 1.6's separate towers: what it costs against the diagonal Gaussian on the same towers and against gSDE on
the shared trunk, at 2^20 envs, every case alternated with the others in one run after a warm-up of every shape.

  - the policy kernel per call, modes 0 / 2 / 3, stochastic: separate diagonal (r6_policy_range), separate gSDE
    (r6_policy_sde_sep_range) and shared gSDE (r6_policy_sde_range);
  - a 16-step collection on two lanes in mode 3: separate diagonal, separate gSDE at sde_sample_freq -1 and 4, shared gSDE;
  - the PPO gradient per 2^20-sample minibatch of a 2^20 x 16 rollout: r6_ppo_grad_sde_sep against r6_ppo_grad on the
    same towers and r6_ppo_grad_sde on the shared trunk.

CUDA events around `--launches` back-to-back calls (collections: one each), per call (the policy also at 10x the
launches, which shows whether the host keeps up); medians over `--reps` alternated
repetitions.  The card name, power limit and max SM clock are read with nvidia-smi in the same run, and the ptxas
registers / stack / spills of the policy and gradient kernels are taken from the library's build log.

    python profiles/sep_sde.py --out profiles/r08_sep_sde.json
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
    """{kernel: 'R registers, S stack, L spill loads'} of the policy and PPO gradient kernels from lib/build.log."""
    path = os.path.join(ROOT, "rl_rocket_6dof_b200", "lib", "build.log")
    if not os.path.exists(path):
        return "build.log not found"
    out, cur, stack = {}, None, None
    for line in open(path):
        m = re.search(r"Compiling entry function '\S*?\d((?:policy|ppo_grad)_\w*?kernel)(?:ILb([01])E)?", line)
        if m:
            cur = m.group(1) + ("" if m.group(2) is None else f"<{'true' if m.group(2) == '1' else 'false'}>")
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
    ap.add_argument("--launches", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    from rl_rocket_6dof_b200 import Rocket6DOFBatch
    from rl_rocket_6dof_b200.ppo import NET_ARCH_SEP, ActorCriticParams, loss_and_grad

    dev = "cuda:0"
    info = gpu_info()
    n = a.envs
    b = Rocket6DOFBatch(n, device=dev, seed=0, lanes=2)
    b.reset()
    nets = {"sep_diag": ActorCriticParams.sb3_init(seed=0, device=dev, net_arch=NET_ARCH_SEP),
            "sep_gsde": ActorCriticParams.sb3_init(seed=0, device=dev, use_sde=True, net_arch=NET_ARCH_SEP),
            "shared_gsde": ActorCriticParams.sb3_init(seed=0, device=dev, use_sde=True)}
    b.reset_noise()
    out = (torch.empty(n, 3, device=dev), torch.empty(n, 3, device=dev), torch.empty(n, device=dev), torch.empty(n, device=dev))

    # ---- policy kernel per call: the C entry points with prebuilt arguments, no Python work per launch but the ctypes
    # call itself (a few microseconds, against 0.1 ms and more of kernel), so the GPU runs ahead of the host ----
    import ctypes as C
    from rl_rocket_6dof_b200 import _lib
    L = _lib.load()
    ptrs = [o.data_ptr() for o in out]
    stream = torch.cuda.current_stream().cuda_stream
    pol = {}
    for k, p in nets.items():
        m = _lib.make_mlp(p.mlp())
        sde = _lib.R6Sde(p.log_std.data_ptr(), b.sde_xi.data_ptr()) if p.use_sde else None
        fn = L.r6_policy_sde_sep_range if p.separate else L.r6_policy_sde_range
        for mode in (0, 2, 3):
            if sde is None:
                pol[f"{k}_mode{mode}"] = (lambda m=m, mode=mode: L.r6_policy_range(C.byref(m), b.obs.data_ptr(), n, 0, n, mode, 1,
                                                                                 0, 0, 0, *ptrs, stream))
            else:
                pol[f"{k}_mode{mode}"] = (lambda m=m, sde=sde, fn=fn, mode=mode: fn(C.byref(m), C.byref(sde), b.obs.data_ptr(), n,
                                                                                  0, n, mode, 1, *ptrs, stream))
    for k, f in pol.items():                                       # every entry point accepts its arguments
        assert f() == 0, (k, L.r6_last_error())
    # ---- 16-step collection, two lanes, mode 3 ----
    col = {"sep_diag": (nets["sep_diag"], -1), "sep_gsde_freq-1": (nets["sep_gsde"], -1),
           "sep_gsde_freq4": (nets["sep_gsde"], 4), "shared_gsde_freq-1": (nets["shared_gsde"], -1)}
    coll = {k: (lambda p=p, f=f: b.collect_rollout(a.steps, p.mlp(), tensor_cores=3, sde_sample_freq=f))
            for k, (p, f) in col.items()}
    # ---- PPO gradient per minibatch ----
    ro = {}
    for k, p in nets.items():
        b.reset()
        ro[k] = b.collect_rollout(a.steps, p.mlp(), tensor_cores=3)
    idx = torch.randperm(a.steps * n, device=dev, generator=torch.Generator(device=dev).manual_seed(0))[:a.minibatch]
    grad = {}
    for k, p in nets.items():
        gs = torch.empty(p.flat.numel(), device=dev)
        grad[k] = (lambda p=p, r=ro[k], gs=gs: loss_and_grad(p, r, idx, grad_sum=gs))
    for fn in (*pol.values(), *coll.values(), *grad.values()):     # warm-up of every shape
        fn()
    times = {**{f"policy_{k}": [] for k in pol}, **{f"policy_{k}_x10": [] for k in pol}, **{f"collect_{k}": [] for k in coll}, **{f"grad_{k}": [] for k in grad}}
    for _ in range(a.reps):
        for k, fn in pol.items():
            times[f"policy_{k}"].append(timed(fn, a.launches))
            times[f"policy_{k}_x10"].append(timed(fn, 10 * a.launches))  # per call at 10x the launches: host-bound if it differs
        for k, fn in coll.items():
            times[f"collect_{k}"].append(timed(fn, 1))
        for k, fn in grad.items():
            times[f"grad_{k}"].append(timed(fn, max(a.launches // 4, 1)))
    med = {k: float(np.median(v)) for k, v in times.items()}
    res = dict(gpu=info, envs=n, steps=a.steps, minibatch=a.minibatch, reps=a.reps, launches_per_rep=a.launches,
               collection="collect_rollout(16, tensor_cores=3) on two lanes, one call per repetition (bootstrap off)",
               policy="r6_policy_range / r6_policy_sde_range / r6_policy_sde_sep_range, stochastic, all outputs written, "
                      "one launch per call; _x10: the same at 10x the launches per timing",
               ms_per_call=times, median_ms_per_call=med, ptxas=ptxas_info())
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()

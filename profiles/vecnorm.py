"""Cost of VecNormalize on the device: a 32-step collection of 2^20 envs on two stream lanes in mode 3 (the
tcgen05 3xTF32 policy, shared trunk, truncation bootstrap on), without VecNormalize, with observation normalization
only, and with observations and rewards, the three cases alternated for 7 repetitions (medians); and the CUDA-event
time of each r6_vn_* entry point at that size.  The card name, power limit and max SM clock are read with nvidia-smi
in the same run, and the ptxas report of the new kernels is taken from the library's build log.

    python profiles/vecnorm.py --out profiles/r10_vecnorm.json
"""
import argparse
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def ptxas_info():
    """{kernel: 'R registers, S stack, spills'} of the vn_* kernels from lib/build.log."""
    path = os.path.join(ROOT, "rl_rocket_6dof_b200", "lib", "build.log")
    if not os.path.exists(path):
        return "build.log not found"
    out, cur, stack = {}, None, None
    for line in open(path):
        m = re.search(r"(?:Compiling entry function|Function properties for) '?\S*?\d(vn_\w*?kernel)", line)
        if m:
            cur = m.group(1)
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            stack = m.groups()
        m = re.search(r"Used (\d+) registers(.*)", line)
        if m and cur and stack:
            out[cur] = f"{m.group(1)} registers{m.group(2)}, {stack[0]} B stack, {stack[1]} B spill stores, {stack[2]} B spill loads"
            cur, stack = None, None
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
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    from rl_rocket_6dof_b200 import _lib
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    from rl_rocket_6dof_b200.ppo import ActorCriticParams
    from rl_rocket_6dof_b200.vec_normalize import VecNormalize
    n, k, dev = a.envs, a.steps, "cuda:0"
    info = gpu_info()
    env = Rocket6DOFBatch(n, device=dev, seed=3, lanes=2)
    env.reset()
    mlp = ActorCriticParams.sb3_init(seed=0, device=dev).mlp()
    vns = {"obs": VecNormalize(env, norm_reward=False), "obs+reward": VecNormalize(env)}
    for vn in vns.values():
        vn.reset()
    cases = {"off": None, **vns}

    def collect(vn):
        env.collect_rollout(k, mlp, tensor_cores=3, bootstrap_truncated=True, vec_normalize=vn)

    for vn in cases.values():                          # warm-up: every shape of the timed window
        collect(vn)
    torch.cuda.synchronize()
    times = {c: [] for c in cases}
    for _ in range(a.reps):
        for c, vn in cases.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            collect(vn)
            torch.cuda.synchronize()
            times[c].append((time.perf_counter() - t0) * 1e3)
    coll = {c: dict(median_ms=float(np.median(v)), all_ms=[round(x, 3) for x in v]) for c, v in times.items()}
    for c in vns:
        coll[c]["extra_ms_per_step"] = (coll[c]["median_ms"] - coll["off"]["median_ms"]) / k

    # each entry point alone, CUDA events over `launches` calls, at the collection's size
    L, s = _lib.load(), torch.cuda.current_stream().cuda_stream
    vn = vns["obs+reward"]
    obs = env.obs.clone()
    out = torch.empty(13, 3, dtype=torch.float64, device=dev)
    work = torch.empty(int(L.r6_vn_moments_work_bytes(n, 13)), dtype=torch.uint8, device=dev)
    rms = vn.obs_rms.clone()
    hist = torch.empty(2, 2, 13, dtype=torch.float64, device=dev)
    dst = torch.empty_like(obs)
    rew = torch.randn(k, n, device=dev)
    done = (torch.rand(k, n, device=dev) < 0.01).to(torch.uint8)
    ret = torch.zeros(n, dtype=torch.float64, device=dev)
    rmom = torch.empty(k, 3, dtype=torch.float64, device=dev)
    rwork = torch.empty(int(L.r6_vn_ret_work_bytes(k, n)), dtype=torch.uint8, device=dev)
    rhist = torch.ones(k + 1, 2, 1, dtype=torch.float64, device=dev)
    rr = vn.ret_rms.clone()
    calls = {
        "r6_vn_moments (13 x 2^20)": lambda: L.r6_vn_moments(obs.data_ptr(), n, 13, 0, n, out.data_ptr(), work.data_ptr(), s),
        "r6_vn_update (1 step)": lambda: L.r6_vn_update(rms.data_ptr(), 13, out.data_ptr(), 1, 1e-8, hist.data_ptr(), s),
        "r6_vn_normalize (whole batch)": lambda: L.r6_vn_normalize(obs.data_ptr(), dst.data_ptr(), n, 0, n, hist.data_ptr(), 1,
                                                                  None, 2, 10.0, s),
        f"r6_vn_ret_moments ({k} x 2^20)": lambda: L.r6_vn_ret_moments(rew.data_ptr(), done.data_ptr(), k, n, ret.data_ptr(),
                                                                      0.99, rmom.data_ptr(), rwork.data_ptr(), s),
        f"r6_vn_update ({k} steps, ret_rms)": lambda: L.r6_vn_update(rr.data_ptr(), 1, rmom.data_ptr(), k,
                                                                     1e-8, rhist.data_ptr(), s),
        f"r6_vn_scale_rewards ({k} x 2^20)": lambda: L.r6_vn_scale_rewards(rew.data_ptr(), k, n, rhist.data_ptr(), 10.0, s),
    }
    kern = {}
    for name, fn in calls.items():
        fn()
        kern[name] = dict(ms_per_call=[round(timed(fn, a.launches), 5) for _ in range(3)])
        kern[name]["median_ms"] = float(np.median(kern[name]["ms_per_call"]))
    res = dict(gpu=info, envs=n, steps=k, lanes=2, tensor_cores=3, reps=a.reps, collection=coll, entry_points=kern,
               ptxas=ptxas_info(),
               note="collection: host clock around collect_rollout + synchronize, cases alternated, medians; entry points: "
                    "CUDA events over back-to-back launches: the 2^20-env observation block (58 MB) fits the 126 MB L2 and "
                    "is read from there after the first launch, the 32-step reward block (134 MB + 34 MB of dones) does not")
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

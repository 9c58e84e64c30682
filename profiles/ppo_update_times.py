"""Times of the PPO update on one GPU: r6_ppo_grad per minibatch size (with achieved FP32 FLOP/s against the FFMA peak
r6_peak_fma measures in the same run), the same loss and gradient by torch autograd in float32 (TF32 off, SB3's
arithmetic; TF32 on for context), one full iteration (collection | update) and a short learning curve from sb3_init.

    python profiles/ppo_update_times.py --out profiles/r03_ppo_update_times.json
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

# per sample: 10 112 MAC forward (13*128 + 128*64 + 64*4), 8 448 MAC backward data (64*4 + 64*128, rounded as stated)
# and 10 112 MAC of weight gradients -> 2 * 28 672 flop
FLOP_PER_SAMPLE = 2 * (10112 + 8448 + 10112)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def cuda_time(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def peak_ffma():
    import ctypes as C
    from rl_rocket_6dof_b200 import _lib
    L = _lib.load()
    sink = torch.zeros(1, dtype=torch.float64, device="cuda")
    blocks, iters = 148 * 64, 4096
    s = torch.cuda.current_stream().cuda_stream
    ms = cuda_time(lambda: _lib.check(L.r6_peak_fma(0, blocks, iters, C.c_void_p(sink.data_ptr()), C.c_void_p(s))), 5)
    return 2.0 * blocks * 256 * iters * 8 / (ms * 1e-3)


def synthetic_rollout(T, n, params, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    dev = "cuda"
    obs = torch.randn(T, n, 13, device=dev, generator=g)
    with torch.no_grad():
        mean, v = torch_forward(params, obs.reshape(-1, 13))
    act = mean + torch.randn(mean.shape, device=dev, generator=g) * torch.exp(params.log_std)
    return dict(obs=obs, actions=act.reshape(T, n, 3).contiguous(),
                log_probs=torch.randn(T, n, device=dev, generator=g) * 0.1 - 3.0,
                advantages=torch.randn(T, n, device=dev, generator=g), returns=v.reshape(T, n) + 1.0,
                values=v.reshape(T, n))


def torch_forward(p, x):
    h = torch.tanh(torch.tanh(x @ p.w0.T + p.b0) @ p.w1.T + p.b1)
    return h @ p.w2.T + p.b2, h @ p.wv + p.bv[0]


def torch_loss_grad(p, ro, idx, clip=0.2, vf=0.5):
    """SB3 1.6's PPO.train loss on one minibatch by autograd (float32)."""
    flat = p.flat.detach().requires_grad_(True)
    from rl_rocket_6dof_b200.ppo import ActorCriticParams
    q = ActorCriticParams.__new__(ActorCriticParams)
    o = 0
    for name, shape in (("w0", (128, 13)), ("b0", (128,)), ("w1", (64, 128)), ("b1", (64,)), ("w2", (3, 64)), ("b2", (3,)),
                        ("wv", (64,)), ("bv", (1,)), ("log_std", (3,))):
        size = int(np.prod(shape))
        setattr(q, name, flat[o:o + size].view(shape))
        o += size
    x = ro["obs"].reshape(-1, 13)[idx]
    mean, v = torch_forward(q, x)
    dist = torch.distributions.Normal(mean, torch.exp(q.log_std))
    logp = dist.log_prob(ro["actions"].reshape(-1, 3)[idx]).sum(1)
    adv = ro["advantages"].reshape(-1)[idx]
    adv = (adv - adv.mean()) / (adv.std() + 1e-8)
    ratio = torch.exp(logp - ro["log_probs"].reshape(-1)[idx])
    pg = -torch.min(adv * ratio, adv * torch.clamp(ratio, 1 - clip, 1 + clip)).mean()
    vl = torch.nn.functional.mse_loss(ro["returns"].reshape(-1)[idx], v)
    (pg + vf * vl).backward()
    return flat.grad


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--curve-iters", type=int, default=12)
    args = ap.parse_args()
    from rl_rocket_6dof_b200 import ppo
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    res = {"gpu": gpu_info(), "flop_per_sample": FLOP_PER_SAMPLE}
    res["ffma_peak_flops"] = peak_ffma()
    params = ppo.ActorCriticParams.sb3_init(0, "cuda")
    T, n = 32, 1 << 15
    ro = synthetic_rollout(T, n, params)
    rows = []
    for lb in range(14, 21):
        B = 1 << lb
        idx = torch.randperm(T * n, device="cuda")[:B]
        gs = torch.empty(ppo.NPARAMS, device="cuda")
        terms = torch.empty(5, dtype=torch.float64, device="cuda")
        work = torch.empty(int(ppo._lib.load().r6_ppo_work_bytes(B)), dtype=torch.uint8, device="cuda")
        ms = cuda_time(lambda: ppo.loss_and_grad(params, ro, idx, grad_sum=gs, terms=terms, work=work), 20)
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
        ms_t = cuda_time(lambda: torch_loss_grad(params, ro, idx), 10)
        torch.backends.cuda.matmul.allow_tf32 = True
        ms_tf = cuda_time(lambda: torch_loss_grad(params, ro, idx), 10)
        torch.backends.cuda.matmul.allow_tf32 = False
        gt = torch_loss_grad(params, ro, idx)
        rel = float((gs / B - gt).abs().max() / gt.abs().max())
        row = dict(B=B, ms=ms, samples_per_s=B / (ms * 1e-3), flops=FLOP_PER_SAMPLE * B / (ms * 1e-3),
                   torch_fp32_ms=ms_t, torch_tf32_ms=ms_tf, speedup_vs_torch_fp32=ms_t / ms,
                   max_rel_diff_vs_torch_fp32=rel)
        row["share_of_ffma_peak"] = row["flops"] / res["ffma_peak_flops"]
        rows.append(row)
        print(json.dumps(row), flush=True)
    res["grad"] = rows
    # one full iteration: 2^20 envs x 32 steps, 4 minibatches x 5 epochs
    env = Rocket6DOFBatch(1 << 20, device="cuda", seed=0)
    tr = ppo.PPOTrainer(env, params, ppo.PPOConfig(n_steps=32, n_epochs=5), seed=0)
    env.reset()
    it = []
    for k in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = env.collect_rollout(32, params.mlp())
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        tr.train(r)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        it.append(dict(collect_s=t1 - t0, update_s=t2 - t1))
        print(json.dumps(it[-1]), flush=True)
    res["iteration_2p20_envs_32_steps_4mb_5ep"] = it
    del env, tr, r
    torch.cuda.empty_cache()
    # learning curve from sb3_init: 2^16 envs x 32 steps per iteration, SB3 defaults otherwise
    env = Rocket6DOFBatch(1 << 16, device="cuda", seed=1)
    p2 = ppo.ActorCriticParams.sb3_init(1, "cuda")
    tr = ppo.PPOTrainer(env, p2, ppo.PPOConfig(n_steps=32), seed=1)
    curve = []
    tr.learn((1 << 16) * 32 * args.curve_iters, callback=lambda d: curve.append(
        {k: d[k] for k in ("time/total_timesteps", "rollout/episodes", "rollout/mean_return", "rollout/landing_rate",
                           "train/value_loss", "train/approx_kl", "train/clip_fraction", "train/std")}))
    for c in curve:
        print(json.dumps(c), flush=True)
    res["learning_curve_2p16_envs"] = curve
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

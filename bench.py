#!/usr/bin/env python
"""bench.py — 6DOF env-steps/s of the batched CUDA env step on N B200s (one process per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--envs E] [--impl b200|reference] [--dump-outputs DIR]

A "step" is one Rocket6DOF env-step for every env of the batch (workload: BASELINE.json configs[2],
2^20 envs per GPU, uniform random actions, auto-reset on).  Rank 0 prints ONE JSON line:
  value      whole-job env-steps/s, one Rocket6DOFBatch.step call per env-step, actions already in HBM, the outputs
             (obs / reward / done) ordered on the caller's stream after EVERY step (what a per-step consumer gets);
             `free_running` = the same K steps with the stream lanes joined only once at the end
  e2e        the same through Rocket6DOFVecEnv.step_host: pinned-host actions in, H2D copy, kernel,
             D2H copy of obs/reward/done/flags every step
  roofline   the step kernel against the measured FP64 FMA-pipe peak (bound "fp64"; the dynamics are
             not a contraction and sit above the HBM ridge) and roofline_hbm against MEASURED_PEAKS
  cpu_baseline  the CPU oracle (C restatement, all host threads) on a bounded sample of the workload
--impl reference times the UNMODIFIED reference env (baseline/_ref) under a SubprocVecEnv-protocol harness on the
host cores (the Python/SciPy port's and the C oracle's numbers are reported beside it).
--dump-outputs DIR writes what the last timed step returned (rank 0's envs) as DIR/<name>.npy, so that two builds run
with the same arguments (same seeds, same inputs) can be compared output for output.
"""
import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True        # the benchmark writes nothing into the tree it runs from (it may be read-only)

METRIC = "6dof_env_steps_per_sec"
UNIT = "env-steps/s"
F_FIX, F_ATT = 985.0, 1850.0          # algorithmic FP64 flops per env-step: 985 + 1850 * attempts (SURVEY §8d)
BYTES_PER_STEP = 336.0                # algorithmic HBM bytes per env-step (SURVEY §8d)
DUMP_ENVS = 1 << 19                   # --dump-outputs: 80 B per env (obs, reward, done, flags, index), 42 MB at most


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--envs", type=int, default=1 << 20, help="envs per GPU")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--preroll", type=int, default=1024,
                    help="untimed env-steps to reach the stationary mix of episode phases: all envs start their first episode "
                         "together and episodes last 143 +- 31 steps, so the step time keeps oscillating by +-4 %% with the "
                         "share of envs that finish per step until ~1000 steps in (profiles/r02_preroll_scan.txt)")
    ap.add_argument("--lanes", type=int, default=2, help="CUDA streams each GPU's env range is stepped on (r6_step_range)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample-envs", type=int, default=32768)
    ap.add_argument("--cpu-sample-steps", type=int, default=100)
    ap.add_argument("--ref-steps-per-worker", type=int, default=1000,
                    help="--impl reference: env-steps per worker process over the whole timed run (BASELINE.md §3)")
    ap.add_argument("--cpu-ref-steps", type=int, default=400,
                    help="cpu_baseline leg of the default run: VecEnv.step calls of the reference env per worker")
    ap.add_argument("--config4-envs", type=int, default=1 << 23,
                    help="envs per GPU of the BASELINE.json configs[3] leg (runs when WORLD_SIZE == 8; 0 = off)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write obs / reward / done / flags of the last timed step for a fixed, "
                         "seeded sample of at most %d envs (all envs below that), and their indices, as DIR/<name>.npy"
                         % DUMP_ENVS)
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return a


# ------------------------------------------------------------------------------------------------
def ncu_traffic(envs_per_launch):
    """dram__bytes_read.sum + dram__bytes_write.sum of one step_kernel launch, from the committed
    `ncu --set full` capture (profiles/step_kernel_traffic.json), scaled to this run's envs per launch."""
    p = os.path.join(ROOT, "profiles", "step_kernel_traffic.json")
    if not os.path.exists(p):
        return None, None
    with open(p) as f:
        d = json.load(f)
    per_env = (d["dram_bytes_read"] + d["dram_bytes_write"]) / d["envs_per_launch"]
    return per_env * envs_per_launch, d.get("source")


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "MEASURED_PEAKS.json"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "50"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None
        atexit.register(self._kill)          # a run that fails before stop() leaves no sampler behind

    def _kill(self):
        if self.p is not None and self.p.poll() is None:
            self.p.kill()

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 7:
                continue
            try:
                sm.append(float(c[0])); mx.append(float(c[1]))
            except ValueError:
                continue
            for nm, v in zip(names, c[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        self.f.close()
        os.unlink(self.f.name)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


def dump_outputs(out_dir, obs, reward, done, flags):
    """What one Rocket6DOFBatch.step returned (obs [14, N] float32, reward [N] float64, done / flags [N] uint8), for a
    fixed sample of the envs drawn with a fixed seed, as float32 / float64 .npy files: env_index [m] (float64),
    obs [m, 14] (float32), reward [m] (float64), done [m] and flags [m] (float32; flags keeps the bit field's value)."""
    import numpy as np
    import torch
    n = reward.shape[0]
    idx = np.arange(n) if n <= DUMP_ENVS else np.sort(np.random.default_rng(0).choice(n, DUMP_ENVS, replace=False))
    sel = torch.from_numpy(idx).to(reward.device)
    arrays = {"env_index": idx.astype(np.float64),
              "obs": obs[:, sel].t().cpu().numpy(),
              "reward": reward[sel].cpu().numpy(),
              "done": done[sel].to(torch.float32).cpu().numpy(),
              "flags": flags[sel].to(torch.float32).cpu().numpy()}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def cpu_oracle_throughput(n_envs, n_steps, threads):
    """C oracle (oracle/r6_oracle.c) on `threads` host threads: bounded sample of the same workload
    (random actions; finished envs are re-seeded with fresh initial conditions on the host)."""
    import numpy as np
    from oracle import c_oracle as co
    from rl_rocket_6dof_b200.params import derive_params, load_config
    sb3, cfg = load_config()
    ep = derive_params(cfg, sb3)
    rng = np.random.default_rng(0)

    def sample(m):
        ic = rng.uniform(ep.ic_low, ep.ic_high, (m, 14)).astype(np.float32)
        q = ic[:, 6:10]
        ic[:, 6:10] = q / np.sqrt((q * q).astype(np.float64).sum(1).astype(np.float32))[:, None]
        return ic
    ob = co.OracleBatch(ep, n_envs, nthreads=threads)
    ic = sample(n_envs)
    ob.set_state(ic.astype(np.float64), ic[:, 13], 0)
    acts = rng.uniform(-1, 1, (8, n_envs, 3)).astype(np.float32)
    ob.step(acts[0])
    t0 = time.perf_counter()
    for k in range(n_steps):
        o = ob.step(acts[k % 8])
        d = np.nonzero(o["done"])[0]
        if len(d):
            ic = sample(len(d))
            ob.set_state(ic.astype(np.float64), ic[:, 13], 0, idx=d)
    dt = time.perf_counter() - t0
    return n_envs * n_steps / dt


# ------------------------------------------------------------------------------------------------
def reference_throughput(vec_steps, warmup):
    """The reference's own CPU implementation of the path: the UNMODIFIED env from baseline/_ref under the
    SubprocVecEnv-protocol harness, one worker per host core (baseline/ref_arm.py; BASELINE.md §3).  Returns
    (result dict, kind); falls back to the Python/SciPy port (kind "port") only when baseline/_ref did not travel."""
    cores = os.cpu_count() or 1
    from baseline import ref_arm
    if ref_arm.available():
        return ref_arm.time_reference(cores, vec_steps, warmup), "reference"
    from oracle import subproc_vec_env as sv
    return sv.time_python_port(n_workers=cores, steps=vec_steps, warmup=warmup), "port"


def run_reference(args):
    """CPU arm (rank 0 only): `--steps K` bench steps, each a block of ceil(1000 / K) VecEnv.step calls over one
    single-env worker process per host core (so the run covers >= 1000 env-steps per worker, BASELINE.md §3), after
    max(50, W) untimed VecEnv.step calls."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    K = max(args.steps, 1)
    block = max(1, -(-args.ref_steps_per_worker // K))
    warm = max(50, args.warmup)
    line = {"impl": "reference", "metric": METRIC, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "gpu_launches": 0}
    res, kind = reference_throughput(K * block, warm)
    value = res["steps_per_s"]
    marks = res.get("marks")
    per_block = None
    if marks:
        import numpy as np
        t = np.asarray(marks)
        per_block = (cores * block / np.diff(t[::block])).tolist()          # env-steps/s of each bench step
    line.update(value=value, ms_per_step=1e3 * res["seconds"] / K,
                config={"workload": "Rocket6DOF config.yaml, uniform random actions, auto-reset, make_env() wrappers "
                                    "(main_6DOF.py:44-53); CPU SubprocVecEnv-protocol harness, one single-env worker "
                                    "process per host core; one bench step = %d VecEnv.step calls" % block,
                           "vec_steps_per_bench_step": block, "workers": cores, "warmup_vec_steps": warm,
                           "episodes_finished": res.get("episodes")},
                cpu_baseline={"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": res["sample"]},
                e2e={"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
    if per_block:
        line["per_step_values"] = {"min": min(per_block), "max": max(per_block), "median": statistics.median(per_block)}
    if not args.no_cpu_baseline:
        # beside it (not the arm's value): the restatements the parity tests use, on the same host cores
        try:
            from oracle import subproc_vec_env as sv
            py = sv.time_python_port(n_workers=cores, steps=200, warmup=20)
            line["cpu_baseline_python_port"] = {"value": py["steps_per_s"], "unit": UNIT, "cores": cores, "kind": "port",
                                                "sample": py["sample"]}
        except Exception as e:  # pragma: no cover
            line["python_port_error"] = repr(e)[:200]
        c_val = cpu_oracle_throughput(args.cpu_sample_envs, args.cpu_sample_steps, cores)
        line["cpu_baseline_c_oracle"] = {"value": c_val, "unit": UNIT, "cores": cores, "kind": "port",
                                         "sample": f"oracle/r6_oracle.c, {args.cpu_sample_envs} envs x "
                                                   f"{args.cpu_sample_steps} steps, pthreads"}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import ctypes as C
    from rl_rocket_6dof_b200 import _lib
    from rl_rocket_6dof_b200.vec_env import Rocket6DOFVecEnv

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from rl_rocket_6dof_b200 import sharding as _sharding
    numa_node = _sharding.bind_to_gpu_numa_node(local) if world > 1 else None    # before any pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    n = args.envs
    K, W = args.steps, max(args.warmup, 3)
    # index-range sharding: rank r owns global envs [r*n, (r+1)*n); no data-path collective
    vec = Rocket6DOFVecEnv(n, device=dev, seed=42, env_offset=rank * n, num_envs_global=world * n,
                           record_attempts=True, lanes=args.lanes)
    env = vec.batch
    L = env.lib
    env.reset()
    env.rollout(args.preroll)                      # untimed: steady-state mix of episode phases
    R = 8
    gen = torch.Generator(device=dev); gen.manual_seed(1234 + rank)
    acts = (torch.rand(R, n, 3, device=dev, generator=gen) * 2 - 1).contiguous()
    acts_h = acts.cpu().pin_memory()
    stream = torch.cuda.current_stream(dev)

    # ---- device-resident throughput: one r6_step launch per env-step -------------------------
    # With stream lanes the K steps run free on the lane streams (each lane forks from `stream` after e0) and are
    # joined back into `stream` before e1; the second measurement joins every step (outputs consumable per step).
    for w in range(W):
        env.step(acts[w % R], join=False)
    env.reset_stats()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    att_sum = torch.zeros((), dtype=torch.float64, device=dev)
    e0.record(stream)
    for k in range(K):
        env.step(acts[k % R], join=False)
    env.join()
    e1.record(stream)
    torch.cuda.synchronize()
    ms_free = max_over_ranks(e0.elapsed_time(e1))
    barrier()
    # headline: every step joined back into the caller's stream (outputs consumable per step)
    for w in range(W):
        env.step(acts[w % R])
    barrier()
    e0.record(stream)
    for k in range(K):
        env.step(acts[k % R])
    e1.record(stream)
    torch.cuda.synchronize()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, env.obs, env.reward, env.done, env.flags)
    barrier()
    ms_step = ms_total / K
    value = world * n * K / (ms_total * 1e-3)
    # realised RK attempts per env-step (sampled outside the timed region)
    for k in range(4):
        env.step(acts[k % R])
        att_sum += env.nattempts.to(torch.float64).mean()
    mean_att = float(att_sum) / 4
    stats = env.stats.clone()
    if world > 1:
        dist.all_reduce(stats)                     # the only collective: 8 doubles of episode statistics
    sd = env.stats_dict(stats)

    # ---- fused rollout kernel (k steps per launch, in-kernel Philox actions) -----------------
    env.rollout(K, fused=True)
    barrier()
    e0.record(stream)
    env.rollout(K, fused=True)
    e1.record(stream)
    torch.cuda.synchronize()
    ms_roll = max_over_ranks(e0.elapsed_time(e1))
    barrier()

    # ---- the same random-action rollout through the integrator | post-step kernel pair (r6_step_random) ----
    env.step_random(W)
    barrier()
    e0.record(stream)
    env.step_random(K)
    e1.record(stream)
    torch.cuda.synchronize()
    ms_rand = max_over_ranks(e0.elapsed_time(e1))
    barrier()

    # ---- optional float32 dynamics path (own error bound, tests/test_gpu_fp32.py): same workload ----
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    env32 = Rocket6DOFBatch(n, device=dev, seed=42, env_offset=rank * n, num_envs_global=world * n, precision="fp32",
                            record_attempts=True, lanes=args.lanes)
    env32.reset()
    env32.rollout(args.preroll)
    for w in range(W):
        env32.step(acts[w % R], join=False)
    env32.join()
    barrier()
    e0.record(stream)
    for k in range(K):
        env32.step(acts[k % R], join=False)
    env32.join()
    e1.record(stream)
    torch.cuda.synchronize()
    ms_f32 = max_over_ranks(e0.elapsed_time(e1))
    mean_att32 = float(env32.nattempts.to(torch.float64).mean())
    barrier()
    del env32

    # ---- fixed-policy closed loop: SB3 MlpPolicy actor fused into the rollout kernel ----------
    from rl_rocket_6dof_b200 import policy as _policy
    from rl_rocket_6dof_b200.batch import ACT_MLP, ACT_MLP_TC
    wpath = os.path.join(ROOT, "tests", "golden", "policy_cl.npz")
    if os.path.exists(wpath):
        wts, wsrc = _policy.load_npz(wpath), "best_model_2bo71j9m actor (tests/golden/policy_cl.npz)"
    else:
        g0 = np.random.default_rng(0)
        wts = {k: (g0.standard_normal(shp) * 0.1).astype(np.float32) for k, shp in _policy.SHAPES.items()}
        wsrc = "random-init actor of the same architecture"
    wdev = _policy.to_device(wts, dev)
    KP = max(K // 2, 1)
    env.rollout(KP, ACT_MLP, mlp=wdev)
    barrier()
    e0.record(stream)
    env.rollout(KP, ACT_MLP, mlp=wdev)
    e1.record(stream)
    torch.cuda.synchronize()
    ms_pol = max_over_ranks(e0.elapsed_time(e1))
    barrier()
    env.rollout(KP, ACT_MLP_TC, mlp=wdev)
    barrier()
    e0.record(stream)
    env.rollout(KP, ACT_MLP_TC, mlp=wdev)
    e1.record(stream)
    torch.cuda.synchronize()
    ms_pol_tc = max_over_ranks(e0.elapsed_time(e1))
    barrier()

    # closed loop as two kernels per env-step (r6_policy + r6_step): what a VecEnv consumer with the policy on
    # the device runs; 2 launches per step
    ms_two = {}
    ms_pol_kernel = {}
    for tc in (0, 1, 2, 3):
        env.step_policy(W, wdev, tensor_cores=tc)
        barrier()
        e0.record(stream)
        env.step_policy(K, wdev, tensor_cores=tc)
        e1.record(stream)
        torch.cuda.synchronize()
        ms_two[tc] = max_over_ranks(e0.elapsed_time(e1))
        barrier()
        e0.record(stream)
        for _ in range(K):
            env.policy_actions(wdev, tensor_cores=tc, out=env._policy_act)
        e1.record(stream)
        torch.cuda.synchronize()
        ms_pol_kernel[tc] = max_over_ranks(e0.elapsed_time(e1)) / K
        barrier()

    # PPO rollout collection on the device: stochastic Gaussian policy (tcgen05 mode) + value head + env step per
    # step, then the GAE scan — what SB3's collect_rollouts / compute_returns_and_advantage do on the host
    wac = dict(wts)
    if "wv" not in wac:
        g1 = np.random.default_rng(1)
        wac.update(wv=(g1.standard_normal(64) * 0.3).astype(np.float32), bv=np.zeros(1, np.float32),
                   log_std=np.array([-1.44, -2.07, -2.01], np.float32))
    wacd = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in wac.items()}
    KC = max(min(K, 32), 1)
    env.collect_rollout(KC, wacd, tensor_cores=3)          # also warms the allocator for the [KC, N, ...] buffers
    barrier()
    e0.record(stream)
    env.collect_rollout(KC, wacd, tensor_cores=3)
    e1.record(stream)
    torch.cuda.synchronize()
    ms_collect = max_over_ranks(e0.elapsed_time(e1))
    barrier()

    # ---- end to end through the VecEnv fast path (host actions in, host obs/reward/done out) --
    for w in range(W):
        vec.step_host(acts_h[w % R])
    barrier()
    e0.record(stream)
    for k in range(K):
        vec.step_host(acts_h[k % R])
    e1.record(stream)
    torch.cuda.synchronize()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    barrier()
    clocks = sampler.stop() if sampler else None
    e2e_value = world * n * K / (ms_e2e * 1e-3)
    h2d_bytes, d2h_bytes = vec.h2d_bytes_per_step, vec.d2h_bytes_per_step

    # ---- BASELINE.json configs[3]: 64 M envs sharded over 8 B200s (2^23 per GPU), NCCL episode-stat reduction ----
    config4 = None
    n4 = args.config4_envs
    if world == 8 and n4 > 0:
        del vec
        torch.cuda.empty_cache()
        env4 = Rocket6DOFBatch(n4, device=dev, seed=42, env_offset=rank * n4, num_envs_global=world * n4,
                               record_attempts=True, lanes=args.lanes)
        env4.reset()
        env4.rollout(args.preroll)
        acts4 = (torch.rand(2, n4, 3, device=dev, generator=gen) * 2 - 1).contiguous()
        for w in range(W):
            env4.step(acts4[w % 2])
        env4.reset_stats()
        barrier()
        K4 = max(K // 2, 4)
        e0.record(stream)
        for k in range(K4):
            env4.step(acts4[k % 2])
        e1.record(stream)
        torch.cuda.synchronize()
        ms4 = max_over_ranks(e0.elapsed_time(e1))
        att4 = float(env4.nattempts.to(torch.float64).mean())
        stats4 = env4.stats.clone()
        dist.all_reduce(stats4)                    # the NCCL episode-statistics reduction of config 4
        sd4 = env4.stats_dict(stats4)
        config4 = {"ms": ms4, "steps": K4, "mean_att": att4, "stats": sd4}
        barrier()
        del env4, acts4

    # ---- FP64 / FP32 FMA-pipe peak, measured here (MEASURED_PEAKS.json has none) -------------
    sink = torch.zeros(1, dtype=torch.float64, device=dev)
    peaks = {}
    for fp64 in (1, 0):
        blocks, iters = 148 * 8, 20000 if fp64 else 40000
        _lib.check(L.r6_peak_fma(fp64, blocks, 100, sink.data_ptr(), stream.cuda_stream), L)
        torch.cuda.synchronize()
        best = 0.0
        for _ in range(3):
            e0.record(stream)
            _lib.check(L.r6_peak_fma(fp64, blocks, iters, sink.data_ptr(), stream.cuda_stream), L)
            e1.record(stream)
            torch.cuda.synchronize()
            fl = 2.0 * blocks * 256 * iters * 8
            best = max(best, fl / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        peaks["fp64" if fp64 else "fp32"] = best

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    hbm_peak, hbm_src = measured_peaks()
    flops_step = F_FIX + F_ATT * mean_att
    per_gpu_steps_s = n / (ms_step * 1e-3)
    ach_tf = per_gpu_steps_s * flops_step / 1e12
    ach_gb = per_gpu_steps_s * BYTES_PER_STEP / 1e9
    traffic, traffic_src = ncu_traffic(n)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"configs[2]: {n} envs/GPU (2^{int(np.log2(n))}), config.yaml, uniform random actions "
                               f"U[-1,1] f32 resident in HBM, auto-reset on, make_env() wrappers fused",
                   "envs_per_gpu": n, "global_envs": world * n, "parallelism": f"index-range shards x{world}",
                   "l2": "per-step working set 336 B x envs = %.0f MB > 126 MB L2" % (n * 336 / 1e6),
                   "preroll_steps": args.preroll, "mean_rk_attempts": mean_att,
                   "stream_lanes": env.lanes, "multipass_integrator": env.work is not None,
                   "value_is": "joined every step: obs/reward/done are ordered on the caller's stream after each step",
                   "streams": (f"each step runs as {env.lanes} contiguous env sub-ranges on {env.lanes} CUDA streams "
                               "(r6_step_range), forked from and joined back into the timed stream around EVERY step"
                               if env.lanes > 1 else "one stream")},
        "gpu_launches": K * (4 if env.work is not None else 2 if env.scratch is not None else 1) * env.lanes,
        "roofline": {"bound": "fp64", "achieved": ach_tf, "peak": peaks["fp64"], "unit": "TFLOP/s",
                     "frac": ach_tf / peaks["fp64"], "traffic": traffic, "traffic_unit": "B/launch",
                     "traffic_source": traffic_src, "algorithmic_bytes_per_launch": BYTES_PER_STEP * n,
                     "note": "algorithmic flops/env-step = 985 + 1850 x RK attempts (SURVEY 8d) x envs per launch; "
                             "peak = DFMA micro-benchmark measured in this run (r6_peak_fma)",
                     "flops_per_env_step": flops_step,
                     "kernel": ((f"integrate_first_kernel + 2 x integrate_resume_kernel + post_kernel (r6_step with the multi-pass "
                                 f"integrator: four launches per lane, {env.lanes} lane(s)); launch_ms = the whole env-step")
                                if env.work is not None else
                                (f"integrate_kernel + post_kernel (r6_step as two launches per lane, {env.lanes} lane(s)); "
                                 "launch_ms = the whole env-step") if env.scratch is not None else "step_kernel"),
                     "launch_ms": ms_step},
        "free_running": {"value": world * n * K / (ms_free * 1e-3), "unit": UNIT, "ms_per_step": ms_free / K,
                         "what": "same K steps with the stream lanes left running and joined into the caller's stream "
                                 "once after the last step (outputs NOT ordered per step; not the headline)"},
        "roofline_hbm": {"bound": "hbm", "achieved": ach_gb, "peak": hbm_peak, "unit": "GB/s",
                         "frac": ach_gb / hbm_peak, "traffic": traffic, "peak_source": hbm_src,
                         "bytes_per_env_step": BYTES_PER_STEP},
        "peaks_measured": {"fp64_tflops": peaks["fp64"], "fp32_tflops": peaks["fp32"]},
        "rollout_fused": {"value": world * n * K / (ms_roll * 1e-3), "unit": UNIT, "ms_per_step": ms_roll / K,
                          "launches": 1, "actions": "in-kernel Philox4x32-10"},
        "rollout_split": {"value": world * n * K / (ms_rand * 1e-3), "unit": UNIT, "ms_per_step": ms_rand / K,
                          "launches": 2 * K, "actions": "in-kernel Philox4x32-10 (r6_step_random: integrator | post-step)"},
        "fp32_path": {"value": world * n * K / (ms_f32 * 1e-3), "unit": UNIT, "ms_per_step": ms_f32 / K, "dtype": "f32",
                      "mean_rk_attempts": mean_att32,
                      "roofline": {"bound": "fp32", "achieved": n / (ms_f32 / K * 1e-3) * (F_FIX + F_ATT * mean_att32) / 1e12,
                                   "peak": peaks["fp32"], "unit": "TFLOP/s",
                                   "frac": n / (ms_f32 / K * 1e-3) * (F_FIX + F_ATT * mean_att32) / 1e12 / peaks["fp32"]},
                      "bytes_per_env_step": 208.0,
                      "note": "R6_PREC_F32: float32 state + integrator, float64 reward/flags; bound stated in tests/test_gpu_fp32.py"},
        "rollout_policy": {"value": world * n * KP / (ms_pol * 1e-3), "unit": UNIT, "ms_per_step": ms_pol / KP,
                           "launches": 1, "actions": "fused MlpPolicy 13-128-64-3 tanh, fp32, deterministic",
                           "weights": wsrc},
        "rollout_policy_tensor_cores": {"value": world * n * KP / (ms_pol_tc * 1e-3), "unit": UNIT,
                                        "ms_per_step": ms_pol_tc / KP, "launches": 1,
                                        "actions": "same network as rollout_policy on mma.sync TF32 tiles, 3xTF32 "
                                                   "compensation, one warp = 32 envs, activations register-chained"},
        "closed_loop_two_kernels": {"value": world * n * K / (ms_two[0] * 1e-3), "unit": UNIT,
                                    "ms_per_step": ms_two[0] / K, "launches_per_step": 2,
                                    "actions": "r6_policy (float32 FMA network) then r6_step"},
        "closed_loop_two_kernels_tensor_cores": {"value": world * n * K / (ms_two[1] * 1e-3), "unit": UNIT,
                                                 "ms_per_step": ms_two[1] / K, "launches_per_step": 2,
                                                 "actions": "r6_policy (mma.sync TF32 tiles, 3xTF32) then r6_step"},
        "closed_loop_two_kernels_tcgen05": {"value": world * n * K / (ms_two[2] * 1e-3), "unit": UNIT,
                                            "ms_per_step": ms_two[2] / K, "launches_per_step": 2,
                                            "actions": "r6_policy (tcgen05.mma kind::tf32, accumulators and activations in TMEM, single-pass TF32: "
                                                       "|d action| ~1e-3) then r6_step"},
        "closed_loop_two_kernels_tcgen05_3xtf32": {"value": world * n * K / (ms_two[3] * 1e-3), "unit": UNIT,
                                                   "ms_per_step": ms_two[3] / K, "launches_per_step": 2,
                                                   "actions": "r6_policy (tcgen05.mma kind::tf32, activations in TMEM, 3xTF32 compensation in one TMEM "
                                                              "accumulator, float32-accurate tanh: |d action| <= 3e-6 vs the "
                                                              "reference's recorded actions) then r6_step — the faithful "
                                                              "closed loop on the 5th-generation tensor cores"},
        "policy_kernel_ms": {"fp32_fma": ms_pol_kernel[0], "mma_sync_3xtf32": ms_pol_kernel[1], "tcgen05_tf32": ms_pol_kernel[2],
                             "tcgen05_3xtf32": ms_pol_kernel[3], "envs": n},
        "ppo_collect_rollout": {"value": world * n * KC / (ms_collect * 1e-3), "unit": UNIT, "ms_per_step": ms_collect / KC,
                                "steps": KC, "what": "stochastic Gaussian policy + value head (r6_policy_ex, faithful tcgen05 3xTF32 mode), r6_step, "
                                                     "[T,N] buffers written on the device, then the GAE scan (r6_gae)"},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
                "d2h_bytes_per_step": d2h_bytes, "ms_per_step": ms_e2e / K,
                "api": "Rocket6DOFVecEnv.step_host (pinned host actions -> obs/reward/done on the host)"},
        "numa_node_rank0": numa_node,
        "config4": None if config4 is None else {
            "workload": f"configs[3]: {world} x {n4} = {world * n4} envs (2^{int(np.log2(world * n4))}), index-range shards, "
                        "uniform random actions resident in HBM, joined every step, NCCL all_reduce of the episode statistics",
            "value": world * n4 * config4["steps"] / (config4["ms"] * 1e-3), "unit": UNIT, "steps": config4["steps"],
            "ms_per_step": config4["ms"] / config4["steps"], "mean_rk_attempts": config4["mean_att"],
            "roofline_frac_fp64": n4 / (config4["ms"] / config4["steps"] * 1e-3) * (F_FIX + F_ATT * config4["mean_att"]) / 1e12 / peaks["fp64"],
            "episode_stats": {k: config4["stats"][k] for k in ("episodes", "mean_return", "mean_length", "landing_rate", "steps")}},
        "episode_stats": {k: sd[k] for k in ("episodes", "mean_return", "mean_length", "landing_rate", "steps")},
        "clocks": clocks,
    }
    if not args.no_cpu_baseline and world == 1:
        cores = os.cpu_count() or 1
        res, kind = reference_throughput(args.cpu_ref_steps, 50)
        line["cpu_baseline"] = {"value": res["steps_per_s"], "unit": UNIT, "cores": cores, "kind": kind,
                                "sample": res["sample"]}
        v = cpu_oracle_throughput(args.cpu_sample_envs, args.cpu_sample_steps, cores)
        line["cpu_baseline_c_oracle"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                         "sample": f"oracle/r6_oracle.c (C restatement), {args.cpu_sample_envs} envs x "
                                                   f"{args.cpu_sample_steps} steps of the same workload, pthreads"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)

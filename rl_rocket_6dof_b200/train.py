"""PPO training with deterministic evaluation and best-model checkpoints on the device: main_6DOF.py's
`model.learn(total_timesteps, callback=EvalCallback(...))` as a command.

    python -m rl_rocket_6dof_b200.train --out run/                       # one GPU
    torchrun --nproc-per-node 8 -m rl_rocket_6dof_b200.train --out run/  # data-parallel, one env shard per GPU
    python -m rl_rocket_6dof_b200.montecarlo --policy run/best_model.npz # the dispersion of the best model

Writes into --out: best_model.npz (the parameters of the best evaluation, `policy.load_npz` format), final_model.npz
(the last iterate), evaluations.npz (SB3's EvalCallback log), progress.csv (one row per iteration of the log dict) and,
with --vecnormalize, best_model_vecnormalize.npz / vecnormalize.npz (the statistics that go with each model; pass them
to the Monte-Carlo CLI's --vecnormalize).
"""
from __future__ import annotations

import csv
import os


def write_progress(path: str, logs: list):
    """SB3's CSV logger output for the log dicts so far: one column per key any row has (sorted), one row per
    iteration, empty where a row lacks the key (eval/ appears only on evaluating iterations)."""
    keys = sorted(set().union(*logs)) if logs else []
    with open(path, "w", newline="") as f:
        wr = csv.DictWriter(f, fieldnames=keys, restval="")
        wr.writeheader()
        wr.writerows(logs)


def main(argv=None) -> int:
    """`python -m rl_rocket_6dof_b200.train` — what `python main_6DOF.py` does in the reference: PPO(seed=42) with the
    reference's policy network, trained for sb3_config's total_timesteps while an EvalCallback keeps the best model."""
    import argparse

    import torch

    from . import sharding
    from .batch import Rocket6DOFBatch
    from .evaluation import EvalCallback
    from .params import load_config
    from .ppo import NET_ARCH_SEP, ActorCriticParams, PPOConfig, PPOTrainer
    from .vec_normalize import VecNormalize

    ap = argparse.ArgumentParser(description=main.__doc__)
    ap.add_argument("--config", default=None, help="config.yaml (default: the packaged reference configuration)")
    ap.add_argument("--total-timesteps", type=int, default=None, help="default: sb3_config's total_timesteps")
    ap.add_argument("--out", default="run", help="output directory")
    ap.add_argument("--seed", type=int, default=42, help="PPO(seed=...): parameters, minibatches and training envs")
    ap.add_argument("--envs", type=int, default=4096, help="training envs per rank")
    ap.add_argument("--lanes", type=int, default=1, help="stream lanes of the training and evaluation batches")
    ap.add_argument("--n-steps", type=int, default=32)
    ap.add_argument("--net-arch", choices=("shared", "separate"), default="shared",
                    help="shared: the reference's net_arch [128, 64]; separate: SB3 1.6's default towers")
    ap.add_argument("--use-sde", action="store_true")
    ap.add_argument("--vecnormalize", action="store_true", help="train inside VecNormalize (SB3 1.6 defaults)")
    ap.add_argument("--eval-freq", type=int, default=640, help="evaluate every this many vec-env steps (SB3's unit)")
    ap.add_argument("--n-eval-episodes", type=int, default=16384, help="episodes per evaluation (all ranks together)")
    ap.add_argument("--eval-seed", type=int, default=None,
                    help="seed of the evaluation envs' initial conditions (default: --seed + 1000)")
    ap.add_argument("--device", default=None, help="default: cuda:LOCAL_RANK")
    a = ap.parse_args(argv)

    rank, local_rank, world = sharding.env_world()
    dev = torch.device(a.device or f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    group = None
    if sharding.init_process_group(dev):
        import torch.distributed as dist
        group = dist.group.WORLD
    try:
        if a.n_eval_episodes % world:
            raise ValueError(f"--n-eval-episodes {a.n_eval_episodes} is not a multiple of the world size {world}")
        sb3_config, env_config = load_config(a.config)
        total = int(a.total_timesteps if a.total_timesteps is not None else float(sb3_config["total_timesteps"]))
        m = a.n_eval_episodes // world
        batch = Rocket6DOFBatch(a.envs, env_config, sb3_config, device=dev, seed=a.seed, lanes=a.lanes,
                                **sharding.shard_batch_kwargs(a.envs, rank, world))
        eval_batch = Rocket6DOFBatch(m, env_config, sb3_config, device=dev,
                                     seed=a.seed + 1000 if a.eval_seed is None else a.eval_seed, auto_reset=False,
                                     time_limit=True, split_step=True, lanes=min(a.lanes, m),
                                     **sharding.shard_batch_kwargs(m, rank, world))
        net_arch = NET_ARCH_SEP if a.net_arch == "separate" else [128, 64]
        params = ActorCriticParams.sb3_init(seed=a.seed, device=dev, use_sde=a.use_sde, net_arch=net_arch)
        vn = VecNormalize(batch, group=group) if a.vecnormalize else None
        trainer = PPOTrainer(batch, params, PPOConfig(n_steps=a.n_steps, use_sde=a.use_sde), seed=a.seed, group=group,
                             vec_normalize=vn)
        cb = EvalCallback(eval_batch, eval_freq=a.eval_freq, log_path=a.out, best_model_save_path=a.out, group=group)
        writer = rank == 0
        if writer:
            os.makedirs(a.out, exist_ok=True)
        logs = []

        def on_iteration(log):
            logs.append(log)
            if writer:
                write_progress(os.path.join(a.out, "progress.csv"), logs)
                if "eval/mean_reward" in log:
                    print(f"timesteps {log['time/total_timesteps']}: eval mean reward {log['eval/mean_reward']:.3f} "
                          f"(best {log['eval/best_mean_reward']:.3f}), landing rate {log['eval/landing_rate']:.3f}, "
                          f"mean length {log['eval/mean_ep_length']:.1f}", flush=True)

        trainer.learn(total, callback=on_iteration, eval_callback=cb)
        if writer:
            params.save_npz(os.path.join(a.out, "final_model.npz"))
            if vn is not None:
                vn.save(os.path.join(a.out, "vecnormalize.npz"))
            print(f"{trainer.num_timesteps} timesteps, {len(logs)} iterations, best eval mean reward "
                  f"{cb.best_mean_reward:.3f}; models in {a.out}")
    finally:
        if group is not None:
            import torch.distributed as dist
            dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    raise SystemExit(main())

"""Monte-Carlo landing dispersion, closed loop, on the GPU.

Restates /root/reference/montecarlo_script.py:33-81: run the trained policy deterministically for
`n_episodes` episodes from sampled initial conditions, and for each terminal state record
    final_position_error   = ||r||            final_velocity_error  = ||v||
    attitude_error         = 0.5 * deg(acos(q0))   angular_velocity_error = ||omega||
    "used mass"            = terminal_state[13]     (sic: the reference writes the remaining mass)
then print mean / standard deviation of every column.  Here every episode is its own environment:
`n_episodes` envs run in ONE fused rollout kernel per chunk of steps with the policy MLP evaluated
in-kernel (`R6_ACT_MLP`), one episode per env (`auto_reset=False`), no host round trip per step.
"""
from __future__ import annotations

import csv
from typing import Dict, Optional

import numpy as np
import torch

from .batch import SPLIT_MIN_ENVS, ACT_MLP, ACT_MLP_TC, Rocket6DOFBatch
from . import policy as _policy

HEADER = ["final_position_error", "final_velocity_error", "attitude_error", "angular_velocity_error", "used mass"]


def dispersion_columns(terminal_state: torch.Tensor) -> Dict[str, torch.Tensor]:
    """terminal_state: [14, N] float64 -> the five CSV columns of montecarlo_script.py:33-52."""
    ts = terminal_state
    return {
        HEADER[0]: ts[0:3].norm(dim=0),
        HEADER[1]: ts[3:6].norm(dim=0),
        HEADER[2]: 0.5 * torch.rad2deg(torch.acos(ts[6])),
        HEADER[3]: ts[10:13].norm(dim=0),
        HEADER[4]: ts[13],
    }


def run_montecarlo(n_episodes: int, weights: Dict[str, np.ndarray], env_config: Optional[dict] = None,
                   sb3_config: Optional[dict] = None, *, device="cuda", seed: Optional[int] = None,
                   chunk_steps: int = 128, csv_path: Optional[str] = None, ic_table: Optional[np.ndarray] = None,
                   env_offset: int = 0, num_envs_global: Optional[int] = None, tensor_cores: bool = False,
                   two_kernel: Optional[bool] = None, lanes: int = 1) -> dict:
    """Returns {"columns": {name: np.ndarray[n]}, "mean": {...}, "std": {...}, "episode_length", "episode_return",
    "landed", "stats"}.  `std` is the sample standard deviation (pandas' default, ddof=1).
    tensor_cores=True evaluates the policy on the tensor cores at float32 accuracy instead of with float32 FMAs.
    two_kernel (default: batches above 65536 episodes): the closed loop as policy kernel + env-step kernels per step
    (`step_policy`: tcgen05 3xTF32 policy when tensor_cores, multi-pass integrator, stream `lanes`) instead of the one
    fused rollout kernel — about twice the throughput for large dispersions, same one-episode semantics.  SB3 1.6's
    separate policy / value towers (weights with vf_w0 ...) always take the two-kernel path: the fused rollout kernel
    does not run that network."""
    if _policy.is_separate(weights):
        if two_kernel is False:
            raise ValueError("the separate policy / value towers have no fused rollout kernel: two_kernel must be True")
        two_kernel = True
    if two_kernel is None:
        two_kernel = n_episodes > SPLIT_MIN_ENVS
    env = Rocket6DOFBatch(n_episodes, env_config, sb3_config, device=device, seed=seed, auto_reset=False,
                          clip_reward=True, time_limit=True, ic_table=ic_table, env_offset=env_offset,
                          num_envs_global=num_envs_global, lanes=lanes if two_kernel else 1,
                          split_step=True if two_kernel else None)
    w = _policy.to_device(weights, env.device)
    env.reset()
    max_steps = int(env.params.max_episode_steps) if env.params.max_episode_steps else 1500
    steps = 0
    if two_kernel:
        chunk_steps = min(chunk_steps, 64)      # frozen envs still cost a policy launch: look for the end more often
    while steps < max_steps:
        if two_kernel:
            env.step_policy(chunk_steps, w, tensor_cores=3 if tensor_cores else 0)
        else:
            env.rollout(chunk_steps, ACT_MLP_TC if tensor_cores else ACT_MLP, mlp=w)
        steps += chunk_steps
        if bool(env.done.all()):        # one device->host byte per chunk, not per step
            break
    cols = dispersion_columns(env.terminal_state)
    out_cols = {k: v.cpu().numpy() for k, v in cols.items()}
    res = {
        "columns": out_cols,
        "mean": {k: float(np.mean(v)) for k, v in out_cols.items()},
        "std": {k: float(np.std(v, ddof=1)) if len(v) > 1 else 0.0 for k, v in out_cols.items()},
        "episode_return": env.ep_info[0].cpu().numpy(),
        "episode_length": env.ep_info[1].cpu().numpy().astype(np.int64),
        "landed": ((env.flags & 0xF8) == 0xF8).cpu().numpy(),
        "flags": env.flags.cpu().numpy(),
        "terminal_state": env.terminal_state.t().cpu().numpy(),
        "stats": env.stats_dict(),
    }
    if csv_path:
        with open(csv_path, "w", newline="") as f:
            wr = csv.writer(f)
            wr.writerow(HEADER)
            wr.writerows(zip(*[out_cols[h] for h in HEADER]))
    return res


def format_report(res: dict) -> str:
    """The lines montecarlo_script.py:74-81 prints."""
    return "\n".join(f"The {h} has mean:{res['mean'][h]} and standard deviation: {res['std'][h]}" for h in HEADER)


def main(argv=None) -> int:
    """`python -m rl_rocket_6dof_b200.montecarlo --policy best_model_2bo71j9m.zip` — what `python montecarlo_script.py`
    does in the reference (results_montecarlo.csv + the mean / std lines), for any number of episodes."""
    import argparse

    from .params import load_config
    ap = argparse.ArgumentParser(description=main.__doc__)
    ap.add_argument("--policy", required=True, help="SB3 model archive (.zip) or .npz with mlp_w0 .. mlp_b2")
    ap.add_argument("--episodes", type=int, default=30)
    ap.add_argument("--config", default=None, help="config.yaml (default: the packaged reference configuration)")
    ap.add_argument("--csv", default="results_montecarlo.csv")
    ap.add_argument("--seed", type=int, default=None)
    ap.add_argument("--device", default="cuda")
    ap.add_argument("--tensor-cores", action="store_true", help="evaluate the policy with the 3xTF32 MMA tiles")
    a = ap.parse_args(argv)
    w = _policy.load_npz(a.policy) if a.policy.endswith(".npz") else _policy.load_sb3_zip(a.policy)
    sb3_config, env_config = load_config(a.config)
    res = run_montecarlo(a.episodes, w, env_config, sb3_config, device=a.device, seed=a.seed, csv_path=a.csv,
                         tensor_cores=a.tensor_cores)
    print(format_report(res))
    print(f"episodes: {a.episodes}, landed: {int(res['landed'].sum())}, mean length {res['episode_length'].mean():.1f} steps")
    return 0


if __name__ == "__main__":
    raise SystemExit(main())

"""Closed-loop path on the GPU: policy MLP fused into the rollout kernel (R6_ACT_MLP), one-episode
(auto_reset = 0) semantics and the Monte-Carlo dispersion driver, against the closed-loop run the
unmodified reference produced with best_model_2bo71j9m (tests/golden/policy_cl.npz)."""
import os

import numpy as np
import pytest

from parity_utils import env_params, f32_ulp_diff

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "policy_cl.npz")


def _golden_episodes(g):
    starts = [int(s) for s in g["ic_step"]]
    ends = starts[1:] + [len(g["action"])]
    return starts, ends


def test_fused_mlp_actions_match_recorded():
    import torch
    from rl_rocket_6dof_b200 import policy
    from rl_rocket_6dof_b200.batch import ACT_MLP, Rocket6DOFBatch
    g = np.load(GOLD)
    w = policy.load_npz(GOLD)
    starts = set(int(s) for s in g["ic_step"])
    idx = np.array([k for k in range(1, len(g["action"])) if k not in starts])
    n = len(idx)
    ep = env_params()
    env = Rocket6DOFBatch(n, params=ep, device="cuda:0", auto_reset=True, seed=3)
    st = g["state"][idx - 1]
    env.set_state(torch.from_numpy(st.astype(np.float32)))
    env.state.copy_(torch.from_numpy(np.ascontiguousarray(st.T)))       # the float64 state the policy saw
    traj = env.rollout(1, ACT_MLP, mlp=policy.to_device(w, env.device), record=True)
    torch.cuda.synchronize()
    a = traj["act"][0].cpu().numpy()
    assert np.abs(a - g["action"][idx]).max() <= 2e-6
    obs = traj["obs"][0].t().cpu().numpy()
    assert f32_ulp_diff(obs, g["obs"][idx - 1][:, :13]).max() <= 1.0


def test_tensor_core_mlp_matches_cuda_core_mlp():
    """R6_ACT_MLP_TC (mma.sync TF32 tiles, 3xTF32 compensation) against the float32 CUDA-core network and the
    recorded reference actions, on every policy input of the golden closed-loop run; ragged batch size so
    that the last warp has lanes without an env."""
    import torch
    from rl_rocket_6dof_b200 import policy
    from rl_rocket_6dof_b200.batch import ACT_MLP, ACT_MLP_TC, Rocket6DOFBatch
    g = np.load(GOLD)
    w = policy.load_npz(GOLD)
    starts = set(int(s) for s in g["ic_step"])
    idx = np.array([k for k in range(1, len(g["action"])) if k not in starts])
    n = len(idx)
    assert n % 32 != 0
    ep = env_params()
    acts = {}
    for mode in (ACT_MLP, ACT_MLP_TC):
        env = Rocket6DOFBatch(n, params=ep, device="cuda:0", auto_reset=True, seed=3)
        st = g["state"][idx - 1]
        env.set_state(torch.from_numpy(st.astype(np.float32)))
        env.state.copy_(torch.from_numpy(np.ascontiguousarray(st.T)))
        traj = env.rollout(1, mode, mlp=policy.to_device(w, env.device), record=True)
        torch.cuda.synchronize()
        acts[mode] = traj["act"][0].cpu().numpy()
        if mode == ACT_MLP_TC:
            assert f32_ulp_diff(traj["obs"][0].t().cpu().numpy(), g["obs"][idx - 1][:, :13]).max() <= 1.0
            state_tc = env.state.clone()
        else:
            state_cc = env.state.clone()
    d = np.abs(acts[ACT_MLP_TC] - acts[ACT_MLP]).max()
    print(f"tensor-core vs CUDA-core policy: max |d action| = {d:.2e}; vs recorded: "
          f"{np.abs(acts[ACT_MLP_TC] - g['action'][idx]).max():.2e}")
    assert d <= 2e-6
    assert np.abs(acts[ACT_MLP_TC] - g["action"][idx]).max() <= 3e-6
    norm = torch.as_tensor(ep.state_normalizer, device="cuda")[:, None]
    assert float(((state_tc - state_cc).abs() / norm).max()) <= 1e-7      # one env-step downstream of the actions


@pytest.mark.parametrize("tensor_cores", [False, True])
def test_policy_kernel_and_two_kernel_closed_loop(tensor_cores):
    """r6_policy on the recorded observations, then r6_policy + r6_step chained == the fused rollout kernel."""
    import torch
    from rl_rocket_6dof_b200 import policy
    from rl_rocket_6dof_b200.batch import ACT_MLP, ACT_MLP_TC, Rocket6DOFBatch
    g = np.load(GOLD)
    w = policy.load_npz(GOLD)
    starts = set(int(s) for s in g["ic_step"])
    idx = np.array([k for k in range(1, len(g["action"])) if k not in starts])
    ep = env_params()
    env = Rocket6DOFBatch(len(idx), params=ep, device="cuda:0", seed=3)
    wd = policy.to_device(w, env.device)
    env.obs.copy_(torch.from_numpy(np.ascontiguousarray(g["obs"][idx - 1].T)))
    a = env.policy_actions(wd, tensor_cores=tensor_cores).cpu().numpy()
    assert np.abs(a - g["action"][idx]).max() <= 3e-6
    # closed loop, VecEnv semantics: 2k launches vs one fused launch, same seeds => same episodes
    n, k = 3000, 150
    x = Rocket6DOFBatch(n, params=ep, device="cuda:0", seed=17)
    y = Rocket6DOFBatch(n, params=ep, device="cuda:0", seed=17)
    x.reset(); y.reset()
    x.step_policy(k, wd, tensor_cores=tensor_cores)
    y.rollout(k, ACT_MLP_TC if tensor_cores else ACT_MLP, mlp=wd)
    torch.cuda.synchronize()
    assert torch.equal(x.episode_id, y.episode_id) and torch.equal(x.step_count, y.step_count)
    norm = torch.as_tensor(ep.state_normalizer, device="cuda")[:, None]
    # same network code in both kernels; nvcc may contract the surrounding arithmetic differently
    assert float(((x.state - y.state).abs() / norm).max()) <= 1e-6
    sx, sy = x.stats.cpu().numpy(), y.stats.cpu().numpy()
    assert np.array_equal(sx[[0, 2, 3, 4, 5, 6, 7]], sy[[0, 2, 3, 4, 5, 6, 7]])


def test_tcgen05_policy_fast_mode():
    """r6_policy tensor_cores = 2 (tcgen05.mma kind::tf32, accumulators and activations in TMEM, single pass): its own bound — TF32
    operands carry 2^-11 relative rounding, so actions agree with the float32 network to ~1e-3 (asserted 5e-3),
    ragged batch, and a closed loop driven by it has the same episode statistics to within sampling noise."""
    import torch
    from rl_rocket_6dof_b200 import policy
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    g = np.load(GOLD)
    w = policy.load_npz(GOLD)
    starts = set(int(s) for s in g["ic_step"])
    idx = np.array([k for k in range(1, len(g["action"])) if k not in starts])
    ep = env_params()
    env = Rocket6DOFBatch(len(idx), params=ep, device="cuda:0", seed=3)
    assert len(idx) % 128 != 0
    wd = policy.to_device(w, env.device)
    env.obs.copy_(torch.from_numpy(np.ascontiguousarray(g["obs"][idx - 1].T)))
    a2 = env.policy_actions(wd, tensor_cores=2).cpu().numpy()
    a0 = env.policy_actions(wd, tensor_cores=0).cpu().numpy()
    d = np.abs(a2 - a0)
    print(f"tcgen05 TF32 policy vs float32 network: max |d action| {d.max():.2e}, mean {d.mean():.2e}")
    assert d.max() <= 5e-3 and d.mean() <= 1e-3 and np.all(np.abs(a2) <= 1)
    # repeated launches (TMEM alloc / dealloc, barrier phases) are stable and deterministic
    for _ in range(3):
        assert np.array_equal(env.policy_actions(wd, tensor_cores=2).cpu().numpy(), a2)
    stats = {}
    for mode in (0, 2):
        x = Rocket6DOFBatch(8192, params=ep, device="cuda:0", seed=23)
        x.reset()
        x.step_policy(400, wd, tensor_cores=mode)
        torch.cuda.synchronize()
        stats[mode] = x.stats_dict()
    s0, s2 = stats[0], stats[2]
    print("closed loop fp32:", s0, "\nclosed loop tcgen05:", s2)
    assert abs(s0["episodes"] - s2["episodes"]) <= 0.01 * s0["episodes"]
    assert abs(s0["mean_length"] - s2["mean_length"]) <= 0.01 * s0["mean_length"]
    assert abs(s0["mean_return"] - s2["mean_return"]) <= 0.02 * abs(s0["mean_return"]) + 0.05


def test_tcgen05_policy_faithful_mode():
    """r6_policy tensor_cores = 3 (tcgen05.mma kind::tf32 with 3xTF32 error compensation, hi*hi + lo*hi + hi*lo in one TMEM
    accumulator, activations in TMEM, two tile groups per CTA handing an epilogue token back and forth — every batch size
    below must leave both groups with the same number of hand-overs): the reference's recorded closed-loop actions at the bar of the float32 FMA
    network (3e-6, montecarlo_script.py:57-64 via tests/golden/policy_cl.npz), ragged batches and env sub-ranges, repeated
    launches, and a closed loop with the same episodes as the float32 network."""
    import ctypes as C
    import torch
    from rl_rocket_6dof_b200 import _lib, policy
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    g = np.load(GOLD)
    w = policy.load_npz(GOLD)
    starts = set(int(s) for s in g["ic_step"])
    idx = np.array([k for k in range(1, len(g["action"])) if k not in starts])
    ep = env_params()
    env = Rocket6DOFBatch(len(idx), params=ep, device="cuda:0", seed=3)
    assert len(idx) % 256 != 0
    wd = policy.to_device(w, env.device)
    env.obs.copy_(torch.from_numpy(np.ascontiguousarray(g["obs"][idx - 1].T)))
    a3 = env.policy_actions(wd, tensor_cores=3).cpu().numpy()
    a0 = env.policy_actions(wd, tensor_cores=0).cpu().numpy()
    print(f"tcgen05 3xTF32 policy: max |d action| vs reference {np.abs(a3 - g['action'][idx]).max():.2e}, "
          f"vs float32 network {np.abs(a3 - a0).max():.2e}")
    assert np.abs(a3 - g["action"][idx]).max() <= 3e-6
    assert np.abs(a3 - a0).max() <= 3e-6 and np.all(np.abs(a3) <= 1)
    for _ in range(3):
        assert np.array_equal(env.policy_actions(wd, tensor_cores=3).cpu().numpy(), a3)
    # sizes around the tile (128) and tile-pair (256) boundaries, and an env sub-range of a larger batch
    rng = np.random.default_rng(0)
    for n in (1, 127, 128, 129, 255, 256, 257, 1000, 148 * 256 + 77):
        e = Rocket6DOFBatch(n, params=ep, device="cuda:0", seed=5)
        e.obs.copy_(torch.from_numpy(rng.uniform(-1, 1, (14, n)).astype(np.float32)))
        b3, b0 = e.policy_actions(wd, tensor_cores=3), e.policy_actions(wd, tensor_cores=0)
        assert float((b3 - b0).abs().max()) <= 3e-6, n
        assert float((e.policy_actions(wd, tensor_cores=2) - b0).abs().max()) <= 1e-2, n      # the fast mode of the same kernel
        if n >= 1000:
            m = _lib.make_mlp(wd)
            out = torch.full((n, 3), 7.0, device="cuda")
            first, count = 300, n - 555
            _lib.check(e.lib.r6_policy_range(C.byref(m), e.obs.data_ptr(), n, first, count, 3, 0, 0, 0, 0, out.data_ptr(), None,
                                             None, None, torch.cuda.current_stream().cuda_stream), e.lib)
            torch.cuda.synchronize()
            assert torch.equal(out[first:first + count], b3[first:first + count])
            assert bool((out[:first] == 7).all()) and bool((out[first + count:] == 7).all())
    stats = {}
    for mode in (0, 3):
        x = Rocket6DOFBatch(8192, params=ep, device="cuda:0", seed=23)
        x.reset()
        x.step_policy(300, wd, tensor_cores=mode)
        torch.cuda.synchronize()
        stats[mode] = (x.stats_dict(), x.episode_id.clone(), x.step_count.clone())
    # float32 feedback amplifies 1e-6 action differences slowly: after 300 steps almost every env is still in step
    same = (stats[0][1] == stats[3][1]) & (stats[0][2] == stats[3][2])
    assert float(same.float().mean()) > 0.995
    assert abs(stats[0][0]["episodes"] - stats[3][0]["episodes"]) <= 0.002 * stats[0][0]["episodes"] + 2


def test_tcgen05_policy_full_size_1m_envs():
    """The size the closed-loop bench runs at: 2^20 envs whose observations come from 64 closed-loop steps (every phase of
    an episode present), both tcgen05 modes against the float32 FMA network — 148 CTAs x 2 tile groups x 28 tile slots, the
    last slot of the second group past the end of the batch."""
    import torch
    from rl_rocket_6dof_b200 import policy
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    n = (1 << 20) - 77
    env = Rocket6DOFBatch(n, params=env_params(), device="cuda:0", seed=9)
    wd = policy.to_device(policy.load_npz(GOLD), env.device)
    env.reset()
    env.step_policy(64, wd, tensor_cores=3)
    a0 = env.policy_actions(wd, tensor_cores=0)
    a3 = env.policy_actions(wd, tensor_cores=3)
    a2 = env.policy_actions(wd, tensor_cores=2)
    torch.cuda.synchronize()
    d3, d2 = float((a3 - a0).abs().max()), float((a2 - a0).abs().max())
    print(f"2^20 envs: tcgen05 3xTF32 vs float32 network {d3:.2e}, single-pass TF32 {d2:.2e}")
    assert d3 <= 3e-6 and d2 <= 1e-2
    assert bool((a3.abs() <= 1).all()) and bool(torch.isfinite(a3).all())


def test_rollout_mlp_needs_weights():
    from rl_rocket_6dof_b200._lib import R6Error
    from rl_rocket_6dof_b200.batch import ACT_MLP, Rocket6DOFBatch
    env = Rocket6DOFBatch(8, params=env_params(), device="cuda:0")
    env.reset()
    with pytest.raises(ValueError):
        env.rollout(1, ACT_MLP)
    import ctypes as C
    rc = env.lib.r6_rollout(C.byref(env._p), C.byref(env._b), 8, 0, 1, ACT_MLP, None, None, 0, 0, None, None, None,
                            None, None)
    assert rc == -1 and b"policy weights" in env.lib.r6_last_error()
    assert R6Error is not None


@pytest.mark.parametrize("two_kernel,tensor_cores,lanes", [(True, False, 1), (True, True, 2)])
def test_montecarlo_two_kernel_closed_loop_matches_reference_and_fused(two_kernel, tensor_cores, lanes):
    """Monte-Carlo dispersion (montecarlo_script.py:54-64) through the policy kernel + env-step kernels (one-episode
    semantics in the split step path: finished envs stay frozen): the reference's 30 recorded closed-loop episodes at
    the bars of the fused rollout kernel, and a 70 000-episode dispersion equal to the fused kernel's (same Philox
    initial conditions) up to the amplification of float32 round-off in the actions."""
    from rl_rocket_6dof_b200 import montecarlo, policy
    g = np.load(GOLD)
    w = policy.load_npz(GOLD)
    starts, ends = _golden_episodes(g)
    n = len(starts)
    res = montecarlo.run_montecarlo(n, w, device="cuda:0", ic_table=g["ic"], chunk_steps=64, tensor_cores=tensor_cores,
                                    two_kernel=two_kernel, lanes=lanes)
    ref_len = np.array([e - s for s, e in zip(starts, ends)])
    ref_term = np.stack([g["state"][e - 1] for e in ends])
    assert np.abs(res["episode_length"] - ref_len).max() <= 1
    same = res["episode_length"] == ref_len
    assert same.mean() >= 0.8
    assert (np.abs(res["terminal_state"] - ref_term) / env_params().state_normalizer)[same].max() <= 2e-3
    assert res["stats"]["episodes"] == n and res["stats"]["steps"] == res["episode_length"].sum()
    big = 70_000
    a = montecarlo.run_montecarlo(big, w, device="cuda:0", seed=5, tensor_cores=tensor_cores, two_kernel=True, lanes=lanes)
    b = montecarlo.run_montecarlo(big, w, device="cuda:0", seed=5, tensor_cores=tensor_cores, two_kernel=False)
    assert a["stats"]["episodes"] == b["stats"]["episodes"] == big
    same = a["episode_length"] == b["episode_length"]
    print(f"two-kernel vs fused Monte Carlo, {big} episodes: identical lengths {same.mean():.4f}, landed "
          f"{a['landed'].mean():.4f} / {b['landed'].mean():.4f}")
    assert same.mean() > 0.97 and np.abs(a["episode_length"] - b["episode_length"]).max() <= 2
    assert a["stats"]["steps"] == a["episode_length"].sum()
    for k in a["mean"]:
        assert abs(a["mean"][k] - b["mean"][k]) <= 2e-3 * abs(b["mean"][k]) + 1e-6, k
        assert abs(a["std"][k] - b["std"][k]) <= 5e-3 * abs(b["std"][k]) + 1e-6, k


@pytest.mark.parametrize("tensor_cores", [False, True])
def test_closed_loop_montecarlo_matches_reference_episodes(tmp_path, tensor_cores):
    """30 episodes from the reference's own initial conditions, policy in the loop on both sides.
    The loop feeds a float32 network back into the dynamics, so agreement is to the amplification of
    float32 round-off in the actions (SURVEY §7 hard part 8), not to 1e-9: episode lengths within one
    step, terminal states within 2e-3 of the normaliser, dispersion means within 1 %."""
    from rl_rocket_6dof_b200 import montecarlo, policy
    g = np.load(GOLD)
    w = policy.load_npz(GOLD)
    starts, ends = _golden_episodes(g)
    n = len(starts)
    assert g["done"][ends[-1] - 1] or g["truncated"][ends[-1] - 1]
    csv_path = str(tmp_path / "results_montecarlo.csv")
    res = montecarlo.run_montecarlo(n, w, device="cuda:0", ic_table=g["ic"], csv_path=csv_path, chunk_steps=64,
                                    tensor_cores=tensor_cores)
    ref_len = np.array([e - s for s, e in zip(starts, ends)])
    ref_term = np.stack([g["state"][e - 1] for e in ends])
    print("episode length diff:", res["episode_length"] - ref_len)
    assert np.abs(res["episode_length"] - ref_len).max() <= 1
    norm = env_params().state_normalizer
    err = np.abs(res["terminal_state"] - ref_term) / norm
    print("terminal state error / normaliser: max", err.max(0))
    same = res["episode_length"] == ref_len
    assert same.mean() >= 0.8
    assert err[same].max() <= 2e-3
    # dispersion statistics (what montecarlo_script.py prints)
    ref_cols = {
        "final_position_error": np.linalg.norm(ref_term[:, 0:3], axis=1),
        "final_velocity_error": np.linalg.norm(ref_term[:, 3:6], axis=1),
        "attitude_error": 0.5 * np.rad2deg(np.arccos(ref_term[:, 6])),
        "angular_velocity_error": np.linalg.norm(ref_term[:, 10:13], axis=1),
        "used mass": ref_term[:, 13],
    }
    for k, v in ref_cols.items():
        assert abs(res["mean"][k] - v.mean()) <= 0.01 * abs(v.mean()) + 1e-6, k
        assert abs(res["std"][k] - v.std(ddof=1)) <= 0.05 * abs(v.std(ddof=1)) + 1e-6, k
    rows = open(csv_path).read().strip().splitlines()
    assert rows[0].split(",") == montecarlo.HEADER and len(rows) == n + 1
    assert "final_position_error has mean" in montecarlo.format_report(res)
    assert res["stats"]["episodes"] == n


def test_montecarlo_cli(tmp_path, capsys):
    from rl_rocket_6dof_b200 import montecarlo
    out = str(tmp_path / "mc.csv")
    assert montecarlo.main(["--policy", GOLD, "--episodes", "64", "--csv", out, "--device", "cuda:0", "--seed", "3"]) == 0
    text = capsys.readouterr().out
    assert "The final_position_error has mean:" in text and "episodes: 64" in text
    assert len(open(out).read().strip().splitlines()) == 65


def test_one_episode_rollout_freezes_finished_envs():
    import torch
    from rl_rocket_6dof_b200.batch import ACT_PHILOX, Rocket6DOFBatch
    n = 512
    env = Rocket6DOFBatch(n, params=env_params(), device="cuda:0", auto_reset=False, seed=11)
    env.reset()
    for _ in range(8):
        env.rollout(64, ACT_PHILOX)
    torch.cuda.synchronize()
    assert bool(env.done.all())                     # random-action episodes last 99-211 steps
    s = env.stats.cpu().numpy()
    assert s[0] == n and s[7] == s[2]               # one episode per env; steps == sum of lengths
    snap = (env.state.clone(), env.terminal_state.clone(), env.step_count.clone(), env.stats.clone())
    env.rollout(64, ACT_PHILOX)
    torch.cuda.synchronize()
    for a, b in zip(snap, (env.state, env.terminal_state, env.step_count, env.stats)):
        assert torch.equal(a, b)
    assert torch.equal(env.state, env.terminal_state)
    env.reset()                                     # un-freezes
    env.rollout(4, ACT_PHILOX)
    torch.cuda.synchronize()
    assert int(env.step_count.min()) == 4 and not bool(env.done.any())


def _actor_critic_weights():
    from rl_rocket_6dof_b200 import policy
    w = policy.load_npz(GOLD)
    rng = np.random.default_rng(5)
    w["wv"] = (rng.standard_normal(64) * 0.3).astype(np.float32)       # the fixture holds the actor only
    w["bv"] = np.array([0.7], np.float32)
    w["log_std"] = np.array([-0.5, -1.0, 0.2], np.float32)
    return w


@pytest.mark.parametrize("tensor_cores,tol", [(0, 3e-6), (1, 5e-6), (2, 1e-2), (3, 5e-6)])
def test_actor_critic_forward_value_and_gaussian_sampling(tensor_cores, tol):
    """r6_policy_ex: value head on the shared latent, Gaussian sampling with Philox noise, SB3's log-probability."""
    import torch
    from rl_rocket_6dof_b200 import policy
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    g = np.load(GOLD)
    w = _actor_critic_weights()
    n = 8739
    env = Rocket6DOFBatch(n, params=env_params(), device="cuda:0", seed=31)
    wd = {k: torch.from_numpy(v).cuda() for k, v in w.items()}
    x = g["obs"][:n, :13]
    env.obs[:13].copy_(torch.from_numpy(np.ascontiguousarray(x.T)))
    mean_ref, val_ref = policy.forward_full_numpy(w, x)
    # deterministic: action = clipped mean, log-prob of the mean, value
    a, raw, v, lp = (t.cpu().numpy() for t in env.policy_forward(wd, stochastic=False, tensor_cores=tensor_cores))
    assert np.abs(raw - mean_ref).max() <= tol and np.abs(v - val_ref).max() <= 4 * tol
    assert np.array_equal(a, np.clip(raw, -1, 1))
    assert np.allclose(lp, -(w["log_std"].sum() + 3 * 0.9189385332046727), atol=1e-5)
    # stochastic: eps = (raw - mean) / std is standard normal, log-prob is SB3's formula, streams are reproducible
    a, raw, v, lp = (t.cpu().numpy() for t in env.policy_forward(wd, stochastic=True, tensor_cores=tensor_cores, step_index=7))
    std = np.exp(w["log_std"])
    eps = (raw - mean_ref) / std
    if tensor_cores != 2:
        ref_lp = (-0.5 * eps.astype(np.float64) ** 2 - w["log_std"] - 0.9189385332046727).sum(1)
        assert np.abs(lp - ref_lp).max() <= 2e-3
    assert abs(eps.mean()) < 0.02 and abs(eps.std() - 1) < 0.02
    assert abs(np.corrcoef(eps[:, 0], eps[:, 1])[0, 1]) < 0.04 and abs(np.corrcoef(eps[:-1, 2], eps[1:, 2])[0, 1]) < 0.04
    assert (np.abs(eps) > 3).mean() < 0.006
    a2, raw2, _, _ = (t.cpu().numpy() for t in env.policy_forward(wd, stochastic=True, tensor_cores=tensor_cores, step_index=7))
    assert np.array_equal(raw, raw2)
    _, raw3, _, _ = (t.cpu().numpy() for t in env.policy_forward(wd, stochastic=True, tensor_cores=tensor_cores, step_index=8))
    assert not np.array_equal(raw, raw3)


def test_collect_rollout_on_device():
    """collect_rollout = policy_forward + step per env-step, then the GAE scan; checked against the pieces."""
    import torch
    from oracle import gae_oracle
    from rl_rocket_6dof_b200 import policy
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    w = _actor_critic_weights()
    wd = {k: torch.from_numpy(v).cuda() for k, v in w.items()}
    n, k = 2048, 48
    env = Rocket6DOFBatch(n, params=env_params(), device="cuda:0", seed=3)
    env.reset()
    ro = env.collect_rollout(k, wd, gamma=0.99, gae_lambda=0.95, stochastic=True)
    torch.cuda.synchronize()
    assert ro["obs"].shape == (k, n, 13) and ro["actions"].shape == (k, n, 3) and ro["advantages"].shape == (k, n)
    mean, val = policy.forward_full_numpy(w, ro["obs"].cpu().numpy().reshape(-1, 13))
    assert np.abs(val.reshape(k, n) - ro["values"].cpu().numpy()).max() <= 2e-5
    eps = (ro["actions"].cpu().numpy().reshape(-1, 3) - mean) / np.exp(w["log_std"])
    assert abs(eps.mean()) < 0.01 and abs(eps.std() - 1) < 0.01
    adv, ret = gae_oracle.compute_returns_and_advantage(ro["rewards"].cpu().numpy(), ro["values"].cpu().numpy(),
                                                        ro["dones"].cpu().numpy() != 0, ro["last_values"].cpu().numpy(),
                                                        0.99, 0.95)
    assert np.array_equal(adv, ro["advantages"].cpu().numpy()) and np.array_equal(ret, ro["returns"].cpu().numpy())
    assert float(env.stats[7]) == n * k


@pytest.mark.gpu
@pytest.mark.parametrize("lanes,auto_reset", [(1, True), (2, True), (1, False), (2, False)])
def test_collect_rollout_in_place_trajectory_equals_step_by_step(lanes, auto_reset):
    """collect_rollout writes the trajectory in place (the env step's obs / reward / done pointers are redirected into the
    [k, ...] buffers, the policy reads the previous slice): bit-identical to policy_forward + step + copies per step, on one
    stream and on two lanes, with and without auto-reset (where the done flags are an INPUT of the step), and the batch's
    own obs / reward / done tensors end up as after k calls of step()."""
    import torch
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    w = _actor_critic_weights()
    wd = {k: torch.from_numpy(v).cuda() for k, v in w.items()}
    n, k = 3000, (70 if auto_reset else 160)
    kw = dict(params=env_params(), device="cuda:0", seed=11, auto_reset=auto_reset)
    a = Rocket6DOFBatch(n, lanes=lanes, **kw)
    b = Rocket6DOFBatch(n, **kw)
    a.reset(); b.reset()
    ro = a.collect_rollout(k, wd, stochastic=True)
    obs, rew, dn, val, act, lps = [], [], [], [], [], []
    for j in range(k):
        obs.append(b.obs[:13].t().clone())
        ae, raw, v, lp = b.policy_forward(wd, stochastic=True, tensor_cores=3)
        b.step(ae)
        act.append(raw.clone()); val.append(v.clone()); lps.append(lp.clone())
        rew.append(b.reward_f32.clone()); dn.append(b.done.clone())
    torch.cuda.synchronize()
    assert torch.equal(ro["obs"], torch.stack(obs)) and torch.equal(ro["actions"], torch.stack(act))
    assert torch.equal(ro["values"], torch.stack(val)) and torch.equal(ro["rewards"], torch.stack(rew))
    assert torch.equal(ro["dones"], torch.stack(dn)) and torch.equal(ro["log_probs"], torch.stack(lps))
    assert torch.equal(a.obs, b.obs) and torch.equal(a.reward_f32, b.reward_f32) and torch.equal(a.done, b.done)
    assert torch.equal(a.state, b.state) and torch.equal(a.stats, b.stats)
    if not auto_reset:
        assert int(dn[-1].sum()) > 0          # some envs did finish and stayed frozen
    # the batch keeps working normally afterwards (pointers restored)
    a.step_policy(3, wd); b.step_policy(3, wd)
    torch.cuda.synchronize()
    assert torch.equal(a.obs, b.obs) and torch.equal(a.state, b.state)

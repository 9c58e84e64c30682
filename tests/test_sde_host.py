"""gSDE on the host: the per-sample PPO math of r6_ppo_grad_sde (tests/sde_hostsim) against float64 autograd of SB3's
StateDependentNoiseDistribution loss (tests/sde_ref.py), the Philox noise draw against its NumPy restatement, and the
policy loaders with a [64, 3] log_std."""
import numpy as np
import pytest
import torch

import sde_hostsim

import sde_ref
from rl_rocket_6dof_b200 import policy


def _weights(seed):
    rng = np.random.default_rng(seed)
    w = {k: (rng.standard_normal(s) * (0.3 if k.startswith("w") else 0.05)).astype(np.float32) for k, s in sde_ref.LAYOUT_SDE}
    w["log_std"] = (rng.uniform(-1.0, 0.5, (64, 3))).astype(np.float32)      # not constant
    return w


def _flat(w):
    return np.concatenate([np.asarray(w[k], np.float32).reshape(-1) for k, _ in sde_ref.LAYOUT_SDE])


def _minibatch(w, n, seed):
    """Observations, gSDE actions of the policy itself (so ratios near 1), perturbed old log-probs (ratios on both sides
    of the clip range), advantages and returns."""
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((n, 13)) * 0.8).astype(np.float32)
    xi = rng.standard_normal((n, 192))
    raw, logp, _, _ = sde_ref.sample(w, x, xi)
    a = raw.astype(np.float32)
    old = (logp + rng.normal(0.0, 0.4, n)).astype(np.float32)
    adv = rng.standard_normal(n).astype(np.float32)
    ret = rng.standard_normal(n).astype(np.float32)
    return x, a, old, adv, ret


@pytest.mark.parametrize("ent_coef", [0.0, 0.01])
def test_host_sde_grad_matches_autograd(ent_coef):
    """Sum of the host per-sample gradient against float64 autograd.  Tolerance: every per-sample float32 entry carries
    a relative error of a few hundred ulp at most (the 64- and 128-term dot products of the forward and backward pass,
    std's 64-term sum), so the sum is held to 1e-4 of the sum of the per-sample magnitudes of that entry plus 1e-9."""
    w = _weights(1)
    x, a, old, adv, ret = _minibatch(w, 256, 2)
    g, t = sde_hostsim.ppo_sde_sample_grad(_flat(w), x, a, old, adv, ret, clip=0.2, vf_coef=0.5, ent_coef=ent_coef)
    ref, ent = sde_ref.grad_sum(w, x, a, old, adv, ret, clip=0.2, vf_coef=0.5, ent_coef=ent_coef)
    clipped = t[:, 2]
    assert 0 < clipped.sum() < len(clipped), "both clipped and unclipped ratios"
    tol = 1e-4 * np.abs(g.astype(np.float64)).sum(0) + 1e-9
    err = np.abs(g.astype(np.float64).sum(0) - ref)
    worst = (err / tol).max()
    print(f"ent_coef={ent_coef}: worst |host - autograd| / tol = {worst:.3f}")
    assert worst <= 1.0
    ls = slice(10308, 10500)
    assert np.abs(ref[ls]).max() > 0
    assert np.allclose(t[:, 4], ent, rtol=1e-5, atol=1e-5)
    # teeth: the same check against a log_std perturbed in one entry fails
    w2 = dict(w)
    w2["log_std"] = w["log_std"].copy()
    w2["log_std"][5, 1] += 0.05
    ref2, _ = sde_ref.grad_sum(w2, x, a, old, adv, ret, clip=0.2, vf_coef=0.5, ent_coef=ent_coef)
    assert (np.abs(g.astype(np.float64).sum(0) - ref2) / tol).max() > 1.0


def test_host_sde_noise_matches_numpy():
    seed = 0x1234_5678_9ABC
    genv = np.array([0, 1, 7, 2 ** 20 - 1, 2 ** 33 + 5], np.uint64)
    for step in (0, 3, 2 ** 32 + 1):
        xi = sde_hostsim.sde_noise(seed, genv, step).astype(np.float64)
        ref = sde_ref.noise(seed, genv, step)
        assert np.all(np.abs(xi - ref) <= sde_ref.noise_bar(ref))
    xi = sde_hostsim.sde_noise(seed, np.arange(4096, dtype=np.uint64), 0)
    assert abs(xi.mean()) < 0.01 and abs(xi.std() - 1.0) < 0.01
    assert not np.array_equal(sde_hostsim.sde_noise(seed, genv, 0), sde_hostsim.sde_noise(seed, genv, 1))


def test_loaders_accept_sde_log_std(tmp_path):
    rng = np.random.default_rng(0)
    w = {k: rng.standard_normal(s).astype(np.float32) for k, s in policy.SHAPES.items()}
    w.update(wv=rng.standard_normal(64).astype(np.float32), bv=np.zeros(1, np.float32),
             log_std=rng.standard_normal((64, 3)).astype(np.float32))
    p = tmp_path / "sde.npz"
    np.savez(p, **{"mlp_" + k: v for k, v in w.items()})
    got = policy.load_npz(str(p))
    assert got["log_std"].shape == (64, 3) and np.array_equal(got["log_std"], w["log_std"])
    assert policy.load_npz(str(p))["w0"].shape == (128, 13)
    # SB3 archive with a gSDE log_std
    import io
    import zipfile
    sd = {"mlp_extractor.shared_net.0.weight": w["w0"], "mlp_extractor.shared_net.0.bias": w["b0"],
          "mlp_extractor.shared_net.2.weight": w["w1"], "mlp_extractor.shared_net.2.bias": w["b1"],
          "action_net.weight": w["w2"], "action_net.bias": w["b2"], "value_net.weight": w["wv"][None],
          "value_net.bias": w["bv"], "log_std": w["log_std"]}
    buf = io.BytesIO()
    torch.save({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}, buf)
    z = tmp_path / "m.zip"
    with zipfile.ZipFile(z, "w") as f:
        f.writestr("policy.pth", buf.getvalue())
    got = policy.load_sb3_zip(str(z))
    assert got["log_std"].shape == (64, 3)
    # a wrong trunk shape is still rejected, and so is a log_std of neither shape
    bad = dict(w, w1=np.zeros((32, 128), np.float32))
    np.savez(tmp_path / "bad.npz", **{"mlp_" + k: v for k, v in bad.items()})
    with pytest.raises(ValueError):
        policy.load_npz(str(tmp_path / "bad.npz"))
    bad = dict(w, log_std=np.zeros(5, np.float32))
    np.savez(tmp_path / "bad2.npz", **{"mlp_" + k: v for k, v in bad.items()})
    with pytest.raises(ValueError):
        policy.load_npz(str(tmp_path / "bad2.npz"))


def test_sde_config_options_rejected():
    from rl_rocket_6dof_b200.ppo import PPOConfig
    PPOConfig(use_sde=True, sde_sample_freq=4)
    for kw in (dict(full_std=False), dict(use_expln=True), dict(squash_output=True), dict(learn_features=True)):
        with pytest.raises(ValueError):
            PPOConfig(use_sde=True, **kw)

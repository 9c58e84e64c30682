"""Fused policy network (host build of the kernel code) against the actions the reference-side
closed-loop run recorded (tests/golden/policy_cl.npz: numpy float32 forward of best_model_2bo71j9m), against the float64
actor-critic of tests/policy_ref.py within its error bound, and the Gaussian policy head against the NumPy statement of
its Philox noise (tests/philox_ref.py)."""
import os

import numpy as np
import pytest

import hostsim
import philox_ref as pr
import policy_ref
from rl_rocket_6dof_b200 import policy

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "policy_cl.npz")


def _episode_inputs(g):
    """(obs13 the policy saw, action it produced) for every step that is not the first of an episode."""
    starts = set(int(s) for s in g["ic_step"])
    idx = np.array([k for k in range(1, len(g["action"])) if k not in starts])
    return g["obs"][idx - 1][:, :13], g["action"][idx]


def test_weights_roundtrip_and_shapes():
    w = policy.load_npz(GOLD)
    assert {k: v.shape for k, v in w.items()} == policy.SHAPES
    bad = dict(w, w0=w["w0"][:, :12])
    try:
        policy._check(bad)
    except ValueError as e:
        assert "w0" in str(e)
    else:
        raise AssertionError("wrong shapes must be rejected")


def test_kernel_mlp_matches_recorded_actions():
    g = np.load(GOLD)
    w = policy.load_npz(GOLD)
    x, a_ref = _episode_inputs(g)
    a = hostsim.mlp_actions(w, x)
    # float32 network: summation order / tanh implementation differ by a few ulp of the pre-activations
    assert np.abs(a - a_ref).max() <= 2e-6
    assert np.abs(policy.forward_numpy(w, x) - a_ref).max() <= 2e-6
    assert np.all(np.abs(a) <= 1.0)
    # the clip of evaluate_policy / predict: a network with a large output gain saturates at +-1
    big = dict(w, w2=w["w2"] * 1000, b2=w["b2"] * 1000)
    ab = hostsim.mlp_actions(big, x[:256])
    assert np.array_equal(ab, policy.forward_numpy(big, x[:256])) or np.abs(ab - policy.forward_numpy(big, x[:256])).max() <= 1e-3
    assert (np.abs(ab) == 1.0).mean() > 0.5


def test_sb3_zip_loader_roundtrip(tmp_path):
    """policy.load_sb3_zip reads the actor (+ critic head and log_std of the shared-trunk policy) out of a
    stable-baselines3 archive layout: a zip with a `policy.pth` state dict."""
    import io
    import zipfile

    import torch
    w = policy.load_npz(GOLD)
    rng = np.random.default_rng(2)
    sd = {
        "mlp_extractor.shared_net.0.weight": torch.from_numpy(w["w0"]), "mlp_extractor.shared_net.0.bias": torch.from_numpy(w["b0"]),
        "mlp_extractor.shared_net.2.weight": torch.from_numpy(w["w1"]), "mlp_extractor.shared_net.2.bias": torch.from_numpy(w["b1"]),
        "action_net.weight": torch.from_numpy(w["w2"]), "action_net.bias": torch.from_numpy(w["b2"]),
        "value_net.weight": torch.from_numpy(rng.standard_normal((1, 64)).astype(np.float32)),
        "value_net.bias": torch.zeros(1), "log_std": torch.full((3,), -1.5),
    }
    buf = io.BytesIO()
    torch.save(sd, buf)
    path = str(tmp_path / "model.zip")
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("policy.pth", buf.getvalue())
        z.writestr("data", "{}")
    got = policy.load_sb3_zip(path[:-4])                 # extension is optional, like PPO.load
    for k in policy.SHAPES:
        assert np.array_equal(got[k], w[k])
    assert got["wv"].shape == (64,) and got["bv"].shape == (1,) and np.allclose(got["log_std"], -1.5)
    mean, value = policy.forward_full_numpy(got, np.zeros((2, 13), np.float32))
    assert mean.shape == (2, 3) and value.shape == (2,)
    a = hostsim.mlp_actions(got, np.zeros((2, 13), np.float32))
    assert np.abs(a - np.clip(mean, -1, 1)).max() <= 1e-6


# seeds, global env ids and step indices on both sides of 2^32 (the high words enter the Philox key and counter)
SEEDS = (0, 31, (1 << 32) - 1, (1 << 32) + 5, (1 << 64) - 3)
STEPS = (0, 7, (1 << 32) - 1, 1 << 32, (3 << 32) + 11)


def _genv_grid():
    return np.concatenate([np.arange(0, 300), np.arange((1 << 32) - 150, (1 << 32) + 150),
                           np.arange((5 << 40) + 17, (5 << 40) + 117)]).astype(np.uint64)


def test_policy_noise_statement():
    """policy_noise is Box-Muller on the uniforms gaussian_head forms: u1 in (0, 1] with 1.0 for the top grid value (the
    float32 k + 0.5 rounds to even), angles in [0, 2 pi], and it depends on every word of (seed, genv, step)."""
    r = np.array([[0xFFFFFFFF, 0xFFFFFFFF, 0x000000FF, 0], [0xFFFFFEFF, 0x80000000, 0xFF, 0xFFFFFF7F]], np.uint32)
    u1, u2, u3, u4 = pr.policy_uniforms(r)
    assert u1[0] == 1.0 and u2[0] == 1.0 and u4[0] == 0.0
    assert u1[1] == np.float32(16777214 / 16777216) and u2[1] == 0.5 and u4[1] == np.float32(4294967040 / 4294967296)
    assert u3[0] == np.float32(0.5 / 16777216)
    z = pr.policy_noise(7, np.arange(1 << 16), 3)
    assert np.all(np.isfinite(z)) and abs(z.mean()) < 0.01 and abs(z.std() - 1) < 0.01
    base = pr.policy_noise(7, np.array([5], np.uint64), 9)
    for other in (pr.policy_noise(7 + (1 << 32), [5], 9), pr.policy_noise(7, [5 + (1 << 32)], 9),
                  pr.policy_noise(7, [5], 9 + (1 << 32)), pr.policy_noise(7, [6], 9), pr.policy_noise(7, [5], 10)):
        assert not np.any(other == base)


@pytest.mark.parametrize("seed", SEEDS)
def test_host_gaussian_head_matches_policy_noise(seed):
    """Host build of gaussian_head (libm log / cos / sin) against policy_noise and SB3's float64 log-probability.
    Bars: z within philox_ref.policy_noise_bar (3 ulp).  raw = mean + RN(RN(expf(ls)) z) adds 1 ulp of exp and 0.5 ulp
    of each operation.  log_prob sums three terms of four float32 operations each: 12 roundings of at most 2^-24 of the
    running magnitude, plus |z| |dz| per term."""
    genv = _genv_grid()
    for step in STEPS:
        z_ref = pr.policy_noise(seed, genv, step)
        n = len(genv)
        z, lp = hostsim.gaussian_head(np.zeros((n, 3)), None, True, seed, genv, step)
        dz = pr.policy_noise_bar(z_ref, seed, genv, step)
        assert np.all(np.abs(z - z_ref) <= dz), (seed, step)
        ref_lp = pr.gaussian_log_prob(z_ref, None)
        mag = (0.5 * z_ref ** 2 + pr.LOG_SQRT_2PI).sum(1)
        assert np.all(np.abs(lp - ref_lp) <= 12 * 2.0 ** -24 * mag + (np.abs(z_ref) * dz).sum(1) + 1e-30)
        # mean and log_std
        rng = np.random.default_rng(seed % 1000 + step % 1000)
        mean = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
        ls = np.array([-5.0, 0.0, 2.0], np.float32)
        raw, lp2 = hostsim.gaussian_head(mean, ls, True, seed, genv, step)
        std = np.exp(ls.astype(np.float64))
        ref_raw = mean + std * z_ref
        tol = 2.0 ** -24 * (np.abs(mean) + np.abs(ref_raw)) + std * (dz + 3 * 2.0 ** -24 * np.abs(z_ref))
        assert np.all(np.abs(raw - ref_raw) <= tol)
        ref_lp2 = pr.gaussian_log_prob(z_ref, ls)
        mag2 = (0.5 * z_ref ** 2 + np.abs(ls) + pr.LOG_SQRT_2PI).sum(1)
        assert np.all(np.abs(lp2 - ref_lp2) <= 12 * 2.0 ** -24 * mag2 + (np.abs(z_ref) * dz).sum(1))


def test_host_gaussian_head_deterministic():
    """stochastic = 0: raw = mean bit for bit, log_prob = -(sum log_std + 3 ln(2 pi) / 2) in the kernel's float32 order."""
    rng = np.random.default_rng(1)
    mean = rng.uniform(-3, 3, (64, 3)).astype(np.float32)
    for ls in (None, np.array([-0.5, -1.0, 0.2], np.float32), np.array([-5.0, 0.0, 2.0], np.float32)):
        raw, lp = hostsim.gaussian_head(mean, ls, False, 3, np.arange(64, dtype=np.uint64), 5)
        assert np.array_equal(raw, mean)
        assert np.all(lp == pr.log_prob_at_mean(ls))


@pytest.mark.parametrize("family", policy_ref.FAMILIES)
def test_host_mlp_forward_within_float64_bound(family):
    """The float32 FMA network (mlp_forward, the code of tensor_cores = 0 and R6_ACT_MLP) against forward64 within the
    mode-0 bound, mean and value, on every observation set; the bound is what the GPU tests hold the kernels to."""
    w = policy_ref.weights(family)
    worst = 0.0
    for name, x in policy_ref.obs_sets(2048).items():
        mean, val = hostsim.mlp_forward(w, x)
        m64, v64 = policy_ref.forward64(w, x)
        b = policy_ref.bound(w, x, 0)
        err = np.abs(np.concatenate([mean, val[:, None]], 1) - np.concatenate([m64, v64[:, None]], 1))
        assert np.all(err <= b), (family, name)
        worst = max(worst, float((err / b).max()))
        assert np.all(hostsim.mlp_actions(w, x) == np.clip(mean, -1, 1))
        actor = {k: v for k, v in w.items() if k not in ("wv", "bv")}
        mean2, val2 = hostsim.mlp_forward(actor, x[:64])
        assert np.array_equal(mean2, mean[:64]) and np.all(val2 == 0)
        assert np.all(policy_ref.bound(actor, x[:64], 0)[:, 3] == 0)
    print(f"{family}: worst |host - forward64| / bound(mode 0) = {worst:.3f}")


def test_weight_families_cover_their_edges():
    """The families hold what their names promise."""
    x = policy_ref.obs_sets(1024)["uniform"]
    w = policy_ref.weights("saturating")
    a0 = x.astype(np.float64) @ w["w0"].T.astype(np.float64) + w["b0"]
    assert (np.abs(a0) > 10).mean() > 0.5 and (a0 > 10).any() and (a0 < -10).any()
    h0 = np.tanh(a0)
    a1 = h0 @ w["w1"].T.astype(np.float64) + w["b1"]
    assert (np.abs(a1) > 10).mean() > 0.5 and (a1 > 10).any() and (a1 < -10).any()
    e = policy_ref.weights("tf32_edges")
    bits = np.concatenate([e[k].ravel() for k in ("w0", "w1", "w2")]).view(np.uint32)
    low = bits & 0x1FFF
    vals = np.concatenate([e[k].ravel() for k in ("w0", "w1", "w2")])
    assert (low == 0x1000).mean() > 0.1 and ((low == 0) & (vals != 0)).mean() > 0.1
    assert (vals.view(np.uint32) == 0x80000000).any() and (vals.view(np.uint32) == 0).any()
    assert ((np.abs(vals) < 2.0 ** -100) & (vals != 0)).mean() > 0.1
    assert np.array_equal(e["log_std"], np.array([-5, 0, 2], np.float32))
    s = policy_ref.weights("sb3_init")
    q = s["w1"].astype(np.float64)
    assert np.allclose(q @ q.T, 2 * np.eye(64), atol=1e-5) and np.all(s["b0"] == 0) and np.all(s["log_std"] == 0)


def test_bound_can_fail():
    """A network evaluated with single-pass TF32 operands (what tensor_cores = 2 does, without its tanh.approx error)
    misses the bar of the faithful 3xTF32 mode: the bar is tight enough to catch dropped correction terms."""
    w = policy_ref.weights("golden")
    x = policy_ref.obs_sets(2048)["golden"]
    rt = policy_ref.round_tf32
    h = rt(x)
    h = rt(np.tanh(h @ rt(w["w0"]).T + w["b0"]))
    h = rt(np.tanh(h @ rt(w["w1"]).T + w["b1"]))
    mean = h @ rt(w["w2"]).T + w["b2"]
    m64, _ = policy_ref.forward64(w, x)
    ratio = (np.abs(mean - m64) / policy_ref.bound(w, x, 3)[:, :3]).max()
    print(f"single-pass TF32 / bound(mode 3) = {ratio:.2f}")
    assert ratio > policy_ref.C_BAR

"""SB3 1.6's default separate policy / value towers (net_arch [dict(pi=[64, 64], vf=[64, 64])]) on the host: the
loaders, the flat layout and SB3's initialisation, and the per-sample PPO math of r6_ppo_grad for that network (host
build, tests/sep_hostsim) against float64 autograd of SB3's loss (tests/sep_ref.py)."""
import io
import math
import zipfile

import numpy as np
import pytest
import torch

import policy_ref
import sep_hostsim
import sep_ref
from rl_rocket_6dof_b200 import _lib, policy
from rl_rocket_6dof_b200.ppo import LAYOUT, LAYOUT_SEP, NPARAMS_SEP, ActorCriticParams


def _zip(tmp_path, sd, name="model.zip"):
    buf = io.BytesIO()
    torch.save({k: torch.as_tensor(np.asarray(v)) for k, v in sd.items()}, buf)
    path = tmp_path / name
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("policy.pth", buf.getvalue())
    return str(path)


def _sb3_sep_state(w):
    """policy.pth of SB3 1.6 PPO("MlpPolicy") without policy_kwargs"""
    return {"log_std": w["log_std"],
            "mlp_extractor.policy_net.0.weight": w["w0"], "mlp_extractor.policy_net.0.bias": w["b0"],
            "mlp_extractor.policy_net.2.weight": w["w1"], "mlp_extractor.policy_net.2.bias": w["b1"],
            "mlp_extractor.value_net.0.weight": w["vf_w0"], "mlp_extractor.value_net.0.bias": w["vf_b0"],
            "mlp_extractor.value_net.2.weight": w["vf_w1"], "mlp_extractor.value_net.2.bias": w["vf_b1"],
            "action_net.weight": w["w2"], "action_net.bias": w["b2"],
            "value_net.weight": np.asarray(w["wv"]).reshape(1, 64), "value_net.bias": w["bv"]}


def test_sb3_16_separate_zip_loads_in_full(tmp_path):
    w = sep_ref.weights(0)
    got = policy.load_sb3_zip(_zip(tmp_path, _sb3_sep_state(w)))
    assert set(got) == {k for k, _ in LAYOUT_SEP}
    for k, shape in LAYOUT_SEP:
        assert got[k].dtype == np.float32 and got[k].shape == shape
        assert np.array_equal(got[k], np.asarray(w[k]).reshape(shape)), k
    assert policy.is_separate(got)


def test_separate_npz_round_trip_is_bit_exact(tmp_path):
    w = sep_ref.weights(1)
    path = str(tmp_path / "w.npz")
    np.savez(path, **{"mlp_" + k: v for k, v in w.items()})
    got = policy.load_npz(path)
    assert set(got) == set(w)
    for k in w:
        assert got[k].tobytes() == np.asarray(w[k], np.float32).tobytes(), k


def test_shared_trunk_and_sb3_18_towers_load_as_before(tmp_path):
    rng = np.random.default_rng(2)
    r = lambda *s: rng.standard_normal(s).astype(np.float32)
    shared = {"mlp_extractor.shared_net.0.weight": r(128, 13), "mlp_extractor.shared_net.0.bias": r(128),
              "mlp_extractor.shared_net.2.weight": r(64, 128), "mlp_extractor.shared_net.2.bias": r(64),
              "action_net.weight": r(3, 64), "action_net.bias": r(3), "value_net.weight": r(1, 64),
              "value_net.bias": r(1), "log_std": r(3)}
    got = policy.load_sb3_zip(_zip(tmp_path, shared, "shared.zip"))
    assert set(got) == {"w0", "b0", "w1", "b1", "w2", "b2", "wv", "bv", "log_std"} and not policy.is_separate(got)
    assert np.array_equal(got["w0"], shared["mlp_extractor.shared_net.0.weight"])
    # SB3 >= 1.8 default: separate towers of [128, 64] -> actor only (and log_std)
    v18 = {k.replace("shared_net", "policy_net"): v for k, v in shared.items() if "shared_net" in k}
    v18.update({k.replace("shared_net", "value_net"): v for k, v in shared.items() if "shared_net" in k})
    v18.update({k: shared[k] for k in ("action_net.weight", "action_net.bias", "value_net.weight", "value_net.bias", "log_std")})
    got = policy.load_sb3_zip(_zip(tmp_path, v18, "v18.zip"))
    assert set(got) == {"w0", "b0", "w1", "b1", "w2", "b2", "log_std"}
    assert np.array_equal(got["w1"], shared["mlp_extractor.shared_net.2.weight"])


@pytest.mark.parametrize("key,shape", [("vf_w0", (64, 12)), ("vf_w1", (64, 128)), ("w1", (64, 128)), ("vf_b1", (32,)),
                                       ("w0", (128, 13))])
def test_malformed_separate_shapes_raise(tmp_path, key, shape):
    w = sep_ref.weights(3)
    w[key] = np.zeros(shape, np.float32)
    with pytest.raises(ValueError):
        policy.to_device(w, "cpu")
    path = str(tmp_path / "bad.npz")
    np.savez(path, **{"mlp_" + k: v for k, v in w.items()})
    with pytest.raises(ValueError):
        policy.load_npz(path)


def test_separate_layout_offsets():
    offs, o = {}, 0
    for k, shape in LAYOUT_SEP:
        offs[k] = o
        o += int(np.prod(shape))
    assert o == NPARAMS_SEP == _lib.PPO_NPARAMS_SEP == 10375
    assert offs == {"w0": 0, "vf_w0": 832, "b0": 1664, "vf_b0": 1728, "w1": 1792, "b1": 5888, "vf_w1": 5952,
                    "vf_b1": 10048, "w2": 10112, "b2": 10304, "wv": 10307, "bv": 10371, "log_std": 10372}
    assert offs["w1"] % 4 == 0 and offs["vf_w1"] % 4 == 0                 # 16-byte aligned for tensor_cores 2 / 3
    # the stacked layer 0 is the shared layout's [128][13] + [128]
    shared = dict(zip([k for k, _ in LAYOUT], np.cumsum([0] + [int(np.prod(s)) for _, s in LAYOUT])[:-1]))
    assert shared["b0"] == offs["b0"] and shared["w1"] == offs["w1"]


def test_sb3_init_gains_and_reproducibility():
    arch = [dict(pi=[64, 64], vf=[64, 64])]
    w = ActorCriticParams.sb3_init_weights(seed=5, net_arch=arch)
    gains = {"w0": math.sqrt(2), "w1": math.sqrt(2), "vf_w0": math.sqrt(2), "vf_w1": math.sqrt(2), "w2": 0.01, "wv": 1.0}
    shapes = dict(LAYOUT_SEP)
    assert set(w) == set(gains)
    for k, g in gains.items():
        W = w[k].double().reshape(shapes[k] if k != "wv" else (1, 64)).numpy()
        G = W @ W.T if W.shape[0] <= W.shape[1] else W.T @ W          # orthonormal on the short side
        assert np.allclose(G, g * g * np.eye(len(G)), atol=1e-5 * g * g), k
    again = ActorCriticParams.sb3_init_weights(seed=5, net_arch=arch)
    other = ActorCriticParams.sb3_init_weights(seed=6, net_arch=arch)
    assert all(torch.equal(w[k], again[k]) for k in w)
    assert not torch.equal(w["vf_w1"], other["vf_w1"])
    assert not torch.equal(w["w0"], w["vf_w0"])
    # the shared trunk draws exactly as before (w0, w1, w2, wv from one generator)
    s = ActorCriticParams.sb3_init_weights(seed=5)
    gen = torch.Generator().manual_seed(5)
    for k, shape, g in (("w0", (128, 13), math.sqrt(2)), ("w1", (64, 128), math.sqrt(2)), ("w2", (3, 64), 0.01),
                        ("wv", (1, 64), 1.0)):
        t = torch.empty(shape)
        torch.nn.init.orthogonal_(t, gain=g, generator=gen)
        assert torch.equal(s[k], t.reshape(-1)), k


@pytest.mark.parametrize("net_arch", [[64, 64], [dict(pi=[128, 64], vf=[128, 64])], [dict(pi=[64], vf=[64])]])
def test_other_architectures_raise(net_arch):
    with pytest.raises(ValueError):
        ActorCriticParams.sb3_init_weights(net_arch=net_arch)
    with pytest.raises(ValueError):
        ActorCriticParams.sb3_init(net_arch=net_arch, device="cpu")


def test_host_forward_within_mode0_bound():
    """mlp_forward_sep (the mode-0 kernel's network) against float64, each tower held to tests/policy_ref's mode-0
    forward bound for its own layers."""
    w = sep_ref.weights(4)
    x = (np.random.default_rng(5).standard_normal((512, 13)) * 0.8).astype(np.float32)
    out = sep_hostsim.forward(sep_ref.flat(w), x).astype(np.float64)
    mean, value = sep_ref.forward64(w, x)
    pol, val = sep_ref.towers(w)
    bp, bv = policy_ref.bound(pol, x, 0)[:, :3], policy_ref.bound(val, x, 0)[:, 0]
    assert np.all(np.abs(out[:, :3] - mean) <= bp)
    assert np.all(np.abs(out[:, 3] - value) <= bv)


@pytest.mark.parametrize("normalize,ent_coef,clip", [(True, 0.0, 0.2), (False, 0.01, 0.2), (False, 0.0, 0.05)])
def test_host_sep_grad_matches_autograd(normalize, ent_coef, clip):
    """Sum of the host per-sample gradient against float64 autograd of SB3's loss, within sep_ref.bound: the first-order
    error of the float32 chain of r6_ppo.cuh, with no accumulation chain (the host sums the float32 products in
    float64)."""
    w = sep_ref.weights(6)
    x, a, old, adv, ret = sep_ref.minibatch(w, 256, 7)
    stats = None
    adv_n = adv.astype(np.float64)
    if normalize:
        a64 = adv.astype(np.float64)
        stats = np.array([a64.mean(), 1.0 / (a64.std(ddof=1) + 1e-8)])
        adv_n = np.array([np.float32((v - stats[0]) * stats[1]) for v in a64], np.float64)
    g, t = sep_hostsim.sample_grad(sep_ref.flat(w), x, a, old, adv, ret, adv_stats=stats, clip=clip, vf_coef=0.5,
                                   ent_coef=ent_coef)
    ref, terms, mag = sep_ref.grad_sum(w, x, a, old, adv_n, ret, clip=clip, vf_coef=0.5, ent_coef=ent_coef)
    clipped = t[:, 2]
    assert 0 < clipped.sum() < len(clipped), "both clipped and unclipped ratios"
    g64 = g.astype(np.float64)
    tol = sep_ref.bound(w, x, a, old, adv_n, ret, clip=clip, vf_coef=0.5, ent_coef=ent_coef, samples_per_cta=0) + 1e-300
    worst = (np.abs(g64.sum(0) - ref) / tol).max()
    print(f"normalize={normalize} ent_coef={ent_coef} clip={clip}: worst |host - autograd| / tol = {worst:.3f}")
    assert worst <= 1.0
    assert np.allclose(t.astype(np.float64).sum(0), terms, rtol=1e-4, atol=1e-3)
    # the reference's magnitude sums are those of the host's per-sample products
    assert np.allclose(mag, np.abs(g64).sum(0), rtol=1e-4, atol=1e-7)
    for k in ("vf_w0", "vf_w1", "w1", "wv"):          # every block carries gradient
        o = sum(int(np.prod(s)) for kk, s in LAYOUT_SEP[:[n for n, _ in LAYOUT_SEP].index(k)])
        assert np.abs(ref[o:o + int(np.prod(dict(LAYOUT_SEP)[k]))]).max() > 0, k
    # teeth: the value tower's gradient differs from what a swapped tower would give
    w2 = dict(w, vf_w1=w["w1"], w1=w["vf_w1"])
    ref2, _, _ = sep_ref.grad_sum(w2, x, a, old, adv_n, ret, clip=clip, vf_coef=0.5, ent_coef=ent_coef)
    assert (np.abs(g64.sum(0) - ref2) / tol).max() > 10

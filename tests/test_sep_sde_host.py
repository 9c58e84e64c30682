"""gSDE on SB3 1.6's separate towers, on the host: the per-sample PPO math of r6_ppo_grad_sde_sep (host build,
tests/sepsde_hostsim) against float64 autograd of SB3's loss (tests/sepsde_ref.py), the flat layout, SB3's
initialisation, the loaders and the options that stay refused."""
import io
import zipfile

import numpy as np
import pytest
import torch

import sepsde_hostsim
import sepsde_ref
from rl_rocket_6dof_b200 import _lib, policy
from rl_rocket_6dof_b200.ppo import (LAYOUT_SEP, LAYOUT_SEP_SDE, NET_ARCH_SEP, NPARAMS_SEP_SDE, ActorCriticParams,
                                     PPOConfig)


@pytest.mark.parametrize("vfc", [None, 0.15])
@pytest.mark.parametrize("normalize", [False, True])
@pytest.mark.parametrize("ent_coef", [0.0, 0.01])
def test_host_grad_matches_autograd(ent_coef, normalize, vfc):
    """Sum of the host per-sample gradient against float64 autograd of SB3's loss, with the bar of test_sde_host (1e-4 of
    the per-entry sum of per-sample magnitudes, plus 1e-9).  The samples lie on both sides of the ratio clip and, with
    clip_range_vf, inside and outside the value band."""
    w = sepsde_ref.weights(1)
    x, a, old, adv, ret, vold = sepsde_ref.minibatch(w, 256, 2)
    stats = None
    adv_n = adv.astype(np.float64)
    if normalize:
        a64 = adv.astype(np.float64)
        stats = np.array([a64.mean(), 1.0 / (a64.std(ddof=1) + 1e-8)])
        adv_n = ((a64 - stats[0]) * stats[1]).astype(np.float32).astype(np.float64)
    g, t = sepsde_hostsim.sample_grad(sepsde_ref.flat(w), x, a, old, adv, ret, vold, vfc or 0.0, adv_stats=stats,
                                      ent_coef=ent_coef)
    ref, terms, ent = sepsde_ref.grad_sum(w, x, a, old, adv_n, ret, ent_coef=ent_coef, clip_range_vf=vfc, old_values=vold)
    assert 0 < t[:, 2].sum() < len(t), "both clipped and unclipped ratios"
    if vfc is not None:
        _, v64, _, _ = sepsde_ref.forward({k: torch.tensor(np.asarray(w[k], np.float64)) for k, _ in LAYOUT_SEP_SDE}, x)
        d = np.abs(v64.numpy() - vold)
        assert (d < vfc).sum() > 20 and (d > vfc).sum() > 20, "samples inside and outside the value band"
    tol = 1e-4 * np.abs(g.astype(np.float64)).sum(0) + 1e-9
    err = np.abs(g.astype(np.float64).sum(0) - ref)
    worst = (err / tol).max()
    print(f"ent={ent_coef} normalize={normalize} vfc={vfc}: worst |host - autograd| / tol = {worst:.3f}")
    assert worst <= 1.0
    ls = slice(sepsde_ref.LOG_STD, NPARAMS_SEP_SDE)
    assert np.abs(ref[ls]).max() > 0
    assert np.allclose(t[:, 4], ent, rtol=1e-5, atol=1e-5)
    assert np.allclose(t[:, :4].astype(np.float64).sum(0), terms, rtol=1e-4, atol=1e-3)
    # teeth: the value latent as h, the gradient let through std, and one perturbed log_std entry all fail the bar
    for kw in (dict(latent="value"), dict(detach=False)):
        bad, _, _ = sepsde_ref.grad_sum(w, x, a, old, adv_n, ret, ent_coef=ent_coef, clip_range_vf=vfc, old_values=vold, **kw)
        assert (np.abs(g.astype(np.float64).sum(0) - bad) / tol).max() > 1.0, kw
    w2 = dict(w, log_std=w["log_std"].copy())
    w2["log_std"][5, 1] += 0.05
    bad, _, _ = sepsde_ref.grad_sum(w2, x, a, old, adv_n, ret, ent_coef=ent_coef, clip_range_vf=vfc, old_values=vold)
    assert (np.abs(g.astype(np.float64).sum(0) - bad) / tol).max() > 1.0


def test_layout_offsets():
    assert _lib.PPO_NPARAMS_SEP_SDE == NPARAMS_SEP_SDE == 10564
    assert LAYOUT_SEP_SDE[:-1] == LAYOUT_SEP[:-1] and LAYOUT_SEP_SDE[-1] == ("log_std", (64, 3))
    assert sepsde_ref.LOG_STD == 10372 and sepsde_ref.LOG_STD % 4 == 0      # 16-byte aligned in an aligned buffer
    assert sepsde_hostsim.lib().hs_sepsde_nparams() == NPARAMS_SEP_SDE
    with open(_lib.os.path.join(_lib.PKG, "..", "include", "r6dof.h")) as f:
        assert "#define R6_PPO_NPARAMS_SEP_SDE 10564" in f.read()


def test_sb3_init_draws_the_separate_matrices():
    """use_sde=True draws exactly the matrices of the diagonal separate-tower init; log_std is zeros [64, 3]."""
    if not torch.cuda.is_available():
        w = ActorCriticParams.sb3_init_weights(5, NET_ARCH_SEP)
        assert set(w) == {"w0", "w1", "vf_w0", "vf_w1", "w2", "wv"}
        pytest.skip("the flat parameters live on a CUDA device")
    p = ActorCriticParams.sb3_init(seed=5, device="cuda", use_sde=True, net_arch=NET_ARCH_SEP)
    q = ActorCriticParams.sb3_init(seed=5, device="cuda", net_arch=NET_ARCH_SEP)
    assert p.separate and p.use_sde and p.flat.numel() == NPARAMS_SEP_SDE
    assert torch.equal(p.flat[:sepsde_ref.LOG_STD], q.flat[:sepsde_ref.LOG_STD])
    assert p.log_std.shape == (64, 3) and not bool(p.log_std.any())


def _sb3_sep_sde_zip(tmp_path, w):
    """policy.pth of SB3 1.6 PPO("MlpPolicy", use_sde=True) without policy_kwargs"""
    sd = {"log_std": w["log_std"],
          "mlp_extractor.policy_net.0.weight": w["w0"], "mlp_extractor.policy_net.0.bias": w["b0"],
          "mlp_extractor.policy_net.2.weight": w["w1"], "mlp_extractor.policy_net.2.bias": w["b1"],
          "mlp_extractor.value_net.0.weight": w["vf_w0"], "mlp_extractor.value_net.0.bias": w["vf_b0"],
          "mlp_extractor.value_net.2.weight": w["vf_w1"], "mlp_extractor.value_net.2.bias": w["vf_b1"],
          "action_net.weight": w["w2"], "action_net.bias": w["b2"],
          "value_net.weight": np.asarray(w["wv"]).reshape(1, 64), "value_net.bias": w["bv"]}
    buf = io.BytesIO()
    torch.save({k: torch.as_tensor(np.asarray(v)) for k, v in sd.items()}, buf)
    path = tmp_path / "model.zip"
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("policy.pth", buf.getvalue())
    return str(path)


def test_sb3_zip_loads_in_full_and_round_trips(tmp_path):
    w = sepsde_ref.weights(3)
    got = policy.load_sb3_zip(_sb3_sep_sde_zip(tmp_path, w))
    assert set(got) == {k for k, _ in LAYOUT_SEP_SDE} and policy.is_separate(got)
    for k, shape in LAYOUT_SEP_SDE:
        assert got[k].shape == shape and np.array_equal(got[k], np.asarray(w[k]).reshape(shape)), k
    path = str(tmp_path / "w.npz")
    np.savez(path, **{"mlp_" + k: v for k, v in got.items()})
    back = policy.load_npz(path)
    assert set(back) == set(got) and all(back[k].tobytes() == got[k].tobytes() for k in got)
    if torch.cuda.is_available():
        P = ActorCriticParams.from_weights(got, "cuda")
        assert P.separate and P.use_sde and P.layout == LAYOUT_SEP_SDE
        assert np.array_equal(P.flat.cpu().numpy(), sepsde_ref.flat(w))
        P.save_npz(str(tmp_path / "p.npz"))
        Q = ActorCriticParams.from_weights(policy.load_npz(str(tmp_path / "p.npz")), "cuda")
        assert torch.equal(P.flat, Q.flat) and Q.use_sde and Q.separate


def test_remaining_refusals():
    from rl_rocket_6dof_b200.batch import _check_separate
    mlp = {k: torch.zeros(s) for k, s in LAYOUT_SEP_SDE}
    _check_separate(mlp, 0)
    _check_separate(mlp, 3)
    with pytest.raises(ValueError, match="mma.sync"):
        _check_separate(mlp, 1)
    for kw in (dict(full_std=False), dict(use_expln=True), dict(squash_output=True), dict(learn_features=True)):
        with pytest.raises(ValueError):
            PPOConfig(use_sde=True, **kw)
    with pytest.raises(ValueError):
        ActorCriticParams.sb3_init(use_sde=True, net_arch=[dict(pi=[128, 64], vf=[128, 64])])

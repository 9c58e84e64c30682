"""gSDE on the B200: the noise buffer, the policy kernels' gSDE head (modes 0, 2, 3), sde_sample_freq in collection, the
r6_ppo_grad_sde kernel against float64 autograd of SB3's loss, and a short gSDE training run."""
import ctypes as C

import numpy as np
import pytest
import torch

import sde_hostsim
import policy_ref
import sde_ref
from rl_rocket_6dof_b200 import Rocket6DOFBatch, _lib
from rl_rocket_6dof_b200.ppo import ActorCriticParams, PPOConfig, PPOTrainer, loss_and_grad

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _params(seed=0):
    p = ActorCriticParams.sb3_init(seed=seed, device=DEV, use_sde=True)
    g = torch.Generator().manual_seed(seed + 1)
    p.log_std.copy_((torch.rand(64, 3, generator=g) * 1.5 - 1.0).to(DEV))     # not constant
    p.w2.mul_(50.0)                                                             # a mean that is not ~0
    return p


def _w(p):
    return {k: v.detach().cpu().numpy() for k, v in p.mlp().items()}


def test_noise_buffer_matches_host_and_is_layout_independent():
    n = 3000
    b1 = Rocket6DOFBatch(n, device=DEV, seed=7)
    b2 = Rocket6DOFBatch(n, device=DEV, seed=7, lanes=2)
    for b in (b1, b2):
        b.steps_done = 11
        b.reset_noise()
    torch.cuda.synchronize()
    xi = b1.sde_xi.cpu().numpy().T.astype(np.float64)
    # device (sincospif, 1 ulp) and host build (double sin / cos rounded) may differ by an ulp: both against NumPy
    ref = sde_ref.noise(7, np.arange(n, dtype=np.uint64), 11)
    host = sde_hostsim.sde_noise(7, np.arange(n, dtype=np.uint64), 11).astype(np.float64)
    assert np.all(np.abs(xi - ref) <= sde_ref.noise_bar(ref))
    assert np.all(np.abs(host - ref) <= sde_ref.noise_bar(ref))
    print(f"noise: {np.mean(xi == host):.4f} of the entries bit-equal to the host build, worst |device - numpy| / bar = "
          f"{(np.abs(xi - ref) / sde_ref.noise_bar(ref)).max():.3f}")
    assert torch.equal(b1.sde_xi, b2.sde_xi)
    # two shards of the same global envs
    s0 = Rocket6DOFBatch(1000, device=DEV, seed=7, env_offset=0, num_envs_global=n)
    s1 = Rocket6DOFBatch(n - 1000, device=DEV, seed=7, env_offset=1000, num_envs_global=n)
    for s in (s0, s1):
        s.reset_noise(step_index=11)
    assert torch.equal(torch.cat([s0.sde_xi, s1.sde_xi], 1), b1.sde_xi)


@pytest.mark.parametrize("mode", [0, 2, 3])
def test_policy_sde_sampling(mode):
    """raw = mean + h (sigma xi) and the log-prob, against float64.  Bounds: |mean - mean64| is within the mode's own
    bound (policy_ref.bound, derived as tests/test_gpu_policy_ref.py derives it); the noise h E adds the error of each
    activation h_k times |E_ka| (4e-6 in modes 0 / 3, 2e-3 in mode 2: tanh.approx and the TF32 rounding of h) and 64
    float32 roundings of the sum, 64 u sum_k |h_k E_ka|, plus 1e-6 for sigma xi's own rounding."""
    n = 4096
    b = Rocket6DOFBatch(n, device=DEV, seed=3)
    b.reset()
    p = _params()
    mlp = p.mlp()
    b.reset_noise()
    act, raw, val, logp = b.policy_forward(mlp, stochastic=True, tensor_cores=mode)
    torch.cuda.synchronize()
    w = _w(p)
    x = b.obs[:13].T.cpu().numpy()
    xi = b.sde_xi.cpu().numpy().T.astype(np.float64)
    raw64, logp64, mean64, h64 = sde_ref.sample(w, x, xi)
    E = np.exp(w["log_std"].astype(np.float64))[None] * xi.reshape(-1, 64, 3)
    hE = np.abs(h64[:, :, None] * E).sum(1)
    mb = policy_ref.bound(w, x, mode)[:, :3]
    act_acc = 2e-3 if mode == 2 else 4e-6
    bar = mb + 64 * 2.0 ** -24 * hE + act_acc * np.abs(E).sum(1) + 1e-6
    err = np.abs(raw.cpu().numpy() - raw64)
    print(f"mode {mode}: worst |raw - raw64| / bar = {(err / bar).max():.3f}")
    assert np.all(err <= bar)
    # log-prob: SB3's Normal(mean, std).log_prob; float32 evaluation at the kernel's own raw
    lp = logp.cpu().numpy()
    lerr = np.abs(lp - logp64)
    lbar = 1e-4 * (1 + np.abs(logp64)) + (2e-2 if mode == 2 else 1e-3)
    print(f"mode {mode}: worst |logp - logp64| / bar = {(lerr / lbar).max():.3f}")
    assert np.all(lerr <= lbar)
    # deterministic outputs bit-identical to the non-gSDE call
    d = b.policy_forward(mlp, stochastic=False, tensor_cores=mode)
    plain = dict(mlp, log_std=torch.zeros(3, device=DEV))
    e = b.policy_forward(plain, stochastic=False, tensor_cores=mode)
    assert torch.equal(d[0], e[0]) and torch.equal(d[1], e[1]) and torch.equal(d[2], e[2])
    assert torch.equal(val, e[2])


def test_policy_sde_mode1_rejected():
    b = Rocket6DOFBatch(256, device=DEV, seed=3)
    b.reset()
    with pytest.raises(_lib.R6Error, match="mma.sync"):
        b.policy_forward(_params().mlp(), stochastic=True, tensor_cores=1)


@pytest.mark.parametrize("freq", [-1, 4])
def test_sde_sample_freq(freq):
    """The noise each env used, recovered from raw - mean, is the draw keyed steps_done + j of the last resample."""
    n, k = 2048, 16
    b = Rocket6DOFBatch(n, device=DEV, seed=5, lanes=2)
    b.reset()
    p = _params()
    s0 = b.steps_done
    ro = b.collect_rollout(k, p.mlp(), tensor_cores=0, sde_sample_freq=freq)
    torch.cuda.synchronize()
    w = _w(p)
    for j in range(k):
        x = ro["obs"][j].cpu().numpy()
        key = s0 + (j - j % freq if freq > 0 else 0)
        xi = sde_hostsim.sde_noise(5, np.arange(n, dtype=np.uint64), key).astype(np.float64)
        raw64, _, _, _ = sde_ref.sample(w, x, xi)
        err = np.abs(ro["actions"][j].cpu().numpy() - raw64).max()
        assert err < 1e-3, (j, err)
        if freq > 0 and j % freq:
            xi_other = sde_hostsim.sde_noise(5, np.arange(n, dtype=np.uint64), key + 1).astype(np.float64)
            assert np.abs(ro["actions"][j].cpu().numpy() - sde_ref.sample(w, x, xi_other)[0]).max() > 1e-2


def test_grad_sde_kernel_matches_autograd():
    n, T = 2048, 8
    b = Rocket6DOFBatch(n, device=DEV, seed=9)
    b.reset()
    p = _params(2)
    ro = b.collect_rollout(T, p.mlp(), tensor_cores=0)
    g = torch.Generator(device=DEV).manual_seed(0)
    idx = torch.randperm(T * n, generator=g, device=DEV)
    idx[5] = -1
    idx[77] = T * n + 3                                  # bad indices: skipped and counted
    for ent in (0.0, 0.01):
        gs, terms = loss_and_grad(p, ro, idx, ent_coef=ent, normalize_advantage=False)
        gs2, terms2 = loss_and_grad(p, ro, idx, ent_coef=ent, normalize_advantage=False)
        torch.cuda.synchronize()
        assert torch.equal(gs, gs2) and torch.equal(terms, terms2)
        assert terms[4].item() == 2
        q = idx.cpu().numpy()
        q = q[(q >= 0) & (q < T * n)]
        x = ro["obs"].reshape(-1, 13)[q].cpu().numpy()
        a = ro["actions"].reshape(-1, 3)[q].cpu().numpy()
        old, adv, ret = (ro[k].reshape(-1)[q].cpu().numpy() for k in ("log_probs", "advantages", "returns"))
        ref, ent_s = sde_ref.grad_sum(_w(p), x, a, old, adv, ret, ent_coef=ent)
        g32 = gs.cpu().numpy().astype(np.float64)
        # 1e-4 of the gradient scale per layer block (float32 per-sample terms summed over 2^14 samples)
        scale = np.abs(ref).max() + 1e-6
        err = np.abs(g32 - ref)
        print(f"ent={ent}: worst |kernel - autograd| / max|grad| = {err.max() / scale:.2e}, log_std block "
              f"{err[10308:].max() / (np.abs(ref[10308:]).max() + 1e-12):.2e}")
        assert err.max() <= 1e-4 * scale
        assert err[10308:].max() <= 1e-3 * np.abs(ref[10308:]).max()
        assert abs(terms[5].item() - ent_s.sum()) <= 1e-5 * abs(ent_s.sum()) + 1e-3


def test_trainer_sde_short_learn():
    b = Rocket6DOFBatch(1 << 14, device=DEV, seed=0)
    p = ActorCriticParams.sb3_init(seed=0, device=DEV, use_sde=True)
    with pytest.raises(ValueError):
        PPOTrainer(b, ActorCriticParams.sb3_init(seed=0, device=DEV), PPOConfig(use_sde=True))
    with pytest.raises(ValueError):
        PPOTrainer(b, p, PPOConfig())
    tr = PPOTrainer(b, p, PPOConfig(use_sde=True, sde_sample_freq=4, n_steps=8, n_epochs=2, ent_coef=0.01), seed=0)
    logs = tr.learn(2 * 8 * (1 << 14))
    assert len(logs) == 2
    for log in logs:
        for k, v in log.items():
            assert np.isfinite(v), (k, v)
    assert abs(logs[0]["train/std"] - 1.0) < 0.05


def test_trainer_sde_steps_match_sb3():
    """One PPOTrainer.train with use_sde=True (2048 envs x 16 steps, batch_size 10,000: three full minibatches and one
    of 2,768, one epoch, entropy bonus) against sde_ref.reference_step, one Adam step at a time from the kernels' own
    pre-step state, and the train/ logs; perturbing one log_std entry of the reference breaks the check."""
    from rl_rocket_6dof_b200 import ppo
    n_envs, T, bs = 2048, 16, 10000
    b = Rocket6DOFBatch(n_envs, device=DEV, seed=4)
    b.reset()
    p = _params(4)
    p.w2.div_(50.0)
    cfg = PPOConfig(use_sde=True, n_steps=T, batch_size=bs, n_epochs=1, ent_coef=0.01)
    ro = b.collect_rollout(T, p.mlp(), tensor_cores=3)
    host = {k: ro[k].contiguous().cpu().numpy().reshape(T * n_envs, -1) for k in ("obs", "actions")}
    host.update({k: ro[k].cpu().numpy().reshape(-1) for k in ("log_probs", "advantages", "returns", "values")})
    trainer = PPOTrainer(b, p, cfg, seed=4)
    steps = []
    real = ppo.adam_step

    def adam_step(params, grad_sum, m, v, **kw):
        rec = dict(params=params.cpu().numpy(), m=m.cpu().numpy(), v=v.cpu().numpy(), **kw)
        real(params, grad_sum, m, v, **kw)
        rec["post"] = params.cpu().numpy()
        steps.append(rec)

    perms = []
    real_lg = ppo.loss_and_grad

    def loss_and_grad(params, rollout, idx, **kw):
        perms.append(idx.cpu().numpy())
        return real_lg(params, rollout, idx, **kw)

    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(ppo, "adam_step", adam_step)
        mp.setattr(ppo, "loss_and_grad", loss_and_grad)
        log = trainer.train(ro)
    assert [len(q) for q in perms] == [bs, bs, bs, T * n_envs - 3 * bs] and len(steps) == 4
    worst, ents = 0.0, []
    for st, idx in zip(steps, perms):
        adv_n = sde_ref.tr.normalized_advantages(host["advantages"][idx], True)
        err = np.zeros(sde_ref.NPARAMS_SDE)
        for c in range(0, len(idx), 1000):                   # per-sample magnitudes from the host build, in chunks
            q = idx[c:c + 1000]
            g, _ = sde_hostsim.ppo_sde_sample_grad(st["params"], host["obs"][q], host["actions"][q], host["log_probs"][q],
                                                   adv_n[c:c + 1000], host["returns"][q], clip=cfg.clip_range,
                                                   vf_coef=cfg.vf_coef, ent_coef=cfg.ent_coef)
            err += np.abs(g.astype(np.float64)).sum(0)
        ref = sde_ref.reference_step(st["params"], st["m"], st["v"], st["step"], host, idx, st["lr"], cfg, err_sum=err)
        r = np.abs(st["post"].astype(np.float64) - ref["p"]) / ref["bound"]
        worst = max(worst, r.max())
        ents.append(ref["entropy"])
        assert r.max() <= 1.0, (st["step"], r.max(), int(r.argmax()))
        if st["step"] == 1:                                  # teeth: one log_std entry off by 1e-3
            bad = st["params"].copy()
            bad[10308 + 3 * 7 + 2] += 1e-3
            ref2 = sde_ref.reference_step(bad, st["m"], st["v"], st["step"], host, idx, st["lr"], cfg, err_sum=err)
            r2 = (np.abs(st["post"].astype(np.float64) - ref2["p"]) / ref2["bound"]).max()
            print(f"teeth (log_std[7][2] + 1e-3): {r2:.1f} x bound")
            assert r2 > 1.0
    print(f"gSDE trainer: worst |post-step - reference| / bound = {worst:.3f}")
    assert abs(log["train/entropy_loss"] + np.mean(ents)) <= 1e-5 * abs(np.mean(ents))
    assert log["train/std"] == pytest.approx(float(np.exp(p.log_std.double().cpu().numpy()).mean()), rel=1e-12)

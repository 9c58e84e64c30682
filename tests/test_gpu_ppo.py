"""r6_ppo_grad / r6_adam_step and the PPO trainer on the GPU, against the float64 reference of tests/ppo_ref.py."""
import numpy as np
import pytest
import torch

import policy_ref as pr
import ppo_ref as rf

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _params(w):
    from rl_rocket_6dof_b200.ppo import ActorCriticParams
    return ActorCriticParams.from_weights(w, DEV)


def _rollout(x, a, old, adv, ret, T, strided):
    """[T, N] rollout tensors over n = T * N samples; obs dense [T, N, 13] or the strided view of a [T + 1, 14, N] buffer."""
    n = len(x) // T
    t = lambda v, *s: torch.from_numpy(np.ascontiguousarray(v, np.float32)).to(DEV).reshape(*s)
    obs = t(x, T, n, 13)
    if strided:
        buf = torch.full((T + 1, 14, n), float("nan"), device=DEV)
        buf[:T, :13] = obs.permute(0, 2, 1)
        obs = buf[:T, :13].permute(0, 2, 1)
    return dict(obs=obs, actions=t(a, T, n, 3), log_probs=t(old, T, n), advantages=t(adv, T, n), returns=t(ret, T, n),
                values=t(ret, T, n))


def _check(w, x, a, old, adv, ret, idx, T=4, strided=False, ent=0.0):
    from rl_rocket_6dof_b200 import ppo
    ro = _rollout(x, a, old, adv, ret, T, strided)
    g, terms = ppo.loss_and_grad(_params(w), ro, torch.from_numpy(idx).to(DEV), ent_coef=ent,
                                 normalize_advantage=len(idx) > 1)
    g, terms = g.cpu().numpy().astype(np.float64), terms.cpu().numpy()
    xs, As = x[idx], adv[idx]
    st = rf.adv_stats(As) if len(idx) > 1 else np.array([0.0, 1.0])
    q = rf.per_sample(w, xs, a[idx], old[idx], (As.astype(np.float64) - st[0]) * st[1], ret[idx], ent_coef=ent)
    g64, t64 = rf.grad_sum(q)
    bnd, tb = rf.bound(q, ent_coef=ent, samples_per_cta=rf.samples_per_cta(len(idx)))
    return g, terms, g64, t64, bnd, tb


SIZES = [1, 31, 128, 129, 2 * 148 * 128 + 129]


@pytest.mark.parametrize("family", pr.FAMILIES)
@pytest.mark.parametrize("B", SIZES)
def test_grad_within_bound(family, B):
    w = pr.weights(family)
    T, n = 4, 10000
    rng = np.random.default_rng(B)
    x = pr.obs_sets(T * n, seed=B)["golden" if B % 2 else "normal5"]
    a, old, adv, ret = rf.minibatch(w, x, seed=B)
    idx = rng.choice(T * n, B, replace=B > T * n // 2)
    if B > 200:
        idx[:50] = idx[50:100]                         # duplicates
        idx[100:300].sort()                            # a sorted stretch
    for strided in (False, True):
        g, terms, g64, t64, bnd, tb = _check(w, x, a, old, adv, ret, idx, T, strided)
        r = np.abs(g - g64) / bnd
        assert np.all(r <= rf.C_BAR), (family, B, strided, float(r.max()), int(r.argmax()))
        assert terms[2] == t64[2] and terms[4] == 0
        assert np.all(np.abs(terms[[0, 1, 3]] - t64[[0, 1, 3]]) <= rf.C_BAR * tb[[0, 1, 3]])
        if strided:
            assert np.array_equal(g, g_dense)
        g_dense = g


def test_grad_at_training_minibatch_sizes():
    """B = 2^18 + 129, the size class of the trainer's minibatches (2^16 envs x 32 steps / 4 = 2^19): every CTA
    accumulates 14 tiles with dW1 parked in shared memory between them, where the SIZES above reach about 2.  Drawn
    without replacement from a T = 32 rollout; dense and strided obs.  Not in the SIZES cross-product: the reference
    costs about 35 s of CPU here.  It is summed in chunks (grad_sum and bound are sums over samples, with the global
    samples_per_cta), so host memory stays near 1 GB."""
    from rl_rocket_6dof_b200 import ppo
    w = pr.weights("golden")
    B, T, n = 2 ** 18 + 129, 32, 8400
    x = pr.obs_sets(T * n, seed=11)["golden"]
    a, old, adv, ret = rf.minibatch(w, x, seed=11)
    idx = np.random.default_rng(11).choice(T * n, B, replace=False)
    st = rf.adv_stats(adv[idx])
    spc = rf.samples_per_cta(B)
    assert spc == 14 * 128
    g64, t64, bnd, tb = 0.0, 0.0, 0.0, 0.0
    for s in range(0, B, 1 << 15):
        j = idx[s:s + (1 << 15)]
        q = rf.per_sample(w, x[j], a[j], old[j], (adv[j].astype(np.float64) - st[0]) * st[1], ret[j])
        g_c, t_c = rf.grad_sum(q)
        b_c, tb_c = rf.bound(q, samples_per_cta=spc)
        g64, t64, bnd, tb = g64 + g_c, t64 + t_c, bnd + b_c, tb + tb_c
    for strided in (False, True):
        ro = _rollout(x, a, old, adv, ret, T, strided)
        g, terms = ppo.loss_and_grad(_params(w), ro, torch.from_numpy(idx).to(DEV))
        g, terms = g.cpu().numpy().astype(np.float64), terms.cpu().numpy()
        r = np.abs(g - g64) / bnd
        print(f"B {B} strided {strided}: max |kernel - ref| / bound {r.max():.3g}, median bound / |g| "
              f"{np.median(bnd / np.maximum(np.abs(g64), 1e-30)):.3g}")
        assert np.all(r <= rf.C_BAR), (strided, float(r.max()), int(r.argmax()))
        assert terms[2] == t64[2] and terms[4] == 0
        assert np.all(np.abs(terms[[0, 1, 3]] - t64[[0, 1, 3]]) <= rf.C_BAR * tb[[0, 1, 3]])
        if strided:
            assert np.array_equal(g, g_dense)
        g_dense = g


def test_bound_has_teeth_and_runs_are_reproducible():
    from rl_rocket_6dof_b200 import ppo
    w = pr.weights("golden")
    B = 256                  # the bound is first order and conservative (~1e-3 of sum |contribution|): small B for teeth
    x = pr.obs_sets(4 * B, seed=9)["golden"]
    a, old, adv, ret = rf.minibatch(w, x, seed=9)
    idx = np.random.default_rng(1).permutation(4 * B)[:B]
    g, terms, g64, _, bnd, _ = _check(w, x, a, old, adv, ret, idx)
    assert np.all(np.abs(g - g64) <= rf.C_BAR * bnd)
    g1, *_ = _check(w, x, a, old, adv, ret, idx[1:])
    assert np.any(np.abs(g1 - g64) > rf.C_BAR * bnd)              # one sample dropped
    ro = _rollout(x, a, old, adv, ret, 4, True)
    p = _params(w)
    it = torch.from_numpy(idx).to(DEV)
    g_raw, _ = ppo.loss_and_grad(p, ro, it, normalize_advantage=False)
    assert np.any(np.abs(g_raw.cpu().numpy() - g64) > rf.C_BAR * bnd)   # normalisation omitted
    ga, ta = ppo.loss_and_grad(p, ro, it)
    gb, tb_ = ppo.loss_and_grad(p, ro, it)
    assert torch.equal(ga, gb) and torch.equal(ta, tb_)
    # the two halves sum to the whole (same normalisation stats: raw advantages, no normalisation)
    g_h1, _ = ppo.loss_and_grad(p, ro, it[:B // 2], normalize_advantage=False)
    g_h2, _ = ppo.loss_and_grad(p, ro, it[B // 2:], normalize_advantage=False)
    q = rf.per_sample(w, x[idx], a[idx], old[idx], adv[idx].astype(np.float64), ret[idx])
    bnd_raw, _ = rf.bound(q, samples_per_cta=rf.samples_per_cta(B))
    assert np.all(np.abs((g_h1 + g_h2).double().cpu().numpy() - g_raw.double().cpu().numpy()) <= 2 * rf.C_BAR * bnd_raw)
    # an index outside the rollout is counted and skipped
    bad = it.clone()
    bad[3] = 4 * B
    _, tbad = ppo.loss_and_grad(p, ro, bad)
    assert float(tbad[4]) == 1.0


@pytest.mark.parametrize("max_norm", [0.5, 1e6])
def test_adam_step_matches_torch(max_norm):
    from rl_rocket_6dof_b200 import ppo
    rng = np.random.default_rng(2)
    P, B = ppo.NPARAMS, 256
    p = torch.from_numpy(rng.standard_normal(P).astype(np.float32)).to(DEV)
    pt = torch.nn.Parameter(p.clone())
    opt = torch.optim.Adam([pt], lr=3e-4, eps=1e-5)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    norm = torch.zeros(1, dtype=torch.float64, device=DEV)
    for step in range(1, 4):
        gs = torch.from_numpy((rng.standard_normal(P) * 0.05 * B).astype(np.float32)).to(DEV)
        ppo.adam_step(p, gs, m, v, lr=3e-4, step=step, scale=1.0 / B, max_grad_norm=max_norm, grad_norm=norm)
        pt.grad = gs * np.float32(1.0 / B)
        tn = torch.nn.utils.clip_grad_norm_([pt], max_norm)
        opt.step()
        assert abs(float(norm) - float(tn)) <= 1e-5 * float(tn)
        # float32 on both sides, different rounding order: 8 ulp of the parameter
        ulp = torch.abs(pt.detach()) * 2.0 ** -23
        assert torch.all(torch.abs(p - pt.detach()) <= 8 * ulp + 1e-9), float((torch.abs(p - pt.detach()) / ulp).max())
    assert (float(norm) > max_norm) == (max_norm == 0.5)


def _trainer(seed):
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    from rl_rocket_6dof_b200.ppo import ActorCriticParams, PPOConfig, PPOTrainer
    env = Rocket6DOFBatch(4096, device=DEV, seed=seed)
    params = ActorCriticParams.sb3_init(seed, DEV)
    return env, params, PPOTrainer(env, params, PPOConfig(n_steps=16, n_epochs=2, batch_size=4096 * 16 // 4), seed=seed)


def test_trainer_end_to_end(tmp_path):
    from rl_rocket_6dof_b200 import policy
    runs = []
    for _ in range(2):
        env, params, tr = _trainer(3)
        env.reset()
        ro = env.collect_rollout(16, params.mlp())
        k0 = torch.zeros(5, dtype=torch.float64, device=DEV)
        from rl_rocket_6dof_b200 import ppo
        idx = torch.randperm(4096 * 16, generator=torch.Generator(device=DEV).manual_seed(0), device=DEV)[:16384]
        _, t0 = ppo.loss_and_grad(params, ro, idx)
        assert float(t0[2]) == 0 and float(t0[3]) / 16384 < 1e-8       # collected with the same weights
        log = tr.train(ro)
        logs = tr.learn(4096 * 16 * 2)
        runs.append((params.flat.clone(), log, logs))
        for d in [log] + logs:
            assert all(np.isfinite(v) for v in d.values() if isinstance(v, float)), d
    assert torch.equal(runs[0][0], runs[1][0]) and runs[0][1] == runs[1][1]
    assert runs[0][1]["train/n_updates"] == 2
    env.reset()
    ro = env.collect_rollout(4, params.mlp(), tensor_cores=3)
    assert torch.isfinite(ro["actions"]).all() and torch.isfinite(ro["values"]).all()
    path = str(tmp_path / "trained.npz")
    params.save_npz(path)
    w = policy.load_npz(path)
    for k, v in params.mlp().items():
        assert np.array_equal(w[k], v.cpu().numpy().reshape(w[k].shape)), k


def test_grad_on_collected_rollout():
    """Observations, actions and log-probs from a real collect_rollout (strided obs view) within the bound."""
    from rl_rocket_6dof_b200 import ppo
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    w = pr.weights("golden")
    env = Rocket6DOFBatch(2048, device=DEV, seed=5)
    env.reset()
    p = _params(w)
    ro = env.collect_rollout(8, p.mlp(), tensor_cores=0)
    B = 8 * 2048
    idx = torch.randperm(B, device=DEV, generator=torch.Generator(device=DEV).manual_seed(1))
    g, terms = ppo.loss_and_grad(p, ro, idx)
    i = idx.cpu().numpy()
    f = lambda t, c: t.reshape(-1, c).cpu().numpy()[i] if c > 1 else t.reshape(-1).cpu().numpy()[i]
    x, a, old, adv, ret = f(ro["obs"].contiguous(), 13), f(ro["actions"], 3), f(ro["log_probs"], 1), f(ro["advantages"], 1), f(ro["returns"], 1)
    st = rf.adv_stats(adv)
    q = rf.per_sample(w, x, a, old, (adv.astype(np.float64) - st[0]) * st[1], ret)
    g64, t64 = rf.grad_sum(q)
    bnd, _ = rf.bound(q, samples_per_cta=rf.samples_per_cta(B))
    assert np.all(np.abs(g.cpu().numpy().astype(np.float64) - g64) <= rf.C_BAR * bnd)
    assert float(terms[2]) == t64[2] == 0

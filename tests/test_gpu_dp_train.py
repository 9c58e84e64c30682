"""Data-parallel PPO training (PPOTrainer(..., group=...)) on the GPU.

1. r6_rank_sum is numpy's float64 rank-order sum rounded to float32, bit for bit, and writes nothing on R6_EINVAL.
2. Collection is shard-invariant: two shards side by side are the rollout of one batch of both shards' envs.
3. One data-parallel Adam step (two shards on one GPU: per-shard gradient with the global advantage statistics,
   r6_rank_sum, adam_step) against tests/ppo_train_ref.py on the union minibatch, within the sum of the per-shard
   ppo_ref bounds plus the rank sum's one float32 rounding; the other layouts and value clipping at the gradient level
   against their existing float64 references.
4. Two spawned ranks on gloo (both on cuda:0) run learn on every layout: replicas, logs and reruns bit-identical, a
   size-1 group bit-identical to group=None, an inconsistent shard refused on both ranks.
5. With two GPUs: the same run on NCCL over cuda:0 / cuda:1 is bit-identical to the gloo run.
The multi-process harness rendezvous through a FileStore under tmp_path, sets timeouts, destroys its process group in a
finally, and joins (or terminates) every child."""
import datetime
import os
import time

import numpy as np
import pytest
import torch

import ppo_ref as rf
import ppo_train_ref as tr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U = 2.0 ** -24
SEP = [dict(pi=[64, 64], vf=[64, 64])]
LAYOUTS = {"shared": {}, "sde": dict(use_sde=True), "sep": dict(net_arch=SEP), "sepsde": dict(use_sde=True, net_arch=SEP)}


# ---------------------------------------------------------------------------------------------------- 1. r6_rank_sum

def _ref_sum(rows):
    acc = np.zeros(rows.shape[1])
    for r in rows:
        acc = acc + r.astype(np.float64)
    return acc


@pytest.mark.parametrize("P", [1, 3, 10375, 10564, (1 << 20) + 5])
@pytest.mark.parametrize("W", [1, 2, 3, 8])
def test_rank_sum_is_the_rank_order_float64_sum(W, P):
    from rl_rocket_6dof_b200 import ppo
    rng = np.random.default_rng(W * 7919 + P)
    g = (rng.standard_normal((W, P)) * 10.0 ** rng.integers(-6, 7, (W, P))).astype(np.float32)
    t = rng.standard_normal((W, 6)) * 10.0 ** rng.integers(-8, 9, (W, 6))
    want_g, want_t = _ref_sum(g).astype(np.float32), _ref_sum(t)
    got_g, got_t = ppo.rank_sum(torch.from_numpy(g).to(DEV), torch.from_numpy(t).to(DEV))
    assert np.array_equal(got_g.cpu().numpy().view(np.int32), want_g.view(np.int32))
    assert np.array_equal(got_t.cpu().numpy().view(np.int64), want_t.view(np.int64))


def test_rank_sum_base_pointers_need_only_element_alignment():
    """Rows of P = 10375 start at 4 g P bytes; base pointers one float / one double past an allocation work too."""
    from rl_rocket_6dof_b200 import _lib
    L = _lib.load()
    W, P, NT = 3, 10375, 5
    rng = np.random.default_rng(3)
    g = torch.from_numpy(rng.standard_normal(W * P + 1).astype(np.float32)).to(DEV)
    t = torch.from_numpy(rng.standard_normal(W * NT + 1)).to(DEV)
    go, to = torch.zeros(P + 1, dtype=torch.float32, device=DEV), torch.zeros(NT + 1, dtype=torch.float64, device=DEV)
    _lib.check(L.r6_rank_sum(g.data_ptr() + 4, t.data_ptr() + 8, W, P, NT, go.data_ptr() + 4, to.data_ptr() + 8,
                             torch.cuda.current_stream().cuda_stream), L)
    want_g = _ref_sum(g[1:].cpu().numpy().reshape(W, P)).astype(np.float32)
    want_t = _ref_sum(t[1:].cpu().numpy().reshape(W, NT))
    assert np.array_equal(go[1:].cpu().numpy(), want_g) and go[0] == 0
    assert np.array_equal(to[1:].cpu().numpy(), want_t) and to[0] == 0


def test_rank_sum_einval_writes_nothing():
    from rl_rocket_6dof_b200 import _lib
    L = _lib.load()
    W, P, NT = 2, 64, 5
    g = torch.ones(W * P + 4, dtype=torch.float32, device=DEV)
    t = torch.ones(W * NT + 2, dtype=torch.float64, device=DEV)
    go = torch.full((P + 4,), 7.0, dtype=torch.float32, device=DEV)
    to = torch.full((NT + 2,), 7.0, dtype=torch.float64, device=DEV)
    gp, tp, gop, top = g.data_ptr(), t.data_ptr(), go.data_ptr(), to.data_ptr()
    s = torch.cuda.current_stream().cuda_stream
    cases = {"world 0": (gp, tp, 0, P, NT, gop, top), "world -1": (gp, tp, -1, P, NT, gop, top),
             "P 0": (gp, tp, W, 0, NT, gop, top), "nterms -1": (gp, tp, W, P, -1, gop, top),
             "W P overflows": (gp, tp, 8, 1 << 62, NT, gop, top),
             "grads NULL": (None, tp, W, P, NT, gop, top), "grad_out NULL": (gp, tp, W, P, NT, None, top),
             "terms NULL": (gp, None, W, P, NT, gop, top), "terms_out NULL": (gp, tp, W, P, NT, gop, None),
             "grads misaligned": (gp + 2, tp, W, P, NT, gop, top), "grad_out misaligned": (gp, tp, W, P, NT, gop + 1, top),
             "terms misaligned": (gp, tp + 4, W, P, NT, gop, top), "terms_out misaligned": (gp, tp, W, P, NT, gop, top + 4)}
    for name, args in cases.items():
        assert L.r6_rank_sum(*args, s) == -1, name
        torch.cuda.synchronize()
        assert bool((go == 7).all()) and bool((to == 7).all()), name
    # nterms = 0 takes NULL terms pointers and writes the gradient half only
    assert L.r6_rank_sum(gp, None, W, P, 0, gop, None, s) == 0
    torch.cuda.synchronize()
    assert bool((go[:P] == W).all()) and bool((go[P:] == 7).all()) and bool((to == 7).all())


def test_rank_sum_reversed_order_fails_on_crafted_rows():
    """1 + 1e30 - 1e30: the kernel's rank order gives 0, the reverse 1 (and the same for the float64 terms)."""
    from rl_rocket_6dof_b200 import ppo
    g = np.array([[1.0], [1e30], [-1e30]], np.float32)
    t = np.array([[1.0], [1e20], [-1e20]])
    got_g, got_t = ppo.rank_sum(torch.from_numpy(g).to(DEV), torch.from_numpy(t).to(DEV))
    assert float(got_g[0]) == 0.0 and float(got_t[0]) == 0.0
    assert _ref_sum(g[::-1])[0] == 1.0 and _ref_sum(t[::-1])[0] == 1.0      # what a reversed sum would give


# ---------------------------------------------------------------------------------------------- 2. shard invariance

N_SH, T_SH = 1024, 8
_SHARDS = {}
KEYS = ("obs", "actions", "log_probs", "values", "rewards", "dones", "advantages", "returns")


def _shards(kind):
    """(params, [shard 0 rollout, shard 1 rollout], rollout of one batch of both shards' 2 N_SH envs) for a layout."""
    if kind not in _SHARDS:
        from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
        from rl_rocket_6dof_b200.ppo import ActorCriticParams
        from rl_rocket_6dof_b200.sharding import shard_batch_kwargs
        p = ActorCriticParams.sb3_init(seed=11, device=DEV, **LAYOUTS[kind])
        envs = [Rocket6DOFBatch(N_SH, device=DEV, seed=21, **shard_batch_kwargs(N_SH, r, 2)) for r in range(2)]
        envs.append(Rocket6DOFBatch(2 * N_SH, device=DEV, seed=21))
        ros = []
        for e in envs:
            e.reset()
            ros.append(e.collect_rollout(T_SH, p.mlp(), bootstrap_truncated=True,
                                         sde_sample_freq=3 if p.use_sde else -1))
        _SHARDS[kind] = (p, ros[:2], ros[2])
    return _SHARDS[kind]


@pytest.mark.parametrize("kind", list(LAYOUTS))
def test_collection_is_shard_invariant(kind):
    _, (a, b), full = _shards(kind)
    for k in KEYS:
        assert torch.equal(torch.cat([a[k], b[k]], dim=1), full[k]), k


# ------------------------------------------------------------------------------ 3. one data-parallel step vs SB3

def _host(ro):
    T, n = ro["advantages"].shape
    h = {k: ro[k].contiguous().cpu().numpy().reshape(T * n, -1) for k in ("obs", "actions")}
    h.update({k: ro[k].cpu().numpy().reshape(-1) for k in ("log_probs", "advantages", "returns", "values")})
    return h


def _minibatch(seed, B_local):
    """Each shard's local indices (a seeded draw without replacement) and their union's global sample ids."""
    rng = np.random.default_rng(seed)
    idx = [rng.permutation(T_SH * N_SH)[:B_local] for _ in range(2)]
    glob = np.concatenate([(i // N_SH) * (2 * N_SH) + r * N_SH + i % N_SH for r, i in enumerate(idx)])
    return [torch.from_numpy(i).to(DEV) for i in idx], idx, glob


def _dp_gradient(p, ros, idx, per_shard_std=False, drop=None, **kw):
    """What PPOTrainer.train does per minibatch with a group, on one GPU: the global advantage statistics from the
    shards' (count, mean, M2), each shard's gradient sum, r6_rank_sum.  Returns (grad, terms, adv_stats)."""
    from rl_rocket_6dof_b200 import ppo
    moms = torch.stack([ppo.local_moments(ro["advantages"].reshape(-1)[i].double()) for ro, i in zip(ros, idx)])
    n, mean, m2 = ppo.combine_moments(moms)
    st = torch.stack([mean, 1.0 / (torch.sqrt(m2 / (n - 1)) + 1e-8)])
    gs, ts = [], []
    for r, (ro, i) in enumerate(zip(ros, idx)):
        if r == drop:
            continue
        g, t = ppo.loss_and_grad(p, ro, i, adv_stats=None if per_shard_std else st, **kw)
        gs.append(g.clone())
        ts.append(t.clone())
    g, t = ppo.rank_sum(torch.stack(gs), torch.stack(ts))
    return g, t, st


def _shard_bound(per_sample, bound, grad, w, host, idx, st, B_local):
    """Bound on |rank-summed kernel gradient - exact gradient of the union|: the per-shard bounds plus one float32
    rounding of the float64 rank sum of the two kernel sums (|sum| <= |G_0| + |G_1| + b_0 + b_1)."""
    b_tot, mag = 0.0, 0.0
    for h, i in zip(host, idx):
        adv_n = (h["advantages"][i].astype(np.float64) - st[0]) * st[1]
        q = per_sample(w, h["obs"][i], h["actions"][i], h["log_probs"][i], adv_n, h["returns"][i], h, i)
        b = bound(q, B_local)
        b_tot, mag = b_tot + b, mag + np.abs(grad(q)) + b
    return b_tot + U * mag


def _weights(p):
    return {k: v.detach().cpu().numpy() for k, v in p.mlp().items()}


def test_dp_adam_steps_match_sb3_on_the_union():
    """Two consecutive data-parallel Adam steps (the second from the kernels' own m, v) against SB3's step on the
    union minibatch of the concatenated rollout; dropping one shard's gradient, or normalising each shard with its own
    std, fails the same bound."""
    from rl_rocket_6dof_b200 import ppo
    from rl_rocket_6dof_b200.ppo import PPOConfig
    p0, ros, full = _shards("shared")
    hfull, hs = _host(full), [_host(r) for r in ros]
    cfg = PPOConfig()
    p = ppo.ActorCriticParams(p0.flat.clone())
    m, v = torch.zeros_like(p.flat), torch.zeros_like(p.flat)
    B_local, lr = 2048, 3e-4
    b1, b2 = tr.BETAS
    for step in (1, 2):
        idx_t, idx, glob = _minibatch(step, B_local)
        B = 2 * B_local
        pre = dict(p=p.flat.cpu().numpy(), m=m.cpu().numpy(), v=v.cpu().numpy())
        g, t, st = _dp_gradient(p, ros, idx_t)
        st_ref = rf.adv_stats(hfull["advantages"][glob])
        assert np.allclose(st.cpu().numpy(), st_ref, rtol=1e-12, atol=0)
        ref = tr.reference_step(pre["p"], pre["m"], pre["v"], step, hfull, glob, lr, cfg)
        w = tr.unflat(pre["p"])
        e_sum = _shard_bound(lambda w, x, a, o, an, r, h, i: rf.per_sample(w, x, a, o, an, r),
                             lambda q, Bl: rf.bound(q, samples_per_cta=rf.samples_per_cta(Bl))[0],
                             lambda q: rf.grad_sum(q)[0], w, hs, idx, st_ref, B_local)
        m64, v64 = pre["m"].astype(np.float64), pre["v"].astype(np.float64)
        gc = ref["clip"] * ref["grad"]
        mp, vp = m64 + (1 - b1) * (gc - m64), b2 * v64 + (1 - b2) * gc * gc
        bound = tr.step_bound(ref["grad"], e_sum / B, ref["norm"], cfg.max_grad_norm, gc, m64, mp, vp, ref["p"], lr, step)

        def ratio(grad):
            q = p.flat.clone()
            mm, vv = m.clone(), v.clone()
            ppo.adam_step(q, grad, mm, vv, lr=lr, step=step, scale=1.0 / B, max_grad_norm=cfg.max_grad_norm)
            return float(np.max(np.abs(q.cpu().numpy().astype(np.float64) - ref["p"]) / bound)), q, mm, vv

        r, q, mm, vv = ratio(g)
        print(f"step {step}: B {B} max |dp step - SB3 step| / bound {r:.3g}")
        assert r <= rf.C_BAR
        if step == 2:
            r_drop = ratio(_dp_gradient(p, ros, idx_t, drop=1)[0])[0]
            r_std = ratio(_dp_gradient(p, ros, idx_t, per_shard_std=True)[0])[0]
            print(f"teeth: one shard dropped {r_drop:.3g}, per-shard std {r_std:.3g}")
            assert min(r_drop, r_std) > rf.C_BAR
        p.flat.copy_(q)
        m.copy_(mm)
        v.copy_(vv)


@pytest.mark.parametrize("kind", ["sep", "vfclip", "sde", "sepsde"])
def test_dp_gradient_of_other_layouts(kind):
    """The rank-summed gradient of the separate towers and of value clipping within the sum of the per-shard bounds of
    sep_ref / vfclip_ref plus the rank sum's rounding; gSDE (both trunks) within tests/test_gpu_vfclip.py's gSDE
    criterion for r6_ppo_grad_sde against sde_ref / sepsde_ref on the union."""
    import sde_ref
    import sep_ref
    import sepsde_ref
    import vfclip_ref as vr
    cvf = 0.2
    p, ros, full = _shards("shared" if kind == "vfclip" else kind)
    hfull, hs = _host(full), [_host(r) for r in ros]
    B_local = 2048
    idx_t, idx, glob = _minibatch(5, B_local)
    kw = dict(clip_range_vf=cvf) if kind == "vfclip" else {}
    g, t, _ = _dp_gradient(p, ros, idx_t, **kw)
    g = g.cpu().numpy().astype(np.float64)
    w = _weights(p)
    st = rf.adv_stats(hfull["advantages"][glob])
    u = lambda k: hfull[k][glob]
    adv_u = (u("advantages").astype(np.float64) - st[0]) * st[1]
    if kind == "sep":
        G = sep_ref.grad_sum(w, u("obs"), u("actions"), u("log_probs"), adv_u, u("returns"))[0]
        tol = _shard_bound(lambda w, x, a, o, an, r, h, i: (w, x, a, o, an, r),
                           lambda q, Bl: sep_ref.bound(*q, samples_per_cta=rf.samples_per_cta(Bl)),
                           lambda q: sep_ref.grad_sum(*q)[0], w, hs, idx, st, B_local)
        worst = float(np.max(np.abs(g - G) / (tol + 1e-300)))
        assert worst <= 1.0, worst
    elif kind == "vfclip":
        q = vr.per_sample(w, u("obs"), u("actions"), u("log_probs"), adv_u, u("returns"), u("values"), cvf)
        G = rf.grad_sum(q)[0]
        tol = _shard_bound(lambda w, x, a, o, an, r, h, i: vr.per_sample(w, x, a, o, an, r, h["values"][i], cvf),
                           lambda q, Bl: vr.bound(q, samples_per_cta=rf.samples_per_cta(Bl))[0],
                           lambda q: rf.grad_sum(q)[0], w, hs, idx, st, B_local)
        worst = float(np.max(np.abs(g - G) / tol))
        assert worst <= rf.C_BAR, worst
    else:
        ref = sde_ref if kind == "sde" else sepsde_ref
        G = ref.grad_sum(w, u("obs"), u("actions"), u("log_probs"), adv_u, u("returns"))[0]
        err, scale = np.abs(g - G), np.abs(G).max() + 1e-6
        worst = float(err.max() / scale)
        assert worst <= 1e-4
    print(f"{kind}: worst {worst:.3g}")


# ------------------------------------------------------------------------------------- 4 / 5. spawned ranks, learn

N_DP, T_DP, ITERS = 256, 8, 2
DP_CASES = {"shared": ({}, dict(clip_range=lambda p: 0.1 + 0.1 * p)),
            "sde": (dict(use_sde=True), dict(use_sde=True, sde_sample_freq=4)),
            "sep": (dict(net_arch=SEP), dict(learning_rate=lambda p: 3e-4 * p)),
            "sepsde": (dict(use_sde=True, net_arch=SEP),
                       dict(use_sde=True, clip_range_vf=0.2, target_kl=0.002, learning_rate=3e-3))}


def _learn(case, rank, world, dev, group, params_seed):
    """A short learn of DP_CASES[case] on rank's shard; returns flat arrays {flat, m, v, logs, adam_steps}."""
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    from rl_rocket_6dof_b200.ppo import ActorCriticParams, PPOConfig, PPOTrainer
    from rl_rocket_6dof_b200.sharding import shard_batch_kwargs
    pk, ck = DP_CASES[case]
    env = Rocket6DOFBatch(N_DP, device=dev, seed=31, **shard_batch_kwargs(N_DP, rank, world))
    params = ActorCriticParams.sb3_init(seed=params_seed, device=dev, **pk)
    trainer = PPOTrainer(env, params, PPOConfig(n_steps=T_DP, n_epochs=2, **ck), seed=9, group=group)
    logs = trainer.learn(ITERS * T_DP * N_DP * world)
    keys = sorted(logs[0])
    return dict(flat=params.flat.cpu().numpy(), m=trainer.m.cpu().numpy(), v=trainer.v.cpu().numpy(),
                logs=np.array([[float(log[k]) for k in keys] for log in logs]), keys=np.array(keys),
                adam_steps=np.array(trainer.adam_steps), timesteps=np.array(trainer.num_timesteps))


def _dp_worker(rank, world, backend, store_path, out_path, devices):
    import torch.distributed as dist
    dev = torch.device(devices[rank])
    torch.cuda.set_device(dev)
    store = dist.FileStore(store_path, world)
    kw = dict(device_id=dev) if backend == "nccl" else {}
    dist.init_process_group(backend, store=store, rank=rank, world_size=world, timeout=datetime.timedelta(seconds=240),
                            **kw)
    try:
        res = {}
        for case in DP_CASES:
            for rep in range(2):      # params drawn per rank: the broadcast from rank 0 must make them agree
                for k, val in _learn(case, rank, world, dev, dist.group.WORLD, params_seed=100 + rank).items():
                    res[f"{case}/dp{rep}/{k}"] = val
        if backend == "gloo":
            singles = [dist.new_group([r]) for r in range(world)]    # every rank creates every group, in order
            for case in DP_CASES:
                for tag, grp in (("one", singles[rank]), ("none", None)):
                    for k, val in _learn(case, 0, 1, dev, grp, params_seed=100).items():
                        res[f"{case}/{tag}/{k}"] = val
        # an inconsistent shard: rank 1 claims rank 0's env range
        from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
        from rl_rocket_6dof_b200.ppo import ActorCriticParams, PPOConfig, PPOTrainer
        env = Rocket6DOFBatch(N_DP, device=dev, seed=31, env_offset=0, num_envs_global=world * N_DP)
        try:
            PPOTrainer(env, ActorCriticParams.sb3_init(seed=1, device=dev), PPOConfig(n_steps=T_DP), group=dist.group.WORLD)
            res["bad_shard_error"] = np.array("")
        except ValueError as e:
            res["bad_shard_error"] = np.array(str(e))
        dist.barrier()
        np.savez(out_path, **res)
    finally:
        dist.destroy_process_group()


def _spawn(backend, devices, tmp):
    """Two ranks of _dp_worker; every child is joined, and terminated if it outlives the deadline (which fails)."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    outs = [os.path.join(tmp, f"{backend}_rank{r}.npz") for r in range(2)]
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, backend, os.path.join(tmp, f"store_{backend}"), outs[r], devices))
             for r in range(2)]
    for p in procs:
        p.start()
    deadline = time.monotonic() + 1200
    survivors = []
    try:
        for p in procs:
            p.join(timeout=max(1.0, deadline - time.monotonic()))
    finally:
        survivors = [p for p in procs if p.is_alive()]
        for p in survivors:
            p.terminate()
        for p in survivors:
            p.join(timeout=30)
            if p.is_alive():
                p.kill()
                p.join()
    assert not survivors, f"{len(survivors)} rank(s) did not finish"
    assert [p.exitcode for p in procs] == [0, 0]
    return [dict(np.load(o)) for o in outs]


@pytest.fixture(scope="module")
def gloo_runs(tmp_path_factory):
    return _spawn("gloo", ["cuda:0", "cuda:0"], str(tmp_path_factory.mktemp("dp_gloo")))


def _eq(x, y):
    """Bit equality of two result arrays (strings compared as strings)."""
    x, y = np.atleast_1d(x), np.atleast_1d(y)
    if x.dtype != y.dtype or x.shape != y.shape:
        return False
    return np.array_equal(x.view(np.uint8), y.view(np.uint8)) if x.dtype.kind in "fiub" else np.array_equal(x, y)


@pytest.mark.timeout(1800)
@pytest.mark.parametrize("case", list(DP_CASES))
def test_gloo_ranks_stay_bit_identical(gloo_runs, case):
    r0, r1 = gloo_runs
    for k in ("flat", "m", "v", "logs", "keys", "adam_steps", "timesteps"):
        assert _eq(r0[f"{case}/dp0/{k}"], r1[f"{case}/dp0/{k}"]), k        # replicas and logs agree across ranks
        assert _eq(r0[f"{case}/dp0/{k}"], r0[f"{case}/dp1/{k}"]), k        # a rerun is bit-identical
    assert int(r0[f"{case}/dp0/timesteps"]) == ITERS * T_DP * N_DP * 2
    logs, keys = r0[f"{case}/dp0/logs"], list(r0[f"{case}/dp0/keys"])
    assert logs[-1, keys.index("rollout/steps")] == T_DP * N_DP * 2          # the group's episode statistics
    assert not np.array_equal(r0[f"{case}/dp0/flat"], r0[f"{case}/none/flat"])  # the update is not the one-rank one


@pytest.mark.timeout(1800)
@pytest.mark.parametrize("case", list(DP_CASES))
def test_size_one_group_is_group_none(gloo_runs, case):
    for r in gloo_runs:
        for k in ("flat", "m", "v", "logs", "keys", "adam_steps", "timesteps"):
            assert _eq(r[f"{case}/one/{k}"], r[f"{case}/none/{k}"]), k


@pytest.mark.timeout(1800)
def test_inconsistent_shard_raises_on_every_rank(gloo_runs):
    msgs = [str(r["bad_shard_error"]) for r in gloo_runs]
    assert all("env_offset" in m for m in msgs) and msgs[0] == msgs[1], msgs


@pytest.mark.timeout(1800)
def test_nccl_on_two_gpus_equals_gloo_on_one(gloo_runs, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    nccl = _spawn("nccl", ["cuda:0", "cuda:1"], str(tmp_path))
    for case in DP_CASES:
        for k in ("flat", "m", "v", "logs", "adam_steps"):
            for a, b in zip(nccl, gloo_runs):
                assert _eq(a[f"{case}/dp0/{k}"], b[f"{case}/dp0/{k}"]), (case, k)

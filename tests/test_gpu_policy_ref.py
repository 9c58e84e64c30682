"""The policy kernels (r6_policy_range / r6_policy_ex, tensor_cores = 0..3, and the network copies inside the fused rollout
kernel) against the float64 actor-critic of tests/policy_ref.py within its derived error bound, and their Gaussian
exploration noise and log-probabilities against the NumPy statement of the Philox / Box-Muller head (tests/philox_ref.py)
— on freshly initialised, saturating and TF32-edge networks as well as the trained one, at tile-size edges, env
sub-ranges, shards, poisoned rows, and the tails of the uniform grids."""
import ctypes as C
import functools

import numpy as np
import pytest

import philox_ref as pr
import policy_ref as ref
from parity_utils import env_params

pytestmark = pytest.mark.gpu

MODES = ref.MODES
FAMILIES = ref.FAMILIES


def _lib():
    from rl_rocket_6dof_b200 import _lib
    return _lib, _lib.load()


def _dev(w):
    from rl_rocket_6dof_b200 import policy
    return policy.to_device(w, "cuda:0")


def _obs_cm(x):
    """float32 [n,13] -> the component-major [13, n] device layout the kernels read."""
    import torch
    return torch.from_numpy(np.ascontiguousarray(np.asarray(x, np.float32).T)).cuda()


def launch(wd, obs, mode, stochastic=False, seed=0, env_offset=0, step=0, first=0, count=None, nulls=False, outs=None):
    """One r6_policy_range launch over obs [13, n]; returns (actions, raw, values, log_prob) as float32 NumPy arrays
    (None for the outputs passed as NULL)."""
    import torch
    _l, L = _lib()
    n = obs.shape[1]
    count = n - first if count is None else count
    if outs is None:
        outs = (torch.empty(n, 3, device="cuda"), torch.empty(n, 3, device="cuda"), torch.empty(n, device="cuda"),
                torch.empty(n, device="cuda"))
    act, raw, val, lp = outs
    m = _l.make_mlp(wd)
    ptr = (lambda t: None) if nulls else (lambda t: t.data_ptr())
    _l.check(L.r6_policy_range(C.byref(m), obs.data_ptr(), n, first, count, int(mode), int(bool(stochastic)), int(seed),
                               int(env_offset), int(step), act.data_ptr(), ptr(raw), ptr(val), ptr(lp),
                               torch.cuda.current_stream().cuda_stream), L)
    torch.cuda.synchronize()
    if nulls:
        return act.cpu().numpy(), None, None, None
    return tuple(t.cpu().numpy() for t in (act, raw, val, lp))


def test_whole_batch_entry_points_equal_policy_range():
    """r6_policy (deterministic actions) and r6_policy_ex (actions, raw actions, values, log-probs) give the bits of
    r6_policy_range over (0, n)."""
    import torch
    _l, L = _lib()
    n = 4097
    wd = _dev(ref.weights("golden"))
    x = _obs_cm(ref.obs_sets(n, seed=7)["normal5"])
    m = _l.make_mlp(wd)
    st = torch.cuda.current_stream().cuda_stream
    for mode in (0, 3):
        a = torch.empty(n, 3, device="cuda")
        _l.check(L.r6_policy(C.byref(m), x.data_ptr(), n, mode, a.data_ptr(), st), L)
        torch.cuda.synchronize()
        assert np.array_equal(a.cpu().numpy(), launch(wd, x, mode, nulls=True)[0]), mode
        for stochastic in (False, True):
            outs = (torch.empty(n, 3, device="cuda"), torch.empty(n, 3, device="cuda"), torch.empty(n, device="cuda"),
                    torch.empty(n, device="cuda"))
            _l.check(L.r6_policy_ex(C.byref(m), x.data_ptr(), n, mode, int(stochastic), 5, 100, 3,
                                    *(t.data_ptr() for t in outs), st), L)
            torch.cuda.synchronize()
            for got, want in zip(outs, launch(wd, x, mode, stochastic, 5, 100, 3)):
                assert np.array_equal(got.cpu().numpy(), want), (mode, stochastic)


def noise_bar(seed, genv, step):
    """(z_ref [n,3], bar [n,3]) for the device noise of (seed, genv, step): philox_ref.policy_noise_bar (3 ulp)."""
    z = pr.policy_noise(seed, genv, step)
    return z, pr.policy_noise_bar(z, seed, genv, step)


def log_prob_bar(z, dz, ls):
    """|log_prob_kernel - SB3 float64 log_prob(z_ref)|: per term -0.5 z z - ls - c, four float32 roundings, plus the
    running sum of three terms (12 roundings of at most 2^-24 of the magnitudes), and the first-order effect of the
    noise error |z| dz + dz^2 / 2."""
    lsa = np.zeros(3) if ls is None else np.abs(np.asarray(ls, np.float64))
    mag = (0.5 * z * z + lsa + pr.LOG_SQRT_2PI).sum(1)
    return 12 * 2.0 ** -24 * mag + (np.abs(z) * dz + 0.5 * dz * dz).sum(1)


# ---- fixtures -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def obs_all():
    """The observation sets of policy_ref plus the observations of a 64-step closed-loop rollout of the trained policy
    (every phase of an episode), 2048 rows each."""
    import torch
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    sets = ref.obs_sets(2048, seed=3)
    env = Rocket6DOFBatch(2048, params=env_params(), device="cuda:0", seed=9)
    env.reset()
    env.step_policy(64, _dev(ref.weights("golden")), tensor_cores=3)
    torch.cuda.synchronize()
    sets["rollout64"] = env.obs[:13].t().contiguous().cpu().numpy()
    return np.concatenate([sets[k] for k in ("golden", "uniform", "normal5", "rollout64")])


@pytest.fixture(scope="module")
def refs(obs_all):
    """{family: (mean64, value64, {mode: bound})} on obs_all."""
    out = {}
    for fam in FAMILIES:
        w = ref.weights(fam)
        m, v = ref.forward64(w, obs_all)
        out[fam] = (m, v, {mode: ref.bound(w, obs_all, mode) for mode in MODES})
    return out


# ---- the network ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", MODES)
def test_forward_within_float64_bound(mode, obs_all, refs):
    """Mean, value, clipped action and log-prob of every mode on every family, deterministic and stochastic, against
    forward64 within C_BAR x bound; outputs without log_std / critic; NULL outputs leave the actions unchanged."""
    x = _obs_cm(obs_all)
    seed, off, step = (1 << 32) + 77, 12345, 9
    genv = np.arange(off, off + len(obs_all), dtype=np.uint64)
    z_ref, dz = noise_bar(seed, genv, step)
    for fam in FAMILIES:
        w = ref.weights(fam)
        m64, v64, bnd = refs[fam]
        b = bnd[mode]
        wd = _dev(w)
        a, raw, val, lp = launch(wd, x, mode)
        err = np.abs(np.concatenate([raw, val[:, None]], 1) - np.concatenate([m64, v64[:, None]], 1))
        ratio = err / b
        print(f"mode {mode} {fam:10s}: worst |kernel - forward64| / bound = {ratio.max():.3f} (mean {ratio[:, :3].max():.3f}, "
              f"value {ratio[:, 3].max():.3f})")
        assert np.all(np.isfinite(raw)) and np.all(err <= ref.C_BAR * b), (mode, fam, ratio.max())
        assert np.array_equal(a, np.clip(raw, -1, 1))
        assert np.all(lp == pr.log_prob_at_mean(w["log_std"]))
        # stochastic: same network, mean + std z, SB3's log-prob at the noise
        a_s, raw_s, val_s, lp_s = launch(wd, x, mode, True, seed, off, step)
        std = np.exp(w["log_std"].astype(np.float32)).astype(np.float64)
        assert np.array_equal(val_s, val) and np.array_equal(a_s, np.clip(raw_s, -1, 1))
        target = m64 + std * z_ref
        tol = ref.C_BAR * b[:, :3] + std * dz + 2.0 ** -24 * (np.abs(m64) + 2 * np.abs(target)) + 2.0 ** -23 * std * np.abs(z_ref)
        assert np.all(np.abs(raw_s - target) <= tol), (mode, fam)
        assert np.all(np.abs(lp_s - pr.gaussian_log_prob(z_ref, w["log_std"])) <= log_prob_bar(z_ref, dz, w["log_std"]))
        # NULL raw / values / log_prob: the actions are the same bits
        for stoch, ref_a in ((False, a), (True, a_s)):
            an, _, _, _ = launch(wd, x, mode, stoch, seed, off, step, nulls=True)
            assert np.array_equal(an, ref_a)
    # without log_std: std 1; without the critic: values exactly 0
    w = ref.weights("golden")
    bare = {k: v for k, v in w.items() if k not in ("wv", "bv", "log_std")}
    m64, _, bnd = refs["golden"]
    a, raw, val, lp = launch(_dev(bare), x, mode, True, seed, off, step)
    assert np.all(val == 0)
    assert np.all(np.abs(raw - (m64 + z_ref)) <= ref.C_BAR * bnd[mode][:, :3] + dz + 2.0 ** -23 * (np.abs(m64) + np.abs(z_ref) + 1))
    assert np.all(np.abs(lp - pr.gaussian_log_prob(z_ref, None)) <= log_prob_bar(z_ref, dz, None))
    _, _, _, lp_d = launch(_dev(bare), x, mode)
    assert np.all(lp_d == pr.log_prob_at_mean(None))


def test_bar_can_fail(obs_all, refs):
    """The single-pass TF32 mode (2) misses the faithful bar of mode 3 on the trained and the freshly initialised network:
    the bound is tight enough to catch a dropped 3xTF32 correction term."""
    x = _obs_cm(obs_all)
    for fam in ("golden", "sb3_init"):
        m64, v64, bnd = refs[fam]
        _, raw, val, _ = launch(_dev(ref.weights(fam)), x, 2)
        err = np.abs(np.concatenate([raw, val[:, None]], 1) - np.concatenate([m64, v64[:, None]], 1))
        r = (err / bnd[3]).max()
        print(f"mode 2 {fam}: worst error / bound(mode 3) = {r:.2f}")
        assert r > ref.C_BAR, fam


# ---- the noise ----------------------------------------------------------------------------------------------------------
def _noise_check(mode, seed, env_offset, step, n, x_row, w):
    """Launch n envs with identical observations; z = (raw_stochastic - raw_deterministic) / std against policy_noise.
    Returns (worst |dz| / bar, #non-finite, genv of the worst, z)."""
    import torch
    wd = _dev(w)
    x = torch.from_numpy(np.ascontiguousarray(x_row.reshape(13, 1))).cuda().expand(13, n).contiguous()
    _, raw_d, _, _ = launch(wd, x, mode)
    _, raw_s, _, lp = launch(wd, x, mode, True, seed, env_offset, step)
    std = np.exp(w["log_std"].astype(np.float64))
    genv = np.arange(env_offset, env_offset + n, dtype=np.uint64)
    z_ref, dz = noise_bar(seed, genv, step)
    bad = int((~np.isfinite(raw_s)).sum() + (~np.isfinite(lp)).sum())
    z = (raw_s.astype(np.float64) - raw_d) / std
    # recovering z from raw costs the roundings of mean + RN(std z): 2^-24 (|raw_d| + |raw_s|) / std
    rec = 2.0 ** -24 * (np.abs(raw_d) + np.abs(raw_s)) / std
    r = np.abs(z - z_ref) / (dz + rec)
    worst = float(np.nanmax(np.where(np.isfinite(r), r, np.inf)))
    i = int(np.argmax(np.where(np.isfinite(r), r, np.inf).max(1)))
    assert np.all(np.abs(lp - pr.gaussian_log_prob(z_ref, w["log_std"])) <= log_prob_bar(z_ref, dz, w["log_std"]))
    return worst, bad, int(genv[i]), z


@pytest.mark.parametrize("mode", MODES)
def test_noise_matches_policy_noise(mode):
    """2^22 envs x 3 dims of device noise against policy_noise, with a seed, env ids and a step index above 2^32 (the env
    range straddles 2^32), and the same launch shifted by env_offset: shards draw different, matching noise."""
    w = ref.weights("sb3_init")
    x_row = ref.obs_sets(1)["uniform"][0]
    n = 1 << 22
    worst, bad, g, z = _noise_check(mode, (1 << 32) + 3, (1 << 32) - (1 << 21), (1 << 32) + 5, n, x_row, w)
    print(f"mode {mode}: noise of 2^22 envs: worst |dz| / bar = {worst:.3f} (genv {g}), non-finite {bad}")
    assert bad == 0 and worst <= 1.0
    assert abs(z.mean()) < 2e-3 and abs(z.std() - 1) < 2e-3


@functools.lru_cache(maxsize=None)
def _tail_envs(seed, step, n):
    """Global env ids in [0, n) whose Philox block puts u1 / u3 in the top or bottom 32 values of the 2^24 grid, or
    u2 / u4 within 2^-20 of 0, 1/2 or 1."""
    hits = []
    for lo in range(0, n, 1 << 22):
        genv = np.arange(lo, min(n, lo + (1 << 22)), dtype=np.uint64)
        r = pr.policy_block(seed, genv, step)
        k1, k3 = r[:, 0] >> np.uint32(8), r[:, 2] >> np.uint32(8)
        sel = (k1 < 32) | (k1 >= (1 << 24) - 32) | (k3 < 32) | (k3 >= (1 << 24) - 32)
        for c in (1, 3):
            u = r[:, c].astype(np.float64) / 2.0 ** 32
            sel |= (np.abs(u) < 2.0 ** -20) | (np.abs(u - 0.5) < 2.0 ** -20) | (np.abs(u - 1.0) < 2.0 ** -20)
        hits.append(genv[sel])
    return np.concatenate(hits)


@pytest.mark.parametrize("mode", MODES)
def test_noise_tails(mode):
    """The Box-Muller tails: every env of a 2^24-env launch is finite, and the envs whose uniforms sit at the ends of
    their grids (u1, u3 -> 1, where ln u is tiny and an absolutely accurate log would be off by all of it; u1, u3 -> 0,
    where the radius is largest; angles near 0, pi and 2 pi) are evaluated one env per launch through env_offset and
    checked against policy_noise."""
    import torch
    seed, step, n = 21, 6, 1 << 24
    w = ref.weights("sb3_init")
    x_row = ref.obs_sets(1)["uniform"][0]
    wd = _dev(w)
    x = torch.from_numpy(np.ascontiguousarray(x_row.reshape(13, 1))).cuda().expand(13, n).contiguous()
    _, raw_s, _, lp = launch(wd, x, mode, True, seed, 0, step)
    assert np.all(np.isfinite(raw_s)) and np.all(np.isfinite(lp))
    del x
    tails = _tail_envs(seed, step, n)
    assert len(tails) >= 200
    x1 = _obs_cm(x_row.reshape(1, 13))
    _, raw_d, _, _ = launch(wd, x1, mode)
    z_ref, dz = noise_bar(seed, tails, step)
    std = np.exp(w["log_std"].astype(np.float64))
    z = np.empty_like(z_ref)
    lps = np.empty(len(tails))
    for j, g in enumerate(tails):
        _, rs, _, l1 = launch(wd, x1, mode, True, seed, int(g), step)
        z[j] = (rs[0].astype(np.float64) - raw_d[0]) / std
        lps[j] = l1[0]
        assert np.array_equal(rs[0], raw_s[int(g)])           # the one-env launch is the same env as in the big one
    # recovering z from raw costs the roundings of mean + RN(std z)
    r = np.abs(z - z_ref) / (dz + 2.0 ** -24 * (np.abs(raw_d[0]) + np.abs(raw_s[tails])) / std)
    k1 = pr.policy_block(seed, tails, step)[:, 0] >> np.uint32(8)
    top = k1 >= (1 << 24) - 32
    print(f"mode {mode}: {len(tails)} tail envs, worst |dz| / bar = {r.max():.3f}; u1 at the top of the grid: {int(top.sum())} "
          f"envs, their |z0 - ref| max {np.abs(z - z_ref)[top, 0].max() if top.any() else 0:.2e}")
    assert np.all(np.isfinite(z)) and np.all(r <= 1.0)
    assert np.all(np.abs(lps - pr.gaussian_log_prob(z_ref, w["log_std"])) <= log_prob_bar(z_ref, dz, w["log_std"]))


# ---- ranges, shards, rows -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", MODES)
def test_sub_ranges_bit_identical(mode):
    """r6_policy_range over unaligned sub-ranges: rows inside are the bits of the full launch, rows outside keep a
    sentinel, for every output."""
    import torch
    n = 1000
    w = ref.weights("golden")
    wd = _dev(w)
    x = _obs_cm(ref.obs_sets(n, seed=4)["uniform"])
    full = launch(wd, x, mode, True, 5, 100, 3)
    for first in (1, 31, 300):
        for count in (1, 127, 129, n - first - 3):
            outs = (torch.full((n, 3), 7.0, device="cuda"), torch.full((n, 3), 7.0, device="cuda"),
                    torch.full((n,), 7.0, device="cuda"), torch.full((n,), 7.0, device="cuda"))
            got = launch(wd, x, mode, True, 5, 100, 3, first=first, count=count, outs=outs)
            for g, f in zip(got, full):
                assert np.array_equal(g[first:first + count], f[first:first + count]), (mode, first, count)
                assert np.all(g[:first] == 7) and np.all(g[first + count:] == 7), (mode, first, count)


@pytest.mark.parametrize("mode", MODES)
def test_shards_bit_identical(mode):
    """One batch split into 2 and 3 shards (env_offset, num_envs_global, observation slices): the concatenated
    stochastic outputs are the bits of the unsharded launch."""
    import torch
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    n = 5000
    w = _dev(ref.weights("tf32_edges"))
    obs = _obs_cm(ref.obs_sets(n, seed=5)["normal5"])
    whole = Rocket6DOFBatch(n, params=env_params(), device="cuda:0", seed=77)
    whole.obs[:13].copy_(obs)
    full = [t.cpu().numpy() for t in whole.policy_forward(w, stochastic=True, tensor_cores=mode, step_index=11)]
    for cuts in ((0, 2345, n), (0, 129, 3000, n)):
        parts = []
        for a, b in zip(cuts[:-1], cuts[1:]):
            s = Rocket6DOFBatch(b - a, params=env_params(), device="cuda:0", seed=77, env_offset=a, num_envs_global=n)
            s.obs[:13].copy_(obs[:, a:b])
            parts.append([t.cpu().numpy() for t in s.policy_forward(w, stochastic=True, tensor_cores=mode, step_index=11)])
        torch.cuda.synchronize()
        for k in range(4):
            assert np.array_equal(np.concatenate([p[k] for p in parts]), full[k]), (mode, cuts, k)


@pytest.mark.parametrize("mode", MODES)
def test_poisoned_rows_stay_in_their_rows(mode):
    """NaN, +-inf and 1e30 observations in rows 0, 77, 128 and n - 1: every other row is bit-identical to the launch in
    which those rows are zeros (the tensor-core modes put 16 or 128 rows in one MMA tile)."""
    n = 4097
    x = ref.obs_sets(n, seed=6)["uniform"]
    rows = [0, 77, 128, n - 1]
    clean = x.copy()
    clean[rows] = 0
    dirty = x.copy()
    dirty[0] = np.nan
    dirty[77] = np.inf
    dirty[77, ::2] = -np.inf
    dirty[128] = 1e30
    dirty[n - 1, :6] = np.nan
    dirty[n - 1, 6:] = -1e30
    wd = _dev(ref.weights("golden"))
    keep = np.setdiff1d(np.arange(n), rows)
    for stoch in (False, True):
        a = launch(wd, _obs_cm(clean), mode, stoch, 3, 0, 2)
        b = launch(wd, _obs_cm(dirty), mode, stoch, 3, 0, 2)
        for u, v in zip(a, b):
            assert np.array_equal(u[keep], v[keep]), (mode, stoch)


def test_tile_size_edges(obs_all):
    """Batch sizes around the warp (32), the tile (128) and the tile pair (256), and 2 SMs x 128 + 129 envs, which gives
    each tcgen05 tile group two slots with an odd tile count: every mode within its bound, deterministic and stochastic."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    sizes = (1, 31, 33, 127, 128, 129, 255, 256, 257, 4097, 2 * sms * 128 + 129)
    nmax = max(sizes)
    w = ref.weights("golden")
    x = np.concatenate([obs_all] * (nmax // len(obs_all) + 1))[:nmax]
    x = x + np.float32(1e-3) * np.random.default_rng(8).standard_normal(x.shape).astype(np.float32)
    m64, v64 = ref.forward64(w, x)
    wd = _dev(w)
    for mode in MODES:
        b = ref.bound(w, x, mode)
        for n in sizes:
            xc = _obs_cm(x[:n])
            a, raw, val, lp = launch(wd, xc, mode)
            err = np.abs(np.concatenate([raw, val[:, None]], 1) - np.concatenate([m64[:n], v64[:n, None]], 1))
            assert np.all(err <= ref.C_BAR * b[:n]), (mode, n)
            _, raw_s, _, lp_s = launch(wd, xc, mode, True, 4, 0, 1)
            assert np.all(np.isfinite(raw_s)) and np.all(np.isfinite(lp_s)) and not np.array_equal(raw_s, raw), (mode, n)


# ---- the other callers ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("family", FAMILIES)
def test_fused_rollout_network_within_bound(family):
    """The network inside the fused rollout kernel (R6_ACT_MLP: float32 FMA; R6_ACT_MLP_TC: mma.sync 3xTF32), one
    recorded step from the reference's closed-loop states, against forward64 within the mode-0 / mode-1 bars."""
    import torch
    from rl_rocket_6dof_b200.batch import ACT_MLP, ACT_MLP_TC, Rocket6DOFBatch
    g = np.load(ref.GOLD)
    starts = set(int(s) for s in g["ic_step"])
    idx = np.array([k for k in range(1, len(g["action"])) if k not in starts])
    w = ref.weights(family)
    for act_mode, name, mode in ((ACT_MLP, "R6_ACT_MLP", 0), (ACT_MLP_TC, "R6_ACT_MLP_TC", 1)):
        env = Rocket6DOFBatch(len(idx), params=env_params(), device="cuda:0", auto_reset=True, seed=3)
        st = g["state"][idx - 1]
        env.set_state(torch.from_numpy(st.astype(np.float32)))
        env.state.copy_(torch.from_numpy(np.ascontiguousarray(st.T)))
        traj = env.rollout(1, act_mode, mlp=_dev(w), record=True)
        torch.cuda.synchronize()
        a = traj["act"][0].cpu().numpy()
        x = traj["obs"][0].t().cpu().numpy()[:, :13]
        m64, _ = ref.forward64(w, x)
        b = ref.bound(w, x, mode)[:, :3]
        err = np.abs(a - np.clip(m64, -1, 1))                # the clip is 1-Lipschitz
        print(f"rollout {name} {family}: worst |action - clip(forward64)| / bound(mode {mode}) = {(err / b).max():.3f}")
        assert np.all(err <= ref.C_BAR * b), (family, name)


def test_collect_rollout_log_probs():
    """collect_rollout's log_probs against SB3's float64 formula at policy_noise with step = steps_done + j, and its raw
    actions against forward64 + std * policy_noise within the mode-3 bar."""
    import torch
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    w = ref.weights("golden")
    n, k = 3000, 12
    env = Rocket6DOFBatch(n, params=env_params(), device="cuda:0", seed=(1 << 33) + 5, env_offset=(1 << 32) - 1000,
                          num_envs_global=(1 << 32) + 4000)
    env.reset()
    env.step_policy(3, _dev(w))
    s0 = env.steps_done
    ro = env.collect_rollout(k, _dev(w), stochastic=True)
    torch.cuda.synchronize()
    genv = np.arange(env.env_offset, env.env_offset + n, dtype=np.uint64)
    std = np.exp(w["log_std"].astype(np.float64))
    obs = ro["obs"].cpu().numpy()
    acts = ro["actions"].cpu().numpy()
    lps = ro["log_probs"].cpu().numpy()
    for j in range(k):
        z_ref, dz = noise_bar(env.seed_value, genv, s0 + j)
        assert np.all(np.abs(lps[j] - pr.gaussian_log_prob(z_ref, w["log_std"])) <= log_prob_bar(z_ref, dz, w["log_std"])), j
        m64, _ = ref.forward64(w, obs[j])
        target = m64 + std * z_ref
        tol = ref.C_BAR * ref.bound(w, obs[j], 3)[:, :3] + std * dz + 2.0 ** -24 * (np.abs(m64) + 3 * np.abs(target))
        assert np.all(np.abs(acts[j] - target) <= tol), j

"""Stream lanes (r6_step_range): stepping disjoint env sub-ranges of one batch on several streams gives bit-identical
results to the single-stream kernel pair, joined every step or free-running."""
import ctypes as C

import numpy as np
import pytest

from parity_utils import env_params

pytestmark = pytest.mark.gpu

FIELDS = ("state", "obs", "reward", "reward_f32", "done", "flags", "step_count", "ep_return", "episode_id", "terminal_state",
          "terminal_obs", "ep_info", "m0", "v0")


def _mk(n, lanes, **kw):
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    return Rocket6DOFBatch(n, params=env_params(), seed=11, split_step=True, lanes=lanes, **kw)


def _same(a, b):
    import torch
    torch.cuda.synchronize()
    for f in FIELDS:
        assert torch.equal(getattr(a, f), getattr(b, f)), f
    sa, sb = a.stats.cpu().numpy(), b.stats.cpu().numpy()      # R6_S_*: counts exact, the two float sums to atomics order
    assert np.array_equal(sa[[0, 3, 4, 5, 6, 7]], sb[[0, 3, 4, 5, 6, 7]]) and np.allclose(sa, sb, rtol=1e-12, atol=0)


@pytest.mark.parametrize("lanes,n", [(2, 5000), (3, 4099), (4, 130)])
def test_lanes_equal_single_stream(lanes, n):
    import torch
    one, many = _mk(n, 1), _mk(n, lanes)
    assert sum(c for _, c in many._lane_ranges) == n and many._lane_ranges[0][0] == 0
    one.reset(); many.reset()
    acts = torch.from_numpy(np.random.default_rng(7).uniform(-1, 1, (150, n, 3)).astype(np.float32)).cuda()
    for k in range(150):                       # joined every step: outputs readable right after the call
        o1 = one.step(acts[k])
        o2 = many.step(acts[k])
        if k % 50 == 49:
            torch.cuda.synchronize()
            assert torch.equal(o1[0], o2[0]) and torch.equal(o1[2], o2[2])
    _same(one, many)
    assert float(one.stats[0]) > 0             # episodes ended and restarted on the way
    for k in range(60):                        # free-running, one join at the end
        one.step(acts[k])
        many.step(acts[k], join=False)
    many.join()
    _same(one, many)
    one.step_random(40)
    many.step_random(40)
    _same(one, many)
    one.step_random(30)
    many.step_random(30, join=False)
    many.join()
    _same(one, many)
    assert one.steps_done == many.steps_done


def test_lanes_follow_the_callers_stream():
    """The lanes wait for work enqueued on the caller's stream (the producer of the actions) and `join` orders the
    outputs back onto it."""
    import torch
    n = 3000
    one, many = _mk(n, 1), _mk(n, 2)
    one.reset(); many.reset()
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        for k in range(20):
            a = torch.rand(n, 3, device="cuda", generator=None) * 2 - 1      # produced on `side`
            many.step(a, join=False)
            one.step(a)
            many.join()
            got = many.reward.clone()                                         # consumed on `side`
            assert torch.equal(got, one.reward)
    torch.cuda.synchronize()
    _same(one, many)


def test_step_range_argument_checks():
    import torch
    from rl_rocket_6dof_b200 import _lib
    env = _mk(256, 1)
    env.reset()
    a = torch.zeros(256, 3, device="cuda")
    L = env.lib
    st = torch.cuda.current_stream().cuda_stream
    assert L.r6_step_range(C.byref(env._p), C.byref(env._b), 256, 0, 0, 0, 0, a.data_ptr(), 1, 0, st) == 0     # empty range
    for first, count in ((-1, 4), (0, 257), (200, 100), (0, -1)):
        assert L.r6_step_range(C.byref(env._p), C.byref(env._b), 256, first, count, 0, 0, a.data_ptr(), 1, 0, st) != 0
        assert b"sub-range" in L.r6_last_error()
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    fused = Rocket6DOFBatch(256, params=env_params(), split_step=False)
    fused.reset()
    assert L.r6_step_range(C.byref(fused._p), C.byref(fused._b), 256, 0, 256, 0, 0, a.data_ptr(), 1, 0, st) != 0
    assert b"scratch" in L.r6_last_error()
    assert L.r6_step_range(C.byref(env._p), C.byref(env._b), 256, 0, 256, 32, 0, a.data_ptr(), 1, 0, st) != 0
    assert b"lane" in L.r6_last_error()
    with pytest.raises(ValueError):
        _mk(2, 3)
    torch.cuda.synchronize()


@pytest.mark.parametrize("tc", [0, 1, 2])
def test_closed_loop_on_lanes(tc):
    """policy -> step chains per lane (r6_policy_range + r6_step_range) == the single-stream closed loop."""
    from rl_rocket_6dof_b200 import policy as pol
    rng = np.random.default_rng(4)
    w = {k: (rng.standard_normal(shp) * 0.2).astype(np.float32) for k, shp in pol.SHAPES.items()}
    n = 4099
    one, many = _mk(n, 1), _mk(n, 3)
    wd = pol.to_device(w, one.device)
    one.reset(); many.reset()
    one.step_policy(320, wd, tensor_cores=tc)
    many.step_policy(320, wd, tensor_cores=tc)
    _same(one, many)
    import torch
    assert torch.equal(one._policy_act, many._policy_act)
    assert float(one.stats[0]) > 0
    # free-running, then joined, with the weights dropped by the caller right after the call: the lanes still read them,
    # so their memory must not come back from the allocator (here as zeroed tensors of the same sizes) before the join
    one.step_policy(40, wd, tensor_cores=tc)
    many.step_policy(40, pol.to_device(w, many.device), tensor_cores=tc, join=False)
    zeros = [torch.zeros_like(t) for t in wd.values()]          # noqa: F841 (held until after the join)
    many.join()
    _same(one, many)
    assert torch.equal(one._policy_act, many._policy_act)


def test_collect_rollout_on_lanes():
    """PPO rollout collection per lane == single stream (stochastic policy: Philox noise keyed by global env id)."""
    import torch
    from rl_rocket_6dof_b200 import policy as pol
    rng = np.random.default_rng(5)
    w = {k: (rng.standard_normal(shp) * 0.2).astype(np.float32) for k, shp in pol.SHAPES.items()}
    w.update(wv=(rng.standard_normal(64) * 0.3).astype(np.float32), bv=np.zeros(1, np.float32),
             log_std=np.array([-1.0, -1.5, -2.0], np.float32))
    n, k = 2051, 48
    one, many = _mk(n, 1), _mk(n, 2)
    wd = {key: torch.from_numpy(v).cuda() for key, v in w.items()}
    one.reset(); many.reset()
    a = one.collect_rollout(k, wd)
    b = many.collect_rollout(k, wd)
    torch.cuda.synchronize()
    for key in a:
        assert torch.equal(a[key], b[key]), key
    _same(one, many)


def _close(a, b, tol):
    """Different kernels round differently in places (the compiler contracts a*b+c per instantiation), so two
    integrator variants agree to round-off, not to the bit; every discrete output must still be identical."""
    import torch
    torch.cuda.synchronize()
    norm = torch.as_tensor(np.asarray(a.params.state_normalizer, np.float64), device=a.device)[:, None]
    for f in ("done", "flags", "step_count", "episode_id"):
        assert torch.equal(getattr(a, f), getattr(b, f)), f
    err = float(((a.state.double() - b.state.double()).abs() / norm).max())
    assert err <= tol, err
    assert float((a.reward - b.reward).abs().max()) <= 1e-6
    return err


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
def test_multipass_integrator_equals_single_kernel(precision):
    """The integrator cut at RK-attempt boundaries (work lists, three passes) against the single-kernel integrator:
    identical attempt counts, solver status, done / flags at every step (including the rare 3-4 attempt steps),
    states equal to round-off; with and without stream lanes bit-identical to each other."""
    import torch
    n = 20000
    a = _mk(n, 1, multipass=False, precision=precision, record_attempts=True)
    b = _mk(n, 2, multipass=True, precision=precision, record_attempts=True)
    c = _mk(n, 1, multipass=True, precision=precision, record_attempts=True)
    assert a.work is None and b.work is not None
    for e in (a, b, c):
        e.reset()
    acts = torch.from_numpy(np.random.default_rng(9).uniform(-1, 1, (40, n, 3)).astype(np.float32)).cuda()
    seen = torch.zeros(8, dtype=torch.long, device="cuda")
    tol = 1e-10 if precision == "fp64" else 2e-3
    worst = 0.0
    for k in range(240):
        for e in (a, b, c):
            e.step(acts[k % 40])
        if precision == "fp64":
            assert torch.equal(a.nattempts, b.nattempts), k
            worst = max(worst, _close(a, b, tol))
        seen += torch.bincount(a.nattempts.long(), minlength=8)[:8]
    _same(b, c)
    assert int(seen[1]) > 0 and int(seen[2]) > 0 and int(seen[3]) > 0        # 1, 2 and >= 3 attempts all occurred
    assert int(torch.count_nonzero(b.work[:256])) == 0                        # work-list counters are back to zero
    for e in (a, b, c):
        e.step_random(30)
    _same(b, c)
    if precision == "fp32":                   # float32 round-off flips a few attempt counts / done flags: statistics
        sa, sb = a.stats.cpu().numpy(), b.stats.cpu().numpy()
        assert abs(sa[0] - sb[0]) <= 0.002 * sa[0] + 5
    print(f"multipass vs single kernel ({precision}): worst state difference {worst:.2e} of the normaliser")

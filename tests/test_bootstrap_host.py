"""The NumPy restatement of SB3's timeout bootstrap (tests/timeout_ref.py) on hand-made cases, and the C-ABI argument
checks of r6_trunc_record / r6_trunc_bootstrap (validated before any CUDA call, so no GPU is needed)."""
import numpy as np

import timeout_ref as tr

G = 0.99


def _two_roundings(r, v):
    return np.float32(np.float32(r) + np.float32(np.float32(G) * np.float32(v)))


def test_truncations_at_both_ends_and_twice_in_one_env():
    T, n = 6, 4
    rew = np.arange(T * n, dtype=np.float32).reshape(T, n) * np.float32(0.25) - np.float32(2.0)
    val = np.linspace(-3, 5, T * n, dtype=np.float32).reshape(T, n)
    trunc = np.zeros((T, n), bool)
    trunc[0, 0] = True                     # at t = 0
    trunc[T - 1, 1] = True                 # at t = k - 1
    trunc[1, 2] = trunc[4, 2] = True       # two truncations of one env
    out = tr.bootstrap_timeouts(rew, trunc, val, G)
    assert out.dtype == np.float32 and out.shape == (T, n)
    assert np.array_equal(out[~trunc], rew[~trunc])
    for t, i in zip(*np.nonzero(trunc)):
        assert out[t, i] == _two_roundings(rew[t, i], val[t, i]) and out[t, i] != rew[t, i]
    # no truncation: the rewards come back unchanged, whatever the values hold
    assert np.array_equal(tr.bootstrap_timeouts(rew, np.zeros_like(trunc), np.full_like(val, np.nan), G), rew)
    # the input is not modified
    assert np.array_equal(rew, np.arange(T * n, dtype=np.float32).reshape(T, n) * np.float32(0.25) - np.float32(2.0))


def test_two_roundings_differ_from_a_fused_multiply_add():
    """r = -0.5356694, V = 1.0847852: fl32(r + fl32(0.99f V)) = 0.538268 but the single-rounding fma gives 0.53826797.
    SB3's float32 ops are the former; a kernel that let the compiler contract them would compute the latter."""
    r, v = np.float32("-0.5356694"), np.float32("1.0847852")
    out = tr.bootstrap_timeouts(np.array([[r]]), np.array([[True]]), np.array([[v]]), G)[0, 0]
    assert out == np.float32("0.538268") == _two_roundings(r, v)
    assert tr.fma_f32(r, np.float32(G), v) == np.float32("0.53826797") != out


def test_abi_argument_checks():
    import ctypes as C
    from rl_rocket_6dof_b200 import _lib
    L = _lib.load()
    p = C.c_void_p(16)                      # never dereferenced: every call below fails its checks first
    assert L.r6_trunc_record(None, p, 8, 0, 8, 0, 1, p, p, None) == -1 and b"null" in L.r6_last_error()
    assert L.r6_trunc_record(p, p, -1, 0, 0, 0, 1, p, p, None) == -1 and b"n < 0" in L.r6_last_error()
    assert L.r6_trunc_record(p, p, 8, 4, 5, 0, 1, p, p, None) == -1 and b"sub-range" in L.r6_last_error()
    assert L.r6_trunc_record(p, p, 8, -1, 2, 0, 1, p, p, None) == -1 and b"sub-range" in L.r6_last_error()
    assert L.r6_trunc_record(p, p, 8, 0, 8, 0, -1, p, p, None) == -1 and b">= 0" in L.r6_last_error()
    assert L.r6_trunc_record(p, p, 8, 0, 8, -3, 1, p, p, None) == -1 and b">= 0" in L.r6_last_error()
    assert L.r6_trunc_record(p, p, 8, 0, 0, 0, 1, p, p, None) == 0          # empty range: nothing launched
    assert L.r6_trunc_record(p, p, 8, 0, 8, 0, 0, p, p, None) == 0          # no slots (no TimeLimit): nothing launched
    assert L.r6_trunc_bootstrap(p, 4, 8, 1, None, p, G, None) == -1 and b"null" in L.r6_last_error()
    assert L.r6_trunc_bootstrap(p, -1, 8, 1, p, p, G, None) == -1 and b"negative" in L.r6_last_error()
    assert L.r6_trunc_bootstrap(p, 4, 8, -2, p, p, G, None) == -1 and b"negative" in L.r6_last_error()
    assert L.r6_trunc_bootstrap(p, 4, 0, 1, p, p, G, None) == 0 and L.r6_trunc_bootstrap(p, 4, 8, 0, p, p, G, None) == 0

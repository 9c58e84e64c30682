"""TEST-ONLY host build of the CUDA kernels' per-environment math (see hostsim.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
LIB = os.path.join(HERE, "_build", "libhostsim.so")
DEPS = [os.path.join(HERE, "hostsim.cpp"), os.path.join(ROOT, "rl_rocket_6dof_b200", "csrc", "r6_core.cuh"),
        os.path.join(ROOT, "include", "r6dof.h")]


class HsEnv(C.Structure):
    _fields_ = [("y", C.c_double * 14), ("m0", C.c_float), ("v0", C.c_float), ("k", C.c_int32),
                ("episode", C.c_uint32), ("ep_return", C.c_double), ("tgo", C.c_float), ("pad", C.c_float)]


class HsOut(C.Structure):
    _fields_ = [("state", C.c_double * 14), ("obs", C.c_float * 14), ("reward", C.c_double),
                ("terms", C.c_double * 7), ("flags", C.c_int32), ("finished", C.c_int32), ("natt", C.c_int32),
                ("status", C.c_int32), ("tgo_missing", C.c_int32)]


ENV_DTYPE = np.dtype(HsEnv)
OUT_DTYPE = np.dtype(HsOut)
_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB) or any(os.path.getmtime(d) > os.path.getmtime(LIB) for d in DEPS):
            os.makedirs(os.path.dirname(LIB), exist_ok=True)
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                                   "-DR6_HOST_BUILD", "-o", LIB, DEPS[0], "-lm"])
        L = C.CDLL(LIB)
        assert L.hs_sizeof_env() == C.sizeof(HsEnv) and L.hs_sizeof_out() == C.sizeof(HsOut)
        L.hs_tgo.restype = C.c_double
        L.hs_tgo.argtypes = [C.c_double] * 4
        L.hs_tgo_warm.restype = C.c_double
        L.hs_tgo_warm.argtypes = [C.c_double] * 5
        L.hs_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
        L.hs_reset.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_uint64]
        L.hs_sim_step_raw.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_double, C.POINTER(C.c_int)]
        L.hs_sim_step_raw_passes.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_double, C.POINTER(C.c_int),
                                             C.POINTER(C.c_int)]
        L.hs_euler_tests.argtypes = [C.c_void_p] * 3 + [C.POINTER(C.c_int)] * 2
        L.hs_philox.argtypes = [C.c_uint32] * 6 + [C.c_void_p]
        L.hs_philox_action.argtypes = [C.c_uint64] * 3 + [C.c_void_p]
        L.hs_mlp_pack.argtypes = [C.c_void_p, C.c_void_p]
        L.hs_mlp.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
        L.hs_mlp_forward.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
        L.hs_gaussian_head.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_uint64, C.c_void_p, C.c_void_p, C.c_int64,
                                       C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


class HostSimBatch:
    """N envs stepped by the host build of the kernel code (mirrors oracle.c_oracle.OracleBatch)."""

    def __init__(self, ep, n, **struct_kw):
        self.ep = ep
        self.p = ep.to_struct(**struct_kw)
        self.t_table = np.ascontiguousarray(ep.t_table, np.float64)
        self.n = n
        self.envs = np.zeros(n, ENV_DTYPE)
        self.outs = np.zeros(n, OUT_DTYPE)

    def set_state(self, y, m0, k, v0=0.0, idx=None):
        idx = np.arange(self.n) if idx is None else np.atleast_1d(idx)
        self.envs["y"][idx] = y
        self.envs["m0"][idx] = m0
        self.envs["k"][idx] = k
        self.envs["v0"][idx] = v0
        self.envs["tgo"][idx] = 0.0          # a new episode starts cold

    def step(self, actions):
        a = np.ascontiguousarray(actions, np.float32).reshape(self.n, 3)
        lib().hs_step(C.byref(self.p), self.t_table.ctypes.data, self.envs.ctypes.data, self.n, a.ctypes.data,
                      self.outs.ctypes.data)
        return self.outs


def _packed(weights):
    from rl_rocket_6dof_b200._lib import make_mlp
    L = lib()
    w = {k: np.ascontiguousarray(v, np.float32) for k, v in weights.items()}
    m = make_mlp(w)
    W = np.zeros(L.hs_mlp_floats(), np.float32)
    L.hs_mlp_pack(C.byref(m), W.ctypes.data)
    return W


def mlp_actions(weights, obs13):
    """Fused-policy network of the kernels (host build) on packed weights: obs [n,13] f32 -> actions [n,3]."""
    W = _packed(weights)
    x = np.ascontiguousarray(obs13, np.float32).reshape(-1, 13)
    out = np.zeros((len(x), 3), np.float32)
    lib().hs_mlp(W.ctypes.data, x.ctypes.data, len(x), out.ctypes.data)
    return out


def mlp_forward(weights, obs13):
    """Raw outputs of the same network: (unclipped mean [n,3], value [n]; 0 without a critic head)."""
    W = _packed(weights)
    x = np.ascontiguousarray(obs13, np.float32).reshape(-1, 13)
    out = np.zeros((len(x), 4), np.float32)
    lib().hs_mlp_forward(W.ctypes.data, x.ctypes.data, len(x), out.ctypes.data)
    return out[:, :3], out[:, 3]


def gaussian_head(mean, log_std, stochastic, seed, genv, step):
    """Host build of the kernels' Gaussian policy head: (raw action [n,3], log-prob [n]) for mean [n,3] and per-row
    global env ids / step indices (uint64)."""
    mean = np.asarray(mean, np.float32).reshape(-1, 3)
    n = len(mean)
    m4 = np.zeros((n, 4), np.float32)
    m4[:, :3] = mean
    g = np.ascontiguousarray(np.broadcast_to(np.asarray(genv, np.uint64), (n,)))
    s = np.ascontiguousarray(np.broadcast_to(np.asarray(step, np.uint64), (n,)))
    ls = None if log_std is None else np.ascontiguousarray(log_std, np.float32)
    raw = np.zeros((n, 3), np.float32)
    logp = np.zeros(n, np.float32)
    lib().hs_gaussian_head(m4.ctypes.data, None if ls is None else ls.ctypes.data, int(bool(stochastic)), int(seed),
                           g.ctypes.data, s.ctypes.data, n, raw.ctypes.data, logp.ctypes.data)
    return raw, logp

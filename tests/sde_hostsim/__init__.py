"""TEST-ONLY host build of the gSDE noise draw and per-sample PPO math (see sde_hostsim.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
LIB = os.path.join(HERE, "_build", "libsde_hostsim.so")
CSRC = os.path.join(ROOT, "rl_rocket_6dof_b200", "csrc")
DEPS = [os.path.join(HERE, "sde_hostsim.cpp"), os.path.join(CSRC, "r6_ppo.cuh"), os.path.join(CSRC, "r6_core.cuh"),
        os.path.join(ROOT, "include", "r6dof.h")]
_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB) or any(os.path.getmtime(d) > os.path.getmtime(LIB) for d in DEPS):
            os.makedirs(os.path.dirname(LIB), exist_ok=True)
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                                   "-DR6_HOST_BUILD", "-o", LIB, DEPS[0], "-lm"])
        L = C.CDLL(LIB)
        L.hs_sde_noise.argtypes = [C.c_uint64, C.c_void_p, C.c_uint64, C.c_int64, C.c_void_p]
        L.hs_ppo_sde_sample_grad.argtypes = [C.c_void_p] * 6 + [C.c_int64, C.c_void_p, C.c_float, C.c_float, C.c_float,
                                                                 C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def sde_noise(seed, genv, step):
    """Host build of the gSDE noise draw: xi [n, 192] for global env ids genv [n] and draw step `step`."""
    g = np.ascontiguousarray(np.atleast_1d(np.asarray(genv, np.uint64)))
    xi = np.zeros((len(g), 192), np.float32)
    lib().hs_sde_noise(int(seed), g.ctypes.data, int(step), len(g), xi.ctypes.data)
    return xi


def ppo_sde_sample_grad(params, obs13, act3, old_logp, adv, ret, adv_stats=None, clip=0.2, vf_coef=0.5, ent_coef=0.0):
    """Host build of the gSDE per-sample PPO math: (grad [n, R6_PPO_NPARAMS_SDE], terms [n, 5] = pg, vloss, clipped, kl,
    entropy)."""
    L = lib()
    f = lambda a, *shape: np.ascontiguousarray(np.asarray(a, np.float32).reshape(*shape))
    x, a = f(obs13, -1, 13), f(act3, -1, 3)
    n = len(x)
    old, ad, rt, p = f(old_logp, n), f(adv, n), f(ret, n), f(params, -1)
    st = None if adv_stats is None else np.ascontiguousarray(adv_stats, np.float64)
    grad = np.zeros((n, L.hs_ppo_sde_nparams()), np.float32)
    terms = np.zeros((n, 5), np.float32)
    L.hs_ppo_sde_sample_grad(p.ctypes.data, x.ctypes.data, a.ctypes.data, old.ctypes.data, ad.ctypes.data, rt.ctypes.data, n,
                             None if st is None else st.ctypes.data, clip, vf_coef, ent_coef, grad.ctypes.data,
                             terms.ctypes.data)
    return grad, terms

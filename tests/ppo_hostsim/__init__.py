"""TEST-ONLY host build of the PPO update's per-sample math and Adam step (see ppo_hostsim.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
LIB = os.path.join(HERE, "_build", "libppo_hostsim.so")
CSRC = os.path.join(ROOT, "rl_rocket_6dof_b200", "csrc")
DEPS = [os.path.join(HERE, "ppo_hostsim.cpp"), os.path.join(CSRC, "r6_ppo.cuh"), os.path.join(CSRC, "r6_core.cuh"),
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
        L.hs_ppo_sample_grad.argtypes = [C.c_void_p] * 6 + [C.c_int64, C.c_void_p, C.c_float, C.c_float, C.c_float,
                                                             C.c_void_p, C.c_void_p]
        L.hs_adam_step.argtypes = [C.c_void_p] * 4 + [C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
        _lib = L
    return _lib


def ppo_sample_grad(params, obs13, act3, old_logp, adv, ret, adv_stats=None, clip=0.2, vf_coef=0.5, ent_coef=0.0):
    """Host build of the per-sample PPO math: (grad [n, R6_PPO_NPARAMS], terms [n, 4] = pg, vloss, clipped, kl)."""
    L = lib()
    f = lambda a, *shape: np.ascontiguousarray(np.asarray(a, np.float32).reshape(*shape))
    x, a = f(obs13, -1, 13), f(act3, -1, 3)
    n = len(x)
    old, ad, rt, p = f(old_logp, n), f(adv, n), f(ret, n), f(params, -1)
    st = None if adv_stats is None else np.ascontiguousarray(adv_stats, np.float64)
    P = L.hs_ppo_nparams()
    grad = np.zeros((n, P), np.float32)
    terms = np.zeros((n, 4), np.float32)
    L.hs_ppo_sample_grad(p.ctypes.data, x.ctypes.data, a.ctypes.data, old.ctypes.data, ad.ctypes.data, rt.ctypes.data, n,
                         None if st is None else st.ctypes.data, clip, vf_coef, ent_coef, grad.ctypes.data, terms.ctypes.data)
    return grad, terms


def adam_step(params, grad_sum, m, v, coef, step):
    """Host build of r6_adam_step, in place on float32 numpy arrays; returns the pre-clip norm."""
    norm = C.c_double()
    lib().hs_adam_step(params.ctypes.data, np.ascontiguousarray(grad_sum, np.float32).ctypes.data, m.ctypes.data,
                       v.ctypes.data, len(params), C.byref(coef), int(step), C.byref(norm))
    return norm.value

"""TEST-ONLY host build of the per-sample PPO math of r6_ppo_grad_sde_sep (see sepsde_hostsim.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
LIB = os.path.join(HERE, "_build", "libsepsde_hostsim.so")
CSRC = os.path.join(ROOT, "rl_rocket_6dof_b200", "csrc")
DEPS = [os.path.join(HERE, "sepsde_hostsim.cpp"), os.path.join(CSRC, "r6_ppo.cuh"), os.path.join(CSRC, "r6_core.cuh"),
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
        f = C.c_float
        L.hs_sepsde_sample_grad.argtypes = [C.c_void_p] * 7 + [C.c_int64, C.c_void_p, f, f, f, f, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def sample_grad(params, obs13, act3, old_logp, adv, ret, vold=None, vfc=0.0, adv_stats=None, clip=0.2, vf_coef=0.5,
                ent_coef=0.0):
    """Per-sample gradient [n, R6_PPO_NPARAMS_SEP_SDE] and terms [n, 5] = pg, vloss, clipped, kl, entropy of the separate
    towers with gSDE; vfc > 0 clips the value around vold."""
    L = lib()
    f = lambda a, *shape: np.ascontiguousarray(np.asarray(a, np.float32).reshape(*shape))
    x = f(obs13, -1, 13)
    n = len(x)
    a, od, ad, rt, p = f(act3, n, 3), f(old_logp, n), f(adv, n), f(ret, n), f(params, -1)
    vo = f(np.zeros(n) if vold is None else vold, n)
    st = None if adv_stats is None else np.ascontiguousarray(adv_stats, np.float64)
    grad = np.zeros((n, L.hs_sepsde_nparams()), np.float32)
    terms = np.zeros((n, 5), np.float32)
    L.hs_sepsde_sample_grad(p.ctypes.data, x.ctypes.data, a.ctypes.data, od.ctypes.data, ad.ctypes.data, rt.ctypes.data,
                            vo.ctypes.data, n, None if st is None else st.ctypes.data, clip, vf_coef, ent_coef, float(vfc),
                            grad.ctypes.data, terms.ctypes.data)
    return grad, terms


def magnitudes(params, obs13, act3, old_logp, adv, ret, vold=None, vfc=0.0, chunk=4096, **kw):
    """Sum over the samples of |per-sample gradient| [R6_PPO_NPARAMS_SEP_SDE] (float64), in chunks of samples."""
    n = len(np.asarray(ret))
    out = 0.0
    for i in range(0, n, chunk):
        s = slice(i, min(i + chunk, n))
        g, _ = sample_grad(params, np.asarray(obs13)[s], np.asarray(act3)[s], np.asarray(old_logp)[s], np.asarray(adv)[s],
                           np.asarray(ret)[s], None if vold is None else np.asarray(vold)[s], vfc, **kw)
        out = out + np.abs(g.astype(np.float64)).sum(0)
    return out

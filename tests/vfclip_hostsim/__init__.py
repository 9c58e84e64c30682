"""TEST-ONLY host build of the value clipping of r6_ppo.cuh after the shared, gSDE and separate-tower heads (see
vfclip_hostsim.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
LIB = os.path.join(HERE, "_build", "libvfclip_hostsim.so")
CSRC = os.path.join(ROOT, "rl_rocket_6dof_b200", "csrc")
DEPS = [os.path.join(HERE, "vfclip_hostsim.cpp"), os.path.join(CSRC, "r6_ppo.cuh"), os.path.join(CSRC, "r6_core.cuh"),
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
        L.hs_vf_head.argtypes = [C.c_int] + [C.c_void_p] * 6 + [C.c_int64, C.c_void_p, f, f, f, f, C.c_void_p, C.c_void_p]
        for name in ("hs_vf_shared_grad", "hs_vf_sep_grad"):
            getattr(L, name).argtypes = [C.c_void_p] * 7 + [C.c_int64, C.c_void_p, f, f, f, f, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def _f(a, *shape):
    return np.ascontiguousarray(np.asarray(a, np.float32).reshape(*shape))


def head(out4, act3, old, adv, ret, vold, ls_or_var, vfc, sde=False, clip=0.2, vf_coef=0.5, ent_coef=0.0):
    """ppo_head (or ppo_head_sde with var [n, 3]) then ppo_value_clip: (g [n, 7], vloss [n])."""
    o = _f(out4, -1, 4)
    n = len(o)
    a, od, ad, rt, vo = _f(act3, n, 3), _f(old, n), _f(adv, n), _f(ret, n), _f(vold, n)
    lv = _f(ls_or_var, n, 3) if sde else _f(ls_or_var, 3)
    g, vl = np.zeros((n, 7), np.float32), np.zeros(n, np.float32)
    lib().hs_vf_head(int(sde), o.ctypes.data, a.ctypes.data, od.ctypes.data, ad.ctypes.data, rt.ctypes.data, vo.ctypes.data,
                     n, lv.ctypes.data, clip, vf_coef, ent_coef, vfc, g.ctypes.data, vl.ctypes.data)
    return g, vl


def sample_grad(params, obs13, act3, old, adv, ret, vold, vfc, adv_stats=None, clip=0.2, vf_coef=0.5, ent_coef=0.0):
    """Per-sample gradient [n, P] and terms [n, 4] of the kVfClip kernels; the layout (shared or separate towers) by
    the size of params."""
    p = _f(params, -1)
    sep = p.size == 10375
    x = _f(obs13, -1, 13)
    n = len(x)
    a, od, ad, rt, vo = _f(act3, n, 3), _f(old, n), _f(adv, n), _f(ret, n), _f(vold, n)
    st = None if adv_stats is None else np.ascontiguousarray(adv_stats, np.float64)
    grad, terms = np.zeros((n, p.size), np.float32), np.zeros((n, 4), np.float32)
    getattr(lib(), "hs_vf_sep_grad" if sep else "hs_vf_shared_grad")(
        p.ctypes.data, x.ctypes.data, a.ctypes.data, od.ctypes.data, ad.ctypes.data, rt.ctypes.data, vo.ctypes.data, n,
        None if st is None else st.ctypes.data, clip, vf_coef, ent_coef, vfc, grad.ctypes.data, terms.ctypes.data)
    return grad, terms

"""ctypes binding of libr6dof.so (C ABI declared in include/r6dof.h).

There is no CPU fallback: if the CUDA library is missing or does not match the header the import
of the batched env raises.  `R6_AUTOBUILD=1` (default) compiles it in-tree with nvcc when absent.
"""
from __future__ import annotations

import ctypes as C
import os

from .params import R6Params

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, "lib", "libr6dof.so")
ABI_VERSION = 22

u8p = C.c_void_p


class R6Buffers(C.Structure):
    """Mirror of `struct R6Buffers` (device pointers, all owned by torch tensors)."""

    _fields_ = [
        ("state", C.c_void_p), ("m0", C.c_void_p), ("v0", C.c_void_p), ("step_count", C.c_void_p),
        ("episode_id", C.c_void_p), ("ep_return", C.c_void_p),
        ("obs", C.c_void_p), ("reward", C.c_void_p), ("done", C.c_void_p), ("flags", C.c_void_p),
        ("terminal_obs", C.c_void_p), ("terminal_state", C.c_void_p), ("reward_terms", C.c_void_p),
        ("nattempts", C.c_void_p), ("status", C.c_void_p), ("ep_info", C.c_void_p), ("reward_f32", C.c_void_p),
        ("t_table", C.c_void_p), ("ic_table", C.c_void_p),
        ("ic_table_len", C.c_int64), ("n_global", C.c_int64),
        ("stats", C.c_void_p),
        ("scratch", C.c_void_p),
        ("work", C.c_void_p),
        ("tgo", C.c_void_p),
    ]


class R6Mlp(C.Structure):
    _fields_ = [("w0", C.c_void_p), ("b0", C.c_void_p), ("w1", C.c_void_p), ("b1", C.c_void_p),
                ("w2", C.c_void_p), ("b2", C.c_void_p),
                ("wv", C.c_void_p), ("bv", C.c_void_p), ("log_std", C.c_void_p),    # nullable: critic head, Gaussian log-std
                ("vf_w0", C.c_void_p), ("vf_b0", C.c_void_p), ("vf_w1", C.c_void_p), ("vf_b1", C.c_void_p)]  # nullable: value tower


class R6PpoRollout(C.Structure):
    _fields_ = [("obs", C.c_void_p), ("obs_stride_step", C.c_int64), ("obs_stride_comp", C.c_int64),
                ("obs_stride_env", C.c_int64), ("actions", C.c_void_p), ("log_probs", C.c_void_p),
                ("advantages", C.c_void_p), ("returns", C.c_void_p), ("T", C.c_int64), ("n", C.c_int64),
                ("old_values", C.c_void_p)]                  # nullable: read only with R6PpoCoef.clip_range_vf > 0


class R6PpoCoef(C.Structure):
    _fields_ = [("clip_range", C.c_double), ("vf_coef", C.c_double), ("ent_coef", C.c_double), ("adv_stats", C.c_void_p),
                ("clip_range_vf", C.c_double)]               # 0 = no value clipping


class R6AdamCoef(C.Structure):
    _fields_ = [("lr", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double),
                ("max_grad_norm", C.c_double), ("scale", C.c_double)]


class R6Sde(C.Structure):
    _fields_ = [("log_std", C.c_void_p), ("xi", C.c_void_p)]     # gSDE log_std [64][3], noise [192][n]


PPO_NPARAMS = 10311
PPO_NTERMS = 5
PPO_NPARAMS_SDE = 10500
PPO_NPARAMS_SEP = 10375
PPO_NPARAMS_SEP_SDE = 10564
PPO_NTERMS_SDE = 6
SDE_NXI = 192


def make_mlp(weights: dict) -> "R6Mlp":
    """R6Mlp from a dict of tensors / arrays exposing data_ptr() or ctypes.data (optional keys: wv, bv, log_std, and
    the separate value tower vf_w0, vf_b0, vf_w1, vf_b1)."""
    def ptr(x):
        if x is None:
            return None
        return x.data_ptr() if hasattr(x, "data_ptr") else x.ctypes.data
    m = R6Mlp(*[ptr(weights[k]) for k in ("w0", "b0", "w1", "b1", "w2", "b2")])
    ls = weights.get("log_std")
    if ls is not None and len(ls.shape) == 2:          # gSDE [64, 3]: passed through R6Sde, never as the Gaussian [3]
        ls = None
    m.wv, m.bv, m.log_std = ptr(weights.get("wv")), ptr(weights.get("bv")), ptr(ls)
    m.vf_w0, m.vf_b0 = ptr(weights.get("vf_w0")), ptr(weights.get("vf_b0"))
    m.vf_w1, m.vf_b1 = ptr(weights.get("vf_w1")), ptr(weights.get("vf_b1"))
    return m


EXPORTS = ["r6_abi_version", "r6_last_error", "r6_params_size", "r6_buffers_size", "r6_reset", "r6_step",
           "r6_rollout", "r6_sim_step_raw", "r6_tgo", "r6_stats_reset", "r6_peak_fma", "r6_gae", "r6_policy", "r6_policy_ex", "r6_step_random", "r6_step_range", "r6_policy_range", "r6_work_bytes",
           "r6_ppo_rollout_size", "r6_ppo_coef_size", "r6_adam_coef_size", "r6_ppo_work_bytes", "r6_ppo_grad", "r6_adam_step",
           "r6_trunc_record", "r6_trunc_bootstrap", "r6_sde_size", "r6_sde_noise", "r6_policy_sde_range",
           "r6_ppo_sde_work_bytes", "r6_ppo_grad_sde", "r6_policy_sde_sep_range", "r6_ppo_grad_sde_sep"]


class R6Error(RuntimeError):
    pass


_lib = None


def load(path: str | None = None):
    """Loads (building first if needed) libr6dof.so and checks ABI version and struct layouts."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or os.environ.get("R6_LIB_PATH") or LIB_PATH      # R6_LIB_PATH: A/B-test another build
    if path == LIB_PATH and os.environ.get("R6_AUTOBUILD", "1") == "1":
        from . import build as _build
        if _build.needs_build():
            _build.build()
    if not os.path.exists(path):
        raise R6Error(f"{path} not found: build it with `python -m rl_rocket_6dof_b200.build` "
                      "(there is no CPU fallback)")
    L = C.CDLL(path)
    for name in EXPORTS:
        if not hasattr(L, name):
            raise R6Error(f"{path} does not export {name}")
    L.r6_last_error.restype = C.c_char_p
    if L.r6_abi_version() != ABI_VERSION:
        raise R6Error(f"ABI version mismatch: library {L.r6_abi_version()}, binding {ABI_VERSION}")
    if L.r6_params_size() != C.sizeof(R6Params):
        raise R6Error(f"R6Params layout mismatch: C {L.r6_params_size()} vs ctypes {C.sizeof(R6Params)}")
    if L.r6_buffers_size() != C.sizeof(R6Buffers):
        raise R6Error(f"R6Buffers layout mismatch: C {L.r6_buffers_size()} vs ctypes {C.sizeof(R6Buffers)}")
    for name, st in (("r6_ppo_rollout_size", R6PpoRollout), ("r6_ppo_coef_size", R6PpoCoef), ("r6_adam_coef_size", R6AdamCoef),
                     ("r6_sde_size", R6Sde)):
        if getattr(L, name)() != C.sizeof(st):
            raise R6Error(f"{st.__name__} layout mismatch: C {getattr(L, name)()} vs ctypes {C.sizeof(st)}")
    pp, bp = C.POINTER(R6Params), C.POINTER(R6Buffers)
    L.r6_reset.argtypes = [pp, bp, C.c_int64, C.c_int64, C.c_void_p, C.c_uint64, C.c_void_p]
    L.r6_step.argtypes = [pp, bp, C.c_int64, C.c_int64, C.c_void_p, C.c_uint64, C.c_void_p]
    L.r6_rollout.argtypes = [pp, bp, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.POINTER(R6Mlp), C.c_void_p,
                             C.c_uint64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.r6_sim_step_raw.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_int64,
                                  C.c_void_p, C.c_void_p, C.c_void_p]
    L.r6_tgo.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    L.r6_stats_reset.argtypes = [C.c_void_p, C.c_void_p]
    L.r6_step_random.argtypes = [pp, bp, C.c_int64, C.c_int64, C.c_uint64, C.c_int64, C.c_void_p]
    L.r6_step_range.argtypes = [pp, bp, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_uint64, C.c_int64,
                                C.c_void_p]
    L.r6_work_bytes.argtypes = [C.c_int64]
    L.r6_work_bytes.restype = C.c_int64
    L.r6_policy_range.argtypes = [C.POINTER(R6Mlp), C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_uint64,
                                  C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.r6_policy_ex.argtypes = [C.POINTER(R6Mlp), C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_uint64, C.c_int64, C.c_int64,
                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.r6_policy.argtypes = [C.POINTER(R6Mlp), C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]
    L.r6_gae.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_double, C.c_double,
                         C.c_void_p, C.c_void_p, C.c_void_p]
    L.r6_trunc_record.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_void_p,
                                  C.c_void_p, C.c_void_p]
    L.r6_trunc_bootstrap.argtypes = [C.c_void_p, C.c_int32, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_double,
                                     C.c_void_p]
    L.r6_ppo_work_bytes.argtypes = [C.c_int64]
    L.r6_ppo_work_bytes.restype = C.c_int64
    L.r6_ppo_grad.argtypes = [C.POINTER(R6Mlp), C.POINTER(R6PpoRollout), C.c_void_p, C.c_int64, C.POINTER(R6PpoCoef),
                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.r6_adam_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(R6AdamCoef), C.c_int64,
                               C.c_void_p, C.c_void_p]
    L.r6_sde_noise.argtypes = [C.c_int64, C.c_int64, C.c_int64, C.c_uint64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]
    L.r6_policy_sde_range.argtypes = [C.POINTER(R6Mlp), C.POINTER(R6Sde), C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int32,
                                      C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.r6_policy_sde_sep_range.argtypes = L.r6_policy_sde_range.argtypes
    L.r6_ppo_sde_work_bytes.argtypes = [C.c_int64]
    L.r6_ppo_sde_work_bytes.restype = C.c_int64
    L.r6_ppo_grad_sde.argtypes = [C.POINTER(R6Mlp), C.POINTER(R6Sde), C.POINTER(R6PpoRollout), C.c_void_p, C.c_int64,
                                  C.POINTER(R6PpoCoef), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.r6_ppo_grad_sde_sep.argtypes = L.r6_ppo_grad_sde.argtypes
    L.r6_peak_fma.argtypes = [C.c_int32, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]
    _lib = L
    return L


def check(rc: int, L=None):
    if rc != 0:
        L = L or load()
        raise R6Error(f"libr6dof error {rc}: {L.r6_last_error().decode()}")

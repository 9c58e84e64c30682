"""Actor weights of the reference's trained PPO agents for the fused closed-loop rollout.

The reference evaluates `PPO.load("best_model_2bo71j9m", env)` with `evaluate_policy(...,
deterministic=True)` (/root/reference/montecarlo_script.py:54-64): SB3's `MlpPolicy` with the default
`net_arch` of SB3 1.6 — a shared tanh MLP 13 -> 128 -> 64 followed by `action_net` 64 -> 3; the
deterministic action is the Gaussian mean clipped to the action space.  `r6_rollout(mode=R6_ACT_MLP)`
runs exactly that network inside the rollout kernel; this module only moves the six tensors around.
"""
from __future__ import annotations

import io
import zipfile
from typing import Dict

import numpy as np
import torch

SHAPES = {"w0": (128, 13), "b0": (128,), "w1": (64, 128), "b1": (64,), "w2": (3, 64), "b2": (3,)}
# SB3 1.6's default MlpPolicy without policy_kwargs: separate tanh towers net_arch [dict(pi=[64, 64], vf=[64, 64])];
# w0 .. b1 are the policy tower, vf_w0 .. vf_b1 the value tower (value_net "wv", "bv" reads the value latent)
SEP_SHAPES = {"w0": (64, 13), "b0": (64,), "w1": (64, 64), "b1": (64,), "w2": (3, 64), "b2": (3,),
              "vf_w0": (64, 13), "vf_b0": (64,), "vf_w1": (64, 64), "vf_b1": (64,)}
# optional: the critic head on the same latent and the Gaussian log-std (needed only to COLLECT training rollouts);
# log_std is [3] (diagonal Gaussian) or, for a gSDE policy (use_sde=True), [64, 3]
OPTIONAL_SHAPES = {"wv": (64,), "bv": (1,), "log_std": (3,)}
SDE_LOG_STD_SHAPE = (64, 3)
_SB3_OPTIONAL = {"wv": "value_net.weight", "bv": "value_net.bias", "log_std": "log_std"}
_SB3_KEYS = {
    "w0": "mlp_extractor.shared_net.0.weight", "b0": "mlp_extractor.shared_net.0.bias",
    "w1": "mlp_extractor.shared_net.2.weight", "b1": "mlp_extractor.shared_net.2.bias",
    "w2": "action_net.weight", "b2": "action_net.bias",
}
# SB3 >= 1.8 has separate policy / value towers: the actor lives under policy_net
_SB3_KEYS_V2 = {**_SB3_KEYS, "w0": "mlp_extractor.policy_net.0.weight", "b0": "mlp_extractor.policy_net.0.bias",
                "w1": "mlp_extractor.policy_net.2.weight", "b1": "mlp_extractor.policy_net.2.bias"}
# SB3 1.6's separate towers (64-wide policy tower): both towers and both heads
_SB3_KEYS_SEP = {**_SB3_KEYS_V2, "vf_w0": "mlp_extractor.value_net.0.weight", "vf_b0": "mlp_extractor.value_net.0.bias",
                 "vf_w1": "mlp_extractor.value_net.2.weight", "vf_b1": "mlp_extractor.value_net.2.bias"}


def is_separate(w) -> bool:
    """True for SB3 1.6's separate policy / value towers (the dict carries the value tower vf_w0 ...)."""
    return w.get("vf_w0") is not None


def _check(w: Dict[str, np.ndarray]) -> Dict[str, np.ndarray]:
    out = {}
    sep = is_separate(w)
    for k, shp in (SEP_SHAPES if sep else SHAPES).items():
        a = np.ascontiguousarray(np.asarray(w[k], dtype=np.float32))
        if a.shape != shp:
            raise ValueError(f"policy tensor {k} has shape {a.shape}, the kernels expect {shp} " +
                             ("(MlpPolicy, separate towers net_arch [dict(pi=[64, 64], vf=[64, 64])], 13 observations, "
                              "3 actions)" if sep else "(MlpPolicy, net_arch [128, 64], 13 observations, 3 actions)"))
        out[k] = a
    for k, shp in OPTIONAL_SHAPES.items():
        if k in w and w[k] is not None:
            a = np.ascontiguousarray(np.asarray(w[k], dtype=np.float32))
            if k == "log_std" and a.size == 64 * 3:
                shp = SDE_LOG_STD_SHAPE
            if a.size != int(np.prod(shp)):
                raise ValueError(f"policy tensor {k} has shape {a.shape}, expected {shp}"
                                 + (f" or {SDE_LOG_STD_SHAPE} (gSDE)" if k == "log_std" else ""))
            out[k] = a.reshape(shp)
    return out


def load_sb3_zip(path: str) -> Dict[str, np.ndarray]:
    """Actor tensors from a stable-baselines3 `model.save()` archive (`policy.pth` member).  SB3 1.6's default separate
    towers (net_arch [dict(pi=[64, 64], vf=[64, 64])]) load in full, the value tower under vf_w0 vf_b0 vf_w1 vf_b1; the
    SB3 >= 1.8 towers of [128, 64] load actor-only."""
    if not path.endswith(".zip"):
        path += ".zip"
    with zipfile.ZipFile(path) as z:
        sd = torch.load(io.BytesIO(z.read("policy.pth")), map_location="cpu", weights_only=True)
    keys = _SB3_KEYS if _SB3_KEYS["w0"] in sd else _SB3_KEYS_V2
    if (keys is _SB3_KEYS_V2 and _SB3_KEYS_SEP["vf_w0"] in sd and _SB3_KEYS_V2["w0"] in sd
            and tuple(sd[_SB3_KEYS_V2["w0"]].shape)[0] == 64):
        keys = _SB3_KEYS_SEP       # SB3 1.6 default towers: the kernels run both, so the critic rides along too
    w = {k: sd[name].numpy() for k, name in keys.items()}
    if keys is not _SB3_KEYS_V2:   # shared trunk / 64-wide towers: the kernels have the critic, so it rides along
        w.update({k: sd[name].numpy() for k, name in _SB3_OPTIONAL.items() if name in sd})
    elif "log_std" in sd:
        w["log_std"] = sd["log_std"].numpy()
    return _check(w)


def load_npz(path: str, prefix: str = "mlp_") -> Dict[str, np.ndarray]:
    """Actor tensors stored as `<prefix>w0` ... `<prefix>b2` in an .npz file (and `<prefix>vf_w0` ... `<prefix>vf_b1` for
    the separate towers)."""
    g = np.load(path, allow_pickle=False)
    keys = SEP_SHAPES if prefix + "vf_w0" in g.files else SHAPES
    w = {k: g[prefix + k] for k in keys}
    w.update({k: g[prefix + k] for k in OPTIONAL_SHAPES if prefix + k in g.files})
    return _check(w)


def to_device(w: Dict[str, np.ndarray], device) -> Dict[str, torch.Tensor]:
    return {k: torch.from_numpy(v).to(device).contiguous() for k, v in _check(w).items()}


def forward_full_numpy(w: Dict[str, np.ndarray], obs13: np.ndarray):
    """Host statement of the actor-critic forward: (unclipped mean [..., 3], value [...]).  With the separate towers
    the value is value_net on the value tower's latent."""
    x = np.asarray(obs13, np.float32)
    h = np.tanh(x @ w["w0"].T + w["b0"]).astype(np.float32)
    h = np.tanh(h @ w["w1"].T + w["b1"]).astype(np.float32)
    mean = (h @ w["w2"].T + w["b2"]).astype(np.float32)
    if is_separate(w):
        h = np.tanh(x @ w["vf_w0"].T + w["vf_b0"]).astype(np.float32)
        h = np.tanh(h @ w["vf_w1"].T + w["vf_b1"]).astype(np.float32)
    value = (h @ w["wv"] + w["bv"][0]).astype(np.float32) if "wv" in w else np.zeros(mean.shape[:-1], np.float32)
    return mean, value


def forward_numpy(w: Dict[str, np.ndarray], obs13: np.ndarray) -> np.ndarray:
    """Host statement of the network (float32), for tests and tiny batches: obs [..., 13] -> actions [..., 3] (the
    policy tower of the separate towers)."""
    x = np.asarray(obs13, np.float32)
    h = np.tanh(x @ w["w0"].T + w["b0"]).astype(np.float32)
    h = np.tanh(h @ w["w1"].T + w["b1"]).astype(np.float32)
    a = (h @ w["w2"].T + w["b2"]).astype(np.float32)
    return np.clip(a, -1.0, 1.0).astype(np.float32)

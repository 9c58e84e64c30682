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


def _check(w: Dict[str, np.ndarray]) -> Dict[str, np.ndarray]:
    out = {}
    for k, shp in SHAPES.items():
        a = np.ascontiguousarray(np.asarray(w[k], dtype=np.float32))
        if a.shape != shp:
            raise ValueError(f"policy tensor {k} has shape {a.shape}, the fused kernel expects {shp} "
                             "(MlpPolicy, net_arch [128, 64], 13 observations, 3 actions)")
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
    """Actor tensors from a stable-baselines3 `model.save()` archive (`policy.pth` member)."""
    if not path.endswith(".zip"):
        path += ".zip"
    with zipfile.ZipFile(path) as z:
        sd = torch.load(io.BytesIO(z.read("policy.pth")), map_location="cpu", weights_only=True)
    keys = _SB3_KEYS if _SB3_KEYS["w0"] in sd else _SB3_KEYS_V2
    w = {k: sd[name].numpy() for k, name in keys.items()}
    if keys is _SB3_KEYS:          # shared trunk: the critic reads the same latent, so it can ride along in the kernel
        w.update({k: sd[name].numpy() for k, name in _SB3_OPTIONAL.items() if name in sd})
    elif "log_std" in sd:
        w["log_std"] = sd["log_std"].numpy()
    return _check(w)


def load_npz(path: str, prefix: str = "mlp_") -> Dict[str, np.ndarray]:
    """Actor tensors stored as `<prefix>w0` ... `<prefix>b2` in an .npz file."""
    g = np.load(path, allow_pickle=False)
    w = {k: g[prefix + k] for k in SHAPES}
    w.update({k: g[prefix + k] for k in OPTIONAL_SHAPES if prefix + k in g.files})
    return _check(w)


def to_device(w: Dict[str, np.ndarray], device) -> Dict[str, torch.Tensor]:
    return {k: torch.from_numpy(v).to(device).contiguous() for k, v in _check(w).items()}


def forward_full_numpy(w: Dict[str, np.ndarray], obs13: np.ndarray):
    """Host statement of the actor-critic forward: (unclipped mean [..., 3], value [...])."""
    x = np.asarray(obs13, np.float32)
    h = np.tanh(x @ w["w0"].T + w["b0"]).astype(np.float32)
    h = np.tanh(h @ w["w1"].T + w["b1"]).astype(np.float32)
    mean = (h @ w["w2"].T + w["b2"]).astype(np.float32)
    value = (h @ w["wv"] + w["bv"][0]).astype(np.float32) if "wv" in w else np.zeros(mean.shape[:-1], np.float32)
    return mean, value


def forward_numpy(w: Dict[str, np.ndarray], obs13: np.ndarray) -> np.ndarray:
    """Host statement of the network (float32), for tests and tiny batches: obs [..., 13] -> actions [..., 3]."""
    x = np.asarray(obs13, np.float32)
    h = np.tanh(x @ w["w0"].T + w["b0"]).astype(np.float32)
    h = np.tanh(h @ w["w1"].T + w["b1"]).astype(np.float32)
    a = (h @ w["w2"].T + w["b2"]).astype(np.float32)
    return np.clip(a, -1.0, 1.0).astype(np.float32)

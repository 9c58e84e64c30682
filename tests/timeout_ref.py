"""NumPy restatement of stable-baselines3 1.6.0 `OnPolicyAlgorithm.collect_rollouts`' timeout handling (SB3 issue #633)
— TEST INFRASTRUCTURE ONLY.  SB3 is not in the image, so, like `oracle/gae_oracle.py`'s GAE recursion, this follows its
published code from memory (unpinned):

    # Handle timeout by bootstraping with value function
    for idx, done in enumerate(dones):
        if done and infos[idx].get("terminal_observation") is not None and infos[idx].get("TimeLimit.truncated", False):
            terminal_obs = self.policy.obs_to_tensor(infos[idx]["terminal_observation"])[0]
            with th.no_grad():
                terminal_value = self.policy.predict_values(terminal_obs)[0]
            rewards[idx] += self.gamma * terminal_value

`rewards` is the float32 array the VecEnv returned, `terminal_value` a float32 torch value and `self.gamma` a python
float: python float times float32 tensor is a float32 product (gamma rounded to float32 first), and the sum is rounded to
float32 again.  Two roundings, never one fused multiply-add.
"""
from fractions import Fraction

import numpy as np


def bootstrap_timeouts(rewards, truncated, terminal_values, gamma=0.99):
    """rewards: [T, n]; truncated: bool [T, n] (TimeLimit.truncated of step t, which implies a terminal observation);
    terminal_values: [T, n], V of the terminal observation of step t (read only where truncated).  Returns the new
    float32 rewards fl32(r + fl32(fl32(gamma) V)) where truncated, r elsewhere.  (NumPy float32 array arithmetic rounds
    every operation and never fuses them.)"""
    out = np.array(rewards, np.float32)
    truncated = np.asarray(truncated, bool)
    v = np.asarray(terminal_values, np.float32)
    g = np.float32(gamma)
    for t in range(out.shape[0]):
        m = truncated[t]
        out[t, m] = out[t, m] + g * v[t, m]
    return out


def fma_f32(r, g, v):
    """fl32(r + g v) with ONE rounding (a fused multiply-add), elementwise on float32 inputs: the wrong answer the
    restatement must tell apart from SB3's two roundings.  The float64 product of two float32 values is exact; the
    float64 sum is exact or, when it is not, is resolved against the exact rational sum below."""
    r, g, v = (np.asarray(x, np.float32) for x in (r, g, v))
    r, g, v = np.broadcast_arrays(r, g, v)
    out = np.empty(r.shape, np.float32)
    for k in np.ndindex(r.shape):
        exact = Fraction(float(r[k])) + Fraction(float(g[k])) * Fraction(float(v[k]))
        c = np.float32(float(exact))
        cand = (np.nextafter(c, np.float32(-np.inf)), c, np.nextafter(c, np.float32(np.inf)))
        out[k] = min(cand, key=lambda x: (abs(Fraction(float(x)) - exact), int(np.asarray(x).view(np.uint32)) & 1))
    return out

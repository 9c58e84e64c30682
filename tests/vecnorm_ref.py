"""A float64 numpy restatement of stable-baselines3 1.6's `RunningMeanStd` and `VecNormalize.reset / step_wait`
([memory]: SB3 is not installed here), the reference the VecNormalize tests compare the device against.

One deviation from SB3 is the project's on purpose: SB3 takes the observation batch's mean and variance of the float32
array (numpy reduces in float32); here `batch_moments` is float64 (two-pass).  `update_from_moments` and everything
after it is SB3's arithmetic in SB3's order (numpy float64 does no contraction)."""
import numpy as np


def batch_moments(x: np.ndarray) -> tuple:
    """(mean, population var, count) of x [count, dim] in float64, two-pass."""
    x = np.asarray(x, np.float64)
    m = x.mean(axis=0)
    return m, ((x - m) ** 2).mean(axis=0), x.shape[0]


class RunningMeanStd:
    def __init__(self, epsilon: float = 1e-4, shape=()):
        self.mean = np.zeros(shape, np.float64)
        self.var = np.ones(shape, np.float64)
        self.count = epsilon

    def update(self, x: np.ndarray):
        bm, bv, bc = batch_moments(x)
        self.update_from_moments(bm, bv, bc)

    def update_from_moments(self, batch_mean, batch_var, batch_count):
        delta = batch_mean - self.mean
        tot_count = self.count + batch_count
        new_mean = self.mean + delta * batch_count / tot_count
        m_a = self.var * self.count
        m_b = batch_var * batch_count
        m_2 = m_a + m_b + np.square(delta) * self.count * batch_count / (self.count + batch_count)
        new_var = m_2 / (self.count + batch_count)
        new_count = batch_count + self.count
        self.mean, self.var, self.count = new_mean, new_var, new_count

    def as_row(self) -> np.ndarray:
        """[mean, var, count] as the device's layout."""
        return np.concatenate([np.ravel(self.mean), np.ravel(self.var), [self.count]])


def normalize_obs(obs: np.ndarray, mean, var, eps: float, clip: float) -> np.ndarray:
    """fl32(clip((fl64(obs) - mean) / sqrt(var + eps), +-clip)); obs [count, 13]."""
    return np.clip((np.asarray(obs, np.float32).astype(np.float64) - mean) / np.sqrt(var + eps), -clip, clip).astype(np.float32)


def normalize_reward(rew: np.ndarray, var, eps: float, clip: float) -> np.ndarray:
    """fl32(clip(fl64(r) / sqrt(var + eps), +-clip)) — the rounding the rollout buffer applies."""
    return np.clip(np.asarray(rew, np.float32).astype(np.float64) / np.sqrt(var + eps), -clip, clip).astype(np.float32)


class VecNormalizeRef:
    """VecNormalize(training, norm_obs, norm_reward, clip_obs, clip_reward, gamma, epsilon) over raw per-step arrays.
    `moments` (optional callable obs -> (mean, var, count)) replaces the float64 two-pass batch moments, so a test can
    feed the device's moments and check everything downstream bit for bit."""

    def __init__(self, num_envs: int, *, training=True, norm_obs=True, norm_reward=True, clip_obs=10.0, clip_reward=10.0,
                 gamma=0.99, epsilon=1e-8, dim=13):
        self.obs_rms, self.ret_rms = RunningMeanStd(shape=(dim,)), RunningMeanStd(shape=())
        self.returns = np.zeros(num_envs)
        self.training, self.norm_obs, self.norm_reward = training, norm_obs, norm_reward
        self.clip_obs, self.clip_reward, self.gamma, self.epsilon = clip_obs, clip_reward, gamma, epsilon

    def _obs_update(self, obs, moments=None):
        if self.training and self.norm_obs:
            if moments is None:
                self.obs_rms.update(obs)
            else:
                self.obs_rms.update_from_moments(*moments(obs))

    def normalize_obs(self, obs):
        if not self.norm_obs:
            return np.asarray(obs, np.float32)
        return normalize_obs(obs, self.obs_rms.mean, self.obs_rms.var, self.epsilon, self.clip_obs)

    def reset(self, obs, moments=None):
        """obs [num_envs, 13] raw reset observations -> normalized."""
        self.returns = np.zeros(len(self.returns))
        self._obs_update(obs, moments)
        return self.normalize_obs(obs)

    def step_wait(self, obs, rewards, dones, terminal_obs=None, moments=None, ret_moments=None):
        """One step of raw (obs [n, 13], float32 rewards [n], dones [n], terminal_obs {env: [13]}) -> (normalized obs,
        normalized float32 rewards, normalized terminal obs {env: [13]})."""
        self._obs_update(obs, moments)
        obs_n = self.normalize_obs(obs)
        if self.training:
            self.returns = self.returns * self.gamma + np.asarray(rewards, np.float32).astype(np.float64)
            if ret_moments is None:
                self.ret_rms.update(self.returns)
            else:
                self.ret_rms.update_from_moments(*ret_moments(self.returns))
        rew_n = (normalize_reward(rewards, self.ret_rms.var, self.epsilon, self.clip_reward) if self.norm_reward
                 else np.asarray(rewards, np.float32))
        term = {i: self.normalize_obs(np.asarray(o)[None])[0] for i, o in (terminal_obs or {}).items()}
        self.returns[np.asarray(dones, bool)] = 0
        return obs_n, rew_n, term


def combine_moments(rows: np.ndarray) -> np.ndarray:
    """numpy twin of ppo.combine_moments: (count, mean, M2) rows [W, 3] combined in row order."""
    n, mean, m2 = rows[0]
    for nb, mb, m2b in rows[1:]:
        tot = n + nb
        d = mb - mean
        mean = mean + d * (nb / tot)
        m2 = m2 + m2b + d * d * (n * nb / tot)
        n = tot
    return np.array([n, mean, m2])


def moments_bound(x: np.ndarray, parts: int, per_thread: int) -> tuple:
    """Bounds on |mean - mean64| and |M2 - M2_64| for r6_vn_moments / r6_vn_ret_moments on x [count]: a thread sums
    per_thread shifted values (x - K) and (x - K)^2, a warp adds its lanes in 5 levels and converts once, a CTA chains its
    8 warps, and the final kernel chains ceil(parts / 256) CTA results per thread, then 5 shuffle levels and 8 warps.
    Every rounding on that path is relative to a quantity no larger than max|x| (mean) or count (2 max|x|)^2 (M2), and
    one Chan step rounds at most 8 times, so the error is at most 8 u depth times that scale."""
    u = 2.0 ** -53
    depth = per_thread + 5 + 2 + 8 + -(-parts // 256) + 5 + 8
    a = float(np.max(np.abs(x))) if x.size else 0.0
    return 8 * depth * u * a, 8 * depth * u * x.size * (2 * a) ** 2

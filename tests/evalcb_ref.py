"""A restatement of stable-baselines3 1.6's `evaluate_policy` loop and `EvalCallback._on_step` [memory], for the host
tests of rl_rocket_6dof_b200.evaluation.  Written from SB3's structure, step by step, not from the module under test.

evaluate_policy(model, env, n_eval_episodes, deterministic=True) with a VecEnv of n_envs envs:
    episode_counts = zeros(n_envs); episode_count_targets = [(n_eval_episodes + i) // n_envs for i in range(n_envs)]
    while (episode_counts < episode_count_targets).any():
        actions = predict(observations); observations, rewards, dones, infos = env.step(actions)
        for i in range(n_envs):
            if episode_counts[i] < episode_count_targets[i]:
                if dones[i]:   # Monitor-wrapped: the episode's info["episode"]
                    episode_rewards.append(info["episode"]["r"]); episode_lengths.append(info["episode"]["l"])
                    episode_counts[i] += 1
    return episode_rewards, episode_lengths

EvalCallback._on_step (called once per vec-env step, n_calls counting them):
    if eval_freq > 0 and n_calls % eval_freq == 0:
        sync_envs_normalization(training_env, eval_env)
        episode_rewards, episode_lengths = evaluate_policy(...)
        if log_path is not None:
            evaluations_timesteps.append(num_timesteps); evaluations_results.append(episode_rewards)
            evaluations_length.append(episode_lengths)
            np.savez(log_path, timesteps=..., results=..., ep_lengths=...)
        mean_reward, std_reward = np.mean(episode_rewards), np.std(episode_rewards)
        mean_ep_length, std_ep_length = np.mean(episode_lengths), np.std(episode_lengths)
        if mean_reward > best_mean_reward:          # best_mean_reward starts at -np.inf
            model.save(best_model_save_path / "best_model"); best_mean_reward = mean_reward
"""
import numpy as np


def monitor_r(ep_return: float) -> float:
    """Monitor: info["episode"]["r"] = round(sum of the episode's rewards, 6)."""
    return round(float(ep_return), 6)


def evaluate_policy(episodes, n_eval_episodes):
    """episodes[i] = the successive (return, length) episodes env i would play (an auto-resetting eval env); all envs
    start at step 0.  Returns (episode_rewards, episode_lengths) in SB3's append order."""
    n_envs = len(episodes)
    counts = np.zeros(n_envs, np.int64)
    targets = np.array([(n_eval_episodes + i) // n_envs for i in range(n_envs)], np.int64)
    ends = [np.cumsum([l for _, l in eps]) for eps in episodes]     # the step at which each episode ends
    nxt = np.zeros(n_envs, np.int64)                                 # index of each env's running episode
    rewards, lengths = [], []
    step = 0
    while (counts < targets).any():
        step += 1
        for i in range(n_envs):
            done = nxt[i] < len(ends[i]) and ends[i][nxt[i]] == step
            if counts[i] < targets[i] and done:
                r, l = episodes[i][nxt[i]]
                rewards.append(monitor_r(r))
                lengths.append(int(l))
                counts[i] += 1
            if done:
                nxt[i] += 1
    return rewards, lengths


class EvalCallbackRef:
    """_on_step's bookkeeping with `evaluate` supplying (episode_rewards, episode_lengths) for the call."""

    def __init__(self, eval_freq):
        self.eval_freq = eval_freq
        self.n_calls = 0
        self.best_mean_reward = -np.inf
        self.timesteps, self.results, self.ep_lengths = [], [], []
        self.saved = []             # the n_calls at which best_model was saved

    def on_step(self, num_timesteps, evaluate):
        self.n_calls += 1
        if not (self.eval_freq > 0 and self.n_calls % self.eval_freq == 0):
            return None
        rewards, lengths = evaluate()
        self.timesteps.append(num_timesteps)
        self.results.append(rewards)
        self.ep_lengths.append(lengths)
        mean_reward = np.mean(rewards)
        logs = {"mean_reward": float(mean_reward), "std_reward": float(np.std(rewards)),
                "mean_ep_length": float(np.mean(lengths)), "std_ep_length": float(np.std(lengths))}
        if mean_reward > self.best_mean_reward:
            self.saved.append(self.n_calls)
            self.best_mean_reward = mean_reward
        return logs

    def npz(self):
        return dict(timesteps=np.array(self.timesteps), results=np.array(self.results),
                    ep_lengths=np.array(self.ep_lengths))

"""TEST INFRASTRUCTURE (oracle) -- numpy restatement of the two Stable-Baselines3 wrappers every trainer of the
reference puts directly after the VecEnv (SURVEY 8f rank 1):

    envs = VecFrameStack(envs, n_stack=frame_stack)                        scripts/train_flat_ppo.py:384-388
    envs = VecNormalize(envs, norm_obs=True, norm_reward=False,            scripts/train_flat_ppo.py:392-399
                        clip_obs=10.0, clip_reward=10.0, gamma=gamma)
    env = VecNormalize.load(path, env); env.training = False               inference.py:455-471

PARITY UNPINNED: stable-baselines3 is a third-party dependency that is neither vendored under /root/reference
(rl_system/requirements.txt:2 `stable-baselines3>=2.0.0`, unpinned; the only lock in the tree,
deprecated/poetry.lock, has 2.7.0) nor importable in the build container, and the reference has no test that
pins results at this boundary.  The algorithm below restates SB3 2.x's published source:
  * common/vec_env/stacked_observations.py  StackedObservations.reset / .update  (channels-last, 1-D obs)
  * common/running_mean_std.py              RunningMeanStd(epsilon=1e-4).update / update_from_moments
  * common/vec_env/vec_normalize.py         VecNormalize.reset / step_wait / normalize_obs / _update_reward
Only tests/ and __graft_entry__.smoke() may import this module.
"""
import numpy as np


class RunningMeanStd:
    def __init__(self, epsilon=1e-4, shape=()):
        self.mean = np.zeros(shape, np.float64)
        self.var = np.ones(shape, np.float64)
        self.count = epsilon

    def update(self, arr):
        batch_mean = np.mean(arr, axis=0)
        batch_var = np.var(arr, axis=0)
        self.update_from_moments(batch_mean, batch_var, arr.shape[0])

    def update_from_moments(self, batch_mean, batch_var, batch_count):
        delta = batch_mean - self.mean
        tot_count = self.count + batch_count
        new_mean = self.mean + delta * batch_count / tot_count
        m_a = self.var * self.count
        m_b = batch_var * batch_count
        m_2 = m_a + m_b + np.square(delta) * self.count * batch_count / (self.count + batch_count)
        self.mean, self.var, self.count = new_mean, m_2 / (self.count + batch_count), batch_count + self.count


class StackedObservations:
    """VecFrameStack for a flat (d,) observation: stacks along the last axis, newest frame last."""

    def __init__(self, num_envs, n_stack, obs_dim):
        self.n_stack, self.d = n_stack, obs_dim
        self.stacked_obs = np.zeros((num_envs, obs_dim * n_stack), np.float32)

    def reset(self, observation):
        self.stacked_obs[...] = 0
        self.stacked_obs[..., -self.d:] = observation
        return self.stacked_obs

    def update(self, observations, dones, infos):
        """infos: dict env_index -> info dict (only finished envs need an entry with 'terminal_observation')."""
        shift = -self.d
        self.stacked_obs = np.roll(self.stacked_obs, shift, axis=-1)
        for env_idx in np.nonzero(dones)[0]:
            info = infos.get(int(env_idx))
            if info is not None and "terminal_observation" in info:
                previous_stack = self.stacked_obs[env_idx, :shift]
                info["terminal_observation"] = np.concatenate((previous_stack, info["terminal_observation"]), axis=-1)
            self.stacked_obs[env_idx] = 0
        self.stacked_obs[..., shift:] = observations
        return self.stacked_obs, infos


class VecNormalize:
    def __init__(self, num_envs, obs_shape, training=True, norm_obs=True, norm_reward=False, clip_obs=10.0,
                 clip_reward=10.0, gamma=0.99, epsilon=1e-8):
        self.obs_rms = RunningMeanStd(shape=obs_shape)
        self.ret_rms = RunningMeanStd(shape=())
        self.clip_obs, self.clip_reward, self.gamma, self.epsilon = clip_obs, clip_reward, gamma, epsilon
        self.training, self.norm_obs, self.norm_reward = training, norm_obs, norm_reward
        self.returns = np.zeros(num_envs)
        self.old_obs = None

    def normalize_obs(self, obs):
        if not self.norm_obs:
            return obs
        return np.clip((obs - self.obs_rms.mean) / np.sqrt(self.obs_rms.var + self.epsilon),
                       -self.clip_obs, self.clip_obs).astype(np.float32)

    def normalize_reward(self, reward):
        if self.norm_reward:
            reward = np.clip(reward / np.sqrt(self.ret_rms.var + self.epsilon), -self.clip_reward, self.clip_reward)
        return reward

    def reset(self, obs):
        self.old_obs = obs
        self.returns = np.zeros(obs.shape[0])
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
        return self.normalize_obs(obs)

    def update(self, obs, rewards, dones):
        """The statistics half of step: obs_rms, the discounted returns and ret_rms, returns[dones] = 0.  Nothing in step
        reads returns between SB3's update and its reset of the finished envs' returns, so the two can sit together here."""
        self.old_obs = obs
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
        if self.training:
            self.returns = self.returns * self.gamma + rewards
            self.ret_rms.update(self.returns)
        self.returns[dones.astype(bool)] = 0

    def step(self, obs, rewards, dones, infos):
        self.update(obs, rewards, dones)
        obs = self.normalize_obs(obs)
        rewards = self.normalize_reward(rewards)
        for idx in np.nonzero(dones)[0]:
            info = infos.get(int(idx))
            if info is not None and "terminal_observation" in info:
                info["terminal_observation"] = self.normalize_obs(info["terminal_observation"])
        return obs, rewards, dones, infos


def compute_returns_and_advantage(rewards, values, episode_starts, last_values, dones, gamma, gae_lambda):
    """RolloutBuffer.compute_returns_and_advantage (common/buffers.py), float32 arrays [T, N]."""
    T = rewards.shape[0]
    advantages = np.zeros_like(rewards)
    last_gae_lam = 0
    for step in reversed(range(T)):
        if step == T - 1:
            next_non_terminal = 1.0 - dones.astype(np.float32)
            next_values = last_values
        else:
            next_non_terminal = 1.0 - episode_starts[step + 1]
            next_values = values[step + 1]
        delta = rewards[step] + gamma * next_values * next_non_terminal - values[step]
        last_gae_lam = delta + gamma * gae_lambda * next_non_terminal * last_gae_lam
        advantages[step] = last_gae_lam
    return advantages, advantages + values

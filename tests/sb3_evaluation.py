"""Numpy restatement of stable-baselines3 2.x `common/evaluation.py` `evaluate_policy` (Monitor-wrapped env,
deterministic=True, return_episode_rewards=True), the reference that DeviceEvaluator (hlynr_intercept_b200/evaluation.py) is
compared against.  PARITY UNPINNED like oracle/sb3_post.py: SB3 is not importable here; this restates its published source.

    n_envs = env.num_envs
    episode_counts = np.zeros(n_envs, dtype="int")
    episode_count_targets = np.array([(n_eval_episodes + i) // n_envs for i in range(n_envs)], dtype="int")
    observations = env.reset()
    while (episode_counts < episode_count_targets).any():
        actions, states = model.predict(observations, deterministic=True)
        new_observations, rewards, dones, infos = env.step(actions)
        for i in range(n_envs):
            if episode_counts[i] < episode_count_targets[i]:
                if dones[i] and "episode" in infos[i].keys():       # is_monitor_wrapped
                    episode_rewards.append(infos[i]["episode"]["r"])
                    episode_lengths.append(infos[i]["episode"]["l"])
                    episode_counts[i] += 1
        observations = new_observations
"""
import numpy as np


def episode_count_targets(n_envs, n_eval_episodes):
    return np.array([(n_eval_episodes + i) // n_envs for i in range(n_envs)], dtype=np.int64)


def evaluate_policy(reset_fn, step_fn, predict_fn, n_envs, n_eval_episodes):
    """reset_fn() -> obs; step_fn(actions) -> (obs, dones [n_envs] bool, infos: indexable by env, entries needed for the
    finished envs); predict_fn(obs) -> actions.  Returns (episode_rewards, episode_lengths, episode_infos): the lists in append
    order, and the info dict of each counted episode (the same order) for comparisons beyond 'r' and 'l'."""
    episode_rewards, episode_lengths, episode_infos = [], [], []
    episode_counts = np.zeros(n_envs, dtype=np.int64)
    targets = episode_count_targets(n_envs, n_eval_episodes)
    observations = reset_fn()
    while (episode_counts < targets).any():
        actions = predict_fn(observations)
        new_observations, dones, infos = step_fn(actions)
        for i in range(n_envs):
            if episode_counts[i] < targets[i] and dones[i] and "episode" in infos[i]:
                episode_rewards.append(infos[i]["episode"]["r"])
                episode_lengths.append(infos[i]["episode"]["l"])
                episode_infos.append(infos[i])
                episode_counts[i] += 1
        observations = new_observations
    return episode_rewards, episode_lengths, episode_infos

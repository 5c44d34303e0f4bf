/*
 * hlynr_rollout.h -- C ABI of the device-side pieces of PPO rollout collection that consume the tensor API of the
 * simulator (SURVEY 8f rank 4, BASELINE config 5 "train.py PPO rollout collection").  The policy network itself is the
 * caller's (torch); these are the two non-GEMM steps stable-baselines3 runs in Python/NumPy around env.step:
 *
 *   reference interface (third party: stable-baselines3 2.x, see oracle/sb3_post.py)             replaced by
 *   ------------------------------------------------------------------------------------------  ------------------------
 *   OnPolicyAlgorithm.collect_rollouts: "if done and infos[idx]['TimeLimit.truncated']:          hlynr_bootstrap_timeouts
 *       rewards[idx] += gamma * policy.predict_values(terminal_observation)"
 *   RolloutBuffer.compute_returns_and_advantage (GAE(lambda), called at rl_system/scripts/       hlynr_gae
 *       train_flat_ppo.py:431-448 through model.learn)
 *   evaluate_policy's per-env episode quotas (EvalCallback, train_flat_ppo.py:497-504):          hlynr_eval_record
 *       "if episode_counts[i] < episode_count_targets[i] and dones[i]: append info['episode']"
 *   inference.py:535-606 logging every tick of each evaluated episode (UnifiedLogger, logger.py:148-273)  hlynr_eval_trace
 *
 * Conventions as in hlynr.h.
 */
#ifndef HLYNR_ROLLOUT_H
#define HLYNR_ROLLOUT_H

#include "hlynr.h"

#ifdef __cplusplus
extern "C" {
#endif

/* rewards_dev[env] += gamma * terminal_values_dev[r] for every record r < min(*counter_dev, rows) of the step's done list
 * that was truncated but not terminated (info['TimeLimit.truncated']).  terminal_values_dev has `rows` entries (the value
 * net evaluated on the first `rows` stacked terminal observations).  If the step finished more than `rows` episodes,
 * *overflow_dev (int32, device, may be NULL) is incremented by the number of truncated-and-not-terminated records left out
 * (timeouts that went without their bootstrap value): callers pass rows = N, or check *overflow_dev once per rollout. */
int hlynr_bootstrap_timeouts(float* rewards_dev, const HlynrDoneRecord* records_dev, const int32_t* counter_dev,
                             int32_t rows, const float* terminal_values_dev, double gamma, int32_t* overflow_dev,
                             int device, void* stream);

/* GAE(lambda) over a [T, N] rollout, float32 arithmetic in SB3's order (one thread per env, reverse scan over T):
 *   rewards_dev, values_dev, episode_starts_dev : float[T, N] (episode_starts = 1.0 where the step begins an episode)
 *   last_values_dev float[N], last_dones_dev uint8[N] : value / done flag of the observation after the last step
 *   advantages_dev, returns_dev : float[T, N] outputs (returns = advantages + values) */
int hlynr_gae(const float* rewards_dev, const float* values_dev, const float* episode_starts_dev,
              const float* last_values_dev, const uint8_t* last_dones_dev, int64_t T, int64_t N, double gamma,
              double gae_lambda, float* advantages_dev, float* returns_dev, int device, void* stream);

/* SB3 evaluate_policy's episode accounting: env e counts its first target_e = (n_episodes + e) / n_envs finished episodes.
 * For each record r < min(*counter_dev, n_envs) of the step's done list (records_dev has n_envs entries) whose env e has
 * counts_dev[e] < target_e:
 *   ticks_dev[e] += steps;  k = offset_e + counts_dev[e];  results_dev[k] = record;  end_tick_dev[k] = ticks_dev[e];
 *   counts_dev[e] += 1;     *remaining_dev -= 1
 * offset_e = e*q + max(0, e - (n_envs - rem)), q = n_episodes / n_envs, rem = n_episodes % n_envs  (= sum of targets before e).
 * Every env starts at the same reset and auto-reset starts its next episode on the following step, so end_tick_dev[k] is the
 * step on which episode k ended, counted from that reset; SB3's list order is the sort by (end_tick, env).  The table does not
 * depend on the order of the records within a step.  The caller zeroes counts_dev (int32[n_envs]) and ticks_dev (int64[n_envs])
 * and sets *remaining_dev (int64) to n_episodes; results_dev / end_tick_dev have n_episodes entries.
 * n_episodes must be in [1, INT32_MAX]. */
int hlynr_eval_record(const HlynrDoneRecord* records_dev, const int32_t* counter_dev, int64_t n_envs, int64_t n_episodes,
                      int32_t* counts_dev, int64_t* ticks_dev, HlynrDoneRecord* results_dev, int64_t* end_tick_dev,
                      int64_t* remaining_dev, int device, void* stream);

/* One tick of one evaluated episode: the values of the reference's info dict for that tick (environment.py:829-857) that its
 * offline inference logs per tick (inference.py:535-548), plus the action, reward and done bits. */
typedef struct HlynrTraceRow {
    float interceptor_pos[3], missile_pos[3];   /* info['interceptor_pos'], info['missile_pos'] */
    float action[6];                            /* the clipped action the env received */
    float reward, distance, fuel_remaining, radar_quality;
    uint32_t flags;                             /* HLYNR_INFO_* bits of the tick; | HLYNR_DONE_TERMINATED / _TRUNCATED on the last row */
    int32_t step;                               /* info['steps'], 1-based */
} HlynrTraceRow;                                /* 18 words = 72 bytes */
size_t hlynr_trace_row_size(void);

/* Files the tick's row of every env still inside its evaluate_policy quota (counts_dev[e] < target_e, targets and offset_e as
 * in hlynr_eval_record) at table_dev[(offset_e + counts_dev[e]) * max_steps + steps[e] - 1]; a row whose steps[e] lies outside
 * [1, max_steps] is not written.  Launch once per tick after hlynr_step (+ hlynr_post_step) and BEFORE hlynr_eval_record of the
 * same tick, which increments counts_dev: the terminal tick is then still addressed to the episode it ends.  No argument changes
 * between ticks, so a CUDA graph of the tick replays correctly.
 *   info: host struct of the tick's device info arrays (what hlynr_step wrote); distance, fuel_remaining, steps, flags,
 *         interceptor_pos, missile_pos and radar_quality must be set, the other fields are not read
 *   actions_dev float[n_envs, 6], rewards_dev float[n_envs], terminated_dev / truncated_dev uint8[n_envs] (the step's outputs)
 *   table_dev: n_episodes * max_steps rows; rows past an episode's length are left untouched
 * n_envs and n_episodes must be in [1, INT32_MAX], max_steps positive. */
int hlynr_eval_trace(const HlynrInfoSoA* info, const float* actions_dev, const float* rewards_dev, const uint8_t* terminated_dev,
                     const uint8_t* truncated_dev, const int32_t* counts_dev, int64_t n_envs, int64_t n_episodes,
                     int32_t max_steps, HlynrTraceRow* table_dev, int device, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HLYNR_ROLLOUT_H */

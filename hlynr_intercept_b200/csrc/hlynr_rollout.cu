// hlynr_rollout.cu -- timeout bootstrapping, GAE(lambda) and evaluation episode quotas on the device (C ABI:
// include/hlynr_rollout.h).  Restated from stable-baselines3 2.x: common/on_policy_algorithm.py collect_rollouts,
// common/buffers.py RolloutBuffer.compute_returns_and_advantage (float32 arrays, Python-float gamma / gae_lambda),
// common/evaluation.py evaluate_policy.
#include <cuda_runtime.h>

#include "../../include/hlynr_rollout.h"
#include "hlynr_host.cuh"

namespace {

__global__ void bootstrap_kernel(float* __restrict__ rewards, const HlynrDoneRecord* __restrict__ recs, const int32_t* __restrict__ counter,
                                 int32_t rows, const float* __restrict__ tv, float gamma, int32_t* overflow) {
    const int32_t count = *counter;
    const int32_t m = count < rows ? count : rows;
    for (int32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < m; r += gridDim.x * blockDim.x) {
        const uint32_t fl = recs[r].flags;
        if ((fl & HLYNR_DONE_TRUNCATED) && !(fl & HLYNR_DONE_TERMINATED)) {
            const int32_t e = recs[r].env;  // one record per env per step: no write conflict
            rewards[e] = __fadd_rn(rewards[e], __fmul_rn(gamma, tv[r]));
        }
    }
    // records beyond `rows` got no value: count the ones that NEEDED one (truncated and not terminated) -- a non-zero *overflow
    // means timeouts went without their gamma * V(terminal_observation)
    if (overflow && count > rows) {
        int32_t missed = 0;
        for (int32_t r = rows + blockIdx.x * blockDim.x + threadIdx.x; r < count; r += gridDim.x * blockDim.x) {
            const uint32_t fl = recs[r].flags;
            missed += ((fl & HLYNR_DONE_TRUNCATED) && !(fl & HLYNR_DONE_TERMINATED)) ? 1 : 0;
        }
        if (missed) atomicAdd(overflow, missed);
    }
}

// evaluate_policy's quota accounting: an env has at most one record per step, so its counts / ticks words are touched by one
// thread only; results are addressed by (env, episode index) instead of appended, which makes the table independent of the
// unspecified order of the records within a step
__global__ void eval_record_kernel(const HlynrDoneRecord* __restrict__ recs, const int32_t* __restrict__ counter, int64_t n_envs,
                                   int64_t q, int64_t rem, int32_t* __restrict__ counts, int64_t* __restrict__ ticks,
                                   HlynrDoneRecord* __restrict__ results, int64_t* __restrict__ end_tick,
                                   unsigned long long* remaining) {
    const int64_t count = *counter;
    const int64_t m = count < n_envs ? count : n_envs;
    const int64_t full = n_envs - rem;   // targets: q for envs [0, full), q + 1 for envs [full, n_envs)
    int taken = 0;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < m; r += (int64_t)gridDim.x * blockDim.x) {
        const int64_t e = recs[r].env;
        const int32_t c = counts[e];
        if (c >= (e < full ? q : q + 1)) continue;   // past the env's quota: SB3 ignores the episode
        const int64_t t = ticks[e] + recs[r].steps;   // auto-reset starts the next episode on the following step
        const int64_t k = e * q + (e > full ? e - full : 0) + c;
        results[k] = recs[r];
        end_tick[k] = t;
        ticks[e] = t;
        counts[e] = c + 1;
        ++taken;
    }
    taken = __reduce_add_sync(0xffffffffu, taken);   // every lane of every warp leaves the loop: blockDim is a multiple of 32
    if (taken && (threadIdx.x & 31) == 0) atomicAdd(remaining, (unsigned long long)(-(long long)taken));
}

static_assert(sizeof(HlynrTraceRow) == 72, "HlynrTraceRow is 18 words");

// the info arrays a trace row reads (hlynr_step writes them; the step kernel skips a NULL field)
struct TraceInfo {
    const float *distance, *fuel_remaining, *radar_quality, *interceptor_pos, *missile_pos;
    const int32_t* steps;
    const uint8_t* flags;
};

// One thread per env.  The row is addressed by the env's episode index counts[e] (not yet incremented for the terminal tick:
// eval_record_kernel runs after this one) and the tick's info['steps'], so no cursor is kept and nothing in the arguments
// changes from tick to tick: a recorded chunk graph writes the same rows as eager launches.
__global__ void __launch_bounds__(256) eval_trace_kernel(TraceInfo in, const float* __restrict__ actions, const float* __restrict__ rewards,
                                                         const uint8_t* __restrict__ terminated, const uint8_t* __restrict__ truncated,
                                                         const int32_t* __restrict__ counts, int64_t n_envs, int64_t q, int64_t rem,
                                                         int32_t max_steps, HlynrTraceRow* __restrict__ table) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_envs) return;
    const int64_t full = n_envs - rem;   // targets and offsets as in eval_record_kernel
    const int32_t c = counts[e];
    if (c >= (e < full ? q : q + 1)) return;   // past the env's quota: SB3 ignores the episode
    const int32_t s = in.steps[e];
    if (s < 1 || s > max_steps) return;
    HlynrTraceRow* r = table + (e * q + (e > full ? e - full : 0) + c) * max_steps + (s - 1);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        r->interceptor_pos[k] = in.interceptor_pos[3 * e + k];
        r->missile_pos[k] = in.missile_pos[3 * e + k];
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) r->action[k] = actions[6 * e + k];
    r->reward = rewards[e];
    r->distance = in.distance[e];
    r->fuel_remaining = in.fuel_remaining[e];
    r->radar_quality = in.radar_quality[e];
    r->flags = (uint32_t)in.flags[e] | (terminated[e] ? HLYNR_DONE_TERMINATED : 0u) | (truncated[e] ? HLYNR_DONE_TRUNCATED : 0u);
    r->step = s;
}

// one thread per env, reverse scan over T; every access is coalesced over N
__global__ void __launch_bounds__(256) gae_kernel(const float* __restrict__ rew, const float* __restrict__ val, const float* __restrict__ starts,
                                                  const float* __restrict__ last_val, const uint8_t* __restrict__ last_done, int64_t T,
                                                  int64_t N, float gamma, float gamma_lambda, float* __restrict__ adv, float* __restrict__ ret) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= N) return;
    float next_val = last_val[e];
    float next_nonterm = 1.f - (last_done[e] ? 1.f : 0.f);
    float lam = 0.f;
    for (int64_t t = T - 1; t >= 0; --t) {
        const int64_t k = t * N + e;
        const float v = val[k];
        // delta = r + gamma * next_values * next_non_terminal - values;  last = delta + gamma * lambda * next_non_terminal * last
        const float delta = __fsub_rn(__fadd_rn(rew[k], __fmul_rn(__fmul_rn(gamma, next_val), next_nonterm)), v);
        lam = __fadd_rn(delta, __fmul_rn(__fmul_rn(gamma_lambda, next_nonterm), lam));  // gamma * gae_lambda is a Python-float product
        adv[k] = lam;
        ret[k] = __fadd_rn(lam, v);
        next_val = v;
        next_nonterm = 1.f - starts[k];
    }
}

}  // namespace

extern "C" {

int hlynr_bootstrap_timeouts(float* rewards_dev, const HlynrDoneRecord* records_dev, const int32_t* counter_dev, int32_t rows,
                             const float* terminal_values_dev, double gamma, int32_t* overflow_dev, int device, void* stream) {
    if (!rewards_dev || !records_dev || !counter_dev || !terminal_values_dev) return fail("hlynr_bootstrap_timeouts: null argument");
    if (rows <= 0) return fail("hlynr_bootstrap_timeouts: rows must be positive");
    DeviceGuard g(device);
    const int blocks = rows < 256 * 64 ? (rows + 255) / 256 : 64;
    bootstrap_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(rewards_dev, records_dev, counter_dev, rows, terminal_values_dev, (float)gamma, overflow_dev);
    CK(cudaGetLastError());
    return 0;
}

int hlynr_gae(const float* rewards_dev, const float* values_dev, const float* episode_starts_dev, const float* last_values_dev,
              const uint8_t* last_dones_dev, int64_t T, int64_t N, double gamma, double gae_lambda, float* advantages_dev,
              float* returns_dev, int device, void* stream) {
    if (!rewards_dev || !values_dev || !episode_starts_dev || !last_values_dev || !last_dones_dev || !advantages_dev || !returns_dev)
        return fail("hlynr_gae: null argument");
    if (T <= 0 || N <= 0) return fail("hlynr_gae: T and N must be positive");
    DeviceGuard g(device);
    gae_kernel<<<(unsigned)((N + 255) / 256), 256, 0, (cudaStream_t)stream>>>(rewards_dev, values_dev, episode_starts_dev, last_values_dev,
                                                                            last_dones_dev, T, N, (float)gamma, (float)(gamma * gae_lambda),
                                                                            advantages_dev, returns_dev);
    CK(cudaGetLastError());
    return 0;
}

int hlynr_eval_record(const HlynrDoneRecord* records_dev, const int32_t* counter_dev, int64_t n_envs, int64_t n_episodes,
                      int32_t* counts_dev, int64_t* ticks_dev, HlynrDoneRecord* results_dev, int64_t* end_tick_dev,
                      int64_t* remaining_dev, int device, void* stream) {
    if (!records_dev || !counter_dev || !counts_dev || !ticks_dev || !results_dev || !end_tick_dev || !remaining_dev)
        return fail("hlynr_eval_record: null argument");
    if (n_envs <= 0 || n_envs > INT32_MAX) return fail("hlynr_eval_record: n_envs must be in [1, INT32_MAX]");
    if (n_episodes <= 0 || n_episodes > INT32_MAX) return fail("hlynr_eval_record: n_episodes must be in [1, INT32_MAX]");
    DeviceGuard g(device);
    const int blocks = n_envs < 256 * 64 ? (int)((n_envs + 255) / 256) : 64;
    eval_record_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(records_dev, counter_dev, n_envs, n_episodes / n_envs, n_episodes % n_envs,
                                                                 counts_dev, ticks_dev, results_dev, end_tick_dev,
                                                                 reinterpret_cast<unsigned long long*>(remaining_dev));
    CK(cudaGetLastError());
    return 0;
}

size_t hlynr_trace_row_size(void) { return sizeof(HlynrTraceRow); }

int hlynr_eval_trace(const HlynrInfoSoA* info, const float* actions_dev, const float* rewards_dev, const uint8_t* terminated_dev,
                     const uint8_t* truncated_dev, const int32_t* counts_dev, int64_t n_envs, int64_t n_episodes,
                     int32_t max_steps, HlynrTraceRow* table_dev, int device, void* stream) {
    if (!info || !actions_dev || !rewards_dev || !terminated_dev || !truncated_dev || !counts_dev || !table_dev)
        return fail("hlynr_eval_trace: null argument");
    if (!info->distance || !info->fuel_remaining || !info->steps || !info->flags || !info->interceptor_pos || !info->missile_pos ||
        !info->radar_quality)
        return fail("hlynr_eval_trace: null argument (info: distance, fuel_remaining, steps, flags, interceptor_pos, missile_pos "
                    "and radar_quality are read)");
    if (n_envs <= 0 || n_envs > INT32_MAX) return fail("hlynr_eval_trace: n_envs must be in [1, INT32_MAX]");
    if (n_episodes <= 0 || n_episodes > INT32_MAX) return fail("hlynr_eval_trace: n_episodes must be in [1, INT32_MAX]");
    if (max_steps <= 0) return fail("hlynr_eval_trace: max_steps must be positive");
    DeviceGuard g(device);
    const TraceInfo in{info->distance, info->fuel_remaining, info->radar_quality, info->interceptor_pos, info->missile_pos,
                       info->steps, info->flags};
    eval_trace_kernel<<<(unsigned)((n_envs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        in, actions_dev, rewards_dev, terminated_dev, truncated_dev, counts_dev, n_envs, n_episodes / n_envs, n_episodes % n_envs,
        max_steps, table_dev);
    CK(cudaGetLastError());
    return 0;
}

}  // extern "C"

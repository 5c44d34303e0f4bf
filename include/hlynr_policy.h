/*
 * hlynr_policy.h -- C ABI of the fused actor-critic forward used by on-device rollout collection (SURVEY 8f rank 4,
 * BASELINE config 5 "train.py PPO rollout collection").
 *
 *   reference interface                                                                    replaced by
 *   ------------------------------------------------------------------------------------  ----------------------
 *   CustomMLP.forward            rl_system/scripts/train_flat_ppo.py:37-85                 hlynr_policy_forward
 *     (in_dim -> Linear 512 -> LayerNorm -> ReLU -> Linear 512 -> LayerNorm -> ReLU -> Linear 256 -> LayerNorm -> ReLU)
 *   SB3 ActorCriticPolicy heads with net_arch=[] (train_flat_ppo.py:419-429): action_net
 *     Linear(256, 6), value_net Linear(256, 1), state-independent log_std; forward() samples
 *     a = mean + exp(log_std) * eps and returns (a, V, log pi(a))                          hlynr_policy_forward
 *   policy.predict_values(terminal_observation) of collect_rollouts' TimeLimit bootstrap   hlynr_policy_forward with
 *                                                                                          n_rows_dev = the done counter
 *
 * One sm_100a kernel does the whole forward for a tile of 128 observation rows: the three GEMMs and the two heads run on
 * the tcgen05 tensor cores (bf16 operands, fp32 accumulators in TMEM), weight tiles arrive by TMA into a shared-memory
 * ring, and bias + LayerNorm + ReLU is the epilogue that turns the TMEM accumulators of one layer into the bf16 A operand
 * of the next without leaving the SM.  Conventions as in hlynr.h (plain pointers, 0 = success, hlynr_last_error()).
 * The hidden layers and heads are the reference's default (train_flat_ppo.py:410 net_arch [512, 512, 256], 6 actions); the
 * input width in_dim is that of the stacked observation, 1-256: 104 = frame_stack 4 x 26-D (the default), 68 = 4 x 17-D, and
 * every other frame_stack of either frame width.  Other shapes are rejected.
 */
#ifndef HLYNR_POLICY_H
#define HLYNR_POLICY_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HLYNR_POLICY_IN 104   /* 4 stacked 26-D frames: the default input width */
#define HLYNR_POLICY_MAX_IN 256   /* widest input: four 64-wide K blocks of the first GEMM */
#define HLYNR_POLICY_H1 512
#define HLYNR_POLICY_H2 512
#define HLYNR_POLICY_H3 256
#define HLYNR_POLICY_ACT 6

typedef struct hlynr_policy hlynr_policy_t;

/* fp32 parameters in PyTorch layout (nn.Linear.weight is [out, in]); device pointers, copied (as bf16 for the GEMM operands)
 * by hlynr_policy_set_weights, so the caller's tensors may change afterwards. */
typedef struct HlynrPolicyWeights {
    const float *w1, *b1, *ln1_g, *ln1_b;   /* [512,in_dim], [512] x3 */
    const float *w2, *b2, *ln2_g, *ln2_b;   /* [512,512], [512] x3 */
    const float *w3, *b3, *ln3_g, *ln3_b;   /* [256,512], [256] x3 */
    const float *wa, *ba;                   /* action_net [6,256], [6] */
    const float *wv, *bv;                   /* value_net  [1,256], [1] */
    const float *log_std;                   /* [6] */
    float ln_eps;                           /* nn.LayerNorm eps (1e-5) */
} HlynrPolicyWeights;

/* A network with input width in_dim in [1, HLYNR_POLICY_MAX_IN]. */
int hlynr_policy_create_dim(int device, int in_dim, hlynr_policy_t** out);
/* hlynr_policy_create_dim with in_dim = HLYNR_POLICY_IN (104). */
int hlynr_policy_create(int device, hlynr_policy_t** out);
void hlynr_policy_destroy(hlynr_policy_t* p);
int hlynr_policy_set_weights(hlynr_policy_t* p, const HlynrPolicyWeights* w, void* stream);

/* Forward of rows [0, n_rows) of obs_dev float[n_rows, in_dim]: rows of pitch in_dim floats.  obs_dev must be 16-byte aligned
 * for in_dim = 104 and 4-byte aligned for every other width (a row of a [T + 1, N, in_dim] rollout buffer).
 *   n_rows_dev   NULL, or a device int32: only min(n_rows, *n_rows_dev) rows are computed (tiles beyond it exit at once);
 *                lets the value net run on "the finished episodes of this step" without a host round trip
 *   actions_dev  float[n_rows, 6] or NULL: mean + exp(log_std) * eps (deterministic != 0: the mean)
 *   values_dev   float[n_rows]    or NULL
 *   logp_dev     float[n_rows]    or NULL: log-probability of the sampled action under the diagonal Gaussian
 *   mean_dev     float[n_rows, 6] or NULL
 *   actions_clipped_dev float[n_rows, 6] or NULL: the sampled action clipped to the action space [-1, 1]^6 -- what SB3's
 *                collect_rollouts passes to env.step while the rollout buffer keeps the unclipped one
 *   seed, counter: eps comes from Philox4x32-10 keyed by seed with counter (row, counter): pass a new counter per call.
 * This entry never reads or changes the handle's device-resident counter (hlynr_policy_forward_dev). */
int hlynr_policy_forward(hlynr_policy_t* p, const float* obs_dev, int64_t n_rows, const int32_t* n_rows_dev,
                         float* actions_dev, float* values_dev, float* logp_dev, float* mean_dev, float* actions_clipped_dev,
                         uint64_t seed, uint64_t counter, int deterministic, void* stream);

/* hlynr_policy_forward with the call counter kept on the device: every launch draws at counter = *dev_counter + 1 and stores
 * that value, for every kind of call (deterministic, value only, any *n_rows_dev, zero included), so a forward captured in a CUDA
 * graph draws fresh noise on every replay.  The handle owns the counter (0 after hlynr_policy_create*).  Forwards through the
 * device counter of one handle must be ordered on one stream: each launch reads the value the previous one stored. */
int hlynr_policy_forward_dev(hlynr_policy_t* p, const float* obs_dev, int64_t n_rows, const int32_t* n_rows_dev,
                             float* actions_dev, float* values_dev, float* logp_dev, float* mean_dev, float* actions_clipped_dev,
                             uint64_t seed, int deterministic, void* stream);
/* Sets the device-resident counter, ordered on `stream` (a one-thread kernel: value is a kernel argument, no host buffer). */
int hlynr_policy_set_counter(hlynr_policy_t* p, uint64_t value, void* stream);
/* Synchronises `stream` and returns the device-resident counter: the counter of the last forward_dev that ran on it. */
int hlynr_policy_get_counter(hlynr_policy_t* p, uint64_t* out, void* stream);

/* Options.  "cluster": CTAs per thread-block cluster, 1 (default), 2 or 4: the CTAs of a cluster share every weight tile through
 * TMA multicast, which divides the L2 -> SM weight traffic (the kernel's bottleneck without it) by the cluster size. */
int hlynr_policy_set_option(hlynr_policy_t* p, const char* name, int64_t value);

/* Debug: with option "timing" = 1 the kernel records SM-clock timestamps of the phases of CTA 0's first 8 tiles; host_out is
 * long long[8][16]: 0 tile start, 1 x loaded, 2/4/6 accumulators of layer 1/2/3 ready, 3/5/7 epilogue of layer 1/2/3 done,
 * 8 head accumulators ready, 9 tile done. */
int hlynr_policy_get_timing(hlynr_policy_t* p, long long* host_out);

/* Kernel launches issued by this handle so far. */
int hlynr_policy_launch_count(const hlynr_policy_t* p, int64_t* out);

#ifdef __cplusplus
}
#endif
#endif /* HLYNR_POLICY_H */

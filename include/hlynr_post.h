/*
 * hlynr_post.h -- C ABI of the on-device observation post-processing that directly follows the env step in every
 * trainer of the reference (SURVEY 8f rank 1):
 *
 *   reference interface (third party: stable-baselines3, see oracle/sb3_post.py)      replaced by
 *   -------------------------------------------------------------------------------  -------------------------
 *   VecFrameStack(envs, n_stack)             rl_system/scripts/train_flat_ppo.py:384-388   hlynr_post_create / _reset / _step
 *   VecNormalize(envs, norm_obs=True, norm_reward=False, clip_obs=10, gamma)   :392-399     hlynr_post_create / _reset / _step
 *   VecNormalize.load(...); env.training = False       rl_system/inference.py:455-471      hlynr_post_set_stats, training = 0
 *   VecNormalize.normalize_obs / get_original_obs                                           hlynr_post_normalize / _original
 *
 * Layout: the last n_stack raw frames live in a ring of [n_stack][N][F] planes, F = the frame width: 26 (the full
 * observation) or 17 (the leading radar channels obs[0:17] a sim with option "obs_dim" = 17 writes); hlynr_step /
 * hlynr_reset write their observation STRAIGHT into the ring slot hlynr_post_obs_target returns (no copy), a per-env age
 * byte says how many older frames are valid since the env's last reset (SB3 zeroes the stack of a finished env), and the
 * stacked, normalised [N, F*n_stack] observation is produced in one pass.  The running mean/variance (float64, SB3's
 * RunningMeanStd) is updated from per-lag column sums that are maintained incrementally: only the new frame is summed
 * (4F B per env) and the frames of the few finished envs are subtracted.
 *
 * Conventions as in hlynr.h: 0 = ok, message from hlynr_last_error(); device pointers are caller-owned; all work is
 * ordered on `stream`.
 */
#ifndef HLYNR_POST_H
#define HLYNR_POST_H

#include "hlynr.h"

#ifdef __cplusplus
extern "C" {
#endif

#define HLYNR_POST_MAX_STACK 8

typedef struct hlynr_post hlynr_post_t;

/* frame_dim = F, the width of one frame: 26, or 17 for a sim created with option "obs_dim" = 17;
 * n_stack = VecFrameStack n_stack (1 = no stacking); clip_obs / epsilon / gamma = VecNormalize's (10.0, 1e-8, 0.99). */
int hlynr_post_create_frames(int64_t n_envs, int device, int frame_dim, int n_stack, double clip_obs, double epsilon,
                             double gamma, hlynr_post_t** out);
/* hlynr_post_create_frames with frame_dim = 26. */
int hlynr_post_create(int64_t n_envs, int device, int n_stack, double clip_obs, double epsilon, double gamma,
                      hlynr_post_t** out);
void hlynr_post_destroy(hlynr_post_t* post);
int hlynr_post_obs_dim(const hlynr_post_t* post, int* out); /* F * n_stack */

/* Device pointer (float[N,F]) the NEXT hlynr_reset / hlynr_step call must pass as obs_dev. */
int hlynr_post_obs_target(hlynr_post_t* post, float** obs_dev);

/* VecFrameStack.reset + VecNormalize.reset, after hlynr_reset(all envs) wrote into the target.
 * out_dev float[N, F*n_stack]; training != 0 updates the running statistics with this batch. */
int hlynr_post_reset(hlynr_post_t* post, float* out_dev, int training, void* stream);

/* VecFrameStack.step_wait + VecNormalize.step_wait, after hlynr_step wrote into the target.
 *   reward_dev, terminated_dev, truncated_dev : outputs of that hlynr_step call
 *   records_dev, counter_dev, capacity        : its compact done list (hlynr_set_done_list), or NULL
 *   out_dev            float[N, F*n_stack]   : stacked + normalised observation
 *   terminal_out_dev   float[capacity, F*n_stack] or NULL: row r = stacked + normalised info['terminal_observation']
 *                      of records_dev[r]; its newest frame is terminal_obs[0:F] of the record
 *   training           != 0: update obs_rms (and returns / ret_rms) with this batch before normalising */
int hlynr_post_step(hlynr_post_t* post, const float* reward_dev, const uint8_t* terminated_dev,
                    const uint8_t* truncated_dev, const HlynrDoneRecord* records_dev, const int32_t* counter_dev,
                    int32_t capacity, float* out_dev, float* terminal_out_dev, int training, void* stream);

/* VecNormalize.get_original_obs(): the stacked, un-normalised observation of the last reset/step. */
int hlynr_post_original(hlynr_post_t* post, float* out_dev, void* stream);
/* VecNormalize.normalize_obs on `rows` caller-provided stacked rows (float[rows, F*n_stack], in place allowed). */
int hlynr_post_normalize(hlynr_post_t* post, const float* stacked_dev, int64_t rows, float* out_dev, void* stream);

/* obs_rms (mean/var: double[F*n_stack], count) and ret_rms (scalars); host pointers, any may be NULL.
 * These are the fields of SB3's vec_normalize.pkl. */
int hlynr_post_get_stats(hlynr_post_t* post, double* mean, double* var, double* count, double* ret_mean,
                         double* ret_var, double* ret_count, void* stream);
int hlynr_post_set_stats(hlynr_post_t* post, const double* mean, const double* var, double count, double ret_mean,
                         double ret_var, double ret_count, void* stream);

/* Test hook: recomputes the per-lag column sums from the frame ring (reads everything) and returns the largest
 * absolute difference to the incrementally maintained ones; resync != 0 also replaces them. */
int hlynr_post_check_sums(hlynr_post_t* post, int resync, double* max_abs_diff, void* stream);
int hlynr_post_launch_count(const hlynr_post_t* post, int64_t* out);
/* CUDA-graph support (see hlynr_ring_period in hlynr.h): a captured sequence of T steps replays correctly iff T is a
 * multiple of n_stack; after each replay call hlynr_post_note_replayed_steps(post, T). */
int hlynr_post_note_replayed_steps(hlynr_post_t* post, int64_t steps, int64_t launches);

/*
 * Snapshots (see hlynr_snapshot_save in hlynr.h): a descriptor plus one device image in a canonical layout that does not depend
 * on the ring phase t % n_stack.  Sections, each 256-byte aligned:
 *   HLYNR_POST_SNAP_FRAMES   float[n_stack][N][F]: the frame ring from the oldest frame to the newest
 *   HLYNR_POST_SNAP_AGE      uint8[N]: how many older frames belong to each env's episode
 *   HLYNR_POST_SNAP_RETURNS  double[N]: VecNormalize's discounted returns
 *   HLYNR_POST_SNAP_STATS    the device statistics block, stats_bytes long: obs_rms, ret_rms and the per-lag column sums that
 *                            later updates start from
 */
#define HLYNR_POST_SNAPSHOT_VERSION 1
enum { HLYNR_POST_SNAP_FRAMES = 0, HLYNR_POST_SNAP_AGE = 1, HLYNR_POST_SNAP_RETURNS = 2, HLYNR_POST_SNAP_STATS = 3,
       HLYNR_POST_SNAP_SECTIONS = 4 };

typedef struct HlynrPostSnapshotInfo {
    int32_t format_version;   /* HLYNR_POST_SNAPSHOT_VERSION */
    int32_t frame_dim, n_stack;
    int32_t sums_valid;       /* the per-lag column sums describe the ring (hlynr_post_step can train) */
    int64_t n_envs;
    uint64_t t;               /* frames written so far (every reset and step writes one) */
    double clip_obs, epsilon, gamma;
    uint64_t stats_bytes;
    uint64_t section_offset[HLYNR_POST_SNAP_SECTIONS];
    uint64_t device_bytes;
} HlynrPostSnapshotInfo;

size_t hlynr_post_snapshot_info_size(void);
int hlynr_post_snapshot_layout(const hlynr_post_t* post, HlynrPostSnapshotInfo* info, size_t* device_bytes);
/* Writes the image to dev_out and fills `info`; ordered on `stream`.  Refused while `stream` is capturing. */
int hlynr_post_snapshot_save(hlynr_post_t* post, void* dev_out, HlynrPostSnapshotInfo* info, void* stream);
/* Restores a snapshot into a pipeline created with the same n_envs, frame_dim, n_stack, clip_obs, epsilon and gamma (refuses
 * another, naming the first mismatch, and a capturing stream).  Ordered on `stream`. */
int hlynr_post_snapshot_load(hlynr_post_t* post, const HlynrPostSnapshotInfo* info, const void* dev_in, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HLYNR_POST_H */

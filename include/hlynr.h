/*
 * hlynr.h -- C ABI of the B200-native batched Hlynr Intercept simulator.
 *
 * This is the drop-in boundary for the reference's per-step hot path.  Nothing like it
 * exists in the reference (it is pure Python); each entry point below names the reference
 * interface it replaces.  All `file:line` citations are relative to the reference tree
 * (RomanSlack/Hlynr_Intercept).
 *
 *   reference interface                                         replaced by
 *   ---------------------------------------------------------  -------------------------
 *   InterceptEnvironment.__init__   rl_system/environment.py:20  hlynr_create
 *   InterceptEnvironment.reset      rl_system/environment.py:353 hlynr_reset / hlynr_reset_host
 *   InterceptEnvironment.step       rl_system/environment.py:605 hlynr_step / hlynr_step_host
 *   (SB3 DummyVecEnv.step_wait auto-reset, scripts/train_flat_ppo.py:371)   folded into hlynr_step
 *   set_training_step_count / _update_radar_curriculum  environment.py:269-351  hlynr_set_curriculum
 *   get_current_intercept_radius    environment.py:223          (host side, then hlynr_set_curriculum)
 *   observation_generator.seed / np.random.seed  environment.py:357-359       hlynr_seed
 *   env.interceptor_state / missile_state (get_attr, visualize.py:149-196)    hlynr_export_state
 *   Monitor episode statistics (scripts/train_flat_ppo.py:292-303)            hlynr_get_stats
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary.
 *   - every function returns 0 on success, non-zero on failure; the message is available
 *     (per thread) from hlynr_last_error().
 *   - "dev" pointers are device pointers owned by the CALLER (e.g. torch tensors), valid on
 *     the device the handle was created on.  "host" pointers are ordinary host memory.
 *   - all device work is ordered on the `stream` argument (a cudaStream_t passed as void*;
 *     NULL = the legacy default stream).  A handle is single-producer: one host thread at a
 *     time.  Handles on different devices are independent.
 *   - observation layout is the reference's 26-D vector (rl_system/core.py:700-721); the
 *     17-D "radar" layout of the original project is obs[0:17].
 */
#ifndef HLYNR_H
#define HLYNR_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HLYNR_ABI_VERSION 1
#define HLYNR_OBS_DIM 26
#define HLYNR_ACT_DIM 6
#define HLYNR_MAX_ONBOARD_DELAY 10 /* physics_randomizer.py:293 clamps the delay to [1,10] */
#define HLYNR_MAX_GROUND_DELAY 31
#define HLYNR_N_DR 13              /* physics_randomizer.py:166-214: 13 draws per episode */
#define HLYNR_MAX_VOLLEY 8         /* missiles per env in volley mode (environment.py:42-44) */

/* observation_mode, rl_system/environment.py:157-166 */
enum { HLYNR_OBS_WORLD = 0, HLYNR_OBS_BODY = 1, HLYNR_OBS_LOS = 2 };
/* precision of the build that a handle runs (north_star: fp32 build / fp64 build) */
enum { HLYNR_FP32 = 32, HLYNR_FP64 = 64 };

/*
 * Resolved ("effective-key") configuration of one InterceptEnvironment.
 * Produced on the host by hlynr_intercept_b200.config.resolve_config() with the reference's
 * .get(key, default) semantics (rl_system/environment.py:24-186).  All reals are doubles --
 * they are Python floats in the reference and are rounded to the compute type at the point of
 * use exactly where NumPy-2 "weak scalar" promotion does it.
 */
typedef struct HlynrParams {
    int32_t abi_version;  /* must be HLYNR_ABI_VERSION */
    int32_t max_steps;    /* environment.py:26 */
    double dt;            /* environment.py:25 */
    double max_range;     /* environment.py:27 */
    double max_velocity;  /* environment.py:28 */
    double target[3];     /* environment.py:39 (float32-rounded) */

    /* --- spawn, environment.py:375-467 --- */
    int32_t m_spawn_spherical; /* missile_spawn.position_mode == 'spherical' */
    int32_t i_vel_toward_missile; /* interceptor_spawn.velocity_mode == 'toward_missile' */
    double m_pos_lo[3], m_pos_hi[3];
    double m_speed_lo, m_speed_hi;    /* :413-415 (norms of the velocity box unless speed_min/max given) */
    double m_radius_lo, m_radius_hi;  /* spherical mode :392-395 */
    double m_az_lo, m_az_hi;          /* degrees */
    double m_el_lo, m_el_hi;          /* degrees */
    double i_pos_lo[3], i_pos_hi[3];
    double i_vel_lo[3], i_vel_hi[3];
    double i_speed_lo, i_speed_hi;    /* :449-450 */

    /* --- wind, environment.py:71-73 --- */
    double base_wind[3];  /* float32-rounded */
    double wind_variability;

    /* --- physics v2.0 switches, environment.py:52-106 --- */
    int32_t isa_enabled;        /* atmospheric_model is not None */
    int32_t mach_enabled;       /* mach_drag_model is not None */
    int32_t enh_wind_enabled;   /* enhanced_wind_model is not None */
    int32_t thrust_dyn_enabled; /* thrust_dynamics_enabled */
    int32_t dr_enabled;         /* physics_randomizer is not None and .enabled */
    int32_t validate_enabled;   /* physics_validation_enabled :106 */
    int32_t evasion_enabled;    /* config['missile_evasion'] :1104 */
    int32_t onboard_delay;      /* samples; 0 = no onboard delay buffer (core.py:292-293) */
    double sub_mach, sup_mach, peak_mult, sup_mult; /* environment.py:65-68 */
    double blh, turb_intensity, gust_scale;         /* environment.py:81-85 */
    double thrust_tau;                              /* :94 */
    double dr_variation[HLYNR_N_DR]; /* sigma of each draw, in physics_randomizer.py:166-214 order;
                                        [1] is the temperature sigma in kelvin (0.05*20) */

    /* --- onboard radar, environment.py:136-138,171-176; core.py:258-270 --- */
    double radar_range;
    double radar_quality;

    /* --- ground radar + datalink, core.py:295-320 --- */
    int32_t ground_enabled;
    int32_t ground_delay; /* samples; 0 = no ground delay buffer */
    double ground_pos[3]; /* float32-rounded */
    double g_max_range, g_min_el, g_max_el; /* elevations in radians (np.radians of the YAML degrees) */
    double g_sigma_r, g_sigma_v, g_base_quality;
    double max_datalink_range, datalink_packet_loss;

    /* --- modes (SURVEY 8f rank 2) --- */
    int32_t obs_mode;        /* HLYNR_OBS_* */
    int32_t precision_mode;  /* curriculum.precision_mode, environment.py:121 */
    int32_t fuze_enabled;    /* proximity_fuze_enabled :128 */
    int32_t volley_size;     /* 0 = volley_mode off; 1..HLYNR_MAX_VOLLEY = volley_mode with that many missiles (:42-43) */
    double kill_radius;      /* proximity_kill_radius :129 */
} HlynrParams;

/*
 * Host-pushed curriculum scalars (global to all envs): environment.py:223-234, 274-351.
 * Recomputed on the host from training_step_count and pushed with hlynr_set_curriculum.
 */
typedef struct HlynrCurriculum {
    double intercept_radius; /* get_current_intercept_radius() */
    double beam_width_deg;   /* observation_generator.radar_beam_width */
    double onboard_reliability;
    double ground_reliability;
} HlynrCurriculum;

/*
 * The whole curriculum schedule (config.Curriculum): what get_current_intercept_radius and _update_radar_curriculum
 * (environment.py:223-234, 274-351) compute from training_step_count, for hlynr_attach_curriculum.  Steps are doubles because
 * YAML may give them as floats.  A ramp is Curriculum._ramp: `initial` below `start`, `final` from `end` on, linear between.
 * With radar_enabled == 0 the three radar values are the constant `*_initial` ones.
 */
typedef struct HlynrCurriculumSchedule {
    int32_t enabled;          /* curriculum.enabled; 0 = the radius is final_radius at every count */
    int32_t radar_enabled;    /* curriculum.radar_curriculum present, non-empty and enabled */
    double initial_radius, final_radius, curriculum_steps;
    double beam_initial, beam_final, beam_start, beam_end;                 /* degrees */
    double onboard_initial, onboard_final, onboard_start, onboard_end;     /* detection reliability */
    double ground_initial, ground_final, ground_start, ground_end;         /* ground reliability */
} HlynrCurriculumSchedule;

/*
 * Optional per-env info, structure-of-arrays, device pointers (any may be NULL).
 * Field meaning = the reference's info dict, environment.py:829-857.  Values are those of the
 * tick just executed (i.e. of the terminal tick for envs that were auto-reset in this call).
 */
typedef struct HlynrInfoSoA {
    float* distance;          /* [N] info['distance'] */
    float* min_distance;      /* [N] info['min_distance'] */
    float* fuel_remaining;    /* [N] info['fuel_remaining'] */
    float* fuel_used;         /* [N] info['fuel_used'] */
    int32_t* steps;           /* [N] info['steps'] */
    uint8_t* flags;           /* [N] bit0 intercepted, bit1 missile_hit_target, bit2 clamped,
                                 bit3 radar_detected (delayed onboard flag), bit4 ground detected,
                                 bit5 crossed_threshold, bit6 proximity_fuze_triggered,
                                 bit7 kalman initialised */
    float* interceptor_pos;   /* [N,3] info['interceptor_pos'] */
    float* missile_pos;       /* [N,3] info['missile_pos'] */
    float* episode_return;    /* [N] Monitor 'r' of the episode that ended in this call (else running sum) */
    int32_t* episode_length;  /* [N] Monitor 'l' */
    int32_t* missiles_intercepted;  /* [N] info['missiles_intercepted'] (volley: len(intercepted indices); else 0/1) */
    int32_t* missiles_remaining;    /* [N] info['missiles_remaining'] */
    float* missile_min_distances;   /* [N, HLYNR_MAX_VOLLEY] info['missile_min_distances'] (unused slots 0; single mode: [distance]) */
    float* radar_quality;           /* [N] info['radar_quality'] (environment.py:840): the configured quality, 0.0 while the onboard
                                       SensorDelayBuffer is still filling ('sensor_delay_initialization', core.py:579-584) */
} HlynrInfoSoA;

#define HLYNR_INFO_INTERCEPTED 0x01
#define HLYNR_INFO_HIT_TARGET 0x02
#define HLYNR_INFO_CLAMPED 0x04
#define HLYNR_INFO_RADAR_DETECTED 0x08
#define HLYNR_INFO_GROUND_DETECTED 0x10
#define HLYNR_INFO_CROSSED 0x20
#define HLYNR_INFO_FUZE 0x40
#define HLYNR_INFO_KF_INIT 0x80

/*
 * One finished episode (done = terminated | truncated), appended by hlynr_step to an optional compact list so that
 * a VecEnv with many envs fetches `count` small records instead of [N]-sized info / terminal-observation arrays.
 * Fields = the reference's info dict on the terminal tick (environment.py:829-857) + what SB3 adds on done
 * (info['terminal_observation'], info['TimeLimit.truncated'], Monitor's info['episode']).  The order of the
 * records within one call is unspecified (sort by `env` if needed).
 */
typedef struct HlynrDoneRecord {
    int32_t env;             /* local env index */
    int32_t steps;           /* info['steps'] == Monitor 'l' */
    uint32_t flags;          /* HLYNR_INFO_* bits | HLYNR_DONE_TERMINATED | HLYNR_DONE_TRUNCATED */
    float distance, min_distance, fuel_remaining, fuel_used;
    float episode_return;    /* Monitor 'r' */
    float interceptor_pos[3], missile_pos[3];
    float terminal_obs[HLYNR_OBS_DIM];
    int32_t missiles_intercepted, missiles_remaining;      /* info['missiles_intercepted'], ['missiles_remaining'] */
    float missile_min_distances[HLYNR_MAX_VOLLEY];         /* info['missile_min_distances'] (single mode: [distance]) */
} HlynrDoneRecord;           /* 50 words = 200 bytes */
#define HLYNR_DONE_TERMINATED 0x100u
#define HLYNR_DONE_TRUNCATED 0x200u
#define HLYNR_DONE_ONBOARD_FILL 0x400u /* the onboard delay buffer was still filling on the terminal tick: info['radar_quality'] = 0.0 */

/* Episode statistics accumulated on the device since the last reset of the block (per handle). */
typedef struct HlynrStats {
    double episodes;          /* finished episodes (terminated or truncated) */
    double successes;         /* info['intercepted'] on the final tick */
    double return_sum;
    double length_sum;
    double min_distance_sum;
    double final_distance_sum;
    double hit_target;        /* termination causes (first matching, in the reference's reward order) */
    double interceptor_crash;
    double fuel_out;
    double missile_ground;    /* missile z<=0 away from the target */
    double worsening;         /* smart early termination, environment.py:795-811 */
    double timeouts;          /* truncated and not terminated */
    double env_steps;         /* ticks simulated */
    double onboard_locks;     /* ticks with the (delayed) onboard flag set */
    double reserved[2];
} HlynrStats;
#define HLYNR_STATS_WORDS 16

/*
 * Full mutable state of one env, for oracle interchange (SURVEY Appendix B.4).  Always double /
 * int32 regardless of the precision of the handle.
 */
typedef struct HlynrEnvState {
    double ipos[3], ivel[3], quat[4], fuel, fuel_used;
    double mpos[3], mvel[3];
    double wind[3], thrust[3];
    double prev_d, last_d, min_d, episode_return;
    double kf_x[6], kf_P[4]; /* P as (pp, pv, vp, vv) of the per-axis 2x2 block */
    double T0, base_cd, peak;
    double vpos[HLYNR_MAX_VOLLEY * 3], vvel[HLYNR_MAX_VOLLEY * 3], vmin[HLYNR_MAX_VOLLEY]; /* volley: missile_states[], min distances */
    int32_t steps, worsen_count, crossed, kf_init, onboard_delay, episode;
    int32_t vactive[HLYNR_MAX_VOLLEY], vcur, vcount; /* volley: active flags, index of self.missile_state, interceptions */
    int32_t kf_f64;   /* dtype of the reference's Kalman state array: 0 = float32, 1 = float64 (core.py:108 rebinds it at the first
                         float64 measurement); tracked by the fp64 build, always 0 in the fp32 build */
    int32_t reserved;
} HlynrEnvState;

typedef struct hlynr_sim hlynr_t;

/* Error text of the last failing call on this thread. */
const char* hlynr_last_error(void);
int hlynr_abi_version(void);
size_t hlynr_params_size(void);
size_t hlynr_env_state_size(void);
size_t hlynr_curriculum_schedule_size(void);

/* Replaces N x InterceptEnvironment(config) (environment.py:20).  `precision` is HLYNR_FP32 or
 * HLYNR_FP64.  Envs get global ids [env_id_offset, env_id_offset + n_envs): trajectories depend
 * only on (seed, global id), never on how envs are sharded over GPUs. */
int hlynr_create(const HlynrParams* params, int64_t n_envs, int device, uint64_t seed,
                 int64_t env_id_offset, int precision, hlynr_t** out);
void hlynr_destroy(hlynr_t* sim);

int hlynr_num_envs(const hlynr_t* sim, int64_t* out);
int hlynr_set_curriculum(hlynr_t* sim, const HlynrCurriculum* cur);
int hlynr_get_curriculum(const hlynr_t* sim, HlynrCurriculum* out);

/* Device-side training-step counter (SB3's model.num_timesteps, which the reference's callback pushes with
 * env_method('set_training_step_count') after every env step, train_flat_ppo.py:173-177).  While a schedule is attached, every
 * hlynr_step first runs a one-thread kernel that computes the curriculum of the current count into a device slot the step kernel
 * reads, then advances the count by `increment`; hlynr_reset computes the slot without advancing.  So the step at tick t after
 * attaching sees t0 + t*increment, as in SB3, where the callback runs after the step -- and a CUDA graph of steps continues the
 * schedule on every replay instead of repeating the curriculum of its capture.
 *   increment  what one tick adds: the number of envs of the whole run (the shard's n, or the global count of a multi-GPU run).
 * Refuses non-finite fields, curriculum_steps <= 0 while enabled and increment < 0.  While attached, hlynr_set_curriculum,
 * hlynr_step_host and hlynr_rollout fail: the host path is driven by the host-side callback, and the fused k-tick rollout would
 * need one slot per fused tick.  The device block lives until hlynr_destroy, so a captured graph never points at freed memory;
 * the schedule, the increment and whether one is attached at all are baked into captured launches (re-capture after changing them). */
int hlynr_attach_curriculum(hlynr_t* sim, const HlynrCurriculumSchedule* schedule, uint64_t num_timesteps, int64_t increment);
/* Back to the by-value curriculum of hlynr_set_curriculum (unchanged since it was last set). */
int hlynr_detach_curriculum(hlynr_t* sim);
/* Sets the count, ordered on `stream` (a one-thread kernel: graph-capturable).  Fails unless a schedule is attached. */
int hlynr_set_timesteps(hlynr_t* sim, uint64_t num_timesteps, void* stream);
/* Synchronises `stream` and returns the count.  Fails unless a schedule is attached. */
int hlynr_get_timesteps(hlynr_t* sim, uint64_t* out, void* stream);
/* Test hook: the curriculum values the device computes from the attached schedule at `count`, widened to double without rounding:
 * out[0] intercept radius (in the handle's precision), out[1] cosine of the half beam width (float; -2 for a beam of 360 degrees
 * or more), out[2] onboard reliability (float), out[3] ground reliability (float).  Synchronous. */
int hlynr_debug_curriculum_at(hlynr_t* sim, uint64_t count, double out[4]);
/* Re-keys the counter-based RNG (reference: reset(seed=...), environment.py:357-359). */
int hlynr_seed(hlynr_t* sim, uint64_t seed);

/* reset(): environment.py:353.  mask_dev: NULL = all envs, else uint8[N], non-zero = reset.
 * obs_dev float[N,26] receives the initial observation of the envs that were reset (others
 * untouched). */
int hlynr_reset(hlynr_t* sim, const uint8_t* mask_dev, float* obs_dev, void* stream);

/* step(): environment.py:605 + SB3 auto-reset.  One 10 ms tick of every env.
 *   actions_dev      float[N,6] (caller clips to [-1,1] as SB3 does)
 *   obs_dev          float[N,26]: observation after the tick; for envs that finished, the
 *                    observation of the NEW episode (SB3 DummyVecEnv semantics)
 *   reward_dev       float[N]
 *   terminated_dev   uint8[N], truncated_dev uint8[N]   (done = terminated | truncated)
 *   terminal_obs_dev float[N,26] or NULL: last observation of finished episodes
 *                    (info['terminal_observation']); rows of unfinished envs are untouched
 *   info             NULL or a struct of optional device arrays
 *   auto_reset       non-zero: finished envs are reset inside the kernel */
int hlynr_step(hlynr_t* sim, const float* actions_dev, float* obs_dev, float* reward_dev,
               uint8_t* terminated_dev, uint8_t* truncated_dev, float* terminal_obs_dev,
               const HlynrInfoSoA* info, int auto_reset, void* stream);

/* Attaches (records_dev != NULL) or detaches the compact done list used by subsequent hlynr_step calls:
 * records_dev HlynrDoneRecord[capacity], counter_dev int32 (appended count; the CALLER zeroes it, it may end above
 * `capacity`, in which case the excess records were dropped). */
int hlynr_set_done_list(hlynr_t* sim, HlynrDoneRecord* records_dev, int32_t* counter_dev, int32_t capacity);

/* k fused ticks in ONE launch with the state held in registers between ticks.
 *   actions_dev  float[k,N,6] or NULL = in-kernel random actions U(-1,1)^6 from the Philox
 *                stream (synthetic random-policy rollouts)
 *   obs_dev      float[N,obs_dim] (option "obs_dim", 26 by default): observation after the last tick (or NULL)
 *   reward_sum_dev float[N] or NULL: sum of the k rewards;  done_count_dev int32[N] or NULL */
int hlynr_rollout(hlynr_t* sim, int k_steps, const float* actions_dev, float* obs_dev,
                  float* reward_sum_dev, int32_t* done_count_dev, void* stream);

/* Host-buffer variants (what a numpy VecEnv calls): copy in, run, copy out, synchronise.
 * Pinned staging buffers are owned by the handle. */
int hlynr_reset_host(hlynr_t* sim, const uint8_t* mask_host, float* obs_host);
int hlynr_step_host(hlynr_t* sim, const float* actions_host, float* obs_host, float* reward_host,
                    uint8_t* terminated_host, uint8_t* truncated_host, float* terminal_obs_host,
                    int auto_reset);
/* Finished episodes of the last hlynr_step_host call: pointer to `*count` records in pinned host memory owned by
 * the handle.  Two buffers alternate, so the records of a call stay valid during the next hlynr_step_host call and are
 * overwritten by the one after it (SB3 loops hold `infos` of step k while step k+1 runs). */
int hlynr_done_records_host(hlynr_t* sim, const HlynrDoneRecord** records, int32_t* count);
/* Pinned host buffers owned by the handle: float[N,6], float[N,26], float[N], uint8[N], uint8[N].  Passing
 * these very pointers -- or ANY page-locked caller buffer (cudaMallocHost / cudaHostRegister / a torch pin_memory()
 * tensor; detected with cudaPointerGetAttributes) -- to hlynr_step_host skips the staging memcpy: the copy engine
 * and the kernel read and write the caller's memory directly.  Callers that alternate two page-locked output sets get
 * the SB3 loop's "the arrays of step k are still read while step k+1 runs" for free. */
int hlynr_pinned_buffers(hlynr_t* sim, float** actions, float** obs, float** reward, uint8_t** terminated,
                         uint8_t** truncated);
/* SB3 `dones` of the last hlynr_step_host call: uint8[N] = terminated | truncated (environment.py:813-816 combined the way
 * DummyVecEnv.step_wait does), in pinned host memory owned by the handle; the step kernel writes it directly, so the
 * caller does not need a pass over both flag arrays.  Overwritten by the next call. */
int hlynr_pinned_done(hlynr_t* sim, uint8_t** done);
/* Redirects `dones` to a caller-owned PAGE-LOCKED buffer uint8[N] (NULL = back to the handle's own); fails for pageable
 * memory, because the kernel stores into it directly. */
int hlynr_host_done_buffer(hlynr_t* sim, uint8_t* done_pinned);
/* Copies the info arrays of the last hlynr_step_host call to host (each pointer optional, host). */
int hlynr_info_host(hlynr_t* sim, HlynrInfoSoA* host_arrays);

/* Episode statistics block: device pointer (HLYNR_STATS_WORDS doubles, for an in-place NCCL
 * all-reduce), host read-back, and zeroing. */
int hlynr_stats_device_ptr(hlynr_t* sim, double** out_dev);
/* Folds the per-block partial sums into the block hlynr_stats_device_ptr points at (stream-ordered). */
int hlynr_stats_reduce(hlynr_t* sim, void* stream);
int hlynr_get_stats(hlynr_t* sim, HlynrStats* host_out, int zero_after, void* stream);

/* Oracle interchange: copy `count` envs starting at local index `first`. */
int hlynr_export_state(hlynr_t* sim, int64_t first, int64_t count, HlynrEnvState* host_out);
int hlynr_import_state(hlynr_t* sim, int64_t first, int64_t count, const HlynrEnvState* host_in);

/* Test hook: raw Philox4x32-10 block and the derived draws for (env, episode, step, block). */
int hlynr_debug_draws(hlynr_t* sim, int64_t env_global_id, uint32_t episode, uint32_t step,
                      uint32_t block, uint32_t raw_out[4], float uniform_out[4], float normal_out[4]);

/* Options.  "specialise": 1 (default) = use the compile-time feature-specialised step kernels when the configuration matches
 * one (medium scenario with physics v2.0 all on / all off), 0 = always the generic kernel.
 * "host_info": 1 (default) = hlynr_step_host also fills the [N]-sized info arrays read by hlynr_info_host, 0 = skip them
 * (finished episodes are still reported through hlynr_done_records_host).
 * "host_chunks": number of chunks hlynr_step_host pipelines (H2D | kernel | D2H on separate streams), 0 = auto.
 * "pdl": 1 (default) = step kernels are launched with programmatic stream serialization (cudaLaunchAttributeProgrammaticStreamSerialization):
 * a tick's grid is scheduled while the previous kernel of the stream drains and waits (griddepcontrol.wait) for its completion
 * before touching memory, which hides the launch latency between back-to-back ticks; 0 = ordinary launches.
 * "host_chunk_growth": g > 0 (default 12) = a 16384-env first chunk, then every chunk g/8 times the previous one (12 = x1.5,
 * 16 = doubling) up to 196608 envs, for shards of >= 131072 envs when "host_chunks" is 0; 0 = uniform chunks.
 * "host_threads": threads used for staging memcpys of unpinned caller buffers, 0 = auto.
 * "obs_dim": 26 (default) or 17.  With 17 every observation array of this API (obs_dev / obs_host / terminal_obs_*) is float[N,17]:
 * the leading "17-D radar" channels obs[0:17] of the reference's vector (rl_system/hrl/observation_schema.py:13-46 MIN_DIMENSION,
 * the layout of the pre-ground-radar models, rl_system/config_17d_compat.yaml); the ground-radar channels 17-25 are not written and
 * the host path downloads 36 B per env less.  HlynrDoneRecord.terminal_obs always holds all 26 channels.
 * "prefetch_waves": the step kernel prefetches into L2 the state planes of the CTA this many CTAs-per-SM further on
 * (default 1, measured best on B200; 0 = off). */
int hlynr_set_option(hlynr_t* sim, const char* name, int64_t value);

/* CUDA-graph support.  Every launch of this library goes to the caller's stream, so a sequence of hlynr_* calls can be
 * stream-captured (e.g. torch.cuda.graph) once allocations have happened in a warm-up call.  The ring-row indices of a
 * tick are kernel arguments computed from the handle's tick counter, so a captured sequence of T ticks replays correctly
 * iff T is a multiple of hlynr_ring_period(); after each replay the host-side counters are advanced with
 * hlynr_note_replayed_ticks(sim, T) (negative values undo the bookkeeping of calls that were only recorded, not executed).
 * By-value curriculum scalars and the seed are baked into the captured arguments; an attached schedule's count lives on the
 * device and advances on every replay (hlynr_attach_curriculum). */
int hlynr_ring_period(const hlynr_t* sim, int* out);   /* lcm(onboard ring length, ground ring length), >= 1 */
int hlynr_note_replayed_ticks(hlynr_t* sim, int64_t ticks, int64_t launches);
/* Ticks executed (or accounted for by hlynr_note_replayed_ticks) since hlynr_create: a captured sequence may only be replayed
 * when this is congruent, modulo hlynr_ring_period(), to its value when the capture started. */
int hlynr_tick_count(const hlynr_t* sim, int64_t* out);

/* Number of kernel launches issued by this handle so far (bench.py's gpu_launches). */
int hlynr_launch_count(const hlynr_t* sim, int64_t* out);

/*
 * Snapshots: checkpoint and resume a run bit for bit.  A snapshot is a descriptor (HlynrSnapshotInfo, host) plus one device
 * image in a CANONICAL layout that does not depend on the handle's plane layout (compact or wide), on the tick phase of the delay
 * rings or on the ring-row convention, so a checkpoint stays readable when the internal layout changes.  The image holds, each
 * section starting at section_offset[] (256-byte aligned):
 *   HLYNR_SNAP_REAL       R[HLYNR_SNAP_REAL_COLS + 7 K][n_envs], R = the handle's precision: per env, in this order, ipos[3], fuel,
 *                         ivel[3], fuel_used, mpos[3], prev_d, mvel[3], last_d, kf_x[0:3], min_d, kf_x[3:6], episode_return,
 *                         thrust[3], T0, quat[4], wind[3], kf_P pp, kf_P pv, vp, vv, base_cd, peak; then per volley missile m < K
 *                         vpos[3], vmin, vvel[3]
 *   HLYNR_SNAP_INT        int32[HLYNR_SNAP_INT_COLS + K][n_envs]: steps, worsen_count, episode, crossed, kf_init, kf_f64,
 *                         onboard_delay, vcur, vcount; then vactive[m] per volley missile
 *   HLYNR_SNAP_ONBOARD    R[onboard_ring_len][4][n_envs]: onboard delay ring in AGE order, row j = the sample written j ticks
 *                         before the snapshot (relative position xyz, detected)
 *   HLYNR_SNAP_GROUND     R[ground_ring_len][8][n_envs]: ground delay ring in age order (relative position xyz, quality,
 *                         relative velocity xyz, detection flag)
 *   HLYNR_SNAP_STATS      double[HLYNR_STAT_SLOTS + 1][HLYNR_STATS_WORDS]: the statistics block, raw (hlynr_get_stats after a load
 *                         returns the same bits)
 *   HLYNR_SNAP_CURRICULUM uint64: the attached schedule's training-step count (0 when none is attached)
 * Options ("pdl", "specialise", "prefetch_waves", ...) and the attached done list are not part of a snapshot: they do not change
 * results, and the done list belongs to the caller.  A CUDA graph captured before a load bakes in the host counters of its
 * capture: re-capture after loading.
 */
#define HLYNR_SNAPSHOT_VERSION 1
#define HLYNR_SNAP_REAL_COLS 41
#define HLYNR_SNAP_INT_COLS 9
#define HLYNR_STAT_ROWS 65   /* per-block slots + the reduced row */
enum { HLYNR_SNAP_REAL = 0, HLYNR_SNAP_INT = 1, HLYNR_SNAP_ONBOARD = 2, HLYNR_SNAP_GROUND = 3, HLYNR_SNAP_STATS = 4,
       HLYNR_SNAP_CURRICULUM = 5, HLYNR_SNAP_SECTIONS = 6 };

typedef struct HlynrSnapshotInfo {
    int32_t format_version;       /* HLYNR_SNAPSHOT_VERSION */
    int32_t abi_version;          /* HLYNR_ABI_VERSION */
    int32_t precision;            /* HLYNR_FP32 / HLYNR_FP64 */
    int32_t obs_dim;              /* option "obs_dim" */
    int64_t n_envs, env_id_offset;
    uint64_t seed;
    int32_t volley_k;             /* params.volley_size */
    int32_t onboard_ring_len, ground_ring_len;   /* rows of the delay rings (0 = no ring) */
    int32_t curriculum_attached;  /* a schedule was attached (hlynr_attach_curriculum) */
    uint64_t tick;                /* hlynr_tick_count */
    double env_steps;             /* ticks x envs since the statistics were last zeroed (word 12 of hlynr_get_stats) */
    int64_t curriculum_increment; /* of the attached schedule */
    HlynrParams params;
    HlynrCurriculum curriculum;          /* the host-pushed curriculum (hlynr_set_curriculum) */
    HlynrCurriculumSchedule schedule;    /* valid when curriculum_attached */
    uint64_t section_offset[HLYNR_SNAP_SECTIONS];   /* byte offset of each section of the device image */
    uint64_t device_bytes;                          /* size of the device image */
} HlynrSnapshotInfo;

size_t hlynr_snapshot_info_size(void);
/* Fills the descriptor of the handle's current state (format, shape, offsets) and the size of the device image. */
int hlynr_snapshot_layout(const hlynr_t* sim, HlynrSnapshotInfo* info, size_t* device_bytes);
/* Writes the device image to dev_out (device_bytes of hlynr_snapshot_layout) and fills `info`; ordered on `stream`, no host
 * synchronisation.  The host counters in `info` are those of the work enqueued so far.  Refused while `stream` is capturing. */
int hlynr_snapshot_save(hlynr_t* sim, void* dev_out, HlynrSnapshotInfo* info, void* stream);
/* Restores a snapshot into a handle created with the same params, precision, n_envs, env_id_offset, obs_dim: the state of every
 * env, the delay rings, the statistics block, the tick and env_steps counters, the seed, the host-pushed curriculum, and the
 * curriculum schedule (re-attached with its count and increment, or detached, as it was).  Refuses, naming the first mismatch, a
 * descriptor of another format version, precision, shape or configuration, and refuses while `stream` is capturing.  Ordered on
 * `stream`; dev_in may be reused once the stream has passed the load.  A compact-layout snapshot loads into a wide-layout handle
 * and the reverse. */
int hlynr_snapshot_load(hlynr_t* sim, const HlynrSnapshotInfo* info, const void* dev_in, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HLYNR_H */

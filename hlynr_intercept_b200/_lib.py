"""Loader of the C-ABI CUDA library (ctypes).  There is NO CPU fallback: if the library is missing or does
not load, importing the simulator fails loudly."""
import ctypes as C
import os

from . import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
# HLYNR_B200_LIB points the loader at another build of the SAME library (kernel experiments, tools/); there is no other backend
SO_PATH = os.environ.get("HLYNR_B200_LIB") or os.path.join(_HERE, "libhlynr_b200.so")
_LIB = None

# every symbol include/hlynr.h declares
EXPORTS = [
    "hlynr_last_error", "hlynr_abi_version", "hlynr_params_size", "hlynr_env_state_size", "hlynr_create",
    "hlynr_destroy", "hlynr_num_envs", "hlynr_set_curriculum", "hlynr_get_curriculum", "hlynr_seed", "hlynr_reset",
    "hlynr_step", "hlynr_rollout", "hlynr_reset_host", "hlynr_step_host", "hlynr_pinned_buffers", "hlynr_info_host",
    "hlynr_stats_device_ptr", "hlynr_stats_reduce", "hlynr_get_stats", "hlynr_export_state", "hlynr_import_state",
    "hlynr_debug_draws", "hlynr_launch_count", "hlynr_set_option", "hlynr_set_done_list", "hlynr_done_records_host",
    "hlynr_ring_period", "hlynr_note_replayed_ticks", "hlynr_tick_count", "hlynr_pinned_done", "hlynr_host_done_buffer",
    "hlynr_curriculum_schedule_size", "hlynr_attach_curriculum", "hlynr_detach_curriculum", "hlynr_set_timesteps", "hlynr_get_timesteps",
    "hlynr_debug_curriculum_at", "hlynr_snapshot_info_size", "hlynr_snapshot_layout", "hlynr_snapshot_save", "hlynr_snapshot_load",
    # include/hlynr_post.h
    "hlynr_post_create", "hlynr_post_create_frames", "hlynr_post_destroy", "hlynr_post_obs_dim", "hlynr_post_obs_target", "hlynr_post_reset",
    "hlynr_post_step", "hlynr_post_original", "hlynr_post_normalize", "hlynr_post_get_stats", "hlynr_post_set_stats",
    "hlynr_post_check_sums", "hlynr_post_launch_count", "hlynr_post_note_replayed_steps", "hlynr_post_snapshot_info_size",
    "hlynr_post_snapshot_layout", "hlynr_post_snapshot_save", "hlynr_post_snapshot_load",
    # include/hlynr_rollout.h
    "hlynr_bootstrap_timeouts", "hlynr_gae", "hlynr_eval_record", "hlynr_trace_row_size", "hlynr_eval_trace",
    # include/hlynr_policy.h
    "hlynr_policy_create", "hlynr_policy_create_dim", "hlynr_policy_destroy", "hlynr_policy_set_weights", "hlynr_policy_forward", "hlynr_policy_forward_dev",
    "hlynr_policy_set_counter", "hlynr_policy_get_counter", "hlynr_policy_launch_count", "hlynr_policy_set_option", "hlynr_policy_get_timing",
]


class HlynrError(RuntimeError):
    pass


def load(build_if_missing=True):
    """Returns the ctypes handle of libhlynr_b200.so, building it in-tree with nvcc if it is stale/missing."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if build_if_missing and "HLYNR_B200_LIB" not in os.environ:
        from . import build as _build

        try:
            _build.build()
        except RuntimeError as e:   # nvcc ran and rejected the sources: never fall back to a stale library silently
            raise HlynrError(f"libhlynr_b200.so is stale and its sources do not compile: {e}") from e
        except Exception as e:  # no nvcc on this box: fall through to the prebuilt library, if any
            if not os.path.exists(SO_PATH):
                raise HlynrError(f"libhlynr_b200.so is missing and could not be built: {e}") from e
    if not os.path.exists(SO_PATH):
        raise HlynrError("libhlynr_b200.so is missing; run `python -m hlynr_intercept_b200.build`")
    L = C.CDLL(SO_PATH)
    vp, i64, u64, i32, u32 = C.c_void_p, C.c_int64, C.c_uint64, C.c_int, C.c_uint32
    L.hlynr_last_error.restype = C.c_char_p
    L.hlynr_params_size.restype = C.c_size_t
    L.hlynr_env_state_size.restype = C.c_size_t
    L.hlynr_curriculum_schedule_size.restype = C.c_size_t
    L.hlynr_create.argtypes = [C.POINTER(abi.HlynrParams), i64, i32, u64, i64, i32, C.POINTER(vp)]
    L.hlynr_destroy.argtypes = [vp]
    L.hlynr_destroy.restype = None
    L.hlynr_num_envs.argtypes = [vp, C.POINTER(i64)]
    L.hlynr_set_curriculum.argtypes = [vp, C.POINTER(abi.HlynrCurriculum)]
    L.hlynr_get_curriculum.argtypes = [vp, C.POINTER(abi.HlynrCurriculum)]
    L.hlynr_attach_curriculum.argtypes = [vp, C.POINTER(abi.HlynrCurriculumSchedule), u64, i64]
    L.hlynr_detach_curriculum.argtypes = [vp]
    L.hlynr_set_timesteps.argtypes = [vp, u64, vp]
    L.hlynr_get_timesteps.argtypes = [vp, C.POINTER(u64), vp]
    L.hlynr_debug_curriculum_at.argtypes = [vp, u64, C.POINTER(C.c_double)]
    L.hlynr_snapshot_info_size.restype = C.c_size_t
    L.hlynr_snapshot_layout.argtypes = [vp, C.POINTER(abi.HlynrSnapshotInfo), C.POINTER(C.c_size_t)]
    L.hlynr_snapshot_save.argtypes = [vp, vp, C.POINTER(abi.HlynrSnapshotInfo), vp]
    L.hlynr_snapshot_load.argtypes = [vp, C.POINTER(abi.HlynrSnapshotInfo), vp, vp]
    L.hlynr_post_snapshot_info_size.restype = C.c_size_t
    L.hlynr_post_snapshot_layout.argtypes = [vp, C.POINTER(abi.HlynrPostSnapshotInfo), C.POINTER(C.c_size_t)]
    L.hlynr_post_snapshot_save.argtypes = [vp, vp, C.POINTER(abi.HlynrPostSnapshotInfo), vp]
    L.hlynr_post_snapshot_load.argtypes = [vp, C.POINTER(abi.HlynrPostSnapshotInfo), vp, vp]
    L.hlynr_seed.argtypes = [vp, u64]
    L.hlynr_reset.argtypes = [vp, vp, vp, vp]
    L.hlynr_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, C.POINTER(abi.HlynrInfoSoA), i32, vp]
    L.hlynr_rollout.argtypes = [vp, i32, vp, vp, vp, vp, vp]
    L.hlynr_reset_host.argtypes = [vp, vp, vp]
    L.hlynr_step_host.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32]
    L.hlynr_pinned_buffers.argtypes = [vp] + [C.POINTER(vp)] * 5
    L.hlynr_pinned_done.argtypes = [vp, C.POINTER(vp)]
    L.hlynr_host_done_buffer.argtypes = [vp, vp]
    L.hlynr_info_host.argtypes = [vp, C.POINTER(abi.HlynrInfoSoA)]
    L.hlynr_stats_device_ptr.argtypes = [vp, C.POINTER(vp)]
    L.hlynr_stats_reduce.argtypes = [vp, vp]
    L.hlynr_get_stats.argtypes = [vp, C.POINTER(abi.HlynrStats), i32, vp]
    L.hlynr_export_state.argtypes = [vp, i64, i64, vp]
    L.hlynr_import_state.argtypes = [vp, i64, i64, vp]
    L.hlynr_debug_draws.argtypes = [vp, i64, u32, u32, u32, vp, vp, vp]
    L.hlynr_launch_count.argtypes = [vp, C.POINTER(i64)]
    L.hlynr_set_option.argtypes = [vp, C.c_char_p, i64]
    L.hlynr_set_done_list.argtypes = [vp, vp, vp, C.c_int32]
    L.hlynr_done_records_host.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_int32)]
    dbl, pd = C.c_double, C.POINTER(C.c_double)
    L.hlynr_post_create.argtypes = [i64, i32, i32, dbl, dbl, dbl, C.POINTER(vp)]
    L.hlynr_post_create_frames.argtypes = [i64, i32, i32, i32, dbl, dbl, dbl, C.POINTER(vp)]
    L.hlynr_post_destroy.argtypes = [vp]
    L.hlynr_post_destroy.restype = None
    L.hlynr_post_obs_dim.argtypes = [vp, C.POINTER(i32)]
    L.hlynr_post_obs_target.argtypes = [vp, C.POINTER(vp)]
    L.hlynr_post_reset.argtypes = [vp, vp, i32, vp]
    L.hlynr_post_step.argtypes = [vp, vp, vp, vp, vp, vp, C.c_int32, vp, vp, i32, vp]
    L.hlynr_post_original.argtypes = [vp, vp, vp]
    L.hlynr_post_normalize.argtypes = [vp, vp, i64, vp, vp]
    L.hlynr_post_get_stats.argtypes = [vp, vp, vp, pd, pd, pd, pd, vp]
    L.hlynr_post_set_stats.argtypes = [vp, vp, vp, dbl, dbl, dbl, dbl, vp]
    L.hlynr_post_check_sums.argtypes = [vp, i32, pd, vp]
    L.hlynr_post_launch_count.argtypes = [vp, C.POINTER(i64)]
    L.hlynr_post_note_replayed_steps.argtypes = [vp, i64, i64]
    L.hlynr_ring_period.argtypes = [vp, C.POINTER(i32)]
    L.hlynr_note_replayed_ticks.argtypes = [vp, i64, i64]
    L.hlynr_tick_count.argtypes = [vp, C.POINTER(i64)]
    L.hlynr_bootstrap_timeouts.argtypes = [vp, vp, vp, C.c_int32, vp, C.c_double, vp, i32, vp]
    L.hlynr_gae.argtypes = [vp, vp, vp, vp, vp, i64, i64, C.c_double, C.c_double, vp, vp, i32, vp]
    L.hlynr_eval_record.argtypes = [vp, vp, i64, i64, vp, vp, vp, vp, vp, i32, vp]
    L.hlynr_trace_row_size.restype = C.c_size_t
    L.hlynr_eval_trace.argtypes = [C.POINTER(abi.HlynrInfoSoA), vp, vp, vp, vp, vp, i64, i64, C.c_int32, vp, i32, vp]
    L.hlynr_policy_create.argtypes = [i32, C.POINTER(vp)]
    L.hlynr_policy_create_dim.argtypes = [i32, i32, C.POINTER(vp)]
    L.hlynr_policy_destroy.argtypes = [vp]
    L.hlynr_policy_destroy.restype = None
    L.hlynr_policy_set_weights.argtypes = [vp, C.POINTER(abi.HlynrPolicyWeights), vp]
    L.hlynr_policy_forward.argtypes = [vp, vp, i64, vp, vp, vp, vp, vp, vp, u64, u64, i32, vp]
    L.hlynr_policy_forward_dev.argtypes = [vp, vp, i64, vp, vp, vp, vp, vp, vp, u64, i32, vp]
    L.hlynr_policy_set_counter.argtypes = [vp, u64, vp]
    L.hlynr_policy_get_counter.argtypes = [vp, C.POINTER(u64), vp]
    L.hlynr_policy_launch_count.argtypes = [vp, C.POINTER(i64)]
    L.hlynr_policy_set_option.argtypes = [vp, C.c_char_p, i64]
    L.hlynr_policy_get_timing.argtypes = [vp, vp]
    if L.hlynr_abi_version() != abi.ABI_VERSION:
        raise HlynrError("ABI version mismatch between libhlynr_b200.so and hlynr_intercept_b200.abi")
    if L.hlynr_params_size() != C.sizeof(abi.HlynrParams):
        raise HlynrError(f"HlynrParams layout mismatch: C {L.hlynr_params_size()} vs ctypes {C.sizeof(abi.HlynrParams)}")
    if L.hlynr_env_state_size() != C.sizeof(abi.HlynrEnvState):
        raise HlynrError("HlynrEnvState layout mismatch")
    if L.hlynr_curriculum_schedule_size() != C.sizeof(abi.HlynrCurriculumSchedule):
        raise HlynrError(f"HlynrCurriculumSchedule layout mismatch: C {L.hlynr_curriculum_schedule_size()} vs ctypes "
                         f"{C.sizeof(abi.HlynrCurriculumSchedule)}")
    for name, cls in (("hlynr_snapshot_info_size", abi.HlynrSnapshotInfo), ("hlynr_post_snapshot_info_size", abi.HlynrPostSnapshotInfo)):
        if getattr(L, name)() != C.sizeof(cls):
            raise HlynrError(f"{cls.__name__} layout mismatch: C {getattr(L, name)()} vs ctypes {C.sizeof(cls)}")
    if L.hlynr_trace_row_size() != abi.trace_row_numpy_dtype().itemsize:
        raise HlynrError(f"HlynrTraceRow layout mismatch: C {L.hlynr_trace_row_size()} vs numpy {abi.trace_row_numpy_dtype().itemsize}")
    _LIB = L
    return L


def check(rc):
    if rc != 0:
        raise HlynrError(load().hlynr_last_error().decode("utf-8", "replace"))

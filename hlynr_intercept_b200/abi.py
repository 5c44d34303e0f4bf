"""ctypes mirror of include/hlynr.h (the C ABI).  Field order and types must match the header exactly;
`hlynr_params_size()` / `hlynr_env_state_size()` / `hlynr_snapshot_info_size()` are checked at load time."""
import ctypes as C

ABI_VERSION = 1
OBS_DIM = 26
ACT_DIM = 6
N_DR = 13
MAX_VOLLEY = 8
STATS_WORDS = 16
FP32, FP64 = 32, 64
OBS_WORLD, OBS_BODY, OBS_LOS = 0, 1, 2

d3 = C.c_double * 3


class HlynrParams(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("max_steps", C.c_int32),
        ("dt", C.c_double), ("max_range", C.c_double), ("max_velocity", C.c_double),
        ("target", d3),
        ("m_spawn_spherical", C.c_int32), ("i_vel_toward_missile", C.c_int32),
        ("m_pos_lo", d3), ("m_pos_hi", d3),
        ("m_speed_lo", C.c_double), ("m_speed_hi", C.c_double),
        ("m_radius_lo", C.c_double), ("m_radius_hi", C.c_double),
        ("m_az_lo", C.c_double), ("m_az_hi", C.c_double),
        ("m_el_lo", C.c_double), ("m_el_hi", C.c_double),
        ("i_pos_lo", d3), ("i_pos_hi", d3), ("i_vel_lo", d3), ("i_vel_hi", d3),
        ("i_speed_lo", C.c_double), ("i_speed_hi", C.c_double),
        ("base_wind", d3), ("wind_variability", C.c_double),
        ("isa_enabled", C.c_int32), ("mach_enabled", C.c_int32), ("enh_wind_enabled", C.c_int32),
        ("thrust_dyn_enabled", C.c_int32), ("dr_enabled", C.c_int32), ("validate_enabled", C.c_int32),
        ("evasion_enabled", C.c_int32), ("onboard_delay", C.c_int32),
        ("sub_mach", C.c_double), ("sup_mach", C.c_double), ("peak_mult", C.c_double), ("sup_mult", C.c_double),
        ("blh", C.c_double), ("turb_intensity", C.c_double), ("gust_scale", C.c_double),
        ("thrust_tau", C.c_double),
        ("dr_variation", C.c_double * N_DR),
        ("radar_range", C.c_double), ("radar_quality", C.c_double),
        ("ground_enabled", C.c_int32), ("ground_delay", C.c_int32),
        ("ground_pos", d3),
        ("g_max_range", C.c_double), ("g_min_el", C.c_double), ("g_max_el", C.c_double),
        ("g_sigma_r", C.c_double), ("g_sigma_v", C.c_double), ("g_base_quality", C.c_double),
        ("max_datalink_range", C.c_double), ("datalink_packet_loss", C.c_double),
        ("obs_mode", C.c_int32), ("precision_mode", C.c_int32), ("fuze_enabled", C.c_int32),
        ("volley_size", C.c_int32),
        ("kill_radius", C.c_double),
    ]


class HlynrPolicyWeights(C.Structure):   # include/hlynr_policy.h
    _fields_ = [(n, C.c_void_p) for n in ("w1", "b1", "ln1_g", "ln1_b", "w2", "b2", "ln2_g", "ln2_b", "w3", "b3", "ln3_g", "ln3_b",
                                          "wa", "ba", "wv", "bv", "log_std")] + [("ln_eps", C.c_float)]


class HlynrCurriculum(C.Structure):
    _fields_ = [("intercept_radius", C.c_double), ("beam_width_deg", C.c_double),
                ("onboard_reliability", C.c_double), ("ground_reliability", C.c_double)]


class HlynrCurriculumSchedule(C.Structure):
    _fields_ = [("enabled", C.c_int32), ("radar_enabled", C.c_int32),
                ("initial_radius", C.c_double), ("final_radius", C.c_double), ("curriculum_steps", C.c_double)] + [
        (f"{ramp}_{k}", C.c_double) for ramp in ("beam", "onboard", "ground") for k in ("initial", "final", "start", "end")]


INFO_FIELDS = [  # name, numpy dtype, trailing shape: the fields of HlynrInfoSoA, in order
    ("distance", "float32", ()), ("min_distance", "float32", ()), ("fuel_remaining", "float32", ()),
    ("fuel_used", "float32", ()), ("steps", "int32", ()), ("flags", "uint8", ()),
    ("interceptor_pos", "float32", (3,)), ("missile_pos", "float32", (3,)),
    ("episode_return", "float32", ()), ("episode_length", "int32", ()),
    ("missiles_intercepted", "int32", ()), ("missiles_remaining", "int32", ()), ("missile_min_distances", "float32", (MAX_VOLLEY,)),
    ("radar_quality", "float32", ()),
]


class HlynrInfoSoA(C.Structure):   # one device or host pointer per field
    _fields_ = [(name, C.c_void_p) for name, _, _ in INFO_FIELDS]

INFO_INTERCEPTED, INFO_HIT_TARGET, INFO_CLAMPED, INFO_RADAR_DETECTED = 0x01, 0x02, 0x04, 0x08
INFO_GROUND_DETECTED, INFO_CROSSED, INFO_FUZE, INFO_KF_INIT = 0x10, 0x20, 0x40, 0x80

DONE_TERMINATED, DONE_TRUNCATED, DONE_ONBOARD_FILL = 0x100, 0x200, 0x400


def done_record_numpy_dtype():
    """numpy structured dtype with the exact memory layout of HlynrDoneRecord (50 words)."""
    import numpy as np

    dt = np.dtype([("env", np.int32), ("steps", np.int32), ("flags", np.uint32), ("distance", np.float32),
                   ("min_distance", np.float32), ("fuel_remaining", np.float32), ("fuel_used", np.float32),
                   ("episode_return", np.float32), ("interceptor_pos", np.float32, (3,)), ("missile_pos", np.float32, (3,)),
                   ("terminal_obs", np.float32, (OBS_DIM,)), ("missiles_intercepted", np.int32), ("missiles_remaining", np.int32),
                   ("missile_min_distances", np.float32, (MAX_VOLLEY,))])
    assert dt.itemsize == 200, dt.itemsize
    return dt


def trace_row_numpy_dtype():
    """numpy structured dtype with the exact memory layout of HlynrTraceRow (include/hlynr_rollout.h, 18 words)."""
    import numpy as np

    dt = np.dtype([("interceptor_pos", np.float32, (3,)), ("missile_pos", np.float32, (3,)), ("action", np.float32, (ACT_DIM,)),
                   ("reward", np.float32), ("distance", np.float32), ("fuel_remaining", np.float32), ("radar_quality", np.float32),
                   ("flags", np.uint32), ("step", np.int32)])
    assert dt.itemsize == 72, dt.itemsize
    return dt


# the info fields a trace row reads (hlynr_eval_trace): the evaluator asks hlynr_step for these only
TRACE_INFO_FIELDS = ("distance", "fuel_remaining", "steps", "flags", "interceptor_pos", "missile_pos", "radar_quality")


STATS_FIELDS = ["episodes", "successes", "return_sum", "length_sum", "min_distance_sum", "final_distance_sum",
                "hit_target", "interceptor_crash", "fuel_out", "missile_ground", "worsening", "timeouts",
                "env_steps", "onboard_locks", "reserved0", "reserved1"]


class HlynrStats(C.Structure):
    _fields_ = [(n, C.c_double) for n in STATS_FIELDS[:14]] + [("reserved", C.c_double * 2)]


class HlynrEnvState(C.Structure):
    _fields_ = [
        ("ipos", d3), ("ivel", d3), ("quat", C.c_double * 4), ("fuel", C.c_double), ("fuel_used", C.c_double),
        ("mpos", d3), ("mvel", d3), ("wind", d3), ("thrust", d3),
        ("prev_d", C.c_double), ("last_d", C.c_double), ("min_d", C.c_double), ("episode_return", C.c_double),
        ("kf_x", C.c_double * 6), ("kf_P", C.c_double * 4),
        ("T0", C.c_double), ("base_cd", C.c_double), ("peak", C.c_double),
        ("vpos", C.c_double * (MAX_VOLLEY * 3)), ("vvel", C.c_double * (MAX_VOLLEY * 3)), ("vmin", C.c_double * MAX_VOLLEY),
        ("steps", C.c_int32), ("worsen_count", C.c_int32), ("crossed", C.c_int32), ("kf_init", C.c_int32),
        ("onboard_delay", C.c_int32), ("episode", C.c_int32),
        ("vactive", C.c_int32 * MAX_VOLLEY), ("vcur", C.c_int32), ("vcount", C.c_int32),
        ("kf_f64", C.c_int32), ("reserved", C.c_int32),
    ]


ENV_STATE_VEC_FIELDS = {"ipos": 3, "ivel": 3, "quat": 4, "mpos": 3, "mvel": 3, "wind": 3, "thrust": 3,
                        "kf_x": 6, "kf_P": 4, "vpos": MAX_VOLLEY * 3, "vvel": MAX_VOLLEY * 3, "vmin": MAX_VOLLEY}
ENV_STATE_INT_VEC_FIELDS = {"vactive": MAX_VOLLEY}


def env_state_numpy_dtype():
    """numpy structured dtype with the exact memory layout of HlynrEnvState."""
    import numpy as np

    fields = []
    for name, ctype in HlynrEnvState._fields_:
        if name in ENV_STATE_VEC_FIELDS:
            fields.append((name, np.float64, (ENV_STATE_VEC_FIELDS[name],)))
        elif name in ENV_STATE_INT_VEC_FIELDS:
            fields.append((name, np.int32, (ENV_STATE_INT_VEC_FIELDS[name],)))
        elif ctype is C.c_int32:
            fields.append((name, np.int32))
        else:
            fields.append((name, np.float64))
    dt = np.dtype(fields, align=True)
    assert dt.itemsize == C.sizeof(HlynrEnvState), (dt.itemsize, C.sizeof(HlynrEnvState))
    return dt


# ---- snapshots (include/hlynr.h hlynr_snapshot_*, include/hlynr_post.h hlynr_post_snapshot_*) ----
SNAPSHOT_VERSION = 1
SNAP_SECTIONS = ("real", "int", "onboard_ring", "ground_ring", "stats", "curriculum")


class HlynrSnapshotInfo(C.Structure):
    _fields_ = [("format_version", C.c_int32), ("abi_version", C.c_int32), ("precision", C.c_int32), ("obs_dim", C.c_int32),
                ("n_envs", C.c_int64), ("env_id_offset", C.c_int64), ("seed", C.c_uint64),
                ("volley_k", C.c_int32), ("onboard_ring_len", C.c_int32), ("ground_ring_len", C.c_int32),
                ("curriculum_attached", C.c_int32), ("tick", C.c_uint64), ("env_steps", C.c_double),
                ("curriculum_increment", C.c_int64), ("params", HlynrParams), ("curriculum", HlynrCurriculum),
                ("schedule", HlynrCurriculumSchedule), ("section_offset", C.c_uint64 * len(SNAP_SECTIONS)), ("device_bytes", C.c_uint64)]


POST_SNAPSHOT_VERSION = 1
POST_SNAP_SECTIONS = ("frames", "age", "returns", "stats")


class HlynrPostSnapshotInfo(C.Structure):
    _fields_ = [("format_version", C.c_int32), ("frame_dim", C.c_int32), ("n_stack", C.c_int32), ("sums_valid", C.c_int32),
                ("n_envs", C.c_int64), ("t", C.c_uint64), ("clip_obs", C.c_double), ("epsilon", C.c_double), ("gamma", C.c_double),
                ("stats_bytes", C.c_uint64), ("section_offset", C.c_uint64 * len(POST_SNAP_SECTIONS)), ("device_bytes", C.c_uint64)]


def struct_to_dict(s):
    """A ctypes structure as plain Python values (nested structures as dicts, arrays as lists): JSON-serialisable, and exact
    for every double (json writes the shortest repr that reads back to the same bits)."""
    def val(v):
        if isinstance(v, C.Structure):
            return struct_to_dict(v)
        if isinstance(v, C.Array):
            return [val(x) for x in v]
        return v

    return {name: val(getattr(s, name)) for name, _ in s._fields_}


def struct_from_dict(cls, d):
    """The inverse of struct_to_dict; refuses a missing or unknown field."""
    names = [name for name, _ in cls._fields_]
    if set(d) != set(names):
        raise ValueError(f"{cls.__name__}: fields {sorted(set(d) ^ set(names))} are missing or unknown")
    s = cls()
    for name, ctype in cls._fields_:
        v = d[name]
        if isinstance(ctype, type) and issubclass(ctype, C.Structure):
            setattr(s, name, struct_from_dict(ctype, v))
        elif isinstance(ctype, type) and issubclass(ctype, C.Array):
            if len(v) != ctype._length_:
                raise ValueError(f"{cls.__name__}.{name}: {len(v)} values, expected {ctype._length_}")
            setattr(s, name, ctype(*v))
        else:
            setattr(s, name, v)
    return s

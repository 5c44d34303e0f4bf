"""Config resolver: the reference's nested env dict -> flat `HlynrParams` + host-side curriculum.

Mirrors `InterceptEnvironment.__init__` (rl_system/environment.py:20-221) and
`Radar26DObservation.__init__` (rl_system/core.py:258-335) key by key, with the same
`.get(key, default)` semantics, so that a config that means X to the reference means X here --
including the keys the reference silently ignores (SURVEY section 5, "dead keys"), for which
`dead_keys()` produces a warning list instead of changing behaviour.
"""
import math
import warnings

import numpy as np

from . import abi

# keys present in the shipped YAMLs that InterceptEnvironment never reads (SURVEY section 5)
_DEAD_ENV_KEYS = ("gravity", "drag_coefficient", "air_density", "radar_range", "radar_noise", "radar_quality",
                  "radar_beam_width", "min_detection_range")


def dead_keys(env_cfg):
    """Keys of `env_cfg` that the reference accepts and ignores."""
    out = [k for k in _DEAD_ENV_KEYS if k in env_cfg]
    pe = env_cfg.get("physics_enhancements", {}) or {}
    am = pe.get("atmospheric_model", {}) or {}
    out += ["physics_enhancements.atmospheric_model." + k for k in am if k != "enabled"]
    ew = pe.get("enhanced_wind", {}) or {}
    out += ["physics_enhancements.enhanced_wind." + k for k in ("gust_probability", "surface_roughness") if k in ew]
    return out


def _f32(v):
    return [float(np.float32(x)) for x in v]


def _delay_samples(delay_ms, dt):
    # core.py:292,316:  int(ms / (dt * 1000.0)) if ms > 0 else 0 ; SensorDelayBuffer clamps to >= 1 (core.py:164)
    n = int(delay_ms / (dt * 1000.0)) if delay_ms > 0 else 0
    return max(1, n) if n > 0 else 0


def resolve_config(env_cfg=None, warn_dead=True):
    """env dict (what the reference passes to InterceptEnvironment) -> (HlynrParams, Curriculum)."""
    cfg = dict(env_cfg or {})
    if warn_dead:
        dk = dead_keys(cfg)
        if dk:
            warnings.warn("config keys ignored by the reference environment (and therefore here): " + ", ".join(dk),
                          stacklevel=2)
    volley_size = 0   # environment.py:42-43: 0 = volley_mode off, else the number of missiles per episode
    if cfg.get("volley_mode", False):
        volley_size = int(cfg.get("volley_size", 1))
        if not 1 <= volley_size <= abi.MAX_VOLLEY:
            raise NotImplementedError(f"volley_size {volley_size} outside [1, {abi.MAX_VOLLEY}]")

    p = abi.HlynrParams()
    p.abi_version = abi.ABI_VERSION
    p.volley_size = volley_size
    p.dt = float(cfg.get("dt", 0.01))
    p.max_steps = int(cfg.get("max_steps", 1000))
    p.max_range = float(cfg.get("max_range", 10000.0))
    p.max_velocity = float(cfg.get("max_velocity", 1000.0))
    p.target[:] = _f32(cfg.get("target_position", [900, 900, 5]))

    ms = cfg.get("missile_spawn", {"position": [[-500, -500, 200], [500, 500, 500]],
                                   "velocity": [[50, 50, -20], [150, 150, -50]]})
    isp = cfg.get("interceptor_spawn", {"position": [[400, 400, 50], [600, 600, 200]],
                                        "velocity": [[0, 0, 0], [50, 50, 20]]})
    m_pos_lo, m_pos_hi = ms["position"]
    m_vel_lo, m_vel_hi = ms["velocity"]
    p.m_pos_lo[:] = [float(x) for x in m_pos_lo]
    p.m_pos_hi[:] = [float(x) for x in m_pos_hi]
    p.m_speed_lo = float(ms.get("speed_min", np.linalg.norm(m_vel_lo)))
    p.m_speed_hi = float(ms.get("speed_max", np.linalg.norm(m_vel_hi)))
    if ms.get("velocity_mode", "toward_target") != "toward_target":
        pass  # environment.py:412 reads velocity_mode and never uses it
    p.m_spawn_spherical = 1 if ms.get("position_mode", "box") == "spherical" else 0
    p.m_radius_lo = float(ms.get("radius_min", 800.0))
    p.m_radius_hi = float(ms.get("radius_max", 1500.0))
    az = ms.get("azimuth_range", [0, 360])
    el = ms.get("elevation_range", [10, 60])
    p.m_az_lo, p.m_az_hi = float(az[0]), float(az[1])
    p.m_el_lo, p.m_el_hi = float(el[0]), float(el[1])
    i_pos_lo, i_pos_hi = isp["position"]
    i_vel_lo, i_vel_hi = isp["velocity"]
    p.i_pos_lo[:] = [float(x) for x in i_pos_lo]
    p.i_pos_hi[:] = [float(x) for x in i_pos_hi]
    p.i_vel_lo[:] = [float(x) for x in i_vel_lo]
    p.i_vel_hi[:] = [float(x) for x in i_vel_hi]
    p.i_vel_toward_missile = 1 if isp.get("velocity_mode", "box") == "toward_missile" else 0
    p.i_speed_lo = float(isp.get("speed_min", np.linalg.norm(i_vel_lo)))
    p.i_speed_hi = float(isp.get("speed_max", np.linalg.norm(i_vel_hi)))

    wind = cfg.get("wind", {}) or {}
    p.base_wind[:] = _f32(wind.get("velocity", [5.0, 0.0, 0.0]))
    p.wind_variability = float(wind.get("variability", 0.1))

    pe = cfg.get("physics_enhancements", {}) or {}
    on = bool(pe.get("enabled", True))
    p.isa_enabled = int(on and (pe.get("atmospheric_model", {}) or {}).get("enabled", True))
    mach = pe.get("mach_effects", {}) or {}
    p.mach_enabled = int(on and mach.get("enabled", True))
    p.sub_mach = float(mach.get("subsonic_mach", 0.8))
    p.sup_mach = float(mach.get("supersonic_mach", 1.2))
    p.peak_mult = float(mach.get("transonic_peak_multiplier", 3.0))
    p.sup_mult = float(mach.get("supersonic_multiplier", 2.5))
    ew = pe.get("enhanced_wind", {}) or {}
    p.enh_wind_enabled = int(on and ew.get("enabled", True))
    p.blh = float(ew.get("boundary_layer_height", 1000.0))
    p.turb_intensity = float(ew.get("turbulence_intensity", 0.1))
    p.gust_scale = float(ew.get("max_gust_speed", 5.0))
    td = pe.get("thrust_dynamics", {}) or {}
    p.thrust_dyn_enabled = int(on and td.get("enabled", True))
    p.thrust_tau = float(td.get("response_time_constant", 0.1))
    dr = pe.get("domain_randomization", {}) or {}
    p.dr_enabled = int(on and dr.get("enabled", False))
    # physics_randomizer.py:19-41 defaults, :108-117 overrides, :166-214 draw order
    p.dr_variation[:] = [
        float(dr.get("air_density_variation", 0.1)),
        0.05 * 20.0,                                    # temperature offset sigma (K)
        float(dr.get("drag_coefficient_variation", 0.2)),
        0.15,                                           # mach_curve_variation
        float(dr.get("sensor_delay_variation", 0.5)),
        0.3,                                            # radar_noise_variation
        0.1,                                            # radar_quality_variation
        float(dr.get("thrust_response_variation", 0.3)),
        0.2,                                            # fuel_consumption_variation
        float(dr.get("wind_variation", 0.3)),
        0.4,                                            # turbulence_variation
        0.1, 0.1,                                       # mass variation x2
    ]
    p.validate_enabled = int((pe.get("performance", {}) or {}).get("enable_physics_validation", True))
    p.evasion_enabled = int(bool(cfg.get("missile_evasion", False)))

    sd = pe.get("sensor_delays", {}) or {}
    delay_ms = float(sd.get("radar_delay_ms", 30.0)) if (on and sd.get("enabled", True)) else 0.0
    p.onboard_delay = _delay_samples(delay_ms, p.dt)
    if p.onboard_delay > 10:
        raise ValueError("onboard sensor delay > 10 samples is not supported")

    radar = cfg.get("radar", {}) or {}
    p.radar_range = float(radar.get("radar_range", 5000.0))
    p.radar_quality = float(radar.get("radar_quality", 1.0))

    g = cfg.get("ground_radar", {}) or {}
    g_on = bool(g.get("enabled", True)) if g else True
    p.ground_enabled = int(bool(g_on and g))  # core.py:296-320: no config dict -> no station
    p.ground_pos[:] = _f32(g.get("position", [0, 0, 100]))
    p.g_max_range = float(g.get("max_range", 20000.0))
    p.g_min_el = float(np.radians(g.get("min_elevation_angle", 5.0)))
    p.g_max_el = float(np.radians(g.get("max_elevation_angle", 85.0)))
    p.g_sigma_r = float(g.get("range_accuracy", 10.0))
    p.g_sigma_v = float(g.get("velocity_accuracy", 2.0))
    p.g_base_quality = float(g.get("base_quality", 0.95))
    p.max_datalink_range = float(g.get("max_datalink_range", 50000.0))
    p.datalink_packet_loss = float(g.get("datalink_packet_loss", 0.05))
    p.ground_delay = _delay_samples(float(g.get("ground_sensor_delay_ms", 50.0)), p.dt) if p.ground_enabled else 0
    if p.ground_delay > 31:
        raise ValueError("ground sensor delay > 31 samples is not supported")

    mode = cfg.get("observation_mode", "world_frame")
    if cfg.get("rotation_invariant", False) and mode == "world_frame":
        mode = "body_frame"
    p.obs_mode = {"world_frame": abi.OBS_WORLD, "body_frame": abi.OBS_BODY, "los_frame": abi.OBS_LOS}[mode]
    cur = cfg.get("curriculum", {}) or {}
    p.precision_mode = int(bool(cur.get("precision_mode", False)))
    p.fuze_enabled = int(bool(cfg.get("proximity_fuze_enabled", False)))
    p.kill_radius = float(cfg.get("proximity_kill_radius", 20.0))
    return p, Curriculum(cfg)


class Curriculum:
    """Host-side curriculum scalars: get_current_intercept_radius (environment.py:223-234) and
    _update_radar_curriculum (environment.py:274-351).  Global to all envs, pushed to the device with
    hlynr_set_curriculum whenever training_step_count changes."""

    def __init__(self, env_cfg):
        cur = env_cfg.get("curriculum", {}) or {}
        self.use_curriculum = bool(cur.get("enabled", True))
        self.initial_radius = float(cur.get("initial_radius", 200.0))
        self.final_radius = float(cur.get("final_radius", 20.0))
        self.curriculum_steps = cur.get("curriculum_steps", 5000000)
        self.rc = cur.get("radar_curriculum", {}) or {}
        self.use_radar_curriculum = bool(self.rc.get("enabled", True))
        radar = env_cfg.get("radar", {}) or {}
        beam = radar.get("radar_beam_width", 60.0)
        self.onboard_reliability = 1.0   # core.py:286-288 defaults
        self.ground_reliability = 1.0
        self.noise_level = 0.05
        if self.use_radar_curriculum and self.rc:  # environment.py:154,182: empty dict is falsy
            beam = self.rc.get("initial_beam_width", 120.0)
            self.onboard_reliability = self.rc.get("initial_detection_reliability", 1.0)
            self.ground_reliability = self.rc.get("initial_ground_reliability", 1.0)
            self.noise_level = self.rc.get("initial_noise_level", 0.0)
        self.beam_width = float(beam)
        self.training_step_count = 0

    def intercept_radius(self):
        if not self.use_curriculum:
            return self.final_radius
        progress = min(1.0, self.training_step_count / self.curriculum_steps)
        return self.initial_radius * (1.0 - progress) + self.final_radius * progress

    @staticmethod
    def _ramp(step, start, end, a, b):
        if step < start:
            return a
        if step >= end:
            return b
        t = (step - start) / (end - start)
        return a * (1.0 - t) + b * t

    def set_training_step_count(self, n):
        self.training_step_count = n
        if not self.use_radar_curriculum or not self.rc:
            return
        rc = self.rc
        self.beam_width = self._ramp(n, rc.get("beam_width_transition_start", 3000000),
                                     rc.get("beam_width_transition_end", 5000000),
                                     rc.get("initial_beam_width", 120.0), rc.get("final_beam_width", 60.0))
        self.onboard_reliability = self._ramp(n, rc.get("reliability_transition_start", 4500000),
                                              rc.get("reliability_transition_end", 6000000),
                                              rc.get("initial_detection_reliability", 1.0),
                                              rc.get("final_detection_reliability", 0.75))
        self.ground_reliability = self._ramp(n, rc.get("ground_reliability_transition_start", 4500000),
                                             rc.get("ground_reliability_transition_end", 6000000),
                                             rc.get("initial_ground_reliability", 1.0),
                                             rc.get("final_ground_reliability", 0.85))
        self.noise_level = self._ramp(n, rc.get("noise_transition_start", 6000000),
                                      rc.get("noise_transition_end", 7000000),
                                      rc.get("initial_noise_level", 0.0), rc.get("final_noise_level", 0.05))

    def schedule(self):
        """The whole schedule as an abi.HlynrCurriculumSchedule, for HlynrSim.track_training_steps: the device then computes
        intercept_radius() and set_training_step_count() from its own counter, with the same double operations."""
        s = abi.HlynrCurriculumSchedule()
        s.enabled = int(self.use_curriculum)
        s.initial_radius, s.final_radius = self.initial_radius, self.final_radius
        s.curriculum_steps = float(self.curriculum_steps)
        rc = self.rc
        s.radar_enabled = int(self.use_radar_curriculum and bool(rc))
        if s.radar_enabled:
            ramps = dict(beam=("beam_width_transition_start", 3000000, "beam_width_transition_end", 5000000,
                               "initial_beam_width", 120.0, "final_beam_width", 60.0),
                         onboard=("reliability_transition_start", 4500000, "reliability_transition_end", 6000000,
                                  "initial_detection_reliability", 1.0, "final_detection_reliability", 0.75),
                         ground=("ground_reliability_transition_start", 4500000, "ground_reliability_transition_end", 6000000,
                                 "initial_ground_reliability", 1.0, "final_ground_reliability", 0.85))
            for name, (ks, ds, ke, de, ki, di, kf, df) in ramps.items():   # the keys and defaults of set_training_step_count
                setattr(s, name + "_start", float(rc.get(ks, ds)))
                setattr(s, name + "_end", float(rc.get(ke, de)))
                setattr(s, name + "_initial", float(rc.get(ki, di)))
                setattr(s, name + "_final", float(rc.get(kf, df)))
        else:   # the values __init__ chose, constant
            s.beam_initial = s.beam_final = self.beam_width
            s.onboard_initial = s.onboard_final = float(self.onboard_reliability)
            s.ground_initial = s.ground_final = float(self.ground_reliability)
        return s

    def to_struct(self):
        c = abi.HlynrCurriculum()
        c.intercept_radius = float(self.intercept_radius())
        c.beam_width_deg = float(self.beam_width)
        c.onboard_reliability = float(self.onboard_reliability)
        c.ground_reliability = float(self.ground_reliability)
        return c

    def as_dict(self):
        s = self.to_struct()
        return {n: getattr(s, n) for n, _ in abi.HlynrCurriculum._fields_}


def params_as_dict(p):
    out = {}
    for name, _ in abi.HlynrParams._fields_:
        v = getattr(p, name)
        out[name] = list(v) if hasattr(v, "__len__") else v
    return out


# ---- the BASELINE.json configurations (SURVEY 8d "Synthetic inputs per BASELINE config") ---------------
def _scenario_env(name):
    """Scenario env dicts restated from rl_system/configs/scenarios/{easy,medium,hard}.yaml (effective keys
    only; the dead keys of those files are omitted)."""
    ground = dict(enabled=True, position=[0, 0, 100], max_range=20000.0, min_elevation_angle=5.0,
                  max_elevation_angle=85.0, range_accuracy=10.0, velocity_accuracy=2.0, base_quality=0.95,
                  weather_sensitivity=0.2, max_datalink_range=50000.0, datalink_packet_loss=0.05,
                  ground_sensor_delay_ms=50.0)
    if name == "easy":
        ground.update(range_accuracy=8.0, velocity_accuracy=1.5, base_quality=0.98, weather_sensitivity=0.1,
                      datalink_packet_loss=0.02, ground_sensor_delay_ms=40.0)
        return dict(target_position=[0, 0, 0],
                    interceptor_spawn=dict(position=[[0, 0, 0], [30, 30, 10]], velocity=[[30, 30, 50], [50, 50, 90]]),
                    missile_spawn=dict(position=[[1000, 1000, 1200], [2000, 2000, 2000]],
                                       velocity=[[-60, -60, -30], [-90, -90, -50]]),
                    max_steps=2000, wind=dict(velocity=[2.0, 0.0, 0.0], variability=0.05),
                    ground_radar=ground, missile_evasion=False)
    if name == "medium":
        return dict(target_position=[0, 0, 0],
                    interceptor_spawn=dict(position=[[0, 0, 0], [50, 50, 10]], velocity=[[20, 20, 40], [40, 40, 80]]),
                    missile_spawn=dict(position=[[1800, 1800, 1800], [3200, 3200, 3200]],
                                       velocity=[[-110, -110, -55], [-160, -160, -75]]),
                    max_steps=2000, wind=dict(velocity=[8.0, 3.0, 0.0], variability=0.15),
                    ground_radar=ground, missile_evasion=True)
    if name == "hard":
        ground.update(max_range=18000.0, range_accuracy=15.0, velocity_accuracy=3.0, base_quality=0.88,
                      weather_sensitivity=0.3, max_datalink_range=45000.0, datalink_packet_loss=0.10,
                      ground_sensor_delay_ms=60.0)
        return dict(target_position=[0, 0, 0],
                    interceptor_spawn=dict(position=[[0, 0, 0], [70, 70, 15]], velocity=[[10, 10, 30], [35, 35, 70]]),
                    missile_spawn=dict(position=[[2500, 2500, 2500], [4000, 4000, 4000]],
                                       velocity=[[-140, -140, -75], [-200, -200, -100]]),
                    max_steps=2000, wind=dict(velocity=[15.0, 8.0, -2.0], variability=0.25),
                    ground_radar=ground, missile_evasion=True)
    raise KeyError(name)


def baseline_config(name):
    """'cfg1'..'cfg4' of BASELINE.json -> env dict."""
    if name == "cfg1":   # easy.yaml as-is (physics v2.0 on by default, Quirk Q2)
        return _scenario_env("easy")
    if name == "cfg2":   # medium, physics v2.0 off
        e = _scenario_env("medium")
        e["physics_enhancements"] = dict(enabled=False)
        return e
    if name in ("cfg3", "cfg3_radar"):  # hard, v2.0 on + domain randomization
        e = _scenario_env("hard")
        e["physics_enhancements"] = dict(enabled=True, domain_randomization=dict(
            enabled=True, drag_coefficient_variation=0.2, air_density_variation=0.1, sensor_delay_variation=0.5,
            thrust_response_variation=0.3, wind_variation=0.3))
        if name == "cfg3_radar":  # honour "narrow beam, high noise" through the radar: sub-dict the env does read
            e["radar"] = dict(radar_beam_width=45.0, radar_quality=0.75, radar_range=3500.0)
        return e
    if name == "cfg4":   # medium, v2.0 on (defaults)
        return _scenario_env("medium")
    raise KeyError(name)

"""Config resolver: same effective-key semantics as InterceptEnvironment.__init__ / Radar26DObservation.__init__."""
import math
import warnings

import numpy as np
import pytest

from hlynr_intercept_b200 import abi, config
from oracle import ref_harness


def test_defaults_match_reference_defaults():
    P, cur = config.resolve_config({}, warn_dead=False)
    assert P.dt == 0.01 and P.max_steps == 1000 and P.max_range == 10000.0 and P.max_velocity == 1000.0
    assert list(P.target) == [900.0, 900.0, 5.0]
    # Quirk Q2: with no physics_enhancements dict every v2.0 feature is ON, domain randomization OFF
    assert (P.isa_enabled, P.mach_enabled, P.enh_wind_enabled, P.thrust_dyn_enabled, P.dr_enabled) == (1, 1, 1, 1, 0)
    assert P.onboard_delay == 3 and P.ground_enabled == 0 and P.ground_delay == 0   # no ground_radar dict -> no station
    assert cur.intercept_radius() == 200.0 and cur.beam_width == 60.0
    assert P.radar_range == 5000.0 and P.radar_quality == 1.0


def test_dead_keys_are_reported_and_ignored():
    cfg = config.baseline_config("cfg4")
    cfg.update(radar_range=4500.0, radar_beam_width=60.0, radar_quality=0.9, gravity=[0, 0, -9.81], drag_coefficient=0.3)
    assert set(config.dead_keys(cfg)) >= {"radar_range", "radar_beam_width", "radar_quality", "gravity", "drag_coefficient"}
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        P, cur = config.resolve_config(cfg)
    assert any("ignored by the reference" in str(x.message) for x in w)
    assert P.radar_range == 5000.0 and P.radar_quality == 1.0 and cur.beam_width == 60.0   # the dead keys changed nothing
    P2, _ = config.resolve_config(dict(cfg, radar=dict(radar_range=4500.0, radar_quality=0.9)), warn_dead=False)
    assert P2.radar_range == 4500.0 and P2.radar_quality == 0.9                            # the radar: sub-dict is read


def test_curriculum_ramps():
    cfg = dict(curriculum=dict(enabled=True, initial_radius=100.0, final_radius=5.0, curriculum_steps=2000000,
                               radar_curriculum=dict(enabled=True, initial_beam_width=120.0, final_beam_width=60.0,
                                                     beam_width_transition_start=5000000, beam_width_transition_end=8000000)))
    _, cur = config.resolve_config(cfg, warn_dead=False)
    assert cur.intercept_radius() == 100.0 and cur.beam_width == 120.0
    cur.set_training_step_count(1000000)
    assert abs(cur.intercept_radius() - 52.5) < 1e-12
    cur.set_training_step_count(6500000)
    assert abs(cur.beam_width - 90.0) < 1e-12 and cur.intercept_radius() == 5.0
    cur.set_training_step_count(6000000)   # default reliability ramp 4.5M-6M: 1.0 -> 0.75 / 0.85
    assert abs(cur.onboard_reliability - 0.75) < 1e-12 and abs(cur.ground_reliability - 0.85) < 1e-12


def test_volley_mode_resolution_and_limits():
    P, _ = config.resolve_config(dict(volley_mode=True, volley_size=3), warn_dead=False)
    assert P.volley_size == 3
    assert config.resolve_config(dict(volley_size=3), warn_dead=False)[0].volley_size == 0   # volley_mode off: size ignored
    assert config.resolve_config(dict(volley_mode=True), warn_dead=False)[0].volley_size == 1  # environment.py:43 default
    with pytest.raises(NotImplementedError):   # more missiles per env than the kernel's planes hold: fail loudly
        config.resolve_config(dict(volley_mode=True, volley_size=9), warn_dead=False)


@pytest.mark.reference
@pytest.mark.parametrize("name", ["cfg1", "cfg2", "cfg3", "cfg3_radar", "cfg4"])
def test_resolver_matches_reference_constructor(name):
    """Every resolved parameter equals the attribute the unmodified reference computes from the same dict."""
    ref_harness.install_shim()
    env = ref_harness.RefBatch(config.baseline_config(name), 1).envs[0]
    P, cur = config.resolve_config(config.baseline_config(name), warn_dead=False)
    og = env.observation_generator
    assert P.dt == env.dt and P.max_steps == env.max_steps and P.max_range == env.max_range
    np.testing.assert_array_equal(np.array(P.target), env.target_position.astype(np.float64))
    np.testing.assert_array_equal(np.array(P.base_wind), env.base_wind.astype(np.float64))
    assert P.wind_variability == env.wind_variability
    assert bool(P.isa_enabled) == (env.atmospheric_model is not None)
    assert bool(P.mach_enabled) == (env.mach_drag_model is not None)
    assert bool(P.enh_wind_enabled) == (env.enhanced_wind_model is not None)
    assert bool(P.thrust_dyn_enabled) == env.thrust_dynamics_enabled
    assert bool(P.dr_enabled) == (env.physics_randomizer is not None and env.physics_randomizer.enabled)
    assert bool(P.evasion_enabled) == bool(env.config.get("missile_evasion", False))
    assert P.onboard_delay == (og.sensor_delay_buffer.delay_samples if og.sensor_delay_buffer else 0)
    assert P.ground_delay == (og.ground_sensor_delay_buffer.delay_samples if og.ground_sensor_delay_buffer else 0)
    assert P.radar_range == og.radar_range and P.radar_quality == env.radar_quality
    g = og.ground_radar
    assert (P.g_max_range, P.g_min_el, P.g_max_el) == (g.max_range, float(g.min_elevation_angle), float(g.max_elevation_angle))
    assert (P.g_sigma_r, P.g_sigma_v, P.g_base_quality) == (g.range_accuracy, g.velocity_accuracy, g.base_quality)
    assert (P.max_datalink_range, P.datalink_packet_loss) == (og.max_datalink_range, og.datalink_packet_loss)
    if env.physics_randomizer is not None:
        pr = env.physics_randomizer.params
        assert P.dr_variation[0] == pr.air_density_variation and P.dr_variation[2] == pr.drag_coefficient_variation
        assert P.dr_variation[4] == pr.sensor_delay_variation and P.dr_variation[1] == pr.temperature_variation * 20.0
    assert cur.intercept_radius() == env.get_current_intercept_radius()
    assert cur.beam_width == og.radar_beam_width


@pytest.mark.parametrize("scen", ["easy", "medium", "hard"])
def test_restated_scenarios_equal_reference_yaml(scen):
    """config._scenario_env restates configs/scenarios/*.yaml: every effective key must agree with the file.  The file's
    `environment` section is the env dict the yaml_scenario_* fixture was generated from (oracle/gen_golden.reference_yaml_env,
    which adds the top-level curriculum and physics_enhancements sections; these scenario files have neither)."""
    from common import load_golden

    y = dict(load_golden("yaml_scenario_" + scen)["meta"]["env_cfg"])
    assert y.pop("curriculum") == {} and y.pop("physics_enhancements") == {}
    mine = config._scenario_env(scen)
    for k in config._DEAD_ENV_KEYS:
        y.pop(k, None)
    assert mine == y

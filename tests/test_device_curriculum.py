"""The training curriculum advanced on the device (hlynr_attach_curriculum, HlynrSim.track_training_steps).

SB3 raises model.num_timesteps by n_envs per env step and the reference's callback pushes it with
env_method('set_training_step_count') after every step, so the step at tick t sees t0 + t * N.  A tracking sim computes the
same curriculum from a device-side counter, so eager steps and CUDA-graph replays continue the schedule.  Checked here:
  (a) the device arithmetic equals config.Curriculum followed by make_kcur bit for bit, for both precisions;
  (b) a tracking sim equals a twin that pushes set_training_step_count(t0 + t * N) from the host before every tick, bit for bit,
      on a configuration where the radius decides outcomes (a frozen curriculum differs);
  (c) StepGraph and DeviceRolloutCollector replays equal eager host-pushed runs, and the counter ends at t0 + R * T * increment;
  (d) the surface: get/set between replays, detach, the refused calls and the invalid schedules."""
import ctypes as C
import math

import numpy as np
import pytest

from hlynr_intercept_b200 import abi, config

N = 1037   # a ragged tile
TICKS = 120
MAX_STEPS = 40


def _ramps_cfg(unit=N, steps_as_float=False):
    """cfg4 with missiles spawned around the intercept radius, and a curriculum whose four ramps all move within TICKS ticks of
    `unit` env steps each (the radius from 200 m to 5 m over 100 ticks)."""
    e = config.baseline_config("cfg4")
    e["max_steps"] = MAX_STEPS
    # test_evaluation.py's spawn: missiles 170-430 m away, closing at ~300 m/s, and interceptors that may start downwards
    e["missile_spawn"] = dict(position=[[150, 150, 100], [260, 260, 220]], velocity=[[-110, -110, -55], [-160, -160, -75]])
    e["interceptor_spawn"] = dict(position=[[0, 0, 0], [50, 50, 10]], velocity=[[20, 20, -40], [40, 40, 80]])
    f = float if steps_as_float else int
    e["curriculum"] = dict(enabled=True, initial_radius=200.0, final_radius=5.0, curriculum_steps=f(100 * unit + 0.5 * steps_as_float),
                           radar_curriculum=dict(
                               enabled=True, initial_beam_width=120.0, final_beam_width=30.0,
                               beam_width_transition_start=f(10 * unit), beam_width_transition_end=f(90 * unit + 0.25 * steps_as_float),
                               initial_detection_reliability=1.0, final_detection_reliability=0.6,
                               reliability_transition_start=f(20 * unit), reliability_transition_end=f(80 * unit),
                               initial_ground_reliability=1.0, final_ground_reliability=0.5,
                               ground_reliability_transition_start=f(30 * unit), ground_reliability_transition_end=f(110 * unit)))
    return e


def _schedules():
    """name -> env cfg: every kind of schedule config.Curriculum distinguishes."""
    out = {"ramps": _ramps_cfg(), "float_steps": _ramps_cfg(steps_as_float=True)}
    e = _ramps_cfg()
    e["curriculum"]["enabled"] = False
    out["disabled"] = e
    e = _ramps_cfg()
    del e["curriculum"]["radar_curriculum"]
    out["no_radar_curriculum"] = e
    e = _ramps_cfg()
    e["curriculum"]["radar_curriculum"] = {}
    out["empty_radar_curriculum"] = e
    e = _ramps_cfg()
    e["curriculum"]["radar_curriculum"]["enabled"] = False
    e["radar"] = dict(radar_beam_width=400.0)   # beam of 360 degrees or more: make_kcur's cos = -2 case
    out["radar_curriculum_off"] = e
    return out


def make_kcur(c, fp64):
    """make_kcur (csrc/hlynr_capi.cu) of an abi.HlynrCurriculum, widened to float64 like hlynr_debug_curriculum_at."""
    f32 = lambda v: float(np.float32(v))   # noqa: E731
    hb = (c.beam_width_deg / 2.0) * (math.pi / 180.0)
    return (c.intercept_radius if fp64 else f32(c.intercept_radius), -2.0 if hb >= math.pi else f32(math.cos(hb)),
            f32(c.onboard_reliability), f32(c.ground_reliability))


def _counts(cur):
    """~10^4 counts over every ramp, the exact start and end counts and their neighbours, and counts above 2^32."""
    s = cur.schedule()
    edges = [0.0, s.curriculum_steps]
    if s.radar_enabled:
        edges += [s.beam_start, s.beam_end, s.onboard_start, s.onboard_end, s.ground_start, s.ground_end]
    cs = set(np.linspace(0, 120 * N, 10000).astype(np.int64).tolist())
    for e in edges:
        for d in (-1, 0, 1):
            cs.add(max(0, int(math.floor(e)) + d))
            cs.add(max(0, int(math.ceil(e)) + d))
    cs.update([2**32 - 1, 2**32, 2**32 + 1, 3 * 2**40 + 12345, 2**52 + 3])
    return sorted(cs)


# ---- CPU ------------------------------------------------------------------------------------------------------------------------

def test_schedule_mirrors_the_curriculum_keys():
    s = config.resolve_config(_ramps_cfg(), warn_dead=False)[1].schedule()
    assert (s.enabled, s.radar_enabled) == (1, 1)
    assert (s.initial_radius, s.final_radius, s.curriculum_steps) == (200.0, 5.0, 100.0 * N)
    assert (s.beam_initial, s.beam_final, s.beam_start, s.beam_end) == (120.0, 30.0, 10.0 * N, 90.0 * N)
    assert (s.onboard_initial, s.onboard_final, s.onboard_start, s.onboard_end) == (1.0, 0.6, 20.0 * N, 80.0 * N)
    assert (s.ground_initial, s.ground_final, s.ground_start, s.ground_end) == (1.0, 0.5, 30.0 * N, 110.0 * N)
    # defaults: environment.py's curriculum keys absent
    d = config.resolve_config({"curriculum": {"radar_curriculum": {"enabled": True, "initial_beam_width": 90}}}, warn_dead=False)[1]
    s = d.schedule()
    assert (s.initial_radius, s.final_radius, s.curriculum_steps) == (200.0, 20.0, 5e6)
    assert (s.beam_initial, s.beam_final, s.beam_start, s.beam_end) == (90.0, 60.0, 3e6, 5e6)
    assert (s.onboard_final, s.onboard_start, s.onboard_end, s.ground_final) == (0.75, 4.5e6, 6e6, 0.85)
    for name, e in _schedules().items():
        cur = config.resolve_config(e, warn_dead=False)[1]
        s = cur.schedule()
        if not s.radar_enabled:   # the constant values __init__ chose
            assert (s.beam_initial, s.onboard_initial, s.ground_initial) == (cur.beam_width, 1.0, 1.0), name
            assert (s.beam_final, s.onboard_final, s.ground_final) == (s.beam_initial, s.onboard_initial, s.ground_initial), name
    assert abi.HlynrCurriculumSchedule.curriculum_steps.offset == 24 and C.sizeof(abi.HlynrCurriculumSchedule) == 128


def test_entry_points_are_exported_and_check_their_arguments():
    from hlynr_intercept_b200 import _lib

    L = _lib.load(build_if_missing=False)
    assert L.hlynr_curriculum_schedule_size() == C.sizeof(abi.HlynrCurriculumSchedule)
    s = abi.HlynrCurriculumSchedule()
    v, out = C.c_uint64(), (C.c_double * 4)()
    assert L.hlynr_attach_curriculum(None, C.byref(s), 0, 1) != 0
    assert L.hlynr_detach_curriculum(None) != 0
    assert L.hlynr_set_timesteps(None, 5, None) != 0
    assert L.hlynr_get_timesteps(None, C.byref(v), None) != 0
    assert L.hlynr_debug_curriculum_at(None, 5, out) != 0


# ---- GPU: arithmetic -------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "fp64"])
@pytest.mark.parametrize("name", sorted(_schedules()))
def test_device_arithmetic_equals_the_host_curriculum(name, precision):
    from hlynr_intercept_b200.sim import HlynrSim

    e = _schedules()[name]
    sim = HlynrSim(e, n_envs=32, seed=3, warn_dead=False, precision=precision)
    sim.track_training_steps(0)
    host = config.resolve_config(e, warn_dead=False)[1]
    counts = _counts(host) if name == "ramps" else _counts(host)[::4]
    bad = []
    for c in counts:
        host.set_training_step_count(c)
        want = make_kcur(host.to_struct(), precision == "fp64")
        got = sim.debug_curriculum_at(c)
        if got != want:
            bad.append((c, got, want))
    assert not bad, (len(bad), bad[:5])
    sim.close()


# ---- GPU: trajectories -----------------------------------------------------------------------------------------------------------

def _done_list(sim):
    import torch

    recs = torch.zeros(sim.n * 200, dtype=torch.uint8, device=sim.device)
    cnt = torch.zeros(1, dtype=torch.int32, device=sim.device)
    p = lambda x: C.c_void_p(x.data_ptr())   # noqa: E731
    from hlynr_intercept_b200 import _lib

    _lib.check(sim.L.hlynr_set_done_list(sim.h, p(recs), p(cnt), sim.n))
    return recs, cnt


def _records(recs, cnt):
    k = int(cnt.item())
    r = recs[: k * 200].cpu().numpy().view(abi.done_record_numpy_dtype())
    return r[np.argsort(r["env"], kind="stable")]   # the order within one call is unspecified


def _state_equal(a, b):
    sa, sb = a.export_state(), b.export_state()
    return all(np.array_equal(sa[k], sb[k]) for k in sa)


def _twin_cfg(layout):
    e = _ramps_cfg()
    if layout == "los":
        e["observation_mode"] = "los_frame"   # FT_GENERIC_MODES
    return e


@pytest.mark.gpu
@pytest.mark.parametrize("obs_dim", [26, 17])
@pytest.mark.parametrize("layout", ["specialised", "los"])
@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_tracked_trajectory_equals_host_pushed_twin(precision, layout, obs_dim):
    """Twin A tracks on the device; twin B pushes set_training_step_count(t0 + t * N) before every tick; a third twin keeps the
    curriculum of t0.  A reset at tick 60 happens inside every ramp and must not move the counter.  cfg4 runs the specialised
    FT_V2ON instantiation (the compact plane layout in the fp32 build), the LOS frame FT_GENERIC_MODES."""
    import torch

    from hlynr_intercept_b200.sim import HlynrSim

    e = _twin_cfg(layout)
    t0 = 5 * N + 123
    sims = [HlynrSim(e, n_envs=N, seed=29, warn_dead=False, precision=precision, obs_dim=obs_dim) for _ in range(3)]
    a, b, frozen = sims
    a.track_training_steps(t0)
    b.set_training_step_count(t0)
    frozen.set_training_step_count(t0)
    lists = [_done_list(s) for s in sims]
    g = torch.Generator(device="cuda")
    g.manual_seed(7)
    oa, ob_ = a.reset().clone(), b.reset().clone()
    frozen.reset()
    assert torch.equal(oa, ob_)
    assert a.num_timesteps == t0
    n_done = 0
    for t in range(TICKS):
        if t == 60:
            assert a.num_timesteps == t0 + 60 * N
            b.set_training_step_count(t0 + 60 * N)
            oa, ob_ = a.reset().clone(), b.reset().clone()
            frozen.reset()
            assert torch.equal(oa, ob_) and a.num_timesteps == t0 + 60 * N
        act = torch.rand(N, 6, device="cuda", generator=g) * 2 - 1
        b.set_training_step_count(t0 + t * N)
        outs = []
        for s, (recs, cnt) in zip(sims, lists):
            cnt.zero_()
            o = s.step(act)
            outs.append([x.cpu().numpy().copy() for x in o[:5]] + [_records(recs, cnt)])
        for k, name in enumerate(("obs", "reward", "terminated", "truncated", "terminal_obs", "records")):
            assert outs[0][k].tobytes() == outs[1][k].tobytes(), f"{name} at tick {t}"
        n_done += len(outs[0][5])
    assert a.num_timesteps == t0 + TICKS * N
    b.set_training_step_count(t0 + TICKS * N)
    assert a.get_current_intercept_radius() == b.get_current_intercept_radius()
    sa, sb = a.stats(), b.stats()
    assert sa == sb
    assert _state_equal(a, b)
    assert n_done > N   # many episodes ended, at many curriculum values
    assert not _state_equal(a, frozen) and a.stats() != frozen.stats()   # the curriculum decides outcomes here
    for s in sims:
        s.close()


# ---- GPU: graphs -----------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("increment", ["n", "3n+7"])
def test_step_graph_replays_continue_the_schedule(increment):
    import torch

    from hlynr_intercept_b200.sim import HlynrSim

    inc = N if increment == "n" else 3 * N + 7
    e = _ramps_cfg(unit=inc)
    a = HlynrSim(e, n_envs=N, seed=31, warn_dead=False)
    b = HlynrSim(e, n_envs=N, seed=31, warn_dead=False)
    t0 = 2 * inc + 5
    a.track_training_steps(t0, increment=inc)
    b.set_training_step_count(t0)
    a.reset(); b.reset()
    per = a.ring_period()
    T = per * max(1, 10 // per)
    g = torch.Generator(device="cuda")
    g.manual_seed(11)
    acts = [torch.rand(N, 6, device="cuda", generator=g) * 2 - 1 for _ in range(T)]
    tick = 0
    for x in acts:   # eager warm-up: every kernel loaded before the capture
        a.step(x)
        b.set_training_step_count(t0 + tick * inc); b.step(x)
        tick += 1
    graph = a.capture_steps(acts, want_terminal_obs=True)
    assert a.num_timesteps == t0 + tick * inc   # recording runs nothing
    R = 3
    for rep in range(R):
        out = graph.replay()
        for x in acts:
            b.set_training_step_count(t0 + tick * inc)
            ob = b.step(x)
            tick += 1
        torch.cuda.synchronize()
        for k in range(5):   # bytes: rows of terminal_obs no episode has written yet are NaN
            assert out[k].cpu().numpy().tobytes() == ob[k].cpu().numpy().tobytes(), (rep, k)
        assert a.num_timesteps == t0 + tick * inc
    assert tick == T * (R + 1)
    assert _state_equal(a, b) and a.stats() == b.stats()
    # get/set between replays: set the count back and replay; the twin pushes the same counts
    a.set_training_step_count(t0)
    graph.replay()
    for k, x in enumerate(acts):
        b.set_training_step_count(t0 + k * inc)
        ob = b.step(x)
    assert torch.equal(graph.out[0], ob[0]) and _state_equal(a, b)
    assert a.num_timesteps == t0 + T * inc
    a.close(); b.close()


@pytest.mark.gpu
def test_collector_replays_equal_host_pushed_eager_collects():
    """A captured DeviceRolloutCollector with FusedActorCritic on a tracking sim, replayed R times, equals R eager collects of a
    twin whose pipe.step pushes t0 + t * increment first; the fused policies have equal noise counters."""
    import torch

    from hlynr_intercept_b200.post import HlynrObsPipeline
    from hlynr_intercept_b200.rollout import DeviceRolloutCollector
    from test_obs_widths import _fused, _net_d

    from hlynr_intercept_b200.sim import HlynrSim

    inc = 2 * N + 1
    e = _ramps_cfg(unit=inc)
    t0 = 7 * inc
    net = _net_d(104, seed=45)
    cols = []
    for _ in range(2):
        sim = HlynrSim(e, n_envs=N, seed=19, warn_dead=False)
        pipe = HlynrObsPipeline(sim, n_stack=4, training=True)
        T = DeviceRolloutCollector(pipe, None, 1).graph_period() * 3
        cols.append(DeviceRolloutCollector(pipe, _fused(net, seed=77), T, bootstrap_rows=N))
    graphed, eager = cols
    graphed.sim.track_training_steps(t0, increment=inc)
    eager.sim.set_training_step_count(t0)
    clock = {"t": 0}
    step = eager.pipe.step

    def pushed_step(*args, **kw):
        eager.sim.set_training_step_count(t0 + clock["t"] * inc)
        clock["t"] += 1
        return step(*args, **kw)

    eager.pipe.step = pushed_step
    # INTEGRATION.md section 7's trainer loop: the collect capture() runs before recording is the first rollout
    model_num_timesteps = t0
    graphed.capture()   # one real collect (the warm-up) ...
    eager.collect()     # ... matched by one eager collect
    model_num_timesteps += T * inc
    assert graphed.sim.num_timesteps == model_num_timesteps
    R = 3
    for rep in range(R):
        graphed.replay()
        eager.collect()
        model_num_timesteps += T * inc
        torch.cuda.synchronize()
        for name in ("obs", "actions", "rewards", "values", "log_probs", "advantages", "returns", "episode_starts"):
            np.testing.assert_array_equal(getattr(graphed, name).cpu().numpy(), getattr(eager, name).cpu().numpy(),
                                          err_msg=f"{name} after replay {rep + 1}")
        assert graphed.sim.num_timesteps == model_num_timesteps == t0 + (rep + 2) * T * inc
    assert clock["t"] == (R + 1) * T
    assert _state_equal(graphed.sim, eager.sim)
    assert float(graphed.episode_starts[1:].sum()) > 0
    for c in cols:
        c.policy.close(); c.pipe.close(); c.sim.close()


# ---- GPU: surface ----------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_refused_calls_and_invalid_schedules():
    import torch

    from hlynr_intercept_b200 import _lib
    from hlynr_intercept_b200.sim import HlynrSim

    sim = HlynrSim(_ramps_cfg(), n_envs=64, seed=1, warn_dead=False)
    with pytest.raises(_lib.HlynrError, match="no curriculum schedule is attached"):
        sim.debug_curriculum_at(3)
    with pytest.raises(_lib.HlynrError, match="no curriculum schedule is attached"):
        _lib.check(sim.L.hlynr_set_timesteps(sim.h, 3, None))
    sched = sim.curriculum.schedule()
    for field, value in [("final_radius", float("nan")), ("beam_end", float("inf")), ("curriculum_steps", 0.0),
                         ("curriculum_steps", -5.0)]:
        s = abi.HlynrCurriculumSchedule.from_buffer_copy(sched)
        setattr(s, field, value)
        with pytest.raises(_lib.HlynrError, match="hlynr_attach_curriculum"):
            _lib.check(sim.L.hlynr_attach_curriculum(sim.h, C.byref(s), 0, sim.n))
    s = abi.HlynrCurriculumSchedule.from_buffer_copy(sched)
    s.enabled, s.curriculum_steps = 0, 0.0   # a disabled curriculum never divides
    _lib.check(sim.L.hlynr_attach_curriculum(sim.h, C.byref(s), 0, sim.n))
    _lib.check(sim.L.hlynr_detach_curriculum(sim.h))
    with pytest.raises(_lib.HlynrError, match="increment must not be negative"):
        sim.track_training_steps(0, increment=-1)
    assert not sim.tracking

    sim.track_training_steps(10 * N)
    with pytest.raises(_lib.HlynrError, match="hlynr_set_curriculum"):
        sim.push_curriculum()
    with pytest.raises(_lib.HlynrError, match="hlynr_rollout"):
        sim.rollout(4)
    obs = np.zeros((sim.n, 26), np.float32)
    with pytest.raises(_lib.HlynrError, match="hlynr_step_host"):
        _lib.check(sim.L.hlynr_step_host(sim.h, np.zeros((sim.n, 6), np.float32).ctypes.data_as(C.c_void_p),
                                         obs.ctypes.data_as(C.c_void_p), np.zeros(sim.n, np.float32).ctypes.data_as(C.c_void_p),
                                         np.zeros(sim.n, np.uint8).ctypes.data_as(C.c_void_p),
                                         np.zeros(sim.n, np.uint8).ctypes.data_as(C.c_void_p), None, 1))
    # get / set, and the radius read at the counter
    sim.set_training_step_count(50 * N)
    assert sim.num_timesteps == 50 * N
    assert sim.get_current_intercept_radius() == 200.0 * 0.5 + 5.0 * 0.5
    sim.reset()
    sim.step(torch.zeros(sim.n, 6, device="cuda"))
    reached = 50 * N + sim.n   # the default increment is the sim's own env count
    assert sim.num_timesteps == reached

    # detach: back to the by-value path, at the values of the count the device reached
    sim.untrack_training_steps()
    assert not sim.tracking and sim.num_timesteps == reached
    c = abi.HlynrCurriculum()
    _lib.check(sim.L.hlynr_get_curriculum(sim.h, C.byref(c)))
    host = config.resolve_config(_ramps_cfg(), warn_dead=False)[1]
    host.set_training_step_count(reached)
    assert config.Curriculum.as_dict(host) == {k: getattr(c, k) for k, _ in abi.HlynrCurriculum._fields_}
    sim.step(torch.zeros(sim.n, 6, device="cuda"))
    sim.rollout(4)   # allowed again
    with pytest.raises(_lib.HlynrError, match="no curriculum schedule is attached"):
        _lib.check(sim.L.hlynr_set_timesteps(sim.h, 3, None))
    sim.close()


@pytest.mark.gpu
def test_detached_sim_is_the_by_value_path():
    """Attach then detach: the steps that follow equal those of a twin that never attached."""
    import torch

    from hlynr_intercept_b200.sim import HlynrSim

    a = HlynrSim(_ramps_cfg(), n_envs=N, seed=41, warn_dead=False)
    b = HlynrSim(_ramps_cfg(), n_envs=N, seed=41, warn_dead=False)
    a.track_training_steps(12 * N)
    a.untrack_training_steps()
    b.set_training_step_count(12 * N)
    a.reset(); b.reset()
    g = torch.Generator(device="cuda")
    g.manual_seed(3)
    for _ in range(30):
        x = torch.rand(N, 6, device="cuda", generator=g) * 2 - 1
        oa, ob = a.step(x), b.step(x)
        assert torch.equal(oa[0], ob[0]) and torch.equal(oa[1], ob[1])
    assert a.num_timesteps == 12 * N and _state_equal(a, b)
    a.close(); b.close()

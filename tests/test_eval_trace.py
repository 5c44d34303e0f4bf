"""Trajectories of evaluated episodes on the device (hlynr_eval_trace, DeviceEvaluator.evaluate(trace=True)) and their episode
JSONL files (episode_log.write_episodes).

On the GPU, three twin sims with the same seed and statistics: one evaluated with trace=True, one without, and one stepped eagerly
through HlynrObsPipeline.step(..., info=...) by the restatement of SB3's evaluate_policy (tests/sb3_evaluation.py), where the host
builds every counted episode's rows from the tick's info arrays, clipped actions, rewards and done flags.  The traced and untraced
evaluations must agree bit for bit, and the device's rows must equal the host's byte for byte."""
import ctypes as C
import json

import numpy as np
import pytest

import sb3_evaluation
from test_evaluation import EPISODES, MAX_STEPS, N, _cfg, _check_twins, _close, _fused_predict, _mixed, _net, _pipes

MODES = {"eager": None, "graph_1x": 1, "graph_3x": 3}


# ---- CPU ------------------------------------------------------------------------------------------------------------------------

def test_trace_row_dtype_matches_the_library():
    from hlynr_intercept_b200 import _lib, abi

    L = _lib.load()
    dt = abi.trace_row_numpy_dtype()
    assert dt.itemsize == L.hlynr_trace_row_size() == 72
    assert "hlynr_eval_trace" in _lib.EXPORTS and hasattr(L, "hlynr_eval_trace")


def test_eval_trace_rejects_bad_arguments():
    """Argument checks of the C entry point, before any device work."""
    from hlynr_intercept_b200 import _lib, abi

    L = _lib.load()
    p = C.c_void_p(256)
    full = abi.HlynrInfoSoA(**{k: 256 for k in abi.TRACE_INFO_FIELDS})

    def call(info=full, ptrs=(p,) * 5, n=4, E=5, max_steps=10, table=p):
        return L.hlynr_eval_trace(None if info is None else C.byref(info), *ptrs, n, E, max_steps, table, 0, None)

    for n, E, msg in ((4, 0, b"n_episodes"), (4, -1, b"n_episodes"), (4, 2**31, b"n_episodes"), (0, 5, b"n_envs"),
                      (2**31, 5, b"n_envs")):
        assert call(n=n, E=E) != 0
        assert msg in L.hlynr_last_error()
    assert call(max_steps=0) != 0 and b"max_steps" in L.hlynr_last_error()
    assert call(info=None) != 0 and b"null argument" in L.hlynr_last_error()
    assert call(table=None) != 0 and b"null argument" in L.hlynr_last_error()
    for k in range(5):
        ptrs = [p] * 5
        ptrs[k] = None
        assert call(ptrs=tuple(ptrs)) != 0 and b"null argument" in L.hlynr_last_error()
    for field in abi.TRACE_INFO_FIELDS:
        partial = abi.HlynrInfoSoA(**{k: 256 for k in abi.TRACE_INFO_FIELDS if k != field})
        assert call(info=partial) != 0 and b"null argument" in L.hlynr_last_error(), field


def _hand_result():
    """Three episodes: intercepted after 3 ticks, truncated after 2, terminated (failed) after 1."""
    from hlynr_intercept_b200 import abi
    from hlynr_intercept_b200.evaluation import EvalResult

    lengths = [3, 2, 1]
    rows = np.zeros(sum(lengths), dtype=abi.trace_row_numpy_dtype())
    rows["step"] = [1, 2, 3, 1, 2, 1]
    rows["reward"] = np.array([0.1, -0.25, 10.3, 1e-3, 2.5, -7.75], np.float32)
    rows["distance"] = np.array([90.5, 12.25, 30.0, 400.0, 410.5, 55.0], np.float32)
    rows["fuel_remaining"] = np.array([99.5, 99.0, 98.25, 100.0, 99.75, 42.0], np.float32)
    rows["interceptor_pos"] = np.arange(18, dtype=np.float32).reshape(6, 3) * np.float32(1.1)
    rows["missile_pos"] = np.arange(18, dtype=np.float32).reshape(6, 3) * np.float32(-0.3)
    rows["action"] = np.linspace(-1, 1, 36, dtype=np.float32).reshape(6, 6)
    rows["flags"] = [abi.INFO_RADAR_DETECTED, abi.INFO_RADAR_DETECTED, abi.INFO_INTERCEPTED | abi.DONE_TERMINATED, 0,
                     abi.DONE_TRUNCATED, abi.DONE_TERMINATED]
    recs = np.zeros(3, dtype=abi.done_record_numpy_dtype())
    recs["steps"] = lengths
    recs["fuel_used"] = np.array([1.75, 0.25, 58.0], np.float32)
    recs["flags"] = [abi.INFO_INTERCEPTED | abi.DONE_TERMINATED, abi.DONE_TRUNCATED, abi.DONE_TERMINATED]
    return EvalResult(records=recs, end_tick=np.array([3, 2, 1]), episode_rewards=np.zeros(3), episode_lengths=np.array(lengths, np.int32),
                      mean_reward=0.0, std_reward=0.0, success_rate=1 / 3, mean_min_distance=0.0, mean_fuel_used=0.0, ticks=3,
                      trajectories=rows, trajectory_offsets=np.array([0, 3, 5, 6], np.int64))


def test_write_episodes_writes_the_recorder_lines(tmp_path):
    from hlynr_intercept_b200.episode_log import write_episodes

    res, dt = _hand_result(), 0.01
    paths = write_episodes(str(tmp_path), res, dt, metadata={"scenario": "easy"})
    assert [p.split("/")[-1] for p in paths] == ["ep_000001.jsonl", "ep_000002.jsonl", "ep_000003.jsonl"]
    rows, off = res.trajectories, res.trajectory_offsets
    want_outcome = ["intercepted", "failed", "failed"]
    for i, path in enumerate(paths):
        lines = [json.loads(x) for x in open(path)]
        ep = rows[off[i]:off[i + 1]]
        l = len(ep)
        assert len(lines) == 1 + 2 * l + 1
        head, foot, states = lines[0], lines[-1], lines[1:-1]
        assert head["type"] == "header" and head["episode_id"] == f"ep_{i + 1:06d}" and head["metadata"] == {"scenario": "easy"}
        for k in range(l):
            it, ms = states[2 * k], states[2 * k + 1]
            assert it == {"type": "state", "timestamp": k * dt, "entity_id": "interceptor",
                          "state": {"position": ep["interceptor_pos"][k].tolist(), "fuel": float(ep["fuel_remaining"][k]),
                                    "action": ep["action"][k].tolist()}}
            assert ms == {"type": "state", "timestamp": k * dt, "entity_id": "missile", "state": {"position": ep["missile_pos"][k].tolist()}}
        total = 0.0
        for r in ep["reward"]:
            total += float(r)
        assert foot["type"] == "footer" and foot["episode_id"] == head["episode_id"] and foot["outcome"] == want_outcome[i]
        assert foot["metrics"] == {"total_reward": total, "steps": l, "final_distance": float(ep["distance"][-1]),
                                   "min_distance": float(ep["distance"].min()), "fuel_used": float(res.records["fuel_used"][i])}
        assert foot["duration"] == l * dt and foot["end_time"] == head["start_time"] + l * dt
    assert json.loads(open(paths[0]).readlines()[-1])["metrics"]["min_distance"] == np.float32(12.25)


def test_write_episodes_refuses_an_untraced_result(tmp_path):
    from hlynr_intercept_b200.episode_log import write_episodes

    res = _hand_result()
    res.trajectories = res.trajectory_offsets = None
    with pytest.raises(ValueError, match="trace=True"):
        write_episodes(str(tmp_path), res, 0.01)


# ---- GPU ------------------------------------------------------------------------------------------------------------------------

def _third(pipes, frame_dim=26, n_stack=4, seed=17, cfg=None):
    """A third twin of _pipes(): same seed, the same statistics."""
    from hlynr_intercept_b200.evaluation import sync_normalization
    from hlynr_intercept_b200.post import HlynrObsPipeline
    from hlynr_intercept_b200.sim import HlynrSim

    sim = HlynrSim(cfg, n_envs=N, seed=seed, warn_dead=False, obs_dim=frame_dim)
    pipe = HlynrObsPipeline(sim, n_stack=n_stack, training=False)
    sync_normalization(pipes[0], pipe)
    return pipe


def _traced_restatement(pipe, predict, E, pad_to):
    """evaluate_policy restated on an eager twin stepped with info arrays; the host builds each tick's rows.  Returns (rows of
    the counted episodes in SB3's order, their (env, first tick, last tick) spans, per-tick float32 interceptor / missile
    positions and fuel of the twin's state after each tick)."""
    import torch

    from hlynr_intercept_b200 import abi

    n, dev = pipe.sim.n, pipe.sim.device
    tt = {"float32": torch.float32, "int32": torch.int32, "uint8": torch.uint8}
    info = {k: torch.zeros((n,) + shp, dtype=tt[d], device=dev) for k, d, shp in abi.INFO_FIELDS if k in abi.TRACE_INFO_FIELDS}
    ticks, states, start = [], [], np.zeros(n, dtype=np.int64)
    obs_box = {}

    def step_fn(actions):
        act = actions.float().contiguous().cpu().numpy()
        obs, rew, te, tr, _ = pipe.step(actions, info=info)
        h = {k: v.cpu().numpy() for k, v in info.items()}
        te, tr = te.cpu().numpy().astype(bool), tr.cpu().numpy().astype(bool)
        row = np.zeros(n, dtype=abi.trace_row_numpy_dtype())
        row["interceptor_pos"], row["missile_pos"], row["action"] = h["interceptor_pos"], h["missile_pos"], act
        row["reward"], row["distance"] = rew.cpu().numpy(), h["distance"]
        row["fuel_remaining"], row["radar_quality"] = h["fuel_remaining"], h["radar_quality"]
        row["flags"] = h["flags"].astype(np.uint32) | np.where(te, abi.DONE_TERMINATED, 0) | np.where(tr, abi.DONE_TRUNCATED, 0)
        row["step"] = h["steps"]
        t = len(ticks)
        ticks.append(row)
        s = pipe.sim.export_state()
        states.append((s["ipos"].astype(np.float32), s["mpos"].astype(np.float32), s["fuel"].astype(np.float32)))
        dones = te | tr
        infos = [{} for _ in range(n)]
        for e in np.flatnonzero(dones).tolist():
            infos[e] = {"episode": {"r": 0.0, "l": 0}, "span": (e, int(start[e]), t)}
        start[dones] = t + 1
        obs_box["obs"] = obs
        return obs, dones, infos

    _, _, infos = sb3_evaluation.evaluate_policy(pipe.reset, step_fn, predict, n, E)
    obs = obs_box["obs"]
    assert pad_to >= len(ticks)
    for _ in range(pad_to - len(ticks)):   # SB3's envs past their quota keep stepping: the twins end in the same state
        obs = pipe.step(predict(obs))[0]
    table = np.stack(ticks)   # [T, N]
    spans = [i["span"] for i in infos]
    rows = np.concatenate([table[s:t + 1, e] for e, s, t in spans])
    return rows, spans, states


def _check_trace(res, ref, E):
    """The device's rows equal the host's; per-episode invariants against the done records and the twin's states."""
    from hlynr_intercept_b200 import abi

    rows, spans, states = ref
    lengths = res.episode_lengths.astype(np.int64)
    assert res.trajectory_offsets.dtype == np.int64 and res.trajectory_offsets.shape == (E + 1,)
    np.testing.assert_array_equal(res.trajectory_offsets, np.concatenate([[0], np.cumsum(lengths)]))
    assert [t - s + 1 for _, s, t in spans] == lengths.tolist()
    assert res.trajectories.dtype == abi.trace_row_numpy_dtype() and len(res.trajectories) == lengths.sum()
    assert res.trajectories.tobytes() == rows.tobytes()
    off, tr = res.trajectory_offsets, res.trajectories
    for i, (rec, (e, s, t)) in enumerate(zip(res.records, spans)):
        assert rec["env"] == e
        ep = tr[off[i]:off[i + 1]]
        np.testing.assert_array_equal(ep["step"], np.arange(1, len(ep) + 1))
        last = ep[-1]
        for k in ("interceptor_pos", "missile_pos", "fuel_remaining", "distance"):
            assert np.array_equal(last[k], rec[k]), (i, k)
        assert last["flags"] & 0xFF == rec["flags"] & 0xFF
        assert last["flags"] & 0x300 == rec["flags"] & 0x300 != 0
        assert (ep["flags"][:-1] & 0x300 == 0).all()
        for k in range(len(ep) - 1):   # non-terminal ticks: what EpisodeRecorder reads from export_state
            ipos, mpos, fuel = states[s + k]
            assert np.array_equal(ep["interceptor_pos"][k], ipos[e]) and np.array_equal(ep["missile_pos"][k], mpos[e])
            assert ep["fuel_remaining"][k] == fuel[e]


def _check_same(a, b):
    """A traced and an untraced evaluation of twin sims: everything but the trajectories bit for bit."""
    assert a.records.tobytes() == b.records.tobytes()
    np.testing.assert_array_equal(a.end_tick, b.end_tick)
    assert a.episode_rewards.tobytes() == b.episode_rewards.tobytes()
    assert a.episode_lengths.tobytes() == b.episode_lengths.tobytes()
    assert (a.ticks, a.mean_reward, a.std_reward, a.success_rate) == (b.ticks, b.mean_reward, b.std_reward, b.success_rate)
    assert b.trajectories is None and b.trajectory_offsets is None


def _run3(pipes, third, policies, predict, E, mode, deterministic=True):
    """Traced evaluation on pipes[0], untraced on pipes[1], the traced restatement on `third`; all three compared."""
    from hlynr_intercept_b200.evaluation import DeviceEvaluator
    from hlynr_intercept_b200.rollout import graph_period

    mult = MODES[mode]
    chunk = None if mult is None else mult * graph_period(pipes[0])
    graph = mode != "eager"
    evs = [DeviceEvaluator(p, pol, chunk=chunk) for p, pol in zip(pipes, policies)]
    res = evs[0].evaluate(E, graph=graph, deterministic=deterministic, trace=True)
    plain = evs[1].evaluate(E, graph=graph, deterministic=deterministic)
    _check_same(res, plain)
    _check_twins(*pipes)
    ref = _traced_restatement(third, predict, E, res.ticks)
    _check_trace(res, ref, E)
    _check_twins(pipes[0], third)
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("episodes", ["37", "N", "2.5N"])
def test_traced_evaluation_equals_untraced_and_restatement(episodes, mode):
    from hlynr_intercept_b200.policy import FusedActorCritic

    E = EPISODES[episodes]
    cfg = _cfg()
    pipes = _pipes(cfg)
    third = _third(pipes, cfg=cfg)
    fused = FusedActorCritic(_net(104), device=0)
    res = _run3(pipes, third, [fused, fused], _fused_predict(fused), E, mode)
    if E >= N:
        _mixed(res)
    _close(fused, *pipes, third)


@pytest.mark.gpu
def test_volley_trace():
    """A volley of 3: the row's distance is the priority missile's, as in the done record."""
    from hlynr_intercept_b200.policy import FusedActorCritic

    cfg = _cfg(volley=True)
    pipes = _pipes(cfg, seed=31)
    third = _third(pipes, seed=31, cfg=cfg)
    assert third.sim.params.volley_size == 3
    fused = FusedActorCritic(_net(104, seed=8), device=0)
    res = _run3(pipes, third, [fused, fused], _fused_predict(fused), EPISODES["2.5N"], "graph_1x")
    assert len(np.unique(res.records["missiles_intercepted"])) > 1
    _close(fused, *pipes, third)


@pytest.mark.gpu
def test_trace_of_17d_frames_with_the_68_wide_policy():
    from hlynr_intercept_b200.policy import FusedActorCritic

    cfg = _cfg()
    pipes = _pipes(cfg, frame_dim=17, n_stack=4, seed=29)
    third = _third(pipes, frame_dim=17, n_stack=4, seed=29, cfg=cfg)
    fused = FusedActorCritic(_net(68, seed=7), device=0)
    res = _run3(pipes, third, [fused, fused], _fused_predict(fused), EPISODES["2.5N"], "graph_3x")
    _mixed(res)
    _close(fused, *pipes, third)


@pytest.mark.gpu
def test_stochastic_trace():
    """deterministic=False: three handles at the same noise counter draw the same samples."""
    import torch

    from hlynr_intercept_b200.policy import FusedActorCritic

    cfg = _cfg()
    pipes = _pipes(cfg, seed=41)
    third = _third(pipes, seed=41, cfg=cfg)
    net = _net(104, seed=10)
    hs = [FusedActorCritic(net, device=0, seed=77) for _ in range(3)]
    for h in hs:
        h.calls = 1000
    buf = torch.empty(N, 6, device="cuda")

    def sample(obs):
        hs[2].forward(obs, deterministic=False, want=(), out=dict(clipped=buf))
        return buf

    res = _run3(pipes, third, hs[:2], sample, EPISODES["N"], "graph_1x", deterministic=False)
    _mixed(res)
    assert hs[0].calls == hs[1].calls == hs[2].calls
    _close(*hs, *pipes, third)


@pytest.mark.gpu
def test_written_files_of_a_gpu_result(tmp_path):
    """The files of a traced GPU evaluation pass EpisodeRecorder's format checks (tests/test_rollout.py)."""
    from hlynr_intercept_b200.episode_log import write_episodes
    from hlynr_intercept_b200.evaluation import DeviceEvaluator
    from hlynr_intercept_b200.policy import FusedActorCritic

    pipes = _pipes(_cfg(), seed=43)
    fused = FusedActorCritic(_net(104, seed=11), device=0)
    res = DeviceEvaluator(pipes[0], fused).evaluate(64, trace=True)
    dt = float(pipes[0].sim.params.dt)
    paths = write_episodes(str(tmp_path), res, dt, metadata={"scenario": "medium"})
    assert len(paths) == 64
    for i, path in enumerate(paths):
        l = int(res.episode_lengths[i])
        assert 1 <= l <= MAX_STEPS
        lines = [json.loads(x) for x in open(path)]
        assert lines[0]["type"] == "header" and lines[0]["metadata"] == {"scenario": "medium"}
        states = [x for x in lines if x["type"] == "state"]
        assert len(states) == 2 * l and {x["entity_id"] for x in states} == {"interceptor", "missile"}
        assert len(states[0]["state"]["position"]) == 3 and len(states[0]["state"]["action"]) == 6
        assert states[-1]["timestamp"] == (l - 1) * dt
        foot = lines[-1]
        assert foot["type"] == "footer" and foot["outcome"] in ("intercepted", "failed") and foot["metrics"]["steps"] == l
        assert foot["outcome"] == ("intercepted" if res.records["flags"][i] & 1 else "failed")
        assert np.float32(foot["metrics"]["final_distance"]) == res.records["distance"][i]
        assert foot["metrics"]["min_distance"] == float(res.trajectories["distance"][res.trajectory_offsets[i]:][:l].min())
    _close(fused, *pipes)

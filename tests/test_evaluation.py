"""Policy evaluation on the device (hlynr_intercept_b200/evaluation.py over hlynr_eval_record) against the numpy restatement
of SB3's evaluate_policy (tests/sb3_evaluation.py).

The restatement runs on a twin sim with the same seed, stepped eagerly through HlynrObsPipeline.step and done_records() with
the same policy's deterministic clipped action; after it, the twin keeps stepping to the evaluator's tick count (SB3's envs
past their quota keep stepping too), so the two sims must also end in the same state.  Everything is compared bit for bit:
the done records, the step each episode ended on, the order, rewards, lengths, mean and std."""
import ctypes as C

import numpy as np
import pytest

import sb3_evaluation
from hlynr_intercept_b200 import config

N = 1037   # a ragged tile
MAX_STEPS = 40
EPISODES = {"37": 37, "N": N, "2.5N": 5 * N // 2, "3N": 3 * N}


# ---- CPU ------------------------------------------------------------------------------------------------------------------------

def _offsets(n, E):
    """offset_e of hlynr_eval_record (include/hlynr_rollout.h): where env e's results start in the table."""
    q, rem = divmod(E, n)
    e = np.arange(n, dtype=np.int64)
    return e * q + np.maximum(0, e - (n - rem))


@pytest.mark.parametrize("n", [1, 2, 3, 7, 64, 1037, 4096])
def test_quota_offsets_are_prefix_sums_of_the_targets(n):
    for E in sorted({1, max(n - 1, 1), n, n + 1, 5 * n // 2, 7 * n}):
        t = sb3_evaluation.episode_count_targets(n, E)
        assert t.sum() == E, (n, E)
        np.testing.assert_array_equal(_offsets(n, E), np.concatenate([[0], np.cumsum(t)[:-1]]), err_msg=f"n={n} E={E}")


# step -> {env: (r, l)}: the episodes of a 3-env run that end on that step (listed out of env order on purpose)
_SCRIPT = {1: {0: (10.5, 1)}, 2: {2: (22.25, 2), 1: (21.0, 2)}, 3: {0: (30.0, 2)}, 4: {2: (42.0, 2)},
           5: {1: (51.0, 3), 0: (50.0, 2)}, 6: {2: (62.0, 2)}, 7: {0: (70.0, 2), 1: (71.0, 2), 2: (72.0, 1)}}


@pytest.mark.parametrize("E,rewards,lengths,steps", [
    # targets (0, 1, 1): only the last two envs count; env 0 finishes on step 1 with a quota of 0; envs 1 and 2 on one step
    (2, [21.0, 22.25], [2, 2], 2),
    # targets (1, 1, 2): env 0's episode of step 3 is past its quota
    (4, [10.5, 21.0, 22.25, 42.0], [1, 2, 2, 2], 4),
    # targets (2, 2, 3): on step 5 env 0 is past its quota and env 1 is not
    (7, [10.5, 21.0, 22.25, 30.0, 42.0, 51.0, 62.0], [1, 2, 2, 2, 2, 3, 2], 6),
])
def test_restated_evaluate_policy_on_a_script(E, rewards, lengths, steps):
    n, clock, seen = 3, [0], []

    def reset_fn():
        return np.zeros(n)

    def step_fn(actions):
        clock[0] += 1
        ends = _SCRIPT[clock[0]]
        infos = [{"episode": {"r": ends[e][0], "l": ends[e][1]}, "env": e} if e in ends else {} for e in range(n)]
        return np.full(n, float(clock[0])), np.array([e in ends for e in range(n)]), infos

    def predict(obs):
        seen.append(float(obs[0]))
        return obs

    r, l, infos = sb3_evaluation.evaluate_policy(reset_fn, step_fn, predict, n, E)
    assert (r, l) == (rewards, lengths)
    assert [i["episode"]["r"] for i in infos] == rewards
    assert clock[0] == steps and seen == [float(s) for s in range(steps)]


def test_sync_normalization_copies_the_statistics_of_the_same_layout():
    """All six statistics go through unchanged; a pipeline of another width, stack depth, clip or epsilon is refused."""
    import types

    from hlynr_intercept_b200.evaluation import sync_normalization

    stats = dict(mean=np.linspace(-1, 1, 104), var=np.linspace(0.5, 2, 104), count=1234.5, ret_mean=0.25, ret_var=3.5,
                 ret_count=77.0)

    def fake(**kw):
        attrs = dict(obs_dim=104, n_stack=4, clip_obs=10.0, epsilon=1e-8, got=[])
        attrs.update(kw)
        return types.SimpleNamespace(get_stats=lambda: stats, set_stats=lambda *a: attrs["got"].append(a), **attrs)

    dst = fake()
    sync_normalization(fake(), dst)
    assert len(dst.got) == 1
    for got, want in zip(dst.got[0], [stats[k] for k in ("mean", "var", "count", "ret_mean", "ret_var", "ret_count")]):
        assert np.array_equal(got, want)
    for k, v in (("obs_dim", 68), ("n_stack", 2), ("clip_obs", 5.0), ("epsilon", 1e-6)):
        dst = fake(**{k: v})
        with pytest.raises(ValueError, match=k):
            sync_normalization(fake(), dst)
        assert dst.got == []


def test_eval_record_rejects_bad_arguments():
    """Argument checks of the C entry point, before any device work."""
    from hlynr_intercept_b200 import _lib

    L = _lib.load()
    p = C.c_void_p(256)
    for n, E, msg in ((4, 0, b"n_episodes"), (4, -1, b"n_episodes"), (4, 2**31, b"n_episodes"), (0, 5, b"n_envs"),
                      (2**31, 5, b"n_envs")):
        assert L.hlynr_eval_record(p, p, n, E, p, p, p, p, p, 0, None) != 0
        assert msg in L.hlynr_last_error()
    assert L.hlynr_eval_record(p, p, 4, 5, p, None, p, p, p, 0, None) != 0
    assert b"null argument" in L.hlynr_last_error()


# ---- GPU ------------------------------------------------------------------------------------------------------------------------

def _cfg(volley=False):
    e = config.baseline_config("cfg4")
    e["max_steps"] = MAX_STEPS
    # missiles spawn 170-430 m from the interceptor, around the 200 m initial intercept radius and closing at ~300 m/s, and a
    # third of the interceptors start downwards from at most 10 m: intercepts, crashes and truncations at mixed lengths
    e["missile_spawn"] = dict(position=[[150, 150, 100], [260, 260, 220]], velocity=[[-110, -110, -55], [-160, -160, -75]])
    e["interceptor_spawn"] = dict(position=[[0, 0, 0], [50, 50, 10]], velocity=[[20, 20, -40], [40, 40, 80]])
    if volley:
        e.update(volley_mode=True, volley_size=3)
    return e


def _pipes(cfg, frame_dim=26, n_stack=4, seed=17):
    """Twin eval pipelines (training=False) whose statistics come from a short training run through sync_normalization."""
    import torch

    from hlynr_intercept_b200.evaluation import sync_normalization
    from hlynr_intercept_b200.post import HlynrObsPipeline
    from hlynr_intercept_b200.sim import HlynrSim

    tsim = HlynrSim(cfg, n_envs=N, seed=seed + 1000, warn_dead=False, obs_dim=frame_dim)
    train = HlynrObsPipeline(tsim, n_stack=n_stack, training=True)
    train.reset()
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    for _ in range(25):
        train.step(torch.rand(N, 6, device="cuda", generator=g) * 2 - 1)
    src = train.get_stats()
    pipes = []
    for _ in range(2):
        sim = HlynrSim(cfg, n_envs=N, seed=seed, warn_dead=False, obs_dim=frame_dim)
        pipe = HlynrObsPipeline(sim, n_stack=n_stack, training=False)
        sync_normalization(train, pipe)
        _assert_stats_equal(pipe.get_stats(), src)
        pipes.append(pipe)
    train.close()
    tsim.close()
    return pipes


def _assert_stats_equal(a, b):
    assert sorted(a) == sorted(b) == ["count", "mean", "ret_count", "ret_mean", "ret_var", "var"]
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def _fused_predict(fused):
    import torch

    buf = torch.empty(N, 6, device="cuda")

    def predict(obs):
        fused.forward(obs, deterministic=True, want=(), out=dict(clipped=buf))
        return buf

    return predict


def _torch_predict(net):
    import torch

    def predict(obs):
        with torch.no_grad():
            return net.mean(obs).float().clamp(-1.0, 1.0)

    return predict


def _restated(pipe, predict, E, pad_to):
    """evaluate_policy restated on `pipe`, then steps up to `pad_to` ticks in all.  Returns (rewards, lengths, records in
    append order, the step each ended on, ticks of the restated loop)."""
    from hlynr_intercept_b200 import abi

    n, clock = pipe.sim.n, {"t": 0}

    def step_fn(actions):
        obs = pipe.step(actions)[0]
        clock["t"] += 1
        clock["obs"] = obs
        rec = pipe.done_records()
        dones = np.zeros(n, dtype=bool)
        dones[rec["env"]] = True
        ret = rec["episode_return"].astype(np.float64).round(6).tolist()   # Monitor 'r' as HlynrVecEnv reports it
        infos = [{} for _ in range(n)]
        for k, e in enumerate(rec["env"].tolist()):
            infos[e] = {"episode": {"r": ret[k], "l": int(rec["steps"][k])}, "record": rec[k], "tick": clock["t"]}
        return obs, dones, infos

    r, l, infos = sb3_evaluation.evaluate_policy(pipe.reset, step_fn, predict, n, E)
    ticks, obs = clock["t"], clock["obs"]
    assert pad_to >= ticks
    for _ in range(pad_to - ticks):
        obs = pipe.step(predict(obs))[0]
    recs = np.array([i["record"] for i in infos], dtype=abi.done_record_numpy_dtype())
    return r, l, recs, np.array([i["tick"] for i in infos], dtype=np.int64), ticks


def _check(res, ref, E, graph, chunk):
    from hlynr_intercept_b200 import abi

    r, l, recs, ends, ticks = ref
    assert len(r) == E and len(res.records) == E
    np.testing.assert_array_equal(res.end_tick, ends)
    assert res.records.tobytes() == recs.tobytes()   # every field, terminal_obs and the volley counters included
    assert res.episode_rewards.tolist() == r and res.episode_lengths.tolist() == l
    assert res.mean_reward == np.mean(r) and res.std_reward == np.std(r)
    assert ticks == ends.max()
    assert res.ticks == (-(-ticks // chunk) * chunk if graph else ticks)
    assert res.success_rate == np.mean((recs["flags"] & abi.INFO_INTERCEPTED) != 0)
    assert res.mean_min_distance == np.mean(recs["min_distance"].astype(np.float64))
    assert res.mean_fuel_used == np.mean(recs["fuel_used"].astype(np.float64))


def _check_twins(ev_pipe, ref_pipe):
    se, sr = ev_pipe.sim.export_state(), ref_pipe.sim.export_state()
    for k in se:
        assert np.array_equal(se[k], sr[k]), k
    assert ev_pipe.sim.tick_count() == ref_pipe.sim.tick_count()


def _mixed(res):
    """The configuration ends episodes at many lengths, by termination and by truncation."""
    from hlynr_intercept_b200 import abi

    fl = res.records["flags"]
    assert len(np.unique(res.episode_lengths)) >= 8, np.unique(res.episode_lengths)
    assert ((fl & abi.DONE_TERMINATED) != 0).any() and ((fl & abi.DONE_TRUNCATED) != 0).any()


def _run(pipes, policy, predict, E, graph, chunk_mult=None):
    from hlynr_intercept_b200.evaluation import DeviceEvaluator
    from hlynr_intercept_b200.rollout import graph_period

    ev_pipe, ref_pipe = pipes
    chunk = None if chunk_mult is None else chunk_mult * graph_period(ev_pipe)
    ev = DeviceEvaluator(ev_pipe, policy, chunk=chunk)
    before = ev_pipe.get_stats()
    res = ev.evaluate(E, graph=graph)
    _assert_stats_equal(ev_pipe.get_stats(), before)
    ref = _restated(ref_pipe, predict, E, res.ticks)
    _check(res, ref, E, graph, ev.chunk)
    _check_twins(ev_pipe, ref_pipe)
    return ev, res


def _close(*objs):
    for o in objs:
        sim = getattr(o, "sim", None)
        o.close()
        if sim is not None:
            sim.close()


def _net(d, seed=5):
    from test_obs_widths import _net_d

    return _net_d(d, seed=seed)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["eager", "graph_1x", "graph_3x"])
@pytest.mark.parametrize("episodes", list(EPISODES))
def test_fused_policy_evaluation_equals_restatement(episodes, mode):
    from hlynr_intercept_b200.policy import FusedActorCritic

    E = EPISODES[episodes]
    pipes = _pipes(_cfg())
    fused = FusedActorCritic(_net(104), device=0)
    graph = mode != "eager"
    _, res = _run(pipes, fused, _fused_predict(fused), E, graph, {"eager": None, "graph_1x": 1, "graph_3x": 3}[mode])
    if E >= N:
        _mixed(res)
    else:   # E < N: only the last E envs are evaluated, one episode each
        assert sorted(res.records["env"].tolist()) == list(range(N - E, N))
    _close(fused, *pipes)


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [True, False])
def test_torch_policy_evaluation_equals_restatement(graph):
    pipes = _pipes(_cfg(), seed=23)
    net = _net(104, seed=6)
    _, res = _run(pipes, net, _torch_predict(net), EPISODES["2.5N"], graph)
    _mixed(res)
    _close(*pipes)


@pytest.mark.gpu
@pytest.mark.parametrize("frame_dim,n_stack", [(17, 4), (26, 2)])
def test_other_observation_layouts(frame_dim, n_stack):
    """17-D/4 with the 68-wide fused policy, 26-D/2 with the 52-wide one."""
    from hlynr_intercept_b200.policy import FusedActorCritic

    pipes = _pipes(_cfg(), frame_dim=frame_dim, n_stack=n_stack, seed=29)
    fused = FusedActorCritic(_net(frame_dim * n_stack, seed=7), device=0)
    _, res = _run(pipes, fused, _fused_predict(fused), EPISODES["2.5N"], True)
    _mixed(res)
    _close(fused, *pipes)


@pytest.mark.gpu
def test_volley_evaluation_equals_restatement():
    from hlynr_intercept_b200.policy import FusedActorCritic

    pipes = _pipes(_cfg(volley=True), seed=31)
    assert pipes[0].sim.params.volley_size == 3
    fused = FusedActorCritic(_net(104, seed=8), device=0)
    _, res = _run(pipes, fused, _fused_predict(fused), EPISODES["2.5N"], True)
    mi = res.records["missiles_intercepted"]
    assert mi.max() > 0 and len(np.unique(mi)) > 1, np.unique(mi)
    _close(fused, *pipes)


@pytest.mark.gpu
def test_second_evaluate_equals_second_restatement():
    """A second evaluate() on the same evaluator (a new reset, a new graph) against a second restatement on the twin."""
    from hlynr_intercept_b200.policy import FusedActorCritic

    pipes = _pipes(_cfg(), seed=37)
    fused = FusedActorCritic(_net(104, seed=9), device=0)
    predict = _fused_predict(fused)
    ev, _ = _run(pipes, fused, predict, N + 1, True)
    for E in (2 * N, 37):
        res = ev.evaluate(E)
        _check(res, _restated(pipes[1], predict, E, res.ticks), E, True, ev.chunk)
        _check_twins(*pipes)
    _close(fused, *pipes)


@pytest.mark.gpu
def test_invalid_input_is_refused():
    import torch

    from hlynr_intercept_b200.evaluation import DeviceEvaluator
    from hlynr_intercept_b200.policy import FusedActorCritic
    from hlynr_intercept_b200.post import HlynrObsPipeline
    from hlynr_intercept_b200.rollout import graph_period
    from hlynr_intercept_b200.sim import HlynrSim

    sim = HlynrSim(_cfg(), n_envs=64, seed=1, warn_dead=False)
    pipe = HlynrObsPipeline(sim, n_stack=4, training=True)
    fused = FusedActorCritic(_net(104), device=0)
    with pytest.raises(ValueError, match="training=False"):
        DeviceEvaluator(pipe, fused)
    pipe.training = False
    narrow = FusedActorCritic(_net(68), device=0)
    with pytest.raises(ValueError, match="68-wide"):
        DeviceEvaluator(pipe, narrow)
    with pytest.raises(ValueError, match="52-wide"):
        DeviceEvaluator(pipe, _net(52))
    with pytest.raises(ValueError, match="mean"):
        DeviceEvaluator(pipe, torch.nn.Linear(104, 6).cuda())
    with pytest.raises(ValueError, match="multiple"):
        DeviceEvaluator(pipe, fused, chunk=graph_period(pipe) + 1)
    ev = DeviceEvaluator(pipe, fused)
    assert ev.chunk % graph_period(pipe) == 0 and ev.chunk >= 16 and ev.chunk - graph_period(pipe) < 16
    for E in (0, -3, 2**31):
        with pytest.raises(ValueError, match="n_eval_episodes"):
            ev.evaluate(E)
    _close(fused, narrow, pipe)


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [True, False])
def test_unfinished_evaluation_raises_instead_of_spinning(graph):
    """With a host-side max_steps below the device's, the quotas cannot be met within the bound: evaluate() raises."""
    from hlynr_intercept_b200.evaluation import DeviceEvaluator
    from hlynr_intercept_b200.policy import FusedActorCritic
    from hlynr_intercept_b200.post import HlynrObsPipeline
    from hlynr_intercept_b200.sim import HlynrSim

    cfg = config.baseline_config("cfg4")
    cfg["max_steps"] = 200   # cfg4's spawn: no episode ends before it truncates
    sim = HlynrSim(cfg, n_envs=N, seed=3, warn_dead=False)
    pipe = HlynrObsPipeline(sim, n_stack=4, training=False)
    fused = FusedActorCritic(_net(104), device=0)
    ev = DeviceEvaluator(pipe, fused)
    sim.params.max_steps = 5
    with pytest.raises(RuntimeError, match="still unfinished"):
        ev.evaluate(N, graph=graph)
    _close(fused, pipe)

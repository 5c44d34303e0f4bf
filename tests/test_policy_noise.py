"""The fused policy's noise counter on the device (hlynr_policy_forward_dev, hlynr_policy_set_counter / get_counter).

Every forward draws eps at counter c = *counter + 1 and stores c, whatever kind of call it is, so a forward captured in a CUDA
graph draws fresh noise on every replay.  Checked here:
  (a) the counter semantics: set / get round trips; each forward of a mixed sequence (stochastic, deterministic, value only,
      n_rows_dev = 0, 3 and > n) advances `calls` by exactly one, at 1 ... 131 149 rows, cluster 1 / 2 / 4, in_dim 104 and 68,
      and every stochastic output is Philox at the new counter (eps_ref, the 16-ulp bounds of test_policy_reference);
  (b) the device-counter entry and hlynr_policy_forward at the same counter give the same bits, and the by-value entry leaves
      the device counter alone;
  (c) a captured sequence of forwards replayed 3 times equals 15 eager forwards on a twin handle, bit for bit;
  (d) rollout replays equal eager collects bit for bit and draw fresh noise each time;
  (e) stochastic evaluation on the device against the restatement of SB3's evaluate_policy(..., deterministic=False);
  (f) on the CPU: the exports and their argument checks."""
import ctypes as C

import numpy as np
import pytest

import sb3_evaluation
from hlynr_intercept_b200 import config
from test_evaluation import EPISODES, N, _cfg, _check, _check_twins, _close, _mixed, _pipes, _restated
from test_obs_widths import _fused, _net_d, _obs_d
from test_policy_reference import CALLS, LOG_STD, SEED, eps_ref, noise_errors

OUTS = ("actions", "values", "logp", "mean", "clipped")


# ---- CPU ------------------------------------------------------------------------------------------------------------------------

def test_counter_entry_points_are_exported_and_check_their_arguments():
    from hlynr_intercept_b200 import _lib

    L = _lib.load()
    for name in ("hlynr_policy_forward_dev", "hlynr_policy_set_counter", "hlynr_policy_get_counter"):
        assert name in _lib.EXPORTS and hasattr(L, name), name
    fake, v = C.c_void_p(256), C.c_uint64()
    assert L.hlynr_policy_set_counter(None, 5, None) != 0
    assert b"null argument" in L.hlynr_last_error()
    for h, out in ((None, C.byref(v)), (fake, None)):
        assert L.hlynr_policy_get_counter(h, out, None) != 0
        assert b"hlynr_policy_get_counter: null argument" in L.hlynr_last_error()
    for h, obs in ((None, fake), (fake, None)):
        assert L.hlynr_policy_forward_dev(h, obs, 1, None, None, None, None, None, None, 0, 0, None) != 0
        assert b"hlynr_policy_forward_dev: null argument" in L.hlynr_last_error()


# ---- GPU: the counter of one handle ---------------------------------------------------------------------------------------------

def _bufs(n, zero=True):
    import torch

    f = torch.zeros if zero else torch.empty
    return dict(actions=f(n, 6, device="cuda"), values=f(n, device="cuda"), logp=f(n, device="cuda"),
                mean=f(n, 6, device="cuda"), clipped=f(n, 6, device="cuda"))


def _check_noise(out, rows, counter):
    a, lp, m = (out[k][:rows] for k in ("actions", "logp", "mean"))
    da, dl = noise_errors(a, lp, m, LOG_STD, eps_ref(SEED, counter, rows))
    assert da <= 1.0 and dl <= 1.0, (rows, counter, da, dl)
    assert bool((out["clipped"][:rows] == a.clamp(-1.0, 1.0)).all())


@pytest.mark.gpu
def test_counter_set_get_round_trips():
    f = _fused(_net_d(104, seed=40))
    for v in (0, 2**32 + 5, 2**63 + 7, 2**64 - 1):
        f.calls = v
        assert f.calls == v
    f.close()


@pytest.mark.gpu
@pytest.mark.parametrize("in_dim", [104, 68])
@pytest.mark.parametrize("cluster", [1, 2, 4])
@pytest.mark.parametrize("n", [1, 129, 37965, 131072 + 77])
def test_every_forward_advances_the_counter_by_one(n, cluster, in_dim):
    """Stochastic, deterministic, value only, n_rows_dev = 0, 3 and n + 5: calls advances by one each time, and the sampled
    rows are Philox at the new counter.  n_rows_dev = 0 returns from every CTA before any work."""
    import torch

    f = _fused(_net_d(in_dim, seed=41), cluster)
    obs = _obs_d(n, in_dim, seed=n)
    lim = torch.zeros(1, dtype=torch.int32, device="cuda")
    f.calls = CALLS
    c = CALLS
    for kind, rows_dev in (("full", None), ("det", None), ("values", None), ("full", 0), ("full", 3), ("full", n + 5)):
        out = _bufs(n)
        if rows_dev is not None:
            lim.fill_(rows_dev)
        if kind == "full":
            f.forward(obs, n_rows_dev=None if rows_dev is None else lim, want=(), out=out)
        elif kind == "det":
            f.forward(obs, deterministic=True, want=(), out=out)
        else:
            f.forward(obs, want=(), out=dict(values=out["values"]))
        c += 1
        assert f.calls == c, (kind, rows_dev)
        rows = n if rows_dev is None else min(n, rows_dev)
        if kind == "full":
            if rows:
                _check_noise(out, rows, c)
            assert bool((out["values"][rows:] == 0).all())   # rows beyond the device-side count are untouched
        elif kind == "det":
            assert torch.equal(out["actions"], out["mean"])
    f.close()


@pytest.mark.gpu
@pytest.mark.parametrize("in_dim", [104, 68])
@pytest.mark.parametrize("cluster", [1, 2, 4])
def test_device_counter_entry_equals_the_by_value_entry(cluster, in_dim):
    """forward_dev after set_counter(c - 1) and hlynr_policy_forward(counter = c): the same bits in all five outputs; the
    by-value call leaves the device counter where it was."""
    import torch

    n = 37965
    f = _fused(_net_d(in_dim, seed=42), cluster)
    obs = _obs_d(n, in_dim, seed=42)
    dev, val = _bufs(n, zero=False), _bufs(n, zero=False)
    f.calls = CALLS
    f.forward(obs, want=(), out=dev)
    assert f.calls == CALLS + 1
    p = lambda k: C.c_void_p(val[k].data_ptr())  # noqa: E731
    from hlynr_intercept_b200 import _lib

    _lib.check(f.L.hlynr_policy_forward(f.h, C.c_void_p(obs.data_ptr()), n, None, p("actions"), p("values"), p("logp"), p("mean"),
                                        p("clipped"), SEED, CALLS + 1, 0, f._stream()))
    torch.cuda.synchronize()
    for k in OUTS:
        assert torch.equal(dev[k], val[k]), k
    assert f.calls == CALLS + 1
    f.close()


def _sequence(f, obs, bufs, lim):
    """Five forwards of mixed kinds into bufs[0..4]."""
    f.forward(obs, want=(), out=bufs[0])
    f.forward(obs, deterministic=True, want=(), out=dict(actions=bufs[1]["actions"], clipped=bufs[1]["clipped"]))
    f.forward(obs, want=(), out=dict(values=bufs[2]["values"]))
    f.forward(obs, n_rows_dev=lim, want=(), out=bufs[3])
    f.forward(obs, want=(), out=dict(clipped=bufs[4]["clipped"]))


@pytest.mark.gpu
@pytest.mark.parametrize("in_dim", [104, 68])
@pytest.mark.parametrize("cluster", [1, 4])
def test_captured_forwards_replay_with_fresh_noise(cluster, in_dim):
    """5 forwards captured once and replayed 3 times == 15 eager forwards on a twin handle (same weights, seed and counter)."""
    import torch

    n = 5003
    net = _net_d(in_dim, seed=43)
    g, e = _fused(net, cluster), _fused(net, cluster)
    obs = _obs_d(n, in_dim, seed=43)
    lim = torch.full((1,), 777, dtype=torch.int32, device="cuda")
    gb, eb = [_bufs(n) for _ in range(5)], [_bufs(n) for _ in range(5)]
    for f in (g, e):   # first launches (shared-memory attributes, grid size) outside the capture
        f.forward(obs)
        f.calls = CALLS
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        _sequence(g, obs, gb, lim)
    assert g.calls == CALLS   # recorded, not run
    prev = None
    for rep in range(3):
        graph.replay()
        _sequence(e, obs, eb, lim)
        torch.cuda.synchronize()
        for i in range(5):
            for k in OUTS:
                assert torch.equal(gb[i][k], eb[i][k]), (rep, i, k)
        _check_noise(gb[0], n, CALLS + 5 * rep + 1)
        _check_noise(gb[3], 777, CALLS + 5 * rep + 4)
        if prev is not None:
            assert float((gb[0]["logp"] != prev).float().mean()) >= 0.99
        prev = gb[0]["logp"].clone()
    assert g.calls == e.calls == CALLS + 15
    g.close(); e.close()


# ---- GPU: rollout collection -----------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("frame_dim,n_stack", [(26, 4), (17, 4)])
def test_rollout_replays_draw_fresh_noise(frame_dim, n_stack):
    """Twin collectors with equal counters: capture(), then replay() x3 against collect() x4 (the first matching capture's
    eager warm-up).  Each replay equals its eager collect in all eight buffers, and log_probs change from replay to replay:
    log_std does not depend on the state, so log pi is a function of eps alone."""
    import torch

    from hlynr_intercept_b200.post import HlynrObsPipeline
    from hlynr_intercept_b200.rollout import DeviceRolloutCollector
    from hlynr_intercept_b200.sim import HlynrSim

    n, d = 1501, frame_dim * n_stack
    cfg = config.baseline_config("cfg4")
    cfg["max_steps"] = 7
    net = _net_d(d, seed=44)
    cols = []
    for _ in range(2):
        sim = HlynrSim(cfg, n_envs=n, seed=13, warn_dead=False, obs_dim=frame_dim)
        pipe = HlynrObsPipeline(sim, n_stack=n_stack, training=True)
        T = DeviceRolloutCollector(pipe, None, 1).graph_period()
        pol = _fused(net, seed=SEED)
        pol.calls = CALLS
        cols.append(DeviceRolloutCollector(pipe, pol, T, bootstrap_rows=n))
    eager, graphed = cols
    per = 2 * T + 1   # per collect: T forwards, T bootstrap value passes, the last value pass
    graphed.capture()
    eager.collect()
    assert graphed.policy.calls == eager.policy.calls == CALLS + per
    lps = []
    for rep in range(3):
        eager.collect()
        graphed.replay()
        torch.cuda.synchronize()
        for name in ("obs", "actions", "values", "log_probs", "rewards", "episode_starts", "advantages", "returns"):
            a, b = getattr(eager, name).cpu().numpy(), getattr(graphed, name).cpu().numpy()
            assert np.isfinite(a).all(), name
            np.testing.assert_array_equal(a, b, err_msg=f"{name} after replay {rep + 1}")
        assert graphed.policy.calls == eager.policy.calls == CALLS + (rep + 2) * per
        lps.append(graphed.log_probs.clone())
    for a, b in zip(lps, lps[1:]):
        assert float((a != b).float().mean()) >= 0.99
    assert float(eager.episode_starts[1:].sum()) > 0
    for c in cols:
        c.policy.close(); c.pipe.close(); c.sim.close()


# ---- GPU: stochastic evaluation --------------------------------------------------------------------------------------------------

def _fused_sample(fused):
    import torch

    buf = torch.empty(N, 6, device="cuda")

    def predict(obs):   # SB3 predict(deterministic=False): a sample, clipped to the Box bounds
        fused.forward(obs, deterministic=False, want=(), out=dict(clipped=buf))
        return buf

    return predict


def _torch_sample(net):
    import torch

    def predict(obs):
        with torch.no_grad():
            return net(obs)[0].float().clamp(-1.0, 1.0)

    return predict


def _eval_handles(net):
    from hlynr_intercept_b200.policy import FusedActorCritic

    hs = [FusedActorCritic(net, device=0, seed=SEED) for _ in range(2)]
    for h in hs:
        h.calls = CALLS
    return hs


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["eager", "graph_1x", "graph_3x"])
@pytest.mark.parametrize("episodes", ["37", "N", "2.5N"])
def test_fused_stochastic_evaluation_equals_restatement(episodes, mode):
    """The restatement's predict samples from a twin handle with the same seed and counter: every record, end step, order,
    reward and length, the mean and std, both sims' state and both counters agree bit for bit."""
    from hlynr_intercept_b200.evaluation import DeviceEvaluator
    from hlynr_intercept_b200.rollout import graph_period

    E = EPISODES[episodes]
    pipes = _pipes(_cfg())
    fused, twin = _eval_handles(_net_d(104, seed=5))
    mult = {"eager": None, "graph_1x": 1, "graph_3x": 3}[mode]
    ev = DeviceEvaluator(pipes[0], fused, chunk=None if mult is None else mult * graph_period(pipes[0]))
    graph = mode != "eager"
    res = ev.evaluate(E, graph=graph, deterministic=False)
    _check(res, _restated(pipes[1], _fused_sample(twin), E, res.ticks), E, graph, ev.chunk)
    _check_twins(*pipes)
    assert fused.calls == twin.calls == CALLS + res.ticks
    if E >= N:
        _mixed(res)
    _close(fused, twin, *pipes)


@pytest.mark.gpu
def test_stochastic_evaluation_differs_from_deterministic():
    """Same seed, same sims: sampling changes the episodes."""
    from hlynr_intercept_b200.evaluation import DeviceEvaluator

    net = _net_d(104, seed=5)
    out = {}
    for det in (True, False):
        pipes = _pipes(_cfg())
        fused, twin = _eval_handles(net)
        out[det] = DeviceEvaluator(pipes[0], fused).evaluate(N, deterministic=det)
        _close(fused, twin, *pipes)
    assert out[True].records.tobytes() != out[False].records.tobytes()
    assert not np.array_equal(out[True].episode_rewards, out[False].episode_rewards)


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
def test_torch_stochastic_evaluation(graph):
    """ReferenceActorCritic with deterministic=False.  Eager: bit for bit against the restatement, both sides starting from
    the same torch.manual_seed.  Graph: torch's generator advances differently under capture, so the SB3 invariants are checked
    instead: E records, every env's quota, (end step, env) order, the returned statistics."""
    import torch

    from hlynr_intercept_b200.evaluation import DeviceEvaluator

    E = EPISODES["2.5N"]
    pipes = _pipes(_cfg(), seed=23)
    net = _net_d(104, seed=6)
    ev = DeviceEvaluator(pipes[0], net)
    torch.manual_seed(77)
    res = ev.evaluate(E, graph=graph, deterministic=False)
    if not graph:
        torch.manual_seed(77)
        _check(res, _restated(pipes[1], _torch_sample(net), E, res.ticks), E, False, ev.chunk)
        _check_twins(*pipes)
    else:
        assert len(res.records) == E and res.ticks % ev.chunk == 0
        np.testing.assert_array_equal(np.bincount(res.records["env"], minlength=N), sb3_evaluation.episode_count_targets(N, E))
        key = res.end_tick * N + res.records["env"]
        assert (np.diff(key) > 0).all()
        assert res.mean_reward == np.mean(res.episode_rewards) and res.std_reward == np.std(res.episode_rewards)
    _mixed(res)
    _close(*pipes)


@pytest.mark.gpu
def test_gaussian_mlp_policy_evaluates_stochastically_only():
    """A torch module with the collector's interface but no mean(obs) (GaussianMlpPolicy): stochastic evaluation runs,
    deterministic evaluation is refused."""
    import torch

    from hlynr_intercept_b200.evaluation import DeviceEvaluator
    from hlynr_intercept_b200.rollout import GaussianMlpPolicy

    pipes = _pipes(_cfg(), seed=47)
    torch.manual_seed(3)
    ev = DeviceEvaluator(pipes[0], GaussianMlpPolicy(104))
    with pytest.raises(ValueError, match="mean"):
        ev.evaluate(N)
    res = ev.evaluate(N, deterministic=False)
    assert len(res.records) == N and sorted(res.records["env"].tolist()) == list(range(N))
    _close(*pipes)

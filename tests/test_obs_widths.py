"""The device training path for every observation layout the reference trains with: 17-D frames (the leading radar channels
obs[0:17], HlynrSim(obs_dim=17)) and any frame_stack through HlynrObsPipeline, input widths 1-256 through the fused policy
forward, and both together through DeviceRolloutCollector, eager and graph-replayed.

Pipeline results are checked against the numpy restatement of SB3's VecFrameStack + VecNormalize (oracle/sb3_post.py) and
against the 26-D pipeline of a twin sim; policy results against the float64 reference forward64 of test_policy_reference.py
(same bounds) and, for widths below 104, bit for bit against the default 104-wide kernel with zero weight columns."""
import ctypes as C
import types

import numpy as np
import pytest

from hlynr_intercept_b200 import config
from oracle import sb3_post
from test_policy_reference import (ATOL, CALLS, LOG_STD, MEAN_TOL, SEED, VALUE_ATOL, _layers, errors, eps_ref, forward64,
                                   noise_errors)
from test_post import _staggered

IN_DIMS = [17, 26, 34, 51, 52, 68, 78, 119, 136, 208, 256]


# ---- observation pipeline ------------------------------------------------------------------------------------------------------

def _sims(cfg, n, seed, obs_dims):
    from hlynr_intercept_b200.sim import HlynrSim

    return [HlynrSim(cfg, n_envs=n, seed=seed, warn_dead=False, obs_dim=d) for d in obs_dims]


def _truncate_all(sims, max_steps):
    """Every env's next step is its last (max_steps): a step whose done list holds every env."""
    st = sims[0].export_state()
    st["steps"][:] = max_steps - 1
    for s in sims:
        s.import_state(st)


@pytest.mark.gpu
@pytest.mark.parametrize("n_stack", [1, 2, 3, 4, 8])
def test_17d_pipeline_matches_sb3_restatement(n_stack):
    """n = 3001 (ragged), staggered episodes, training, then frozen statistics, then training again; odd 17k (k = 1, 3) gives
    4-byte aligned output rows.  Tolerances of test_post.test_pipeline_matches_sb3_restatement."""
    import torch

    from hlynr_intercept_b200.post import HlynrObsPipeline

    n, max_steps, T, F = 3001, 40, 130, 17
    cfg = config.baseline_config("cfg4")
    cfg["max_steps"] = max_steps
    ref, sim = _sims(cfg, n, 5, (F, F))
    pipe = HlynrObsPipeline(sim, n_stack=n_stack, training=True)
    assert pipe.frame_dim == F and pipe.obs_dim == F * n_stack
    out0 = pipe.reset()
    obs0 = ref.reset().cpu().numpy()
    assert obs0.shape == (n, F)
    rng = np.random.default_rng(1)
    state = _staggered(ref, rng, max_steps)
    ref.import_state(state); sim.import_state(state)
    stack = sb3_post.StackedObservations(n, n_stack, F)
    vn = sb3_post.VecNormalize(n, (F * n_stack,), gamma=0.99)
    np.testing.assert_allclose(out0.cpu().numpy(), vn.reset(stack.reset(obs0).astype(np.float64)), atol=2e-6)
    total_done, all_done = 0, False
    for t in range(T):
        if t == 70:
            pipe.training = vn.training = False
            _truncate_all((ref, sim), max_steps)
        if t == 100:
            pipe.training = vn.training = True
        a = torch.as_tensor(rng.uniform(-1, 1, (n, 6)).astype(np.float32)).cuda()
        o, r, te, tr, tobs, _ = ref.step(a)
        o, r, tobs = o.cpu().numpy(), r.cpu().numpy(), tobs.cpu().numpy()
        dones = (te | tr).cpu().numpy().astype(bool)
        infos = {int(i): {"terminal_observation": tobs[i].copy()} for i in np.nonzero(dones)[0]}
        stacked, infos = stack.update(o, dones, infos)
        want, _, _, infos = vn.step(stacked.astype(np.float64), r.astype(np.float64), dones, infos)
        out, rew, te2, tr2, (records, counter, terminal) = pipe.step(a)
        assert (rew.cpu().numpy() == r).all() and ((te2 | tr2).cpu().numpy().astype(bool) == dones).all()
        np.testing.assert_allclose(out.cpu().numpy(), want, atol=5e-6, err_msg=f"tick {t}")
        np.testing.assert_array_equal(pipe.get_original_obs().cpu().numpy(), stacked)
        rec = pipe.done_records()
        all_done |= len(rec) == n
        assert sorted(rec["env"].tolist()) == sorted(infos.keys())
        term = terminal.cpu().numpy()
        for k, e in enumerate(rec["env"].tolist()):
            np.testing.assert_allclose(term[k], infos[e]["terminal_observation"], atol=5e-6)
        total_done += len(rec)
        s = pipe.get_stats()
        np.testing.assert_allclose(s["mean"], vn.obs_rms.mean, rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(s["var"], vn.obs_rms.var, rtol=1e-8, atol=1e-12)
        assert abs(s["count"] - vn.obs_rms.count) < 1e-6
        np.testing.assert_allclose([s["ret_mean"], s["ret_var"]], [vn.ret_rms.mean, vn.ret_rms.var], rtol=1e-9)
        if t % 16 == 0:
            assert pipe.check_sums() < 1e-6
    assert all_done and total_done > 3 * n
    assert pipe.check_sums() < 1e-6
    x = torch.as_tensor(rng.uniform(-2, 1, (7, F * n_stack)).astype(np.float32)).cuda()
    np.testing.assert_allclose(pipe.normalize_obs(x).cpu().numpy(), vn.normalize_obs(x.cpu().numpy().astype(np.float64)), atol=5e-6)
    pipe.close(); sim.close(); ref.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n_stack", [1, 3, 4])
def test_17d_pipeline_is_the_26d_pipeline_on_the_leading_channels(n_stack):
    """Twin sims, same seed, obs_dim 26 and 17: raw stacks bit for bit, statistics to 1e-12, and with the same statistics
    (training off) the normalised observations and terminal rows bit for bit."""
    import torch

    from hlynr_intercept_b200.post import HlynrObsPipeline

    n, max_steps, T = 2999, 30, 90
    cfg = config.baseline_config("cfg4")
    cfg["max_steps"] = max_steps
    sims = _sims(cfg, n, 7, (26, 17))
    pipes = [HlynrObsPipeline(s, n_stack=n_stack, training=True) for s in sims]
    cols = (np.arange(26 * n_stack) % 26) < 17        # the 17-D features inside the 26-D stack
    for p in pipes:
        p.reset()
    rng = np.random.default_rng(3)
    state = _staggered(sims[0], rng, max_steps)
    for s in sims:
        s.import_state(state)
    frozen = False
    for t in range(T):
        if t == 60:   # the 26-D statistics, restricted to the leading channels, for both; then inference mode
            s26 = pipes[0].get_stats()
            pipes[1].set_stats(s26["mean"][cols], s26["var"][cols], s26["count"])
            for p in pipes:
                p.training = False
            frozen = True
            _truncate_all(sims, max_steps)
        a = torch.as_tensor(rng.uniform(-1, 1, (n, 6)).astype(np.float32)).cuda()
        res = [p.step(a) for p in pipes]
        recs = [p.done_records() for p in pipes]
        order = [np.argsort(r["env"], kind="stable") for r in recs]   # the done lists fill in completion order
        assert np.array_equal(recs[0]["env"][order[0]], recs[1]["env"][order[1]])
        o26, o17 = (p.get_original_obs().cpu().numpy() for p in pipes)
        np.testing.assert_array_equal(o17, o26[:, cols], err_msg=f"tick {t}")
        if frozen:
            np.testing.assert_array_equal(res[1][0].cpu().numpy(), res[0][0].cpu().numpy()[:, cols], err_msg=f"tick {t}")
            m = len(recs[0])
            t26, t17 = res[0][4][2][:m].cpu().numpy()[order[0]], res[1][4][2][:m].cpu().numpy()[order[1]]
            np.testing.assert_array_equal(t17, t26[:, cols], err_msg=f"terminal rows, tick {t}")
        else:
            s26, s17 = pipes[0].get_stats(), pipes[1].get_stats()
            np.testing.assert_allclose(s17["mean"], s26["mean"][cols], rtol=1e-12, atol=1e-300)
            np.testing.assert_allclose(s17["var"], s26["var"][cols], rtol=1e-12, atol=1e-300)
            assert s17["count"] == s26["count"]
    for p in pipes:
        assert p.check_sums() < 1e-6
        p.close()
    for s in sims:
        s.close()


def _fake_pipe(frame_dim, n_stack, stats=None):
    """The attributes save / load / save_sb3_pickle / load_sb3_pickle read, without a device."""
    d = frame_dim * n_stack
    got = []
    s = stats or dict(mean=np.linspace(-1, 1, d), var=np.linspace(0.5, 2, d), count=123.0, ret_mean=0.1, ret_var=2.0, ret_count=9.0)
    return types.SimpleNamespace(frame_dim=frame_dim, n_stack=n_stack, obs_dim=d, clip_obs=10.0, clip_reward=10.0, gamma=0.99,
                                 epsilon=1e-8, norm_obs=True, training=True, sim=types.SimpleNamespace(n=5),
                                 get_stats=lambda: s, set_stats=lambda *a: got.append(a), got=got)


def test_statistics_files_carry_the_frame_width(tmp_path):
    """A 17-D/4 .npz and vec_normalize.pkl (obs_shape (68,)) round-trip; a 26-D file is refused by a 17-D pipeline and the
    reverse; an .npz without the frame width is a 26-D one."""
    from hlynr_intercept_b200.post import HlynrObsPipeline as P

    p17, p26 = _fake_pipe(17, 4), _fake_pipe(26, 4)
    P.save(p17, str(tmp_path / "s17.npz")); P.save(p26, str(tmp_path / "s26.npz"))
    P.save_sb3_pickle(p17, str(tmp_path / "v17.pkl")); P.save_sb3_pickle(p26, str(tmp_path / "v26.pkl"))
    q17, q26 = _fake_pipe(17, 4), _fake_pipe(26, 4)
    P.load(q17, str(tmp_path / "s17.npz"))
    P.load_sb3_pickle(q17, str(tmp_path / "v17.pkl"))
    for mean, var, count, *ret in q17.got:
        np.testing.assert_array_equal(mean, p17.get_stats()["mean"]); np.testing.assert_array_equal(var, p17.get_stats()["var"])
        assert count == 123.0 and list(ret) == [0.1, 2.0, 9.0]
    assert len(q17.got) == 2
    from hlynr_intercept_b200 import sb3_pickle

    assert sb3_pickle.load(str(tmp_path / "v17.pkl"))["obs_shape"] == (68,)
    with pytest.raises(ValueError, match="17-D"):
        P.load(q26, str(tmp_path / "s17.npz"))
    with pytest.raises(ValueError, match="26-D"):
        P.load(q17, str(tmp_path / "s26.npz"))
    with pytest.raises(ValueError, match="shape"):
        P.load_sb3_pickle(q17, str(tmp_path / "v26.pkl"))
    with pytest.raises(ValueError, match="shape"):
        P.load_sb3_pickle(q26, str(tmp_path / "v17.pkl"))
    # a file written before the frame width was saved
    z = dict(np.load(str(tmp_path / "s26.npz")))
    del z["frame_dim"]
    np.savez(str(tmp_path / "old.npz"), **z)
    P.load(q26, str(tmp_path / "old.npz"))
    with pytest.raises(ValueError, match="26-D"):
        P.load(q17, str(tmp_path / "old.npz"))
    with pytest.raises(AssertionError, match="frame_stack"):
        P.load(_fake_pipe(17, 2), str(tmp_path / "s17.npz"))


# ---- policy forward ------------------------------------------------------------------------------------------------------------

def _net_d(d, seed=0, device="cuda"):
    """test_policy_reference._net at input width d."""
    import torch
    from hlynr_intercept_b200.policy import ReferenceActorCritic

    torch.manual_seed(seed)
    net = ReferenceActorCritic(obs_dim=d, device=device)
    lins, lns = _layers(net)
    with torch.no_grad():
        for lin, ln in zip(lins, lns):
            lin.bias.normal_(0, 0.2)
            ln.weight.uniform_(0.5, 1.5); ln.bias.normal_(0, 0.3)
        net.action_net.weight.mul_(40.0); net.action_net.bias.normal_(0, 0.1)
        net.value_net.bias.fill_(0.37)
        net.log_std.copy_(torch.tensor(LOG_STD, device=device))
    return net


def _obs_d(n, d, seed=0):
    import torch

    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    obs = (torch.randn(n, d, device="cuda", generator=g) * 1.5).clamp(-10, 10)
    obs[:, min(7, d - 1)] = 5.0 + 5.0 * torch.rand(n, device="cuda", generator=g)
    return obs.contiguous()


def _fused(net, cluster=1, seed=SEED):
    from hlynr_intercept_b200.policy import FusedActorCritic

    f = FusedActorCritic(net, device=0, seed=seed)
    f.set_option("cluster", cluster)
    return f


def _all_outputs(fused, obs):
    import torch

    n = obs.shape[0]
    clipped = torch.empty(n, 6, device="cuda")
    fused.calls = CALLS
    a, v, lp, m = (t.clone() for t in fused.forward(obs, want=("actions", "values", "logp", "mean"), out=dict(clipped=clipped)))
    torch.cuda.synchronize()
    return dict(actions=a, values=v, logp=lp, mean=m, clipped=clipped)


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", [1, 2, 4])
@pytest.mark.parametrize("in_dim", IN_DIMS)
def test_forward_at_input_width(in_dim, cluster):
    """mean / value against forward64 with the plain-case bounds, sampled actions and log pi within 16 ulp, for 1, 129 and
    37 965 rows; odd widths also from 4-byte aligned rows (a row of a rollout buffer), bit for bit."""
    import torch

    net = _net_d(in_dim, seed=in_dim)
    fused = _fused(net, cluster)
    assert fused.in_dim == in_dim
    for n in (1, 129, 37965):
        obs = _obs_d(n, in_dim, seed=n)
        out = _all_outputs(fused, obs)
        with torch.no_grad():
            rm, rv = forward64(net, obs)
        for name, got, ref, atol in (("mean", out["mean"], rm, ATOL), ("value", out["values"], rv, VALUE_ATOL)):
            assert torch.isfinite(got).all(), name
            worst, mad, dmax = errors(got, ref, atol)
            assert worst <= 1.0, f"{name} at {n} rows: max |diff| {dmax:.3e}"
            assert mad < MEAN_TOL, f"{name} at {n} rows: mean |diff| {mad:.3e}"
        da, dl = noise_errors(out["actions"], out["logp"], out["mean"], LOG_STD, eps_ref(SEED, CALLS + 1, n))
        assert da <= 1.0 and dl <= 1.0, (n, da, dl)
        assert torch.equal(out["clipped"], out["actions"].clamp(-1.0, 1.0))
        if in_dim % 2:
            buf = torch.empty(n * in_dim + 1, device="cuda")
            view = buf[1:].view(n, in_dim)
            assert view.data_ptr() % 16 == 4
            view.copy_(obs)
            got = _all_outputs(fused, view)
            for k in out:
                assert torch.equal(got[k], out[k]), k
    fused.close()


@pytest.mark.gpu
@pytest.mark.parametrize("in_dim", [d for d in IN_DIMS if d < 104])
def test_narrow_input_equals_zero_padded_default_network(in_dim):
    """A d-wide network gives the bits of the default 104-wide kernel whose w1 has the same first d columns and zeros after
    them, fed rows with arbitrary finite values in columns d..103: every output, at the same seed and counter."""
    import torch
    from hlynr_intercept_b200.policy import ReferenceActorCritic

    n = 37965
    net = _net_d(in_dim, seed=100 + in_dim)
    wide = ReferenceActorCritic(obs_dim=104, device="cuda")
    sd = net.state_dict()
    w1 = torch.zeros(512, 104, device="cuda")
    w1[:, :in_dim] = sd["network.0.weight"]
    sd["network.0.weight"] = w1
    wide.load_state_dict(sd)
    obs = _obs_d(n, in_dim, seed=1)
    g = torch.Generator(device="cuda"); g.manual_seed(2)
    junk = torch.randn(n, 104 - in_dim, device="cuda", generator=g) * 1e6
    junk[::3] = 3e37
    obs104 = torch.cat([obs, junk], 1).contiguous()
    a, b = _fused(net), _fused(wide)
    got, want = _all_outputs(a, obs), _all_outputs(b, obs104)
    for k in want:
        assert torch.equal(got[k], want[k]), k
    a.close(); b.close()


@pytest.mark.gpu
def test_default_width_handles_and_resync():
    """hlynr_policy_create_dim(104) and hlynr_policy_create give the same bits; sync_weights() after a change of w1 of a
    68-wide network equals a fresh handle."""
    import torch
    from hlynr_intercept_b200 import _lib

    net = _net_d(104, seed=21)
    obs = _obs_d(5000, 104, seed=21)
    f = _fused(net)
    plain = _fused(net)
    L = _lib.load()
    L.hlynr_policy_destroy(plain.h)
    h = C.c_void_p()
    _lib.check(L.hlynr_policy_create(0, C.byref(h)))
    plain.h = h
    plain.sync_weights()
    got, want = _all_outputs(f, obs), _all_outputs(plain, obs)
    for k in want:
        assert torch.equal(got[k], want[k]), k
    f.close(); plain.close()

    net = _net_d(68, seed=22)
    obs = _obs_d(5000, 68, seed=22)
    f = _fused(net)
    before = _all_outputs(f, obs)
    with torch.no_grad():
        net.network[0].weight.mul_(-1.3).add_(0.01)
    f.sync_weights()
    fresh = _fused(net)
    got, want = _all_outputs(f, obs), _all_outputs(fresh, obs)
    assert not torch.equal(got["mean"], before["mean"])
    for k in want:
        assert torch.equal(got[k], want[k]), k
    f.close(); fresh.close()


def test_input_width_out_of_range_is_refused():
    """in_dim 0 or 257 by the C entry point, 257 by FusedActorCritic; both before any device work."""
    from hlynr_intercept_b200 import _lib
    from hlynr_intercept_b200.policy import FusedActorCritic, ReferenceActorCritic

    L = _lib.load()
    for d in (0, 257, -1):
        h = C.c_void_p()
        assert L.hlynr_policy_create_dim(0, d, C.byref(h)) != 0
        assert b"in_dim must be in [1, 256]" in L.hlynr_last_error()
    FusedActorCritic._modules(types.SimpleNamespace(net=ReferenceActorCritic(obs_dim=256, device="cpu")))
    with pytest.raises(NotImplementedError, match="in_dim"):
        FusedActorCritic._modules(types.SimpleNamespace(net=ReferenceActorCritic(obs_dim=257, device="cpu")))


@pytest.mark.gpu
def test_rows_of_another_width_are_refused():
    """forward with rows of another width, and a 17-D pipeline feeding the default 104-wide policy, raise."""
    import torch

    from hlynr_intercept_b200.post import HlynrObsPipeline
    from hlynr_intercept_b200.rollout import DeviceRolloutCollector

    f = _fused(_net_d(68, seed=3))
    with pytest.raises(ValueError, match="68 wide"):
        f.forward(torch.zeros(52, 136, device="cuda"))   # 104 rows' worth of floats: no silent reshape
    with pytest.raises(ValueError, match="68 wide"):
        f.forward(torch.zeros(10, 104, device="cuda"))
    f.close()
    cfg = config.baseline_config("cfg4")
    (sim,) = _sims(cfg, 200, 1, (17,))
    pipe = HlynrObsPipeline(sim, n_stack=4)
    f = _fused(_net_d(104, seed=3))
    with pytest.raises(ValueError, match="104 wide"):
        DeviceRolloutCollector(pipe, f, 4).collect()
    f.close(); pipe.close(); sim.close()


# ---- end to end ----------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("frame_dim,n_stack", [(17, 4), (26, 2)])
def test_rollout_with_fused_policy_graph_replay_equals_eager(frame_dim, n_stack):
    """Twin collectors on twin sims with the fused policy of width frame_dim * n_stack: capture(); replay() against
    collect(); collect(), bit for bit.  The warm-up collect inside capture() leaves both policies at the same call counter."""
    import torch

    from hlynr_intercept_b200.post import HlynrObsPipeline
    from hlynr_intercept_b200.rollout import DeviceRolloutCollector

    n, d = 1501, frame_dim * n_stack
    cfg = config.baseline_config("cfg4")
    cfg["max_steps"] = 7   # every env truncates inside each collect
    net = _net_d(d, seed=31)
    cols = []
    for _ in range(2):
        (sim,) = _sims(cfg, n, 11, (frame_dim,))
        pipe = HlynrObsPipeline(sim, n_stack=n_stack, training=True)
        T = DeviceRolloutCollector(pipe, None, 1).graph_period()
        cols.append(DeviceRolloutCollector(pipe, _fused(net, seed=9), T, bootstrap_rows=n))
    eager, graphed = cols
    assert eager.obs.shape == (T + 1, n, d)
    graphed.capture()
    graphed.replay()
    eager.collect()
    eager.collect()
    torch.cuda.synchronize()
    for name in ("obs", "actions", "values", "log_probs", "rewards", "episode_starts", "advantages", "returns"):
        a, b = getattr(eager, name).cpu().numpy(), getattr(graphed, name).cpu().numpy()
        assert np.isfinite(a).all(), name
        np.testing.assert_array_equal(a, b, err_msg=name)
    assert float(eager.episode_starts[1:].sum()) > 0   # episodes ended inside the rollout
    for c in cols:
        c.policy.close(); c.pipe.close(); c.sim.close()

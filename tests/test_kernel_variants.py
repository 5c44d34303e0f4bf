"""The kernel variants the per-tick API step does not exercise, bit for bit against that step on a second handle.

The per-tick step (`hlynr_step`, `step_kernel<R, false, F>`) is tied to the NumPy reference by the oracle and golden tests.  The
variants below run the same arithmetic, so every comparison here is exact:

  A. the fused k-tick rollout (`hlynr_rollout`, `step_kernel<R, true, F>`) against k per-tick steps, with episodes that end and
     auto-reset inside a launch, ragged tiles, delay-ring rows carried across launches of every length, caller actions and the
     in-kernel random policy;
  B. the launch options `specialise` (the generic kernel, also on the compact plane layouts), `pdl` and `prefetch_waves`, which
     must change timing only;
  C. the finished-episode lists: the host list past the records fetched together with the count, and a caller-attached device
     list whose capacity is below the number of envs that finish.
"""
import ctypes as C

import numpy as np
import pytest

from hlynr_intercept_b200 import abi, config
from oracle import draws

pytestmark = pytest.mark.gpu

MAX_ONBOARD_DELAY = 10   # include/hlynr.h HLYNR_MAX_ONBOARD_DELAY
INT_STATS = ("episodes", "successes", "length_sum", "hit_target", "interceptor_crash", "fuel_out", "missile_ground", "worsening",
             "timeouts", "env_steps", "onboard_locks")
FLOAT_STATS = ("return_sum", "min_distance_sum", "final_distance_sum")


def _cfg(case, max_steps=None):
    """Env dicts of the feature sets, with the step-kernel instantiation feature_set() (hlynr_capi.cu) picks for each."""
    if case == "cfg2":      # physics v2.0 off: FT_V2OFF
        e = config.baseline_config("cfg2")
    elif case == "cfg4":    # v2.0 on: FT_V2ON; fp32 handles use compact layout 1
        e = config.baseline_config("cfg4")
    elif case == "cfg3":    # v2.0 on + domain randomization: FT_V2ON_DR; fp32 handles use compact layout 2
        e = config.baseline_config("cfg3")
    elif case == "generic":  # precision mode + proximity fuze: FT_GENERIC
        e = config.baseline_config("cfg4")
        e["curriculum"] = dict(precision_mode=True)
        e["proximity_fuze_enabled"] = True
    elif case == "modes":   # los_frame + volley of 3 on cfg3 (per-env onboard delays of domain randomization): FT_GENERIC_MODES
        e = config.baseline_config("cfg3")
        e.update(observation_mode="los_frame", volley_mode=True, volley_size=3)
    elif case == "body":    # body_frame observations: FT_GENERIC_MODES
        e = config.baseline_config("cfg4")
        e["observation_mode"] = "body_frame"
    else:
        raise KeyError(case)
    if max_steps is not None:
        e["max_steps"] = max_steps
    P, _ = config.resolve_config(e, warn_dead=False)
    want = dict(generic=dict(precision_mode=1, fuze_enabled=1, obs_mode=abi.OBS_WORLD, volley_size=0),
                modes=dict(obs_mode=abi.OBS_LOS, volley_size=3, dr_enabled=1),
                body=dict(obs_mode=abi.OBS_BODY, volley_size=0)).get(case, {})
    for k, v in want.items():   # the dict really selects the feature set named above
        assert getattr(P, k) == v, (case, k)
    return e


def _sim(cfg, n, seed, f64=False, offset=0, obs_dim=26, **options):
    from hlynr_intercept_b200.sim import HlynrSim

    s = HlynrSim(cfg, n_envs=n, seed=seed, env_id_offset=offset, precision="fp64" if f64 else "fp32", warn_dead=False,
                 obs_dim=obs_dim)
    for k, v in options.items():
        s.set_option(k, v)
    return s


def _np(x):
    return x.cpu().numpy().copy()


def _assert_same_state(a, b, what):
    sa, sb = a.export_state(), b.export_state()
    for k in sa:
        assert np.array_equal(sa[k], sb[k], equal_nan=True), (what, k)


def _assert_same_stats(a, b, what, float_rtol=1e-12):
    sa, sb = a.stats(), b.stats()
    for k in INT_STATS:
        assert sa[k] == sb[k], (what, k, sa[k], sb[k])
    # double atomics over the statistics slots: the order of the additions is not fixed (on a B200 they came out exact)
    for k in FLOAT_STATS:
        np.testing.assert_allclose(sa[k], sb[k], rtol=float_rtol, atol=0, err_msg=f"{what}: {k}")


# ---------------------------------------------------------------------------------------------------------------------------
# A. fused rollout == k per-tick steps
# ---------------------------------------------------------------------------------------------------------------------------
# ("step",) = one hlynr_step on every handle; k = one fused launch of k ticks.  165 ticks: the launches start at many ring phases
# and none of the lengths is a multiple of every ring length (asserted against ring_period() below).
SCHEDULE = [1, "step", 7, "step", 31, "step", 12, "step"] * 3
MAX_STEPS = 23   # every env auto-resets several times inside fused launches, some twice in one 31-tick launch

A_CASES = [(c, False) for c in ("cfg2", "cfg4", "cfg3", "generic", "modes", "body")] + [(c, True) for c in ("cfg4", "cfg3", "modes")]


def _rollout_vs_steps(case, f64, policy, n=1037, offset=0, seed=4711):
    """Per-tick handle `ref`; fused handles `fus` (obs), `nob` (want_obs=False) and `f17` (obs_dim=17).  Every handle runs the
    same schedule; the fused ones turn each k into one launch."""
    import torch

    cfg = _cfg(case, MAX_STEPS)
    ref = _sim(cfg, n, seed, f64, offset)
    fus = _sim(cfg, n, seed, f64, offset)
    nob = _sim(cfg, n, seed, f64, offset)
    f17 = _sim(cfg, n, seed, f64, offset, obs_dim=17)
    per = ref.ring_period()
    launches = [k for k in SCHEDULE if k != "step"]
    assert any(k % per for k in launches), per
    if ref.params.dr_enabled and ref.params.onboard_delay > 0:
        assert per % (MAX_ONBOARD_DELAY + 1) == 0, per   # per-env delays: the onboard ring has the maximum length
    o_ref = _np(ref.reset())
    assert np.array_equal(_np(fus.reset()), o_ref) and np.array_equal(_np(nob.reset()), o_ref)
    assert np.array_equal(_np(f17.reset()), o_ref[:, :17])
    gids = offset + np.arange(n, dtype=np.int64)
    episode = np.zeros(n, np.int64)
    steps = np.zeros(n, np.int64)
    rng = np.random.default_rng(seed)
    tick, phases, twice, in_launch = 0, set(), False, 0

    def host_actions():
        if policy == "random":
            return draws.random_actions(seed, gids, episode, steps + 1)
        return rng.uniform(-1.2, 1.2, (n, 6)).astype(np.float32)

    def ref_step(a):
        o, r, te, tr, _, _ = ref.step(torch.as_tensor(a).cuda())
        o, r, te, tr = _np(o), _np(r), _np(te), _np(tr)
        done = (te | tr).astype(bool)
        episode[:] += done
        steps[:] = np.where(done, 0, steps + 1)
        return o, r, te, tr, done

    for op in SCHEDULE:
        if op == "step":
            a = host_actions()
            o, r, te, tr, _ = ref_step(a)
            at = torch.as_tensor(a).cuda()
            for h in (fus, nob, f17):
                x = h.step(at)
                assert np.array_equal(_np(x[0]), o[:, :h.obs_dim]), (tick, h.obs_dim)
                assert np.array_equal(_np(x[1]), r) and np.array_equal(_np(x[2]), te) and np.array_equal(_np(x[3]), tr), tick
            tick += 1
            continue
        k = op
        phases.add(tick % per)
        acts = []
        rsum = np.zeros(n, np.float32)
        dcount = np.zeros(n, np.int32)
        for s in range(k):
            a = host_actions()
            acts.append(a)
            o, r, te, tr, done = ref_step(a)
            rsum = rsum + r   # float32, tick order: the kernel's `rsum += t.reward`
            dcount += done
        assert rsum.dtype == np.float32
        at = torch.as_tensor(np.stack(acts)).cuda() if policy == "caller" else None
        of, rf, df = (_np(x) for x in fus.rollout(k, at))
        _, rn, dn = nob.rollout(k, at, want_obs=False)
        o17, r17, d17 = (_np(x) for x in f17.rollout(k, at))
        what = (case, f64, policy, tick, k)
        assert np.array_equal(of, o), what
        assert np.array_equal(rf, rsum), what
        assert np.array_equal(df, dcount), what
        assert np.array_equal(_np(rn), rsum) and np.array_equal(_np(dn), dcount), what
        assert np.array_equal(o17, of[:, :17]) and np.array_equal(r17, rsum) and np.array_equal(d17, dcount), what
        twice |= bool((dcount >= 2).any())
        in_launch += int(dcount.sum())
        tick += k
    assert tick == ref.tick_count() == fus.tick_count()
    assert len(phases) > 1 and in_launch > 2 * n, (phases, in_launch)
    assert twice or n < 64   # a handful of envs may never end two episodes inside one launch
    for h, name in ((fus, "fused"), (nob, "want_obs=False"), (f17, "obs_dim=17")):
        _assert_same_state(ref, h, name)
        _assert_same_stats(ref, h, name)


@pytest.mark.parametrize("policy", ["caller", "random"])
@pytest.mark.parametrize("case,f64", A_CASES, ids=[f"{c}-{'fp64' if f else 'fp32'}" for c, f in A_CASES])
def test_fused_rollout_equals_per_tick_steps(case, f64, policy):
    """1037 envs: a ragged last 128-env tile and a partial 64-thread CTA, whose shadow lanes run the fused loop too."""
    _rollout_vs_steps(case, f64, policy)


def test_fused_rollout_equals_per_tick_steps_single_partial_cta():
    _rollout_vs_steps("cfg3", False, "caller", n=5)


def test_fused_random_policy_with_high_env_ids():
    """Global ids above 2^32 put their high bits into the Philox counter (c3hi): the in-kernel random policy of a real rollout
    must still draw what oracle.draws does for the same ids."""
    _rollout_vs_steps("cfg4", False, "random", offset=2 ** 32 + 5)


# ---------------------------------------------------------------------------------------------------------------------------
# B. launch options and the generic kernel change nothing
# ---------------------------------------------------------------------------------------------------------------------------
VARIANTS = {"specialise=0": dict(specialise=0), "pdl=0": dict(pdl=0), "prefetch_waves=0": dict(prefetch_waves=0),
            "prefetch_waves=4": dict(prefetch_waves=4), "all three": dict(specialise=0, pdl=0, prefetch_waves=0)}


@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
@pytest.mark.parametrize("base", ["cfg2", "cfg3", "cfg4"])
def test_launch_options_and_generic_kernel_are_bit_identical(base, f64):
    """The default handle (feature-specialised kernel, PDL, one prefetch wave) against one handle per option set, 30013 envs: every
    output of every tick, the terminal rows, every info array, the exported state and the statistics -- early in the episode and,
    after aging every handle with a 1700-tick fused rollout under its own options, at the steady state with auto-resets.  In the
    fp32 build cfg4 and cfg3 run compact layouts 1 and 2, so `specialise=0` runs the generic kernel on them."""
    import torch

    cfg = config.baseline_config(base)
    n, seed = 30013, 2718
    ref = _sim(cfg, n, seed, f64)
    sims = {name: _sim(cfg, n, seed, f64, **opts) for name, opts in VARIANTS.items()}
    o = ref.reset()
    for name, s in sims.items():
        assert torch.equal(s.reset(), o), name
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    resets = 0
    for phase, ticks in (("early", 30), ("steady", 60)):
        if phase == "steady":
            for s in [ref] + list(sims.values()):
                s.rollout(1700, None, want_obs=False)
        for t in range(ticks):
            act = (torch.rand(n, 6, device="cuda", generator=g) * 2.4 - 1.2).contiguous()
            want = ref.step(act, want_info=True)
            done = (want[2] | want[3]).bool()
            resets += int(done.sum())
            for name, s in sims.items():
                got = s.step(act, want_info=True)
                for x, y, what in zip(got[:4], want[:4], ("obs", "reward", "terminated", "truncated")):
                    assert torch.equal(x, y), (name, phase, t, what)
                assert torch.equal(got[4][done], want[4][done]), (name, phase, t, "terminal_obs")
                for k in want[5]:
                    assert torch.equal(got[5][k], want[5][k]), (name, phase, t, k)
    assert resets > 0
    for name, s in sims.items():
        _assert_same_state(ref, s, name)
        _assert_same_stats(ref, s, name)


@pytest.mark.parametrize("base", ["cfg4", "cfg3"])
def test_generic_kernel_in_host_chunks_matches_device_api(base):
    """HlynrVecEnv with five host chunks and the generic kernel (chunks that start at first > 0, compact layouts 1 and 2) against
    the default device API: observations, rewards, dones and every finished-episode record."""
    import torch

    from hlynr_intercept_b200.vec_env import HlynrVecEnv

    cfg = config.baseline_config(base)
    n, seed = 30013, 99
    ref = _sim(cfg, n, seed)
    v = HlynrVecEnv(cfg, n_envs=n, seed=seed, warn_dead=False, lazy_infos=True, copy_outputs=True)
    v.sim.set_option("host_chunks", 5)
    v.sim.set_option("specialise", 0)
    assert np.array_equal(v.reset(), _np(ref.reset()))
    rng = np.random.default_rng(seed)
    seen = 0
    for phase, ticks in (("early", 30), ("steady", 60)):
        if phase == "steady":
            ref.rollout(1700, None, want_obs=False)
            v.sim.rollout(1700, None, want_obs=False)
        for t in range(ticks):
            a = rng.uniform(-1.2, 1.2, (n, 6)).astype(np.float32)
            o, r, te, tr, tobs, info = ref.step(torch.as_tensor(a).cuda(), want_info=True)
            obs, rew, dones, infos = v.step(a)
            te, tr = _np(te), _np(tr)
            assert np.array_equal(obs, _np(o)) and np.array_equal(rew, _np(r)), (phase, t)
            assert np.array_equal(dones, (te | tr).astype(bool)), (phase, t)
            seen += _check_records(np.array(infos.records), te, tr, {k: _np(x) for k, x in info.items()}, _np(tobs))
    assert seen > 0
    _assert_same_state(ref, v.sim, "host chunks")
    v.close()


# ---------------------------------------------------------------------------------------------------------------------------
# C. finished-episode lists
# ---------------------------------------------------------------------------------------------------------------------------
def _check_records(rec, te, tr, info, tobs26):
    """Records of one step against the device API's [N]-sized outputs of the same tick: one record per finished env, every field.
    Returns the number of records."""
    done = (te | tr).astype(bool)
    idx = np.nonzero(done)[0]
    rec = np.sort(rec, order="env")
    assert np.array_equal(rec["env"], idx)
    for name in ("steps", "distance", "min_distance", "fuel_remaining", "fuel_used", "episode_return", "interceptor_pos",
                 "missile_pos", "missiles_intercepted", "missiles_remaining", "missile_min_distances"):
        assert np.array_equal(rec[name], info[name][idx]), name
    assert np.array_equal(rec["steps"], info["episode_length"][idx])
    fl = rec["flags"]
    assert np.array_equal(fl & 0xff, info["flags"][idx])
    assert np.array_equal((fl & abi.DONE_TERMINATED) != 0, te[idx].astype(bool))
    assert np.array_equal((fl & abi.DONE_TRUNCATED) != 0, tr[idx].astype(bool))
    assert np.array_equal((fl & abi.DONE_ONBOARD_FILL) != 0, info["radar_quality"][idx] == 0)
    assert np.array_equal(rec["terminal_obs"], tobs26[idx])
    return len(idx)


def _done_records(sim):
    ptr, cnt = C.c_void_p(), C.c_int32()
    from hlynr_intercept_b200 import _lib

    _lib.check(sim.L.hlynr_done_records_host(sim.h, C.byref(ptr), C.byref(cnt)))
    dt = abi.done_record_numpy_dtype()
    if cnt.value == 0:
        return np.zeros(0, dtype=dt)
    return np.frombuffer((C.c_char * (cnt.value * dt.itemsize)).from_address(ptr.value), dtype=dt).copy()


@pytest.mark.parametrize("obs_dim", [26, 17])
def test_host_done_list_past_the_prefix(obs_dim):
    """hlynr_step_host fetches the first 4096 records together with the count and the rest in a second copy.  With max_steps 30,
    all 70001 envs truncate in the same step: every record, and every terminal row hlynr_step_host scatters into the caller's
    buffer, must equal the device API's outputs of that tick."""
    import torch

    from hlynr_intercept_b200 import _lib

    cfg = config.baseline_config("cfg4")
    cfg["max_steps"] = 30
    n, seed = 70001, 5
    ref = _sim(cfg, n, seed)
    host = _sim(cfg, n, seed, obs_dim=obs_dim)
    assert np.array_equal(_np(host.reset()), _np(ref.reset())[:, :obs_dim])
    obs, rew = np.zeros((n, obs_dim), np.float32), np.zeros(n, np.float32)
    te_h, tr_h = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
    p = lambda x: x.ctypes.data_as(C.c_void_p)  # noqa: E731
    rng = np.random.default_rng(1)
    most = 0
    for t in range(32):
        a = rng.uniform(-1, 1, (n, 6)).astype(np.float32)
        tobs_h = np.full((n, obs_dim), np.nan, np.float32)
        o, r, te, tr, tobs, info = ref.step(torch.as_tensor(a).cuda(), want_info=True)
        _lib.check(host.L.hlynr_step_host(host.h, p(a), p(obs), p(rew), p(te_h), p(tr_h), p(tobs_h), 1))
        te, tr, tobs = _np(te), _np(tr), _np(tobs)
        assert np.array_equal(obs, _np(o)[:, :obs_dim]) and np.array_equal(rew, _np(r)), t
        assert np.array_equal(te_h, te) and np.array_equal(tr_h, tr), t
        rec = _done_records(host)
        cnt = _check_records(rec, te, tr, {k: _np(x) for k, x in info.items()}, tobs)
        done = (te | tr).astype(bool)
        assert np.array_equal(tobs_h[done], tobs[done][:, :obs_dim]), t
        assert np.isnan(tobs_h[~done]).all(), t
        most = max(most, cnt)
    assert most > 10 * 4096, most


def test_attached_device_done_list_drops_records_past_capacity():
    """hlynr_set_done_list with a capacity below the number of envs that finish in a step: the counter still counts every
    finished env, exactly `capacity` records are written (each one of a finished env, equal to its info values) and nothing is
    written past them (64 guard records filled with a sentinel stay intact)."""
    import torch

    from hlynr_intercept_b200 import _lib

    cfg = config.baseline_config("cfg4")
    cfg["max_steps"] = 30
    n, cap, guard = 20000, 1500, 64
    dt = abi.done_record_numpy_dtype()
    sim = _sim(cfg, n, 8)
    recs = torch.full(((cap + guard) * dt.itemsize,), 0xA5, dtype=torch.uint8, device="cuda")
    counter = torch.zeros(1, dtype=torch.int32, device="cuda")
    _lib.check(sim.L.hlynr_set_done_list(sim.h, C.c_void_p(recs.data_ptr()), C.c_void_p(counter.data_ptr()), cap))
    sentinel = np.full(guard * dt.itemsize, 0xA5, np.uint8)
    sim.reset()
    rng = np.random.default_rng(2)
    overflowed = 0
    try:
        for t in range(32):
            counter.zero_()
            recs[:cap * dt.itemsize].fill_(0xA5)
            a = torch.as_tensor(rng.uniform(-1, 1, (n, 6)).astype(np.float32)).cuda()
            _, _, te, tr, tobs, info = sim.step(a, want_info=True)
            te, tr, tobs = _np(te), _np(tr), _np(tobs)
            info = {k: _np(x) for k, x in info.items()}
            done = (te | tr).astype(bool)
            total = int(counter.item())
            assert total == int(done.sum()), t
            raw = _np(recs)
            assert np.array_equal(raw[cap * dt.itemsize:], sentinel), t
            written = min(total, cap)
            assert (raw[written * dt.itemsize:cap * dt.itemsize] == 0xA5).all(), t
            rec = raw[:written * dt.itemsize].view(dt)
            env = rec["env"]
            assert len(np.unique(env)) == written and done[env].all(), t
            for name in ("steps", "distance", "min_distance", "fuel_remaining", "fuel_used", "episode_return", "interceptor_pos",
                         "missile_pos", "missiles_intercepted", "missiles_remaining", "missile_min_distances"):
                assert np.array_equal(rec[name], info[name][env]), (t, name)
            assert np.array_equal(rec["flags"] & 0xff, info["flags"][env]), t
            assert np.array_equal((rec["flags"] & abi.DONE_TRUNCATED) != 0, tr[env].astype(bool)), t
            assert np.array_equal(rec["terminal_obs"], tobs[env]), t
            overflowed += total > cap
    finally:
        _lib.check(sim.L.hlynr_set_done_list(sim.h, None, None, 0))
        torch.cuda.synchronize()
    assert overflowed > 0

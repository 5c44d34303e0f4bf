"""Checkpoint and resume (include/hlynr.h hlynr_snapshot_*, include/hlynr_post.h hlynr_post_snapshot_*, checkpoint.py).

CPU: the descriptor mirrors have the library's sizes, the entry points refuse null pointers, and checkpoint.load refuses a file
with a flipped byte in any section, a truncated file and another format version.
GPU: a run that is saved, torn down, rebuilt and loaded continues bit for bit like the uninterrupted run (every layout and
feature set of the step kernels, snapshots taken at ticks off the ring period and while the delay rings refill), across the
compact and wide layouts; saving does not disturb the run; mismatched handles are refused with a message."""
import ctypes as C
import json
import zipfile

import numpy as np
import pytest

from hlynr_intercept_b200 import _lib, abi, checkpoint, config

N = 300   # a ragged tile


# ---- CPU -------------------------------------------------------------------------------------------------------------------------

def test_descriptor_mirrors_have_the_library_sizes():
    L = _lib.load()
    assert L.hlynr_snapshot_info_size() == C.sizeof(abi.HlynrSnapshotInfo)
    assert L.hlynr_post_snapshot_info_size() == C.sizeof(abi.HlynrPostSnapshotInfo)
    assert len(abi.HlynrSnapshotInfo().section_offset) == len(abi.SNAP_SECTIONS)
    info = abi.HlynrSnapshotInfo(tick=2 ** 63 + 5, env_steps=0.1, seed=2 ** 64 - 1)
    info.params.dr_variation[3] = 1.0 / 3.0
    d = json.loads(json.dumps(abi.struct_to_dict(info)))
    assert bytes(abi.struct_from_dict(abi.HlynrSnapshotInfo, d)) == bytes(info)
    d.pop("tick")
    with pytest.raises(ValueError, match="tick"):
        abi.struct_from_dict(abi.HlynrSnapshotInfo, d)


def test_entry_points_refuse_null_pointers():
    L = _lib.load()
    info, pinfo, nb, buf = abi.HlynrSnapshotInfo(), abi.HlynrPostSnapshotInfo(), C.c_size_t(), C.c_void_p(16)
    calls = [("hlynr_snapshot_layout", lambda: L.hlynr_snapshot_layout(None, C.byref(info), C.byref(nb))),
             ("hlynr_snapshot_save", lambda: L.hlynr_snapshot_save(None, buf, C.byref(info), None)),
             ("hlynr_snapshot_load", lambda: L.hlynr_snapshot_load(None, C.byref(info), buf, None)),
             ("hlynr_post_snapshot_layout", lambda: L.hlynr_post_snapshot_layout(None, C.byref(pinfo), C.byref(nb))),
             ("hlynr_post_snapshot_save", lambda: L.hlynr_post_snapshot_save(None, buf, C.byref(pinfo), None)),
             ("hlynr_post_snapshot_load", lambda: L.hlynr_post_snapshot_load(None, C.byref(pinfo), buf, None))]
    for name, call in calls:
        assert call() != 0, name
        assert L.hlynr_last_error().decode() == f"{name}: null argument"


class _Part:
    def __init__(self, state):
        self.state, self.loaded = state, None

    def state_dict(self):
        return self.state

    def load_state_dict(self, state):
        self.loaded = state


def _parts():
    rng = np.random.default_rng(3)
    return dict(sim=_Part({"info": {"tick": 17, "params": {"dt": 0.01}}, "image": rng.integers(0, 255, 4000, dtype=np.uint8)}),
                pipe=_Part({"info": {"t": 9}, "image": rng.integers(0, 255, 3000, dtype=np.uint8), "training": True}),
                collector=_Part({"next_obs": rng.standard_normal((7, 104)).astype(np.float32), "started": True,
                                 "last_dones": np.ones(7, np.uint8), "overflow": np.zeros(1, np.int32)}),
                policy=_Part({"calls": 123, "seed": 77}))


def test_checkpoint_round_trip_and_refusals(tmp_path):
    parts = _parts()
    path = str(tmp_path / "ckpt.npz")
    checkpoint.save(path, **parts)
    fresh = {k: _Part(None) for k in parts}
    assert checkpoint.load(path, **fresh) == sorted(parts)
    for k, p in parts.items():
        for key, v in p.state.items():
            got = fresh[k].loaded[key]
            if isinstance(v, np.ndarray):
                assert got.dtype == v.dtype and got.tobytes() == v.tobytes(), (k, key)
            else:
                assert got == v, (k, key)
    raw = open(path, "rb").read()
    # a flipped byte in the data of every section (every array of the archive) is refused
    with zipfile.ZipFile(path) as z:
        infos = z.infolist()
    assert {i.filename for i in infos} >= {"descriptor.npy", "descriptor_crc32.npy", "sim.image.npy", "pipe.image.npy",
                                           "collector.next_obs.npy"}
    for zi in infos:
        data_start = zi.header_offset + 30 + len(zi.filename.encode()) + len(zi.extra)
        pos = data_start + zi.compress_size - 1   # the member's last byte: array data, past the .npy header
        bad = bytearray(raw)
        bad[pos] ^= 0x40
        p = str(tmp_path / f"bad_{zi.filename}.npz")
        open(p, "wb").write(bytes(bad))
        with pytest.raises(checkpoint.CheckpointError):
            checkpoint.load(p, **{k: _Part(None) for k in parts})
    for cut in (len(raw) // 2, len(raw) - 10):
        p = str(tmp_path / f"cut{cut}.npz")
        open(p, "wb").write(raw[:cut])
        with pytest.raises(checkpoint.CheckpointError):
            checkpoint.load(p, sim=_Part(None))
    # another format version, with a consistent checksum
    with np.load(path) as z:
        files = {k: z[k] for k in z.files}
    desc = json.loads(files["descriptor"].tobytes())
    desc["format_version"] = checkpoint.FORMAT_VERSION + 1
    files["descriptor"] = np.frombuffer(json.dumps(desc).encode(), np.uint8)
    files["descriptor_crc32"] = np.array([checkpoint._crc(files["descriptor"])], np.uint32)
    p = str(tmp_path / "v2.npz")
    np.savez(p, **files)
    with pytest.raises(checkpoint.CheckpointError, match="format version"):
        checkpoint.load(p, sim=_Part(None))
    # a part the caller asks for but the file does not hold
    p = str(tmp_path / "policy_only.npz")
    checkpoint.save(p, policy=parts["policy"])
    with pytest.raises(checkpoint.CheckpointError, match="sim"):
        checkpoint.load(p, sim=_Part(None), policy=_Part(None))


# ---- GPU -------------------------------------------------------------------------------------------------------------------------

ROLLOUT = ("obs", "actions", "values", "log_probs", "rewards", "advantages", "returns", "episode_starts")


def _cfg(name):
    if name == "volley":
        e = config.baseline_config("cfg4")
        e.update(volley_mode=True, volley_size=3, max_steps=60)
        e["missile_spawn"] = dict(position=[[150, 150, 100], [260, 260, 220]], velocity=[[-110, -110, -55], [-160, -160, -75]])
        return e
    if name == "curriculum":
        from test_device_curriculum import _ramps_cfg

        return _ramps_cfg(unit=N)
    e = config.baseline_config(name)
    e["max_steps"] = 200
    return e


def _build(cfg, precision="fp32", obs_dim=26, n_stack=4, track=None, seed=23, n=N, env_id_offset=0):
    from hlynr_intercept_b200.post import HlynrObsPipeline
    from hlynr_intercept_b200.rollout import DeviceRolloutCollector
    from hlynr_intercept_b200.sim import HlynrSim
    from test_obs_widths import _fused, _net_d

    sim = HlynrSim(cfg, n_envs=n, seed=seed, warn_dead=False, precision=precision, obs_dim=obs_dim, env_id_offset=env_id_offset)
    if track is not None:
        sim.track_training_steps(track)
    pipe = HlynrObsPipeline(sim, n_stack=n_stack, training=True)
    fused = _fused(_net_d(pipe.obs_dim, seed=45), seed=77)
    T = DeviceRolloutCollector(pipe, None, 1).graph_period()
    return DeviceRolloutCollector(pipe, fused, T, bootstrap_rows=None)


def _pre(col, k0):
    """k0 eager ticks before the collector's first reset: the rings and the tick go on through that reset, so the snapshot after
    one rollout is taken at tick k0 + T, off the ring period."""
    import torch

    g = torch.Generator(device="cuda")
    g.manual_seed(5)
    col.pipe.reset()
    for _ in range(k0):
        col.pipe.step(torch.rand(col.sim.n, 6, device="cuda", generator=g) * 2 - 1)


def _rollout(col):
    import torch

    torch.cuda.synchronize()
    return {k: getattr(col, k).cpu().numpy().copy() for k in ROLLOUT}


def _end(col):
    return dict(stats=col.sim.stats(), state=col.sim.export_state(), num_timesteps=col.sim.num_timesteps, calls=col.policy.calls,
                tick=col.sim.tick_count(), vecnorm=col.pipe.get_stats())


def _close(col):
    col.policy.close(); col.pipe.close(); col.sim.close()


def _assert_same(a, b):
    ra, ea = a
    rb, eb = b
    for k in ROLLOUT:
        assert ra[k].tobytes() == rb[k].tobytes(), f"second rollout: {k}"
    assert ea["stats"] == eb["stats"]
    for k in ea["state"]:
        assert ea["state"][k].tobytes() == eb["state"][k].tobytes(), f"export_state {k}"
    assert ea["num_timesteps"] == eb["num_timesteps"] and ea["calls"] == eb["calls"] and ea["tick"] == eb["tick"]
    # obs_rms subtracts the frames of a step's finished episodes in done-list order, which the step kernel's atomic appends leave
    # unspecified, so two uninterrupted runs too can differ in the last bits when many episodes end in one step
    for k in ea["vecnorm"]:
        np.testing.assert_allclose(ea["vecnorm"][k], eb["vecnorm"][k], rtol=1e-12, atol=0, err_msg=f"VecNormalize {k}")


def _uninterrupted(make, k0, save_midway=None):
    col = make()
    _pre(col, k0)
    col.capture()   # rollout 1: the warm-up collect
    if save_midway:
        checkpoint.save(save_midway, sim=col.sim, pipe=col.pipe, collector=col, policy=col.policy)
    col.replay()    # rollout 2
    out = (_rollout(col), _end(col))
    _close(col)
    return out


def _interrupted(make, remake, k0, path):
    col = make()
    _pre(col, k0)
    col.capture()
    checkpoint.save(path, sim=col.sim, pipe=col.pipe, collector=col, policy=col.policy)
    _close(col)
    del col
    col = remake()
    checkpoint.load(path, sim=col.sim, pipe=col.pipe, collector=col, policy=col.policy)
    col.capture()   # re-captured after the load; its warm-up collect is rollout 2
    first, end = _rollout(col), _end(col)
    _close(col)
    return first, end


CASES = {   # name -> (cfg, build kwargs, k0)
    "cfg4_compact": ("cfg4", {}, 5),
    "cfg4_wide": ("cfg4", {}, 5),
    "cfg3_dr": ("cfg3", {}, 3),
    "cfg2": ("cfg2", {}, 7),
    "cfg4_fp64": ("cfg4", dict(precision="fp64"), 5),
    "volley3": ("volley", {}, 5),
    "obs17_stack4": ("cfg4", dict(obs_dim=17, n_stack=4), 5),
    "curriculum": ("curriculum", dict(track=7 * N + 3), 5),
    "rings_refilling": ("cfg4", {}, 5),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_resumed_run_continues_bit_for_bit(case, tmp_path, monkeypatch):
    """Twin A collects two rollouts (fused policy, graph replays), then a third by replay; twin B collects one, is saved, torn
    down, rebuilt and loaded, re-captures (its warm-up collect is rollout 2) and replays rollout 3.  B's rollouts 2 and 3 and
    the end state equal A's byte for byte."""
    name, kw, k0 = CASES[case]
    if case == "cfg4_wide":
        monkeypatch.setenv("HLYNR_NO_COMPACT", "1")
    cfg = _cfg(name)
    if case == "rings_refilling":
        # a 12-tick rollout after a reset at tick 5: every env still running truncates at step 11 (tick 16), so at the snapshot
        # (tick 17) it is one tick into a new episode, inside the 3-tick onboard delay
        cfg["max_steps"] = 11
    make = lambda: _build(cfg, **kw)  # noqa: E731
    col = make()
    per, T = col.sim.ring_period(), col.T
    _close(col)
    assert (k0 + T) % per != 0
    # A: rollouts 1, 2 and 3 (compare rollout 2 with B's warm-up, rollout 3 with B's replay)
    a = make()
    _pre(a, k0)
    a.capture()
    a.replay()
    a2 = _rollout(a)
    a.replay()
    a3, a_end = _rollout(a), _end(a)
    _close(a)
    # B
    path = str(tmp_path / "ckpt.npz")
    b = make()
    _pre(b, k0)
    b.capture()
    checkpoint.save(path, sim=b.sim, pipe=b.pipe, collector=b, policy=b.policy)
    _close(b)
    del b
    b = _build(cfg, **{k: v for k, v in kw.items() if k != "track"})   # fresh handles; the load re-attaches a schedule
    checkpoint.load(path, sim=b.sim, pipe=b.pipe, collector=b, policy=b.policy)
    assert b.sim.tick_count() == k0 + T
    b.capture()
    b2 = _rollout(b)
    b.replay()
    b3, b_end = _rollout(b), _end(b)
    _close(b)
    for k in ROLLOUT:
        assert a2[k].tobytes() == b2[k].tobytes(), f"rollout 2: {k}"
    _assert_same((a3, a_end), (b3, b_end))
    if case == "rings_refilling":
        assert float(a2["episode_starts"][0].sum()) == 0 and float(a2["episode_starts"].sum()) > 0   # episodes end inside rollout 2


@pytest.mark.gpu
def test_compact_snapshot_loads_into_a_wide_handle(tmp_path, monkeypatch):
    """The image is canonical: a snapshot of the compact layout continues in the wide layout like the uninterrupted compact run."""
    cfg = _cfg("cfg4")
    make = lambda: _build(cfg)  # noqa: E731
    ref = _uninterrupted(make, 5)

    def wide():
        monkeypatch.setenv("HLYNR_NO_COMPACT", "1")
        try:
            return make()
        finally:
            monkeypatch.delenv("HLYNR_NO_COMPACT")

    _assert_same(ref, _interrupted(make, wide, 5, str(tmp_path / "c.npz")))
    # and back: wide to compact
    _assert_same(ref, _interrupted(wide, make, 5, str(tmp_path / "w.npz")))


@pytest.mark.gpu
def test_saving_does_not_disturb_the_run(tmp_path):
    cfg = _cfg("cfg4")
    make = lambda: _build(cfg)  # noqa: E731
    _assert_same(_uninterrupted(make, 5), _uninterrupted(make, 5, save_midway=str(tmp_path / "m.npz")))


@pytest.mark.gpu
def test_mismatched_handles_are_refused(tmp_path):
    import torch

    from hlynr_intercept_b200.post import HlynrObsPipeline
    from hlynr_intercept_b200.sim import HlynrSim

    cfg = _cfg("cfg4")
    sim = HlynrSim(cfg, n_envs=N, seed=3, warn_dead=False)
    pipe = HlynrObsPipeline(sim, n_stack=4)
    pipe.reset()
    s, p = sim.state_dict(), pipe.state_dict()
    other = dict(cfg, max_steps=cfg["max_steps"] + 1)
    refusals = [(dict(env_cfg=other), "HlynrParams.max_steps"), (dict(precision="fp64"), "precision"),
                (dict(n_envs=N + 1), "n_envs"), (dict(env_id_offset=N), "env_id_offset"), (dict(obs_dim=17), "obs_dim")]
    for kw, what in refusals:
        args = dict(env_cfg=cfg, n_envs=N, seed=3, warn_dead=False)
        args.update(kw)
        t = HlynrSim(**args)
        with pytest.raises(_lib.HlynrError, match=what):
            t.load_state_dict(s)
        t.close()
    for kw, what in ((dict(n_stack=2), "n_stack"), (dict(gamma=0.98), "gamma"), (dict(clip_obs=5.0), "clip_obs")):
        q = HlynrObsPipeline(sim, **kw)
        with pytest.raises(_lib.HlynrError, match=what):
            q.load_state_dict(p)
        q.close()
    pipe.close()
    pipe = HlynrObsPipeline(sim, n_stack=4)
    # a capturing stream: both directions refuse and enqueue nothing
    L = sim.L
    info, pinfo = abi.struct_from_dict(abi.HlynrSnapshotInfo, s["info"]), abi.struct_from_dict(abi.HlynrPostSnapshotInfo, p["info"])
    buf = torch.empty(max(info.device_bytes, pinfo.device_bytes), dtype=torch.uint8, device="cuda")
    x = torch.zeros(4, device="cuda")
    g, side = torch.cuda.CUDAGraph(), torch.cuda.Stream()
    with torch.cuda.graph(g, stream=side):
        st = C.c_void_p(side.cuda_stream)
        rc = [L.hlynr_snapshot_save(sim.h, C.c_void_p(buf.data_ptr()), C.byref(info), st),
              L.hlynr_snapshot_load(sim.h, C.byref(info), C.c_void_p(buf.data_ptr()), st),
              L.hlynr_post_snapshot_save(pipe.h, C.c_void_p(buf.data_ptr()), C.byref(pinfo), st),
              L.hlynr_post_snapshot_load(pipe.h, C.byref(pinfo), C.c_void_p(buf.data_ptr()), st)]
        msg = L.hlynr_last_error().decode()
        x.add_(1)
    assert all(r != 0 for r in rc) and "capturing" in msg, (rc, msg)
    # a descriptor of another format version
    bad = dict(s, info=dict(s["info"], format_version=abi.SNAPSHOT_VERSION + 1))
    with pytest.raises(_lib.HlynrError, match="format version"):
        sim.load_state_dict(bad)
    pipe.close(); sim.close()

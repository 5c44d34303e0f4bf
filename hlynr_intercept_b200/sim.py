"""HlynrSim: the device-resident batched simulator (one GPU shard) behind the C ABI of include/hlynr.h.

`step(actions_cuda)` is the tensor API used for >= 64k envs (no per-env Python objects, no infos);
`HlynrVecEnv` (vec_env.py) layers the Stable-Baselines3 VecEnv contract on top of the host-buffer entry
points.  torch is plumbing only: it owns the caller-side device tensors and the current stream.
"""
import ctypes as C

import numpy as np

from . import _lib, abi, config as _config


class HlynrSim:
    def __init__(self, env_cfg=None, n_envs=1, device=0, seed=1234, env_id_offset=0, precision="fp32",
                 params=None, curriculum=None, warn_dead=True, obs_dim=26):
        import torch

        if not torch.cuda.is_available():
            raise _lib.HlynrError("HlynrSim needs a CUDA device: there is no CPU fallback")
        self.L = _lib.load()
        if params is None:
            params, curriculum = _config.resolve_config(env_cfg, warn_dead=warn_dead)
        self.params, self.curriculum = params, curriculum
        self.n = int(n_envs)
        self.device_index = int(device)
        self.device = torch.device("cuda", self.device_index)
        self.precision = {"fp32": abi.FP32, "fp64": abi.FP64, 32: abi.FP32, 64: abi.FP64}[precision]
        self.seed_value = int(seed)
        self.env_id_offset = int(env_id_offset)
        h = C.c_void_p()
        _lib.check(self.L.hlynr_create(C.byref(params), self.n, self.device_index, self.seed_value, self.env_id_offset,
                                       self.precision, C.byref(h)))
        self.h = h
        self.obs_dim = int(obs_dim)
        if self.obs_dim != 26:   # 17: the leading radar channels obs[0:17] only (include/hlynr.h, option "obs_dim")
            _lib.check(self.L.hlynr_set_option(self.h, b"obs_dim", self.obs_dim))
        self.push_curriculum()
        self.tracking = False
        self._torch = torch
        self._info_t = None
        self._out = None

    # ---- plumbing -------------------------------------------------------------------------------------
    def _stream(self):
        return C.c_void_p(self._torch.cuda.current_stream(self.device).cuda_stream)

    def _alloc_out(self):
        t = self._torch
        if self._out is None:
            n, d = self.n, self.device
            self._out = dict(obs=t.empty((n, self.obs_dim), dtype=t.float32, device=d), reward=t.empty(n, dtype=t.float32, device=d),
                             terminated=t.empty(n, dtype=t.uint8, device=d), truncated=t.empty(n, dtype=t.uint8, device=d),
                             terminal_obs=t.full((n, self.obs_dim), float("nan"), dtype=t.float32, device=d))
        return self._out

    def info_tensors(self):
        t = self._torch
        if self._info_t is None:
            tt = {"float32": t.float32, "int32": t.int32, "uint8": t.uint8}
            self._info_t = {n: t.zeros((self.n,) + shp, dtype=tt[dt], device=self.device) for n, dt, shp in abi.INFO_FIELDS}
            self._info_struct = abi.HlynrInfoSoA(**{n: self._info_t[n].data_ptr() for n, _, _ in abi.INFO_FIELDS})
        return self._info_t

    # ---- reference-facing operations --------------------------------------------------------------------
    def push_curriculum(self):
        c = self.curriculum.to_struct()
        _lib.check(self.L.hlynr_set_curriculum(self.h, C.byref(c)))

    def set_training_step_count(self, n):
        """environment.py:269 set_training_step_count (global to all envs).  While tracking: sets the device counter, ordered on the
        current stream."""
        self.curriculum.set_training_step_count(n)
        if self.tracking:
            _lib.check(self.L.hlynr_set_timesteps(self.h, int(n), self._stream()))
        else:
            self.push_curriculum()

    def get_current_intercept_radius(self):
        """environment.py:223.  While tracking: at the device counter (synchronises the current stream)."""
        if self.tracking:
            self.curriculum.set_training_step_count(self.num_timesteps)
        return self.curriculum.intercept_radius()

    def track_training_steps(self, num_timesteps=0, increment=None):
        """Advance the curriculum on the device, as SB3's per-step set_training_step_count callback would: every step() first
        computes the curriculum of the device counter, then adds `increment` to it (default: this sim's n; a shard of a multi-GPU
        run passes the global env count).  reset() uses the counter without advancing it.  Eager steps, StepGraph replays and
        DeviceRolloutCollector replays all continue the schedule.  step_host-based paths (HlynrVecEnv) and rollout() refuse to run
        while tracking; untrack_training_steps() ends it."""
        increment = self.n if increment is None else int(increment)
        _lib.check(self.L.hlynr_attach_curriculum(self.h, C.byref(self.curriculum.schedule()), int(num_timesteps), increment))
        self.curriculum.set_training_step_count(int(num_timesteps))
        self.tracking, self.increment = True, increment

    def untrack_training_steps(self):
        """Back to the host-pushed curriculum, set to the values of the device counter's current count."""
        if not self.tracking:
            return
        n = self.num_timesteps
        _lib.check(self.L.hlynr_detach_curriculum(self.h))
        self.tracking = False
        self.set_training_step_count(n)

    @property
    def num_timesteps(self):
        """The training-step count: the device counter while tracking (synchronises the current stream), else the last pushed."""
        if not self.tracking:
            return self.curriculum.training_step_count
        v = C.c_uint64()
        _lib.check(self.L.hlynr_get_timesteps(self.h, C.byref(v), self._stream()))
        return v.value

    def debug_curriculum_at(self, count):
        """(intercept radius, cos of the half beam width, onboard reliability, ground reliability) the device computes from the
        tracked schedule at `count`, as float64 (test hook)."""
        out = (C.c_double * 4)()
        _lib.check(self.L.hlynr_debug_curriculum_at(self.h, int(count), out))
        return tuple(out)

    def seed(self, seed):
        self.seed_value = int(seed)
        _lib.check(self.L.hlynr_seed(self.h, self.seed_value))

    def reset(self, mask=None, out=None):
        """reset() of every env (or of mask != 0): returns obs[N,26] float32 on the device."""
        o = self._alloc_out()
        obs = o["obs"] if out is None else out
        m = None
        if mask is not None:
            m = mask.to(device=self.device, dtype=self._torch.uint8).contiguous()
        _lib.check(self.L.hlynr_reset(self.h, C.c_void_p(m.data_ptr()) if m is not None else None,
                                      C.c_void_p(obs.data_ptr()), self._stream()))
        return obs

    def step(self, actions, auto_reset=True, want_info=False, want_terminal_obs=True):
        """One tick of every env.  actions: float32 cuda tensor [N,6].
        Returns (obs, reward, terminated, truncated, terminal_obs_or_None, info_dict_or_None), all device tensors
        that are overwritten by the next call."""
        t = self._torch
        if not (actions.is_cuda and actions.dtype == t.float32 and actions.shape == (self.n, 6) and actions.is_contiguous()):
            actions = actions.to(device=self.device, dtype=t.float32).reshape(self.n, 6).contiguous()
        o = self._alloc_out()
        info = None
        if want_info:
            self.info_tensors()
            info = C.byref(self._info_struct)
        _lib.check(self.L.hlynr_step(self.h, C.c_void_p(actions.data_ptr()), C.c_void_p(o["obs"].data_ptr()),
                                     C.c_void_p(o["reward"].data_ptr()), C.c_void_p(o["terminated"].data_ptr()),
                                     C.c_void_p(o["truncated"].data_ptr()),
                                     C.c_void_p(o["terminal_obs"].data_ptr()) if want_terminal_obs else None,
                                     info, int(auto_reset), self._stream()))
        return (o["obs"], o["reward"], o["terminated"], o["truncated"], o["terminal_obs"] if want_terminal_obs else None,
                self._info_t if want_info else None)

    def rollout(self, k_steps, actions=None, want_obs=True):
        """k fused ticks in one launch (state in registers).  actions: None = in-kernel random policy, or a float32
        cuda tensor [k,N,6].  Returns (obs_after_last_tick[N,obs_dim] or None, reward_sum[N], done_count[N])."""
        t = self._torch
        o = self._alloc_out()
        if not hasattr(self, "_rsum"):
            self._rsum = t.empty(self.n, dtype=t.float32, device=self.device)
            self._dcount = t.empty(self.n, dtype=t.int32, device=self.device)
        ap = None
        if actions is not None:
            assert actions.is_cuda and actions.dtype == t.float32 and actions.shape == (k_steps, self.n, 6)
            actions = actions.contiguous()
            ap = C.c_void_p(actions.data_ptr())
        _lib.check(self.L.hlynr_rollout(self.h, int(k_steps), ap, C.c_void_p(o["obs"].data_ptr()) if want_obs else None,
                                        C.c_void_p(self._rsum.data_ptr()), C.c_void_p(self._dcount.data_ptr()),
                                        self._stream()))
        return (o["obs"] if want_obs else None), self._rsum, self._dcount

    # ---- statistics / state interchange -----------------------------------------------------------------
    def stats(self, zero_after=False):
        s = abi.HlynrStats()
        _lib.check(self.L.hlynr_get_stats(self.h, C.byref(s), int(zero_after), self._stream()))
        return {n: getattr(s, n) for n in abi.STATS_FIELDS[:14]}

    def stats_tensor(self):
        """The reduced statistics block as a float64 cuda tensor view (for an in-place NCCL all-reduce)."""
        import torch

        p = C.c_void_p()
        _lib.check(self.L.hlynr_stats_reduce(self.h, self._stream()))
        _lib.check(self.L.hlynr_stats_device_ptr(self.h, C.byref(p)))
        return _tensor_from_ptr(torch, p.value, (abi.STATS_WORDS,), torch.float64, self.device)

    def export_state(self, first=0, count=None):
        count = self.n - first if count is None else count
        arr = np.zeros(count, dtype=abi.env_state_numpy_dtype())
        _lib.check(self.L.hlynr_export_state(self.h, first, count, arr.ctypes.data_as(C.c_void_p)))
        return {k: arr[k].copy() for k in arr.dtype.names}

    def import_state(self, state, first=0):
        dt = abi.env_state_numpy_dtype()
        count = len(state["steps"])
        arr = np.zeros(count, dtype=dt)
        for k in dt.names:
            arr[k] = state[k]
        _lib.check(self.L.hlynr_import_state(self.h, first, count, arr.ctypes.data_as(C.c_void_p)))

    # ---- snapshots (include/hlynr.h hlynr_snapshot_*, DESIGN.md section 17) ------------------------------------------------
    def state_dict(self):
        """The whole shard's state: {'info': the descriptor as a dict, 'image': its canonical device image as a uint8 CPU tensor,
        'training_step_count': the host curriculum's count}.  Every env (episodes in flight, delay rings, Kalman tracks,
        domain-randomised draws), the statistics block, the tick, the seed, the curriculum and an attached schedule with its device
        count.  Synchronises the current stream."""
        info, nbytes = abi.HlynrSnapshotInfo(), C.c_size_t()
        _lib.check(self.L.hlynr_snapshot_layout(self.h, C.byref(info), C.byref(nbytes)))
        dev = self._torch.empty(nbytes.value, dtype=self._torch.uint8, device=self.device)
        _lib.check(self.L.hlynr_snapshot_save(self.h, C.c_void_p(dev.data_ptr()), C.byref(info), self._stream()))
        return {"info": abi.struct_to_dict(info), "image": image_to_host(self._torch, dev),
                "training_step_count": self.curriculum.training_step_count}

    def load_state_dict(self, state):
        """Restores a state_dict() into this sim, which must have been created with the same configuration, precision, n_envs,
        env_id_offset and obs_dim (refused otherwise, naming the first difference).  Options are kept.  A StepGraph or collector
        graph captured before the load must be captured again."""
        info = abi.struct_from_dict(abi.HlynrSnapshotInfo, state["info"])
        dev = image_to_device(self._torch, state["image"], info.device_bytes, self.device)
        _lib.check(self.L.hlynr_snapshot_load(self.h, C.byref(info), C.c_void_p(dev.data_ptr()), self._stream()))
        self.seed_value = int(info.seed)
        self.curriculum.set_training_step_count(state["training_step_count"])
        self.tracking = bool(info.curriculum_attached)
        if self.tracking:
            self.increment = int(info.curriculum_increment)

    def debug_draws(self, env_global_id, episode, step, block):
        raw, uni, nrm = np.zeros(4, np.uint32), np.zeros(4, np.float32), np.zeros(4, np.float32)
        _lib.check(self.L.hlynr_debug_draws(self.h, env_global_id, episode, step, block, raw.ctypes.data_as(C.c_void_p),
                                            uni.ctypes.data_as(C.c_void_p), nrm.ctypes.data_as(C.c_void_p)))
        return raw, uni, nrm

    def ring_period(self):
        """A captured sequence of T ticks replays correctly iff T is a multiple of this (include/hlynr.h, CUDA-graph support)."""
        per = C.c_int()
        _lib.check(self.L.hlynr_ring_period(self.h, C.byref(per)))
        return per.value

    def tick_count(self):
        v = C.c_int64()
        _lib.check(self.L.hlynr_tick_count(self.h, C.byref(v)))
        return v.value

    def capture_steps(self, actions_seq, want_terminal_obs=False):
        """Captures len(actions_seq) consecutive step() calls into ONE CUDA graph (small batches are launch-bound: a tick of 4096
        envs is ~6 us of GPU work behind ~10 us of Python + launch overhead).  actions_seq: list of persistent float32 cuda
        tensors [N,6] the caller refills between replays; its length must be a multiple of ring_period().  Returns a StepGraph
        whose replay() runs the ticks and leaves the LAST tick's outputs in the tensors step() returns."""
        return StepGraph(self, actions_seq, want_terminal_obs)

    def set_option(self, name, value):
        _lib.check(self.L.hlynr_set_option(self.h, name.encode(), int(value)))

    def launch_count(self):
        v = C.c_int64()
        _lib.check(self.L.hlynr_launch_count(self.h, C.byref(v)))
        return v.value

    def close(self):
        if getattr(self, "h", None):
            self.L.hlynr_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class StepGraph:
    def __init__(self, sim, actions_seq, want_terminal_obs=False):
        torch = sim._torch
        T = len(actions_seq)
        if T == 0 or T % sim.ring_period():
            raise ValueError(f"a step graph needs a multiple of ring_period() = {sim.ring_period()} ticks, got {T}")
        self.sim, self.T = sim, T
        self.period = sim.ring_period()
        self.phase = sim.tick_count() % self.period
        sim._alloc_out()
        torch.cuda.synchronize(sim.device)
        l0 = sim.launch_count()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):   # recorded, not executed: only the host-side tick counter advances ...
            for a in actions_seq:
                self.out = sim.step(a, want_terminal_obs=want_terminal_obs)
        self.launches = sim.launch_count() - l0
        # ... and is put back (ring phases are unchanged: T is a multiple of every ring length)
        _lib.check(sim.L.hlynr_note_replayed_ticks(sim.h, -T, -self.launches))

    def replay(self):
        if self.sim.tick_count() % self.period != self.phase:   # the delay-ring rows are baked into the captured launches
            raise _lib.HlynrError(f"StepGraph captured at tick phase {self.phase} (mod {self.period}) cannot replay at phase "
                                  f"{self.sim.tick_count() % self.period}: step eagerly to the next multiple of ring_period() first")
        self.graph.replay()
        _lib.check(self.sim.L.hlynr_note_replayed_ticks(self.sim.h, self.T, self.launches))
        return self.out


def image_to_host(torch, dev):
    """A snapshot's device image as a CPU tensor, copied through pinned memory (synchronises the current stream)."""
    host = torch.empty(dev.numel(), dtype=torch.uint8, pin_memory=True)
    host.copy_(dev, non_blocking=True)
    torch.cuda.current_stream(dev.device).synchronize()
    return host


def image_to_device(torch, image, nbytes, device):
    """A snapshot's image (CPU tensor or numpy array of bytes) on the device, through pinned memory, ordered on the current stream."""
    image = torch.as_tensor(image).reshape(-1).view(torch.uint8)
    if image.numel() != nbytes:
        raise ValueError(f"the snapshot image has {image.numel()} bytes, its descriptor says {nbytes}")
    host = torch.empty(image.numel(), dtype=torch.uint8, pin_memory=True)
    host.copy_(image)
    return host.to(device, non_blocking=True)


def _tensor_from_ptr(torch, ptr, shape, dtype, device):
    """Zero-copy torch view of raw device memory through __cuda_array_interface__."""
    n = int(np.prod(shape))
    typestr = {torch.float64: "<f8", torch.float32: "<f4"}[dtype]

    class _Holder:
        pass

    h = _Holder()
    h.__cuda_array_interface__ = dict(shape=(n,), typestr=typestr, data=(int(ptr), False), version=3, strides=None)
    return torch.as_tensor(h, device=device).view(shape)

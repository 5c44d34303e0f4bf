"""HlynrObsPipeline: VecFrameStack + VecNormalize fused on the device behind the tensor API (SURVEY 8f rank 1).

The reference wraps its VecEnv as
    envs = VecFrameStack(envs, n_stack=frame_stack)                         rl_system/scripts/train_flat_ppo.py:384-388
    envs = VecNormalize(envs, norm_obs=True, norm_reward=False, clip_obs=10.0, clip_reward=10.0, gamma=gamma)   :392-399
and loads the statistics for inference with VecNormalize.load(...); env.training = False (inference.py:455-471).
This class keeps the same names (n_stack, training, norm_obs, clip_obs, epsilon, gamma, obs_rms, ret_rms,
normalize_obs, get_original_obs) over include/hlynr_post.h: the simulator writes its observation straight into the
frame ring, and one pass produces the stacked, normalised [N, F*n_stack] tensor the policy consumes -- no host round
trip, no np.roll of the stack.  F, the frame width, is the sim's obs_dim: 26, or 17 for the leading radar channels obs[0:17]
of the pre-ground-radar models (HlynrSim(obs_dim=17)).
"""
import ctypes as C

import numpy as np

from . import _lib, abi


class _Rms:
    """Read-only view with the attribute names of SB3's RunningMeanStd."""

    def __init__(self, mean, var, count):
        self.mean, self.var, self.count = mean, var, count


class HlynrObsPipeline:
    def __init__(self, sim, n_stack=4, training=True, norm_obs=True, norm_reward=False, clip_obs=10.0, clip_reward=10.0,
                 gamma=0.99, epsilon=1e-8, want_terminal_obs=True):
        if norm_reward:
            raise NotImplementedError("norm_reward=True is not on the reference's path (train_flat_ppo.py:395)")
        import torch

        frame_dim = int(getattr(sim, "obs_dim", abi.OBS_DIM))
        if frame_dim not in (abi.OBS_DIM, 17):
            raise ValueError(f"HlynrObsPipeline stacks 26-D or 17-D frames, the sim writes {frame_dim}-D ones")
        self.sim, self.L, self._torch = sim, sim.L, torch
        self.frame_dim = frame_dim
        self.n_stack, self.training, self.norm_obs = int(n_stack), bool(training), bool(norm_obs)
        self.clip_obs, self.clip_reward, self.gamma, self.epsilon = float(clip_obs), float(clip_reward), float(gamma), float(epsilon)
        self.obs_dim = frame_dim * self.n_stack
        h = C.c_void_p()
        _lib.check(self.L.hlynr_post_create_frames(sim.n, sim.device_index, frame_dim, self.n_stack, self.clip_obs, self.epsilon,
                                                   self.gamma, C.byref(h)))
        self.h = h
        n, d = sim.n, sim.device
        self._out = torch.empty((n, self.obs_dim), dtype=torch.float32, device=d)
        self._orig = None
        self.want_terminal_obs = bool(want_terminal_obs)
        # compact done list of the step (finished episodes): records + counter live in torch tensors
        self._rec_dtype = abi.done_record_numpy_dtype()
        self._records = torch.zeros(n * self._rec_dtype.itemsize, dtype=torch.uint8, device=d)
        self._counter = torch.zeros(1, dtype=torch.int32, device=d)
        self._terminal = torch.empty((n, self.obs_dim), dtype=torch.float32, device=d) if want_terminal_obs else None
        _lib.check(self.L.hlynr_set_done_list(sim.h, C.c_void_p(self._records.data_ptr()), C.c_void_p(self._counter.data_ptr()), n))
        if not self.norm_obs:  # frame stacking only: identity statistics, never updated
            self.set_stats(np.zeros(self.obs_dim), np.full(self.obs_dim, 1.0 - self.epsilon), 1e-4)

    # ---- plumbing ----
    def _stream(self):
        return C.c_void_p(self._torch.cuda.current_stream(self.sim.device).cuda_stream)

    def _target(self):
        p = C.c_void_p()
        _lib.check(self.L.hlynr_post_obs_target(self.h, C.byref(p)))
        return p

    def _train_flag(self):
        return 1 if (self.training and self.norm_obs) else 0

    # ---- VecEnv-like surface on device tensors ----
    def _check_out(self, out, shape):
        t = self._torch
        if not (out.is_cuda and out.dtype == t.float32 and tuple(out.shape) == shape and out.is_contiguous()):
            raise ValueError(f"output tensor must be a contiguous cuda float32 tensor of shape {shape}")
        return out

    def reset(self, out=None):
        """VecFrameStack.reset + VecNormalize.reset: returns the stacked, normalised observation [N, F*n_stack]
        (written into `out` if given, e.g. a row of a rollout buffer)."""
        dst = self._out if out is None else self._check_out(out, (self.sim.n, self.obs_dim))
        _lib.check(self.L.hlynr_reset(self.sim.h, None, self._target(), self._stream()))
        _lib.check(self.L.hlynr_post_reset(self.h, C.c_void_p(dst.data_ptr()), self._train_flag(), self._stream()))
        return dst

    def step(self, actions, auto_reset=True, out=None, reward_out=None, info=None):
        """One tick + post-processing.  Returns (obs[N, Fk], reward[N], terminated[N], truncated[N], done) where
        `done` = (records uint8 tensor viewable with abi.done_record_numpy_dtype, counter int32[1],
        terminal_obs[capacity, Fk] or None): row r of terminal_obs is the stacked + normalised
        info['terminal_observation'] of record r.  All tensors are overwritten by the next call.
        info: None, an abi.HlynrInfoSoA of device pointers, or a dict of device tensors named as in abi.INFO_FIELDS (any
        subset, each of that field's dtype and shape): hlynr_step writes the tick's info there (for an env reset in this
        call: its terminal tick's)."""
        t, sim = self._torch, self.sim
        if isinstance(info, dict):
            info = self._info_struct(info)
        if not (actions.is_cuda and actions.dtype == t.float32 and actions.shape == (sim.n, 6) and actions.is_contiguous()):
            actions = actions.to(device=sim.device, dtype=t.float32).reshape(sim.n, 6).contiguous()
        o = sim._alloc_out()
        dst = self._out if out is None else self._check_out(out, (sim.n, self.obs_dim))
        rew = o["reward"] if reward_out is None else self._check_out(reward_out, (sim.n,))
        self._counter.zero_()
        st = self._stream()
        _lib.check(self.L.hlynr_step(sim.h, C.c_void_p(actions.data_ptr()), self._target(), C.c_void_p(rew.data_ptr()),
                                     C.c_void_p(o["terminated"].data_ptr()), C.c_void_p(o["truncated"].data_ptr()), None,
                                     None if info is None else C.byref(info), int(auto_reset), st))
        _lib.check(self.L.hlynr_post_step(self.h, C.c_void_p(rew.data_ptr()), C.c_void_p(o["terminated"].data_ptr()),
                                          C.c_void_p(o["truncated"].data_ptr()), C.c_void_p(self._records.data_ptr()),
                                          C.c_void_p(self._counter.data_ptr()), sim.n, C.c_void_p(dst.data_ptr()),
                                          C.c_void_p(self._terminal.data_ptr()) if self._terminal is not None else None,
                                          self._train_flag(), st))
        return dst, rew, o["terminated"], o["truncated"], (self._records, self._counter, self._terminal)

    def _info_struct(self, tensors):
        t, n = self._torch, self.sim.n
        fields = {name: (dt, shp) for name, dt, shp in abi.INFO_FIELDS}
        ptrs = {}
        for name, x in tensors.items():
            if name not in fields:
                raise ValueError(f"unknown info field {name!r}; the fields are {list(fields)}")
            dt, shp = fields[name]
            if not (x.is_cuda and x.device == self.sim.device and x.dtype == getattr(t, dt) and tuple(x.shape) == (n,) + shp
                    and x.is_contiguous()):
                raise ValueError(f"info[{name!r}] must be a contiguous {dt} tensor of shape {(n,) + shp} on {self.sim.device}")
            ptrs[name] = x.data_ptr()
        return abi.HlynrInfoSoA(**ptrs)

    def done_records(self):
        """Host copy of the finished episodes of the last step (synchronises)."""
        cnt = min(int(self._counter.item()), self.sim.n)
        if cnt == 0:
            return np.zeros(0, dtype=self._rec_dtype)
        raw = self._records[: cnt * self._rec_dtype.itemsize].cpu().numpy()
        return raw.view(self._rec_dtype).copy()

    def get_original_obs(self):
        """VecNormalize.get_original_obs(): the stacked, un-normalised observation of the last reset/step."""
        t = self._torch
        if self._orig is None:
            self._orig = t.empty((self.sim.n, self.obs_dim), dtype=t.float32, device=self.sim.device)
        _lib.check(self.L.hlynr_post_original(self.h, C.c_void_p(self._orig.data_ptr()), self._stream()))
        return self._orig

    def normalize_obs(self, stacked):
        """VecNormalize.normalize_obs on a cuda float32 tensor [rows, F*n_stack]."""
        t = self._torch
        x = stacked.to(device=self.sim.device, dtype=t.float32).reshape(-1, self.obs_dim).contiguous()
        out = t.empty_like(x)
        _lib.check(self.L.hlynr_post_normalize(self.h, C.c_void_p(x.data_ptr()), x.shape[0], C.c_void_p(out.data_ptr()), self._stream()))
        return out

    # ---- statistics (the content of SB3's vec_normalize.pkl) ----
    def get_stats(self):
        mean, var = np.zeros(self.obs_dim), np.zeros(self.obs_dim)
        c, rm, rv, rc = C.c_double(), C.c_double(), C.c_double(), C.c_double()
        _lib.check(self.L.hlynr_post_get_stats(self.h, mean.ctypes.data_as(C.c_void_p), var.ctypes.data_as(C.c_void_p), C.byref(c),
                                               C.byref(rm), C.byref(rv), C.byref(rc), self._stream()))
        return dict(mean=mean, var=var, count=c.value, ret_mean=rm.value, ret_var=rv.value, ret_count=rc.value)

    def set_stats(self, mean, var, count, ret_mean=0.0, ret_var=1.0, ret_count=1e-4):
        mean, var = np.ascontiguousarray(mean, np.float64), np.ascontiguousarray(var, np.float64)
        assert mean.shape == (self.obs_dim,) and var.shape == (self.obs_dim,)
        _lib.check(self.L.hlynr_post_set_stats(self.h, mean.ctypes.data_as(C.c_void_p), var.ctypes.data_as(C.c_void_p), float(count),
                                               float(ret_mean), float(ret_var), float(ret_count), self._stream()))

    @property
    def obs_rms(self):
        s = self.get_stats()
        return _Rms(s["mean"], s["var"], s["count"])

    @property
    def ret_rms(self):
        s = self.get_stats()
        return _Rms(s["ret_mean"], s["ret_var"], s["ret_count"])

    def save(self, path):
        """Statistics + hyper-parameters as .npz (the fields VecNormalize.__getstate__ pickles, and the frame width)."""
        s = self.get_stats()
        np.savez(path, n_stack=self.n_stack, frame_dim=self.frame_dim, clip_obs=self.clip_obs, clip_reward=self.clip_reward,
                 gamma=self.gamma, epsilon=self.epsilon, norm_obs=self.norm_obs, **s)

    def load(self, path):
        """Statistics saved by save(); a file without a frame width is from a 26-D pipeline."""
        z = np.load(path)
        frame_dim = int(z["frame_dim"]) if "frame_dim" in z.files else abi.OBS_DIM
        if frame_dim != self.frame_dim:
            raise ValueError(f"the statistics are of {frame_dim}-D frames, this pipeline stacks {self.frame_dim}-D ones")
        assert int(z["n_stack"]) == self.n_stack, "frame_stack of the statistics differs"
        self.set_stats(z["mean"], z["var"], float(z["count"]), float(z["ret_mean"]), float(z["ret_var"]), float(z["ret_count"]))

    def save_sb3_pickle(self, path):
        """`VecNormalize.save(path)` (scripts/train_flat_ppo.py:477,530): a vec_normalize.pkl that `VecNormalize.load` of
        inference.py:163-170 accepts -- the wrapper object pickled under SB3's module paths with the device-side statistics
        (sb3_pickle.py; works without stable_baselines3 installed; parity unpinned, see there)."""
        from . import sb3_pickle

        s = self.get_stats()
        sb3_pickle.dump(path, mean=s["mean"], var=s["var"], count=s["count"], ret_mean=s["ret_mean"], ret_var=s["ret_var"],
                        ret_count=s["ret_count"], obs_shape=(self.obs_dim,), num_envs=self.sim.n, clip_obs=self.clip_obs,
                        clip_reward=self.clip_reward, gamma=self.gamma, epsilon=self.epsilon, training=self.training,
                        norm_obs=self.norm_obs, norm_reward=False)

    def load_sb3_pickle(self, path):
        """Statistics from a vec_normalize.pkl written by the reference's trainer or by save_sb3_pickle()."""
        from . import sb3_pickle

        d = sb3_pickle.load(path)
        if d["obs_shape"] != (self.obs_dim,):
            raise ValueError(f"the pickle normalises observations of shape {d['obs_shape']}, this pipeline {(self.obs_dim,)}")
        if (d["clip_obs"], d["epsilon"]) != (self.clip_obs, self.epsilon):
            raise ValueError("clip_obs / epsilon of the pickle differ from this pipeline's")
        self.set_stats(d["mean"], d["var"], d["count"], d["ret_mean"], d["ret_var"], d["ret_count"])

    # ---- snapshots (include/hlynr_post.h hlynr_post_snapshot_*, DESIGN.md section 17) ----
    def state_dict(self):
        """{'info': descriptor dict, 'image': uint8 CPU tensor, 'training': the training flag}: the frame ring, the per-env ages
        and discounted returns, obs_rms / ret_rms and the running column sums.  Synchronises the current stream."""
        from .sim import image_to_host

        info, nbytes = abi.HlynrPostSnapshotInfo(), C.c_size_t()
        _lib.check(self.L.hlynr_post_snapshot_layout(self.h, C.byref(info), C.byref(nbytes)))
        dev = self._torch.empty(nbytes.value, dtype=self._torch.uint8, device=self.sim.device)
        _lib.check(self.L.hlynr_post_snapshot_save(self.h, C.c_void_p(dev.data_ptr()), C.byref(info), self._stream()))
        return {"info": abi.struct_to_dict(info), "image": image_to_host(self._torch, dev), "training": self.training}

    def load_state_dict(self, state):
        """Restores a state_dict() into a pipeline of the same n_envs, frame width, n_stack, clip_obs, epsilon and gamma."""
        from .sim import image_to_device

        info = abi.struct_from_dict(abi.HlynrPostSnapshotInfo, state["info"])
        dev = image_to_device(self._torch, state["image"], info.device_bytes, self.sim.device)
        _lib.check(self.L.hlynr_post_snapshot_load(self.h, C.byref(info), C.c_void_p(dev.data_ptr()), self._stream()))
        self.training = bool(state["training"])

    def check_sums(self, resync=False):
        d = C.c_double()
        _lib.check(self.L.hlynr_post_check_sums(self.h, int(resync), C.byref(d), self._stream()))
        return d.value

    def launch_count(self):
        v = C.c_int64()
        _lib.check(self.L.hlynr_post_launch_count(self.h, C.byref(v)))
        return v.value

    def close(self):
        if getattr(self, "h", None):
            _lib.check(self.L.hlynr_set_done_list(self.sim.h, None, None, 0))
            self.L.hlynr_post_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

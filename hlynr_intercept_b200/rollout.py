"""On-device PPO rollout collection over the tensor API (SURVEY 8f rank 4, BASELINE config 5).

The reference collects rollouts through stable-baselines3 (`model.learn`, rl_system/scripts/train_flat_ppo.py:431-448):
per step a policy forward, env.step through the VecEnv wrappers, the TimeLimit bootstrap
(`rewards[i] += gamma * V(terminal_observation)`), a NumPy rollout buffer, and GAE(lambda) at the end.  Here the whole
loop stays on the GPU: the simulator writes into the frame ring, `HlynrObsPipeline` writes the stacked + normalised
observation straight into the next row of the rollout buffer, finished episodes are a compact device-side list, and the
two non-GEMM steps (timeout bootstrap, GAE) are CUDA kernels behind include/hlynr_rollout.h.  No host synchronisation
happens inside `collect()`.

The policy network is the caller's torch module (plumbing: cuBLAS GEMMs); `GaussianMlpPolicy` is a minimal stand-in with
SB3's MlpPolicy shape (separate pi / vf MLPs, state-independent log_std) for synthetic rollouts and the benchmark.
"""
import ctypes as C
import math

from . import _lib


def _torch():
    import torch

    return torch


class GaussianMlpPolicy:
    """Factory: returns a torch.nn.Module with forward(obs) -> (actions, values, log_probs) and value(obs)."""

    def __new__(cls, obs_dim, act_dim=6, net_arch=(512, 512, 256), layer_norm=True, log_std_init=0.0, device="cuda", dtype=None):
        torch = _torch()
        nn = torch.nn

        def mlp(out_dim):
            layers, d = [], obs_dim
            for h in net_arch:
                layers.append(nn.Linear(d, h))
                if layer_norm:
                    layers.append(nn.LayerNorm(h))
                layers.append(nn.Tanh())
                d = h
            layers.append(nn.Linear(d, out_dim))
            return nn.Sequential(*layers)

        class _Policy(nn.Module):
            def __init__(self):
                super().__init__()
                self.pi, self.vf = mlp(act_dim), mlp(1)
                self.log_std = nn.Parameter(torch.full((act_dim,), float(log_std_init)))

            def value(self, obs):
                return self.vf(obs).squeeze(-1).float()

            def forward(self, obs):
                mean = self.pi(obs).float()
                std = self.log_std.exp()
                actions = mean + std * torch.randn_like(mean)
                logp = (-0.5 * ((actions - mean) / std) ** 2 - self.log_std - 0.5 * math.log(2 * math.pi)).sum(-1)
                return actions, self.value(obs), logp

        m = _Policy().to(device)
        if dtype is not None:
            m = m.to(dtype)
        return m


class DeviceRolloutCollector:
    """SB3 OnPolicyAlgorithm.collect_rollouts + RolloutBuffer.compute_returns_and_advantage on device tensors."""

    def __init__(self, pipe, policy, n_steps, gamma=0.99, gae_lambda=0.95, bootstrap_rows=None):
        torch = _torch()
        self.pipe, self.policy, self.sim = pipe, policy, pipe.sim
        self.T, self.gamma, self.gae_lambda = int(n_steps), float(gamma), float(gae_lambda)
        n, d, dev = self.sim.n, pipe.obs_dim, self.sim.device
        f32 = torch.float32
        self.obs = torch.empty((self.T + 1, n, d), dtype=f32, device=dev)   # row T = observation after the last step
        self.actions = torch.empty((self.T, n, 6), dtype=f32, device=dev)
        self.rewards = torch.empty((self.T, n), dtype=f32, device=dev)
        self.episode_starts = torch.empty((self.T, n), dtype=f32, device=dev)
        self.values = torch.empty((self.T, n), dtype=f32, device=dev)
        self.log_probs = torch.empty((self.T, n), dtype=f32, device=dev)
        self.advantages = torch.empty((self.T, n), dtype=f32, device=dev)
        self.returns = torch.empty((self.T, n), dtype=f32, device=dev)
        self.last_dones = torch.ones(n, dtype=torch.uint8, device=dev)
        self.overflow = torch.zeros(1, dtype=torch.int32, device=dev)
        # rows of the done list whose terminal observation gets a value (TimeLimit bootstrap).  Default: ALL n -- after a
        # synchronised reset an untrained policy lets most envs time out in the SAME tick, and SB3 bootstraps every one of
        # them.  A smaller bound is a speed knob for the value net; collect() then verifies that no timeout was left out.
        self.rows = min(n, int(bootstrap_rows)) if bootstrap_rows else n
        self._started = False
        self._clipped = None
        self.L = pipe.L
        self._graph = None

    def _stream(self):
        return C.c_void_p(_torch().cuda.current_stream(self.sim.device).cuda_stream)

    def reset(self):
        self.pipe.reset(out=self.obs[0])
        self.last_dones.fill_(1)   # SB3: _last_episode_starts = ones
        self._started = True

    def collect(self):
        """Fills the buffers with n_steps transitions of every env and computes advantages / returns.  Returns self."""
        torch = _torch()
        if not self._started:
            self.reset()
        else:
            self.obs[0].copy_(self.obs[self.T])
        pipe, pol, sim = self.pipe, self.policy, self.sim
        p = lambda x: C.c_void_p(x.data_ptr())  # noqa: E731
        fused = bool(getattr(pol, "fused", False))   # policy.FusedActorCritic: one sm_100a kernel per forward, fp32 rows in
        cast = (lambda x: x) if fused or next(pol.parameters()).dtype == torch.float32 else (lambda x: x.to(next(pol.parameters()).dtype))
        with torch.no_grad():
            for t in range(self.T):
                o = self.obs[t]
                if fused:   # the kernel writes the rollout-buffer rows and the clipped action itself: no copies, no clamp kernel
                    if self._clipped is None:
                        self._clipped = torch.empty((sim.n, 6), dtype=torch.float32, device=sim.device)
                    pol.forward(o, out=dict(actions=self.actions[t], values=self.values[t], logp=self.log_probs[t], clipped=self._clipped))
                    env_actions = self._clipped
                else:
                    a, v, lp = pol(cast(o))
                    self.actions[t].copy_(a)
                    self.values[t].copy_(v)
                    self.log_probs[t].copy_(lp)
                    env_actions = a.float().clamp(-1.0, 1.0)
                self.episode_starts[t].copy_(self.last_dones)
                _, rew, te, tr, (records, counter, terminal) = pipe.step(env_actions, out=self.obs[t + 1], reward_out=self.rewards[t])
                # TimeLimit bootstrap on the first `rows` finished episodes of the step (more only if nearly every env
                # finishes in the same step; counted in self.overflow)
                term_rows = terminal[: self.rows]
                # the fused kernel reads the number of finished episodes from the device-side counter and skips every tile beyond
                # it, so bootstrapping ALL rows costs nothing in the common case of a handful of finished episodes per step
                tv = pol.value_rows(term_rows, counter) if fused else pol.value(cast(term_rows)).contiguous()
                _lib.check(self.L.hlynr_bootstrap_timeouts(p(self.rewards[t]), p(records), p(counter), self.rows, p(tv), self.gamma,
                                                           p(self.overflow), sim.device_index, self._stream()))
                torch.bitwise_or(te, tr, out=self.last_dones)
            o = self.obs[self.T]
            last_values = pol.value(cast(o)).contiguous()
            _lib.check(self.L.hlynr_gae(p(self.rewards), p(self.values), p(self.episode_starts), p(last_values), p(self.last_dones),
                                        self.T, sim.n, self.gamma, self.gae_lambda, p(self.advantages), p(self.returns),
                                        sim.device_index, self._stream()))
        if self.rows < sim.n and not torch.cuda.is_current_stream_capturing():
            missed = int(self.overflow.item())   # one synchronisation per rollout (the caller consumes the rollout next anyway)
            if missed:
                self.overflow.zero_()
                raise RuntimeError(f"{missed} timed-out episodes of this rollout finished beyond bootstrap_rows={self.rows} and got no "
                                   f"gamma * V(terminal_observation): create the collector with bootstrap_rows=None (all envs)")
        return self

    # ---- checkpoints ------------------------------------------------------------------------------------------------------
    def state_dict(self):
        """What the next collect() continues from: obs[T] (its first row), last_dones, whether reset() has run, and the
        bootstrap overflow count, as CPU tensors.  The sim, the pipeline and the policy keep their own state_dict()."""
        return {"next_obs": self.obs[self.T].cpu(), "last_dones": self.last_dones.cpu(), "started": self._started,
                "overflow": self.overflow.cpu()}

    def load_state_dict(self, state):
        """Restores a state_dict() into a collector of the same n_envs and observation width.  A graph captured before the load
        is dropped: capture() again (its warm-up collect is then the first rollout after the resume)."""
        for name, dst in (("next_obs", self.obs[self.T]), ("last_dones", self.last_dones), ("overflow", self.overflow)):
            src = _torch().as_tensor(state[name])
            if tuple(src.shape) != tuple(dst.shape) or src.dtype != dst.dtype:
                raise ValueError(f"collector state {name!r} is {src.dtype} {tuple(src.shape)}, this collector needs {dst.dtype} {tuple(dst.shape)}")
            dst.copy_(src)
        self._started = bool(state["started"])
        self._graph = None

    # ---- CUDA graph: the whole collect() (T x ~20 launches) as one graph launch --------------------------------------
    def graph_period(self):
        """collect() can be captured once and replayed iff n_steps is a multiple of this (see graph_period())."""
        return graph_period(self.pipe)

    def capture(self):
        """Warm-up + stream capture of collect() into a CUDA graph (launch-bound at small n_envs: ~20 launches per step).
        The seed and host-pushed curriculum scalars are baked into the captured kernel arguments: re-capture after changing them.
        A sim that tracks training steps (HlynrSim.track_training_steps) keeps its counter on the device and every captured step
        advances it there, so each replay continues the curriculum schedule; re-capture only after attaching or detaching one.
        The fused policy's noise counter lives on the device and each forward advances it there, so every replay draws fresh
        exploration noise, exactly as the same number of eager collects would."""
        if self.T % self.graph_period():
            raise ValueError(f"n_steps={self.T} must be a multiple of {self.graph_period()} to be graph-captured")
        self._graph = TickGraph(self.pipe, self.T, self.collect)
        return self

    def replay(self):
        """One collect() as a single graph launch."""
        if self._graph is None:
            raise RuntimeError("capture() first (after load_state_dict() too)")
        self._graph.replay()
        return self


def graph_period(pipe):
    """A captured sequence of ticks of `pipe` (HlynrObsPipeline) and its sim replays correctly iff its length is a multiple of
    this: ring rows of the delay buffers, the frame-ring slot and the age ping-pong are kernel arguments derived from host-side
    tick counters."""
    per = C.c_int()
    _lib.check(pipe.L.hlynr_ring_period(pipe.sim.h, C.byref(per)))
    return math.lcm(per.value, pipe.n_stack, 2)


class TickGraph:
    """fn(), which runs `ticks` steps of `pipe` and its sim (and whatever else it launches on the current stream), as one CUDA
    graph.  Construction runs fn() once for real on a side stream (allocations, cuBLAS workspaces, lazy module init), then
    records it.  The recording advances the host-side tick counters although nothing runs; that is undone, and replay()
    advances them by what the graph ran.  Both are consistent only because `ticks` is a multiple of graph_period(pipe): the
    counters come back to the phases the captured kernel arguments were derived from."""

    def __init__(self, pipe, ticks, fn):
        torch = _torch()
        self.pipe, self.sim, self.ticks = pipe, pipe.sim, int(ticks)
        if self.ticks <= 0 or self.ticks % graph_period(pipe):
            raise ValueError(f"{ticks} ticks must be a positive multiple of {graph_period(pipe)} to be graph-captured")
        dev = self.sim.device
        cur = torch.cuda.current_stream(dev)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            fn()
        cur.wait_stream(side)
        torch.cuda.synchronize(dev)
        l0, p0 = self.sim.launch_count(), pipe.launch_count()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            fn()   # recorded, not executed
        self.launches = (self.sim.launch_count() - l0, pipe.launch_count() - p0)
        self._note(-1)

    def _note(self, sign):
        L = self.pipe.L
        _lib.check(L.hlynr_note_replayed_ticks(self.sim.h, sign * self.ticks, sign * self.launches[0]))
        _lib.check(L.hlynr_post_note_replayed_steps(self.pipe.h, sign * self.ticks, sign * self.launches[1]))

    def replay(self):
        self.graph.replay()
        self._note(1)

"""Evaluation of a policy on the device: stable-baselines3's `evaluate_policy` over HlynrObsPipeline.

The reference evaluates with `evaluate_policy(model, eval_env, n_eval_episodes, deterministic=True)` (EvalCallback,
rl_system/scripts/train_flat_ppo.py:497-504; `inference.py --mode offline`) on a Monitor-wrapped, VecNormalize-wrapped eval env
whose statistics were copied from the training env (`sync_envs_normalization`) and are frozen (`training=False`).  SB3 gives
env i the quota `(n_eval_episodes + i) // n_envs` and counts only the first that many episodes each env finishes; the envs keep
stepping until every quota is met.  Counting "the first E episodes that finish" instead would favour short episodes: an
intercept that fails early finishes first.  With fewer episodes than envs only the LAST n_eval_episodes envs are evaluated,
as in SB3.

One tick here is the policy's action clipped to [-1, 1] (the mean with deterministic=True, a sample otherwise), `pipe.step` and
`hlynr_eval_record` (include/hlynr_rollout.h), which files each counted episode's done record in a table addressed by
(env, episode index), with the step it ended on.  The host reads one counter per chunk of ticks; with graph=True a chunk is one CUDA graph launch.
"""
import ctypes as C
import dataclasses

import numpy as np

from . import _lib, abi
from .rollout import TickGraph, graph_period

INT32_MAX = 2**31 - 1


def _torch():
    import torch

    return torch


def sync_normalization(train_pipe, eval_pipe):
    """`sync_envs_normalization(train_env, eval_env)`: the eval pipeline gets the training pipeline's obs_rms and ret_rms."""
    for name in ("obs_dim", "n_stack", "clip_obs", "epsilon"):
        a, b = getattr(train_pipe, name), getattr(eval_pipe, name)
        if a != b:
            raise ValueError(f"{name} differs between the training ({a}) and the eval ({b}) pipeline")
    s = train_pipe.get_stats()
    eval_pipe.set_stats(s["mean"], s["var"], s["count"], s["ret_mean"], s["ret_var"], s["ret_count"])


@dataclasses.dataclass
class EvalResult:
    """The counted episodes in the order of SB3's lists (finishing step first, then env index)."""
    records: np.ndarray           # abi.done_record_numpy_dtype(): every info field of the episode's final step
    end_tick: np.ndarray          # int64: the step the episode ended on, counted from the evaluation's reset
    episode_rewards: np.ndarray   # float64 Monitor 'r', rounded to 6 decimals
    episode_lengths: np.ndarray   # int32 Monitor 'l'
    mean_reward: float            # np.mean / np.std of episode_rewards, what evaluate_policy returns
    std_reward: float
    success_rate: float           # mean of info['intercepted']
    mean_min_distance: float
    mean_fuel_used: float
    ticks: int                    # ticks run


class DeviceEvaluator:
    """evaluate_policy(policy, pipe, n_eval_episodes, deterministic) on device tensors.

    pipe: an HlynrObsPipeline with training=False (load or sync its statistics first).
    policy: a FusedActorCritic (one kernel writes the clipped action), or a torch module with mean(obs) for deterministic
      evaluation and the collector's forward(obs) -> (actions, values, log_probs) for stochastic evaluation, such as
      ReferenceActorCritic (both) or GaussianMlpPolicy (stochastic only); its input width must be pipe.obs_dim.  For a torch
      module, value(obs) only marks the collector's interface: the forward's signature is not checked before the first tick.
    chunk: ticks between two reads of the remaining-episodes counter and the length of the CUDA graph; a multiple of
      graph_period(pipe).  Default: the smallest such multiple that is at least 16."""

    def __init__(self, pipe, policy, chunk=None):
        torch = _torch()
        if pipe.training:
            raise ValueError("the eval pipeline must have training=False: evaluate_policy runs with frozen statistics")
        self.pipe, self.policy, self.sim = pipe, policy, pipe.sim
        self.fused = bool(getattr(policy, "fused", False))
        if self.fused:
            in_dim = policy.in_dim
        elif hasattr(policy, "mean") or hasattr(policy, "value"):
            in_dim = next(p for p in policy.parameters() if p.dim() == 2).shape[1]
        else:
            raise ValueError("policy must be a FusedActorCritic, or a torch module with mean(obs) or the rollout collector's "
                             "forward(obs) -> (actions, values, log_probs) and value(obs)")
        if in_dim != pipe.obs_dim:
            raise ValueError(f"the policy takes {in_dim}-wide observations, the pipeline produces {pipe.obs_dim}-wide ones")
        period = graph_period(pipe)
        self.chunk = period * -(-16 // period) if chunk is None else int(chunk)
        if self.chunk <= 0 or self.chunk % period:
            raise ValueError(f"chunk must be a positive multiple of {period}, got {chunk}")
        n, dev = self.sim.n, self.sim.device
        self.obs = torch.empty((n, pipe.obs_dim), dtype=torch.float32, device=dev)
        self.actions = torch.empty((n, 6), dtype=torch.float32, device=dev) if self.fused else None
        self.counts = torch.zeros(n, dtype=torch.int32, device=dev)
        self.ticks = torch.zeros(n, dtype=torch.int64, device=dev)
        self.remaining = torch.zeros(1, dtype=torch.int64, device=dev)
        self._rec_dtype = abi.done_record_numpy_dtype()
        self._n_episodes, self._results, self._end_tick = 0, None, None
        self._deterministic = True

    def _tick(self):
        torch, sim = _torch(), self.sim
        if self.fused:
            self.policy.forward(self.obs, deterministic=self._deterministic, want=(), out=dict(clipped=self.actions))
            act = self.actions
        elif self._deterministic:
            act = self.policy.mean(self.obs).float().clamp(-1.0, 1.0)
        else:   # SB3's predict(deterministic=False): a sample, clipped to the Box bounds
            act = self.policy(self.obs)[0].float().clamp(-1.0, 1.0)
        _, _, _, _, (records, counter, _) = self.pipe.step(act, out=self.obs)
        p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
        _lib.check(sim.L.hlynr_eval_record(p(records), p(counter), sim.n, self._n_episodes, p(self.counts), p(self.ticks),
                                           p(self._results), p(self._end_tick), p(self.remaining), sim.device_index,
                                           C.c_void_p(torch.cuda.current_stream(sim.device).cuda_stream)))

    def _chunk(self):
        for _ in range(self.chunk):
            self._tick()

    def evaluate(self, n_eval_episodes, graph=True, deterministic=True):
        """Resets the pipeline and runs until every env has finished its quota.  graph=True: chunks of `chunk` ticks, the
        first one eager, the others as replays of one CUDA graph, so `ticks` is a multiple of `chunk`; graph=False: the
        counter is read after every tick and `ticks` is the step on which the last counted episode ended.
        deterministic=False samples the action, as SB3's evaluate_policy(..., deterministic=False): the fused policy draws at
        its device-side noise counter, one step per tick, so every graph replay draws fresh noise; a torch module draws from
        torch's generator."""
        torch = _torch()
        E = int(n_eval_episodes)
        if not 1 <= E <= INT32_MAX:
            raise ValueError(f"n_eval_episodes must be in [1, {INT32_MAX}], got {n_eval_episodes}")
        if not self.fused and not hasattr(self.policy, "mean" if deterministic else "value"):
            raise ValueError("deterministic evaluation of a torch module needs its mean(obs)" if deterministic else
                             "stochastic evaluation of a torch module needs the collector's forward(obs) -> (actions, values, "
                             "log_probs) and value(obs)")
        self._deterministic = bool(deterministic)
        n = self.sim.n
        # every episode ends within max_steps ticks, and an env needs at most ceil(E / n) of them
        limit = -(-E // n) * int(self.sim.params.max_steps) + self.chunk
        self._n_episodes = E
        self._results = torch.empty(E * self._rec_dtype.itemsize, dtype=torch.uint8, device=self.sim.device)
        self._end_tick = torch.empty(E, dtype=torch.int64, device=self.sim.device)
        self.counts.zero_()
        self.ticks.zero_()
        self.remaining.fill_(E)
        ticks = 0
        with torch.no_grad():
            self.pipe.reset(out=self.obs)
            if graph:
                # recorded anew by every call: pipe.reset() moves the frame-ring slot against the age ping-pong, so a graph
                # recorded after an earlier reset would address the wrong ring slots
                g = TickGraph(self.pipe, self.chunk, self._chunk)   # runs the first chunk, then records it
                ticks = self.chunk
                while int(self.remaining.item()) > 0:
                    self._check_limit(ticks, limit)
                    g.replay()
                    ticks += self.chunk
            else:
                while int(self.remaining.item()) > 0:
                    self._check_limit(ticks, limit)
                    self._tick()
                    ticks += 1
        return self._result(ticks)

    def _check_limit(self, ticks, limit):
        if ticks >= limit:
            raise RuntimeError(f"{int(self.remaining.item())} of {self._n_episodes} episodes still unfinished after {ticks} ticks, "
                               f"more than any episode of max_steps={int(self.sim.params.max_steps)} allows")

    def _result(self, ticks):
        recs = self._results.cpu().numpy().view(self._rec_dtype)
        end = self._end_tick.cpu().numpy()
        order = np.lexsort((recs["env"], end))   # SB3 appends in step order, and within a step in env order
        recs, end = recs[order], end[order]
        rewards = recs["episode_return"].astype(np.float64).round(6)
        return EvalResult(records=recs, end_tick=end, episode_rewards=rewards, episode_lengths=recs["steps"].copy(),
                          mean_reward=float(np.mean(rewards)), std_reward=float(np.std(rewards)),
                          success_rate=float(np.mean((recs["flags"] & abi.INFO_INTERCEPTED) != 0)),
                          mean_min_distance=float(np.mean(recs["min_distance"].astype(np.float64))),
                          mean_fuel_used=float(np.mean(recs["fuel_used"].astype(np.float64))), ticks=ticks)

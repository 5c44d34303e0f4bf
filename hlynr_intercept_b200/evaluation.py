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

evaluate(..., trace=True) also keeps every tick of every counted episode: `pipe.step` writes the tick's info arrays and
`hlynr_eval_trace`, launched before `hlynr_eval_record`, files each env's row at (episode slot, info['steps']).  The rows are
what the reference's offline inference logs per tick (inference.py:535-606); episode_log.write_episodes writes them as its
episode JSONL files.
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
    trajectories: np.ndarray = None       # evaluate(trace=True): abi.trace_row_numpy_dtype() rows of every episode, in `records` order
    trajectory_offsets: np.ndarray = None  # int64 [E+1]: episode i is trajectories[offsets[i]:offsets[i+1]], episode_lengths[i] rows


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
        self._trace_dtype = abi.trace_row_numpy_dtype()
        self._table = self._info = self._info_struct = None   # evaluate(trace=True) only

    def _tick(self):
        torch, sim = _torch(), self.sim
        if self.fused:
            self.policy.forward(self.obs, deterministic=self._deterministic, want=(), out=dict(clipped=self.actions))
            act = self.actions
        elif self._deterministic:
            act = self.policy.mean(self.obs).float().clamp(-1.0, 1.0)
        else:   # SB3's predict(deterministic=False): a sample, clipped to the Box bounds
            act = self.policy(self.obs)[0].float().clamp(-1.0, 1.0)
        p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
        stream = C.c_void_p(torch.cuda.current_stream(sim.device).cuda_stream)
        if self._table is None:
            _, _, _, _, (records, counter, _) = self.pipe.step(act, out=self.obs)
        else:
            _, rew, term, trunc, (records, counter, _) = self.pipe.step(act, out=self.obs, info=self._info_struct)
            if not act.is_contiguous():
                act = act.contiguous()
            # before hlynr_eval_record: the terminal tick's row goes to the episode it ends, not to the next slot
            _lib.check(sim.L.hlynr_eval_trace(C.byref(self._info_struct), p(act), p(rew), p(term), p(trunc), p(self.counts), sim.n,
                                              self._n_episodes, self._max_steps, p(self._table), sim.device_index, stream))
        _lib.check(sim.L.hlynr_eval_record(p(records), p(counter), sim.n, self._n_episodes, p(self.counts), p(self.ticks),
                                           p(self._results), p(self._end_tick), p(self.remaining), sim.device_index, stream))

    def _chunk(self):
        for _ in range(self.chunk):
            self._tick()

    def evaluate(self, n_eval_episodes, graph=True, deterministic=True, trace=False):
        """Resets the pipeline and runs until every env has finished its quota.  graph=True: chunks of `chunk` ticks, the
        first one eager, the others as replays of one CUDA graph, so `ticks` is a multiple of `chunk`; graph=False: the
        counter is read after every tick and `ticks` is the step on which the last counted episode ended.
        deterministic=False samples the action, as SB3's evaluate_policy(..., deterministic=False): the fused policy draws at
        its device-side noise counter, one step per tick, so every graph replay draws fresh noise; a torch module draws from
        torch's generator.
        trace=True also records every tick of every counted episode into `trajectories` / `trajectory_offsets` of the result
        (abi.trace_row_numpy_dtype(): positions, clipped action, reward, distance, fuel, radar quality, info flags | done bits,
        info['steps']).  It allocates a device table of E x max_steps rows of 72 bytes (E = 4096, max_steps = 1000: 295 MB)
        and [N]-sized info arrays (41 B per env), and adds one launch and 72 B of writes per env and tick; the evaluation
        itself is unchanged, bit for bit.  trace=False allocates and launches nothing extra."""
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
        self._prepare(E, trace)
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

    def _prepare(self, E, trace):
        """The per-evaluation device state: result table, zeroed quota counters, and with trace the row table and info arrays."""
        torch = _torch()
        self._n_episodes = E
        self._results = torch.empty(E * self._rec_dtype.itemsize, dtype=torch.uint8, device=self.sim.device)
        self._end_tick = torch.empty(E, dtype=torch.int64, device=self.sim.device)
        self.counts.zero_()
        self.ticks.zero_()
        self.remaining.fill_(E)
        self._max_steps = int(self.sim.params.max_steps)
        if trace:
            dev, n = self.sim.device, self.sim.n
            self._table = torch.empty(E * self._max_steps * self._trace_dtype.itemsize, dtype=torch.uint8, device=dev)
            dt = {"float32": torch.float32, "int32": torch.int32, "uint8": torch.uint8}
            self._info = {name: torch.empty((n,) + shp, dtype=dt[d], device=dev) for name, d, shp in abi.INFO_FIELDS
                          if name in abi.TRACE_INFO_FIELDS}
            self._info_struct = abi.HlynrInfoSoA(**{k: v.data_ptr() for k, v in self._info.items()})
        else:
            self._table = self._info = self._info_struct = None

    def _trajectories(self, order, lengths):
        """Rows [0, l) of each episode's max_steps slots, episodes in SB3's order; only those rows leave the device."""
        torch = _torch()
        lengths = lengths.astype(np.int64)
        if len(lengths) and lengths.max() > self._max_steps:
            raise RuntimeError(f"an episode ran {int(lengths.max())} steps, more than the table's max_steps={self._max_steps} rows")
        offsets = np.zeros(len(lengths) + 1, dtype=np.int64)
        np.cumsum(lengths, out=offsets[1:])
        first = order.astype(np.int64) * self._max_steps   # table slot k of the record now at position i is order[i]
        idx = np.repeat(first - offsets[:-1], lengths) + np.arange(offsets[-1], dtype=np.int64)
        table = self._table.view(-1, self._trace_dtype.itemsize)
        rows = table.index_select(0, torch.from_numpy(idx).to(table.device)).cpu().numpy()
        return rows.reshape(-1).view(self._trace_dtype), offsets

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
        rows = offsets = None
        if self._table is not None:
            rows, offsets = self._trajectories(order, recs["steps"])
            self._table = self._info = self._info_struct = None
        return EvalResult(records=recs, end_tick=end, episode_rewards=rewards, episode_lengths=recs["steps"].copy(),
                          trajectories=rows, trajectory_offsets=offsets,
                          mean_reward=float(np.mean(rewards)), std_reward=float(np.std(rewards)),
                          success_rate=float(np.mean((recs["flags"] & abi.INFO_INTERCEPTED) != 0)),
                          mean_min_distance=float(np.mean(recs["min_distance"].astype(np.float64))),
                          mean_fuel_used=float(np.mean(recs["fuel_used"].astype(np.float64))), ticks=ticks)

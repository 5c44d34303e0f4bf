"""Episode JSONL export in the reference's logger format, for the tensor API (SURVEY 8f rank 4, second half).

The reference writes one `<log_dir>/episodes/<episode_id>.jsonl` per episode through `UnifiedLogger`
(rl_system/logger.py:148-273): a `header` line, `state` lines per entity and tick (`interceptor`: position / fuel / action,
`missile`: position -- what inference.py:535-548 logs and the Unity replay tooling reads), optional `event` lines and a
`footer` line with the outcome and the metrics of inference.py:588-606.  When the reference's own scripts drive
`HlynrVecEnv` they keep using their own logger on the `infos`; this recorder is for callers of the tensor API, where
nothing per-env ever reaches the host unless asked: it follows ONE env of the batch (lazy: one 400-byte state export per
tick) and writes the same records.  `write_episodes` writes the same files for every episode of an evaluation traced on the
device (`DeviceEvaluator.evaluate(..., trace=True)`), which steps every env with auto-reset inside CUDA graphs.
"""
import json
import os
import time

import numpy as np

from . import abi


class EpisodeRecorder:
    def __init__(self, sim, log_dir, env_index=0, metadata=None):
        self.sim, self.env = sim, int(env_index)
        self.dir = os.path.join(log_dir, "episodes")
        os.makedirs(self.dir, exist_ok=True)
        self.metadata = dict(metadata or {})
        self.count, self.file, self._buf = 0, None, []
        self._t0 = self._ret = self._steps = self._min_d = None

    # ---- logger.py:148-273 ----
    def begin_episode(self, episode_id=None):
        self.count += 1
        self.episode_id = episode_id or f"ep_{self.count:06d}"
        self._t0, self._ret, self._steps, self._min_d = time.time(), 0.0, 0, float("inf")
        self.file = os.path.join(self.dir, self.episode_id + ".jsonl")
        with open(self.file, "w") as f:
            f.write(json.dumps({"type": "header", "episode_id": self.episode_id, "start_time": self._t0,
                                "metadata": self.metadata}) + "\n")
        self._buf = []

    def _state(self, entity_id, state):
        self._buf.append({"type": "state", "timestamp": time.time() - self._t0, "entity_id": entity_id, "state": state})
        if len(self._buf) >= 100:
            self._flush()

    def _flush(self):
        if self._buf:
            with open(self.file, "a") as f:
                for e in self._buf:
                    f.write(json.dumps(e) + "\n")
            self._buf = []

    def record_tick(self, action, reward, terminated, truncated, distance, intercepted):
        """Call after every sim.step(auto_reset=False) (or before the auto-reset overwrote the env) with the env's action
        and outputs; reads the env's state from the device.  Returns True when the episode ended (footer written)."""
        if self.file is None:
            self.begin_episode()
        s = self.sim.export_state(self.env, 1)
        self._state("interceptor", {"position": s["ipos"][0].astype(np.float32).tolist(), "fuel": float(s["fuel"][0]),
                                    "action": np.asarray(action, np.float32).tolist()})
        self._state("missile", {"position": s["mpos"][0].astype(np.float32).tolist()})
        self._ret += float(reward)
        self._steps += 1
        self._min_d = min(self._min_d, float(distance))
        if not (terminated or truncated):
            return False
        self._flush()
        end = time.time()
        outcome = "intercepted" if intercepted else "failed"     # inference.py:586
        metrics = {"total_reward": self._ret, "steps": self._steps, "final_distance": float(distance),
                   "min_distance": self._min_d, "fuel_used": float(s["fuel_used"][0])}
        with open(self.file, "a") as f:
            f.write(json.dumps({"type": "footer", "episode_id": self.episode_id, "end_time": end, "duration": end - self._t0,
                                "outcome": outcome, "metrics": metrics}) + "\n")
        self.file = None
        return True


def write_episodes(log_dir, result, dt, metadata=None):
    """Writes `<log_dir>/episodes/ep_XXXXXX.jsonl` (ep_000001 first) for every episode of an EvalResult of
    `DeviceEvaluator.evaluate(..., trace=True)`, in SB3's order, with the lines EpisodeRecorder writes: header, per tick an
    `interceptor` state (position, fuel, action) and a `missile` state (position), footer.  The metrics are EpisodeRecorder's:
    total_reward is the float64 sum of the rewards in tick order, min_distance the minimum of the ticks' info['distance'],
    final_distance the last tick's, fuel_used the done record's.

    The ticks ran in batches on the device, not one at a time on the host, so time is simulated time: a state line's
    `timestamp` is (step - 1) * dt (EpisodeRecorder: wall-clock seconds since the episode began), the footer's `duration` is
    steps * dt, and `start_time` / `end_time` are the wall clock at writing and that plus the duration.  `fuel` is
    info['fuel_remaining'] (float32; EpisodeRecorder logs the state's float64).  Returns the paths written."""
    rows, off = result.trajectories, result.trajectory_offsets
    if rows is None or off is None:
        raise ValueError("the result has no trajectories: evaluate with trace=True")
    if len(off) != len(result.records) + 1:
        raise ValueError(f"{len(off) - 1} trajectories for {len(result.records)} episodes")
    dt = float(dt)
    out_dir = os.path.join(log_dir, "episodes")
    os.makedirs(out_dir, exist_ok=True)
    metadata = dict(metadata or {})
    paths = []
    for i, rec in enumerate(result.records):
        ep = rows[off[i]:off[i + 1]]
        episode_id = f"ep_{i + 1:06d}"
        t0 = time.time()
        lines = [{"type": "header", "episode_id": episode_id, "start_time": t0, "metadata": metadata}]
        total, min_d = 0.0, float("inf")
        ipos, mpos, act = ep["interceptor_pos"].tolist(), ep["missile_pos"].tolist(), ep["action"].tolist()
        for k, (step, fuel, reward, dist) in enumerate(zip(ep["step"].tolist(), ep["fuel_remaining"].tolist(), ep["reward"].tolist(),
                                                            ep["distance"].tolist())):
            ts = (step - 1) * dt
            lines.append({"type": "state", "timestamp": ts, "entity_id": "interceptor",
                          "state": {"position": ipos[k], "fuel": fuel, "action": act[k]}})
            lines.append({"type": "state", "timestamp": ts, "entity_id": "missile", "state": {"position": mpos[k]}})
            total += reward
            min_d = min(min_d, dist)
        duration = len(ep) * dt
        outcome = "intercepted" if int(ep["flags"][-1]) & abi.INFO_INTERCEPTED else "failed"     # inference.py:586
        metrics = {"total_reward": total, "steps": len(ep), "final_distance": float(ep["distance"][-1]),
                   "min_distance": min_d, "fuel_used": float(rec["fuel_used"])}
        lines.append({"type": "footer", "episode_id": episode_id, "end_time": t0 + duration, "duration": duration,
                      "outcome": outcome, "metrics": metrics})
        path = os.path.join(out_dir, episode_id + ".jsonl")
        with open(path, "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))
        paths.append(path)
    return paths

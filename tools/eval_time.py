"""Timing of policy evaluation on the device (DESIGN.md section 14), in one GPU call:

  * DeviceEvaluator.evaluate(E = n_envs) at 131 072 envs, cfg4 (max_steps 2000), graph mode with the default chunk:
    26-D frames stacked 4 deep with the 104-wide fused policy, 17-D/4 with the 68-wide one; ticks, wall time around the call
    (it ends in a device synchronise), env-steps/s, episodes/s;
  * the same tick without the episode accounting: deterministic forward + pipe.step for one chunk as a CUDA graph, replayed,
    so the difference is what hlynr_eval_record and the one counter read per chunk cost.

    python tools/eval_time.py [--envs 131072] [--reps 3] [--out FILE]

The card's name and power limit are printed with the results."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def _layout(frame_dim, n, reps):
    import torch
    from hlynr_intercept_b200 import config
    from hlynr_intercept_b200.evaluation import DeviceEvaluator
    from hlynr_intercept_b200.policy import FusedActorCritic, ReferenceActorCritic
    from hlynr_intercept_b200.post import HlynrObsPipeline
    from hlynr_intercept_b200.rollout import TickGraph
    from hlynr_intercept_b200.sim import HlynrSim

    sim = HlynrSim(config.baseline_config("cfg4"), n_envs=n, seed=4321, warn_dead=False, obs_dim=frame_dim)
    pipe = HlynrObsPipeline(sim, n_stack=4, training=False)
    torch.manual_seed(0)
    fused = FusedActorCritic(ReferenceActorCritic(obs_dim=pipe.obs_dim, device="cuda"), device=0)
    ev = DeviceEvaluator(pipe, fused)
    ev.evaluate(n)   # warm-up: module loads, first launches
    runs = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = ev.evaluate(n)
        s = time.perf_counter() - t0
        runs.append({"ticks": res.ticks, "s": s, "env_steps_per_s": n * res.ticks / s, "episodes_per_s": n / s,
                     "us_per_tick": s / res.ticks * 1e6, "mean_reward": res.mean_reward, "max_end_tick": int(res.end_tick.max())})
    # the same tick without the accounting, as graph replays of one chunk
    act = torch.empty(n, 6, device="cuda")

    def chunk():
        for _ in range(ev.chunk):
            fused.forward(ev.obs, deterministic=True, want=(), out=dict(clipped=act))
            pipe.step(act, out=ev.obs)

    with torch.no_grad():
        pipe.reset(out=ev.obs)
        g = TickGraph(pipe, ev.chunk, chunk)
        k = max(1, runs[0]["ticks"] // ev.chunk)
        plain = []
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(k):
                g.replay()
            torch.cuda.synchronize()
            plain.append((time.perf_counter() - t0) / (k * ev.chunk) * 1e6)
    fused.close(); pipe.close(); sim.close()
    med = lambda key: statistics.median(r[key] for r in runs)  # noqa: E731
    return {"envs": n, "in_dim": 4 * frame_dim, "chunk": ev.chunk, "n_eval_episodes": n, "runs": runs,
            "ticks": med("ticks"), "s": med("s"), "env_steps_per_s": med("env_steps_per_s"), "episodes_per_s": med("episodes_per_s"),
            "us_per_tick": med("us_per_tick"), "us_per_tick_without_accounting": statistics.median(plain),
            "us_per_tick_without_accounting_all": plain}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=131072)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    sys.path.insert(0, HERE)
    import torch

    if not torch.cuda.is_available():
        sys.exit("eval_time.py measures on a CUDA device; none is visible")
    res = {"card": _card()}
    print("card (name, power limit, max SM clock):", res["card"], flush=True)
    for f in (26, 17):
        r = _layout(f, args.envs, args.reps)
        res[f"{f}x4"] = r
        print(f"{f}-D/4, {r['in_dim']}-wide policy:", json.dumps({k: v for k, v in r.items() if k != "runs"}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()

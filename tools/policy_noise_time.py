"""Timings of the fused policy's device-side noise counter (DESIGN.md sections 12 and 14), in one GPU call:

  A/B, two builds of the project alternated on the same card, 26-D frames stacked 4 deep:
    * fused policy forward at 131 072 rows, cluster 1, in_dim 104 (CUDA events, median of 7 windows of 100 calls);
    * rollout_collection.cfg5 from `python bench.py` (bench.py run in each tree as it is);
  new figures of this build (not compared):
    * the per-tick cost of DeviceEvaluator.evaluate at 1037 and 131 072 envs, cfg4, 104-wide fused policy, deterministic next to
      stochastic, in alternation: one chunk of the evaluator's tick (forward, pipe.step, hlynr_eval_record) as a CUDA graph,
      replayed (CUDA events over 2400 ticks); and, for reference, the per-call average of a whole evaluate(E = n_envs) (wall
      time around the call over the ticks it ran), which also carries the reset, the eager first chunk and the graph recording
      that every call repeats.

    python tools/policy_noise_time.py [--other DIR [--no-new]] [--reps 3] [--out FILE]

DIR is a checkout of the other build with its library built.  The card's name and power limit are printed with the results."""
import argparse
import json
import os
import statistics
import sys
import time

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(HERE, "tools"))
from obs_layouts_time import _bench, _card, _forward_in  # noqa: E402


def _eval_us_per_tick(n, reps):
    import torch
    from hlynr_intercept_b200 import config
    from hlynr_intercept_b200.evaluation import DeviceEvaluator
    from hlynr_intercept_b200.policy import FusedActorCritic, ReferenceActorCritic
    from hlynr_intercept_b200.post import HlynrObsPipeline
    from hlynr_intercept_b200.rollout import TickGraph
    from hlynr_intercept_b200.sim import HlynrSim

    sim = HlynrSim(config.baseline_config("cfg4"), n_envs=n, seed=4321, warn_dead=False)
    pipe = HlynrObsPipeline(sim, n_stack=4, training=False)
    torch.manual_seed(0)
    fused = FusedActorCritic(ReferenceActorCritic(obs_dim=pipe.obs_dim, device="cuda"), device=0)
    ev = DeviceEvaluator(pipe, fused)
    out = {}
    for det in (True, False):   # warm-up of both kinds
        ev.evaluate(n, deterministic=det)
    for _ in range(reps):
        for det in (True, False):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = ev.evaluate(n, deterministic=det)
            s = time.perf_counter() - t0
            # the steady-state tick: replays of one chunk, recorded after evaluate() left the evaluator in this mode
            with torch.no_grad():
                pipe.reset(out=ev.obs)
                g = TickGraph(pipe, ev.chunk, ev._chunk)
                reps_g = max(1, 2400 // ev.chunk)
                g.replay(); torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps_g):
                    g.replay()
                e1.record(); torch.cuda.synchronize()
            out.setdefault("deterministic" if det else "stochastic", []).append(
                {"us_per_tick": e0.elapsed_time(e1) * 1e3 / (reps_g * ev.chunk), "us_per_tick_per_call": s / res.ticks * 1e6,
                 "ticks": res.ticks, "mean_reward": res.mean_reward})
    fused.close(); pipe.close(); sim.close()
    summ = {"envs": n, "chunk": ev.chunk}
    for k, runs in out.items():
        summ[k] = {"runs": runs}
        for key in ("us_per_tick", "us_per_tick_per_call"):
            us = [r[key] for r in runs]
            summ[k][key] = (statistics.median(us), min(us), max(us))
    return summ


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--other", help="checkout of the other build (A/B); omitted: new figures only")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--bench-steps", type=int, default=100)
    ap.add_argument("--bench-warmup", type=int, default=20)
    ap.add_argument("--no-new", action="store_true", help="the A/B only")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    sys.path.insert(0, HERE)
    import torch

    if not torch.cuda.is_available():
        sys.exit("policy_noise_time.py measures on a CUDA device; none is visible")
    res = {"card": _card(), "ab": [], "new": {}}
    print("card (name, power limit, max SM clock):", res["card"], flush=True)
    if args.other:
        trees = {"other": os.path.abspath(args.other), "this": HERE}
        for rep in range(args.reps):
            for name in (["other", "this"] if rep % 2 == 0 else ["this", "other"]):
                row = {"build": name, "rep": rep, "forward_us": _forward_in(trees[name])}
                row.update(_bench(trees[name], args.bench_steps, args.bench_warmup))
                res["ab"].append(row)
                print(json.dumps(row), flush=True)
        for name in ("other", "this"):
            rows = [r for r in res["ab"] if r["build"] == name]
            summ = {k: (statistics.median(r[k] for r in rows), min(r[k] for r in rows), max(r[k] for r in rows))
                    for k in ("forward_us", "cfg5")}
            res[f"ab_{name}"] = summ
            print(name, "median (min, max):", json.dumps(summ), flush=True)
    if not args.no_new:
        for n in (1037, 131072):
            r = res["new"][f"eval_{n}"] = _eval_us_per_tick(n, args.reps)
            print(f"evaluate() at {n} envs, us per tick (median, min, max) as graph replays and per call:",
                  json.dumps({k: {kk: vv for kk, vv in v.items() if kk != "runs"} if isinstance(v, dict) else v for k, v in r.items()}),
                  flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

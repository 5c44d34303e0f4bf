"""Timings of traced evaluation (DeviceEvaluator.evaluate(trace=True), DESIGN.md section 16), in one GPU call:

  new figures of this build:
    * the per-tick cost of the evaluator's tick with and without the trace (info arrays written by the step kernel +
      hlynr_eval_trace), cfg4, 26-D frames stacked 4 deep, the 104-wide fused policy, at 1037 and 131 072 envs: replays of one
      chunk graph recorded right after a reset with 2 episodes per env to go, so every env is inside its quota while timed
      (CUDA events over 8 replays), the two kinds alternated, 3 windows each;
  A/B, two builds of the project alternated on the same card (--other DIR):
    * the untraced evaluator tick, measured the same way in each tree (a subprocess per tree);
    * rollout_collection.cfg5 from `python bench.py` (bench.py run in each tree as it is).

    python tools/trace_time.py [--other DIR] [--reps 3] [--out FILE]

DIR is a checkout of the other build with its library built.  The card's name and power limit are printed with the results."""
import argparse
import json
import os
import statistics
import subprocess
import sys

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(HERE, "tools"))
from obs_layouts_time import _bench, _card  # noqa: E402

SIZES = (1037, 131072)


def _evaluator(n):
    import torch

    from hlynr_intercept_b200 import config
    from hlynr_intercept_b200.evaluation import DeviceEvaluator
    from hlynr_intercept_b200.policy import FusedActorCritic, ReferenceActorCritic
    from hlynr_intercept_b200.post import HlynrObsPipeline
    from hlynr_intercept_b200.sim import HlynrSim

    sim = HlynrSim(config.baseline_config("cfg4"), n_envs=n, seed=4321, warn_dead=False)
    pipe = HlynrObsPipeline(sim, n_stack=4, training=False)
    torch.manual_seed(0)
    fused = FusedActorCritic(ReferenceActorCritic(obs_dim=pipe.obs_dim, device="cuda"), device=0)
    ev = DeviceEvaluator(pipe, fused)
    ev.evaluate(n)   # warm-up: every launch of the tick has run once
    return ev


def _window(ev, trace, replays=8):
    """us per tick of `replays` chunk-graph replays right after a reset, every env inside a quota of 2 episodes (cfg4's
    episodes are longer than the window).  trace None: the parent's evaluator, set up through the attributes both builds have."""
    import torch

    from hlynr_intercept_b200.rollout import TickGraph

    E = 2 * ev.sim.n
    if trace is None:
        ev.counts.zero_(); ev.ticks.zero_(); ev.remaining.fill_(E)
    else:
        ev._prepare(E, trace)
    with torch.no_grad():
        ev.pipe.reset(out=ev.obs)
        g = TickGraph(ev.pipe, ev.chunk, ev._chunk)
        g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(replays):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
    del g
    return e0.elapsed_time(e1) * 1e3 / (replays * ev.chunk)


def _summary(us):
    return (statistics.median(us), min(us), max(us))


def _traced_vs_untraced(n, reps):
    ev = _evaluator(n)
    runs = {"untraced": [], "traced": []}
    for r in range(reps):
        for kind in (["untraced", "traced"] if r % 2 == 0 else ["traced", "untraced"]):
            runs[kind].append(_window(ev, kind == "traced"))
    ev._prepare(1, False)
    ev.policy.close(); ev.pipe.close(); ev.sim.close()
    out = {"envs": n, "chunk": ev.chunk}
    for k, us in runs.items():
        out[k] = {"us_per_tick": _summary(us), "runs": us}
    out["added_us_per_tick"] = out["traced"]["us_per_tick"][0] - out["untraced"]["us_per_tick"][0]
    return out


def _worker(n):
    ev = _evaluator(n)
    print(json.dumps({"us_per_tick": _window(ev, None)}), flush=True)


def _untraced_in(tree, n):
    r = subprocess.run([sys.executable, os.path.join(HERE, "tools", "trace_time.py"), "--worker", "--envs", str(n)], cwd=tree,
                       env=dict(os.environ, PYTHONPATH=tree), stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    if r.returncode:
        raise RuntimeError(f"worker in {tree} failed:\n{r.stderr[-3000:]}")
    return json.loads(r.stdout.strip().splitlines()[-1])["us_per_tick"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--other", help="checkout of the other build (A/B); omitted: new figures only")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--bench-steps", type=int, default=100)
    ap.add_argument("--bench-warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--envs", type=int, default=0, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:   # runs with cwd and PYTHONPATH at the tree under test
        sys.path.insert(0, os.getcwd())
        return _worker(args.envs)
    sys.path.insert(0, HERE)
    import torch

    if not torch.cuda.is_available():
        sys.exit("trace_time.py measures on a CUDA device; none is visible")
    res = {"card": _card(), "new": {}, "ab": []}

    def save():
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                json.dump(res, f, indent=1)
    print("card (name, power limit, max SM clock):", res["card"], flush=True)
    for n in SIZES:
        r = res["new"][f"eval_{n}"] = _traced_vs_untraced(n, args.reps)
        print(f"evaluator tick at {n} envs, us (median, min, max):",
              json.dumps({k: ({kk: vv for kk, vv in v.items() if kk != "runs"} if isinstance(v, dict) else v) for k, v in r.items()}),
              flush=True)
        save()
    if args.other:
        trees = {"other": os.path.abspath(args.other), "this": HERE}
        for rep in range(args.reps):
            for name in (["other", "this"] if rep % 2 == 0 else ["this", "other"]):
                row = {"build": name, "rep": rep}
                for n in SIZES:
                    row[f"untraced_{n}_us"] = _untraced_in(trees[name], n)
                row["cfg5"] = _bench(trees[name], args.bench_steps, args.bench_warmup)["cfg5"]
                res["ab"].append(row)
                print(json.dumps(row), flush=True)
                save()
        for name in ("other", "this"):
            rows = [r for r in res["ab"] if r["build"] == name]
            res[f"ab_{name}"] = {k: _summary([r[k] for r in rows]) for k in rows[0] if k not in ("build", "rep")}
            print(name, "median (min, max):", json.dumps(res[f"ab_{name}"]), flush=True)
    save()


if __name__ == "__main__":
    main()

"""Timings of the device-side curriculum counter (DESIGN.md section 15), in one GPU call:

  A/B, two builds of the project alternated on the same card (a sim that never attaches a schedule runs the same kernels as
  before, so this is the detached path):
    * bench.py's headline, the API step (cfg4, 2^20 envs, steady state), its ms per step, configs.cfg2@4096 and
      rollout_collection.cfg5 (bench.py run in each tree as it is);
  new figures of this build (not compared):
    * DeviceRolloutCollector replays (cfg4, 26-D frames stacked 4 deep, the 104-wide fused policy, n_steps 24) at 131 072 and
      4 096 envs, a tracking sim next to an untracked one, in alternation: CUDA events over 8 replays, 5 windows each; the
      difference per tick is what the curriculum tick kernel adds.

    python tools/curriculum_time.py [--other DIR [--no-new]] [--reps 3] [--out FILE]

DIR is a checkout of the other build with its library built.  The card's name and power limit are printed with the results."""
import argparse
import json
import os
import statistics
import subprocess
import sys

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(HERE, "tools"))
from obs_layouts_time import _card  # noqa: E402


def _bench(tree, steps, warmup):
    cmd = [sys.executable, "bench.py", "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup), "--no-cpu-baseline",
           "--strong-total", "0", "--fused", "0", "--cfg5-cpu-seconds", "0", "--ref-python-seconds", "0"]
    r = subprocess.run(cmd, cwd=tree, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    if r.returncode:
        raise RuntimeError(f"bench.py in {tree} failed:\n{r.stderr[-3000:]}")
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    return {"api_cfg4": line["value"], "api_ms_per_step": line["ms_per_step"], "cfg2@4096": line["configs"]["cfg2@4096"]["value"],
            "cfg5": line["rollout_collection"]["cfg5"]["value"]}


def _collector(n, track, T):
    import torch

    from hlynr_intercept_b200 import config
    from hlynr_intercept_b200.policy import FusedActorCritic, ReferenceActorCritic
    from hlynr_intercept_b200.post import HlynrObsPipeline
    from hlynr_intercept_b200.rollout import DeviceRolloutCollector
    from hlynr_intercept_b200.sim import HlynrSim

    sim = HlynrSim(config.baseline_config("cfg4"), n_envs=n, seed=4321, warn_dead=False)
    if track:
        sim.track_training_steps(0)
    pipe = HlynrObsPipeline(sim, n_stack=4, training=True)
    torch.manual_seed(0)
    fused = FusedActorCritic(ReferenceActorCritic(obs_dim=pipe.obs_dim, device="cuda"), device=0)
    col = DeviceRolloutCollector(pipe, fused, T)
    col.capture()
    return col


def _collector_us_per_tick(n, windows=5, replays=8, T=24):
    import torch

    cols = {"untracked": _collector(n, False, T), "tracked": _collector(n, True, T)}
    for c in cols.values():
        c.replay()
    torch.cuda.synchronize()
    runs = {k: [] for k in cols}
    for w in range(windows):
        for name in (["untracked", "tracked"] if w % 2 == 0 else ["tracked", "untracked"]):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(replays):
                cols[name].replay()
            e1.record()
            torch.cuda.synchronize()
            runs[name].append(e0.elapsed_time(e1) * 1e3 / (replays * T))
    t = cols["tracked"].sim
    assert t.num_timesteps == (2 + windows * replays) * T * n, t.num_timesteps   # capture's warm-up + the first replay
    out = {"envs": n, "n_steps": T, "launches_per_tick": {k: c._graph.launches[0] / T for k, c in cols.items()}}
    for k, us in runs.items():
        out[k] = {"us_per_tick": (statistics.median(us), min(us), max(us)), "runs": us}
    out["added_us_per_tick"] = out["tracked"]["us_per_tick"][0] - out["untracked"]["us_per_tick"][0]
    for c in cols.values():
        c.policy.close(); c.pipe.close(); c.sim.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--other", help="checkout of the other build (A/B); omitted: new figures only")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--bench-steps", type=int, default=200)
    ap.add_argument("--bench-warmup", type=int, default=50)
    ap.add_argument("--no-new", action="store_true", help="the A/B only")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    sys.path.insert(0, HERE)
    import torch

    if not torch.cuda.is_available():
        sys.exit("curriculum_time.py measures on a CUDA device; none is visible")
    res = {"card": _card(), "ab": [], "new": {}}

    def save():   # after every row: a partial run still leaves its figures
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                json.dump(res, f, indent=1)
    print("card (name, power limit, max SM clock):", res["card"], flush=True)
    if not args.no_new:
        for n in (131072, 4096):
            r = res["new"][f"collector_{n}"] = _collector_us_per_tick(n)
            print(f"collector replay at {n} envs, us per tick (median, min, max):",
                  json.dumps({k: ({kk: vv for kk, vv in v.items() if kk != "runs"} if isinstance(v, dict) else v) for k, v in r.items()}),
                  flush=True)
            save()
    if args.other:
        trees = {"other": os.path.abspath(args.other), "this": HERE}
        for rep in range(args.reps):
            for name in (["other", "this"] if rep % 2 == 0 else ["this", "other"]):
                row = {"build": name, "rep": rep}
                row.update(_bench(trees[name], args.bench_steps, args.bench_warmup))
                res["ab"].append(row)
                print(json.dumps(row), flush=True)
                save()
        for name in ("other", "this"):
            rows = [r for r in res["ab"] if r["build"] == name]
            summ = {k: (statistics.median(r[k] for r in rows), min(r[k] for r in rows), max(r[k] for r in rows))
                    for k in ("api_cfg4", "api_ms_per_step", "cfg2@4096", "cfg5")}
            res[f"ab_{name}"] = summ
            print(name, "median (min, max):", json.dumps(summ), flush=True)
    save()


if __name__ == "__main__":
    main()

"""Timings of the observation layouts of the device training path (DESIGN.md sections 9 and 12), in one GPU call:

  A/B, two builds of the project alternated on the same card, 26-D frames stacked 4 deep:
    * fused policy forward at 131 072 rows, cluster 1 (CUDA events, median of 7 windows of 100 calls);
    * rollout_collection.cfg5 and obs_pipeline from `python bench.py` (bench.py run in each tree as it is);
  new figures of this build (not compared):
    * fused forward at in_dim 26, 52, 68, 78, 104, 136, 208 at 131 072 rows;
    * hlynr_post_step alone at 2^20 envs, 17-D/4 next to 26-D/4 (training on; the step's outputs are replayed);
    * rollout collection at 131 072 envs x 24 steps as one graph replay, 17-D/4 with the 68-wide fused policy next to
      26-D/4 with the default 104-wide one.

    python tools/obs_layouts_time.py [--other DIR [--no-new]] [--reps 3] [--out FILE]

DIR is a checkout of the other build with its library built.  The card's name and power limit are printed with the results."""
import argparse
import json
import os
import statistics
import subprocess
import sys

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROWS = 131072


def _events_us(torch, f, calls=100, windows=7):
    f(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = []
    for _ in range(windows):
        e0.record()
        for _ in range(calls):
            f()
        e1.record(); torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) / calls * 1e3)
    return statistics.median(out), min(out), max(out)


def _forward_us(in_dim, cluster=1):
    """Fused forward of a ReferenceActorCritic of input width in_dim (the default 104 uses only the API of every build)."""
    import torch
    from hlynr_intercept_b200.policy import FusedActorCritic, ReferenceActorCritic

    torch.manual_seed(0)
    net = ReferenceActorCritic(obs_dim=in_dim, device="cuda")
    fused = FusedActorCritic(net, device=0)
    fused.set_option("cluster", cluster)
    obs = torch.randn(ROWS, in_dim, device="cuda")
    r = _events_us(torch, lambda: fused(obs))
    fused.close()
    return r


def worker_forward():
    med, lo, hi = _forward_us(104)
    print(json.dumps({"forward_us": med, "min": lo, "max": hi}))


def _post_step_ms(frame_dim, n=1 << 20, n_stack=4, steps=200):
    import ctypes as C

    import torch
    from hlynr_intercept_b200 import _lib, config
    from hlynr_intercept_b200.post import HlynrObsPipeline
    from hlynr_intercept_b200.sim import HlynrSim

    sim = HlynrSim(config.baseline_config("cfg4"), n_envs=n, seed=1, warn_dead=False, obs_dim=frame_dim)
    pipe = HlynrObsPipeline(sim, n_stack=n_stack, training=True)
    pipe.reset()
    a = torch.rand(n, 6, device="cuda") * 2 - 1
    for _ in range(8):
        out, rew, te, tr, (rec, cnt, term) = pipe.step(a)
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    st = pipe._stream()

    def post():
        _lib.check(pipe.L.hlynr_post_step(pipe.h, p(rew), p(te), p(tr), p(rec), p(cnt), n, p(out), p(term), 1, st))

    med, lo, hi = _events_us(torch, post, calls=steps // 7 + 1)
    pipe.close(); sim.close()
    return {"ms": med / 1e3, "min_ms": lo / 1e3, "max_ms": hi / 1e3, "envs": n, "n_stack": n_stack,
            "done_per_step": int(cnt.item())}


def _rollout(frame_dim, n=ROWS, n_stack=4, T=24):
    import time

    import torch
    from hlynr_intercept_b200 import config
    from hlynr_intercept_b200.policy import FusedActorCritic, ReferenceActorCritic
    from hlynr_intercept_b200.post import HlynrObsPipeline
    from hlynr_intercept_b200.rollout import DeviceRolloutCollector
    from hlynr_intercept_b200.sim import HlynrSim

    sim = HlynrSim(config.baseline_config("cfg4"), n_envs=n, seed=4321, warn_dead=False, obs_dim=frame_dim)
    pipe = HlynrObsPipeline(sim, n_stack=n_stack, training=True)
    torch.manual_seed(0)
    fused = FusedActorCritic(ReferenceActorCritic(obs_dim=frame_dim * n_stack, device="cuda"), device=0)
    col = DeviceRolloutCollector(pipe, fused, T)
    col.capture()
    col.replay(); torch.cuda.synchronize()
    reps = max(1, -(-5_000_000 // (n * T)))
    times = []
    for _ in range(5):
        t0 = time.perf_counter()
        for _ in range(reps):
            col.replay()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    s = statistics.median(times)
    fused.close(); pipe.close(); sim.close()
    return {"env_steps_per_s": n * T * reps / s, "min": n * T * reps / max(times), "max": n * T * reps / min(times),
            "envs": n, "n_steps": T, "in_dim": frame_dim * n_stack}


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def _bench(tree, steps, warmup):
    cmd = [sys.executable, "bench.py", "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup), "--no-cpu-baseline",
           "--no-configs", "--strong-total", "0", "--fused", "0", "--cfg5-cpu-seconds", "0", "--ref-python-seconds", "0"]
    r = subprocess.run(cmd, cwd=tree, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    if r.returncode:
        raise RuntimeError(f"bench.py in {tree} failed:\n{r.stderr[-3000:]}")
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    return {"cfg5": line["rollout_collection"]["cfg5"]["value"], "obs_pipeline": line["obs_pipeline"]["value"],
            "headline": line["value"]}


def _forward_in(tree):
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", "--tree", tree], stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True)
    if r.returncode:
        raise RuntimeError(f"forward worker in {tree} failed:\n{r.stderr[-3000:]}")
    return json.loads(r.stdout.strip().splitlines()[-1])["forward_us"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--other", help="checkout of the other build (A/B); omitted: new figures only")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--bench-steps", type=int, default=100)
    ap.add_argument("--bench-warmup", type=int, default=20)
    ap.add_argument("--no-new", action="store_true", help="the A/B only")
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--tree", default=HERE)
    args = ap.parse_args()
    if args.worker:
        sys.path.insert(0, os.path.abspath(args.tree))
        worker_forward()
        return
    sys.path.insert(0, HERE)
    import torch

    if not torch.cuda.is_available():
        sys.exit("obs_layouts_time.py measures on a CUDA device; none is visible")
    res = {"card": _card(), "ab": [], "new": {}}
    print("card (name, power limit, max SM clock):", res["card"], flush=True)
    if args.other:
        trees = {"other": os.path.abspath(args.other), "this": HERE}
        for rep in range(args.reps):
            order = ["other", "this"] if rep % 2 == 0 else ["this", "other"]
            for name in order:
                row = {"build": name, "rep": rep, "forward_us": _forward_in(trees[name])}
                row.update(_bench(trees[name], args.bench_steps, args.bench_warmup))
                res["ab"].append(row)
                print(json.dumps(row), flush=True)
        for name in ("other", "this"):
            rows = [r for r in res["ab"] if r["build"] == name]
            summ = {k: (statistics.median(r[k] for r in rows), min(r[k] for r in rows), max(r[k] for r in rows))
                    for k in ("forward_us", "cfg5", "obs_pipeline", "headline")}
            res[f"ab_{name}"] = summ
            print(name, "median (min, max):", json.dumps(summ), flush=True)
    if args.no_new:
        args.out and _dump(res, args.out)
        return
    res["new"]["forward_us"] = {d: _forward_us(d)[0] for d in (26, 52, 68, 78, 104, 136, 208)}
    print("forward at 131072 rows, cluster 1 (us):", json.dumps(res["new"]["forward_us"]), flush=True)
    res["new"]["post_step"] = {f"{f}x4": _post_step_ms(f) for f in (26, 17)}
    print("post step at 2^20 envs:", json.dumps(res["new"]["post_step"]), flush=True)
    res["new"]["rollout"] = {f"{f}x4": _rollout(f) for f in (17, 26)}
    print("rollout 131072 x 24, graph:", json.dumps(res["new"]["rollout"]), flush=True)
    if args.out:
        _dump(res, args.out)


def _dump(res, path):
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

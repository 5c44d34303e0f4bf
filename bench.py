#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched Hlynr Intercept step on B200 (BASELINE.json metric).

A "step" is one tick (environment.py:605 step + SB3 auto-reset) of every env of the batch = ONE launch of
the sm_100a step kernel through the C ABI (hlynr_step), actions resident in HBM.  The episodes are aged
(desynchronised by a fused rollout) before the warm-up, so the timed ticks run at the steady-state rate of
finished episodes and in-kernel auto-resets (`done_episodes_per_step`, `episode_stats`).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg4] [--envs-per-gpu 1048576] [--dump-outputs DIR]
  torchrun --nproc-per-node N bench.py --gpus N ...        (one rank per GPU, envs sharded by global id, no
                                                           per-step communication; one NCCL all-reduce of the
                                                           episode-statistics block per rollout, inside the
                                                           timed region)
  python bench.py --impl reference ...                     (reference arm: the C port of the reference step on all
                                                           host cores at the full workload size, plus the unmodified
                                                           Python reference under a SubprocVecEnv clone, bounded)

Prints ONE JSON line (rank 0).  `value` = env-steps/s with inputs resident in HBM (weak scaling: --envs-per-gpu
envs on every GPU); `strong` = the same for BASELINE cfg4's 2^20 envs IN TOTAL sharded over the GPUs; `configs` =
BASELINE cfg2 at 4096 envs and cfg3 at 262144 envs; `e2e` = the metric through the numpy VecEnv API (pinned H2D of
actions, D2H of obs/reward/dones every step); `roofline` = the step kernel against the measured HBM copy bandwidth;
`cpu_baseline` = the C port and the Python reference on the host cores.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# SURVEY 8(d): algorithmic bytes per env-step, fp32 build, API mode (the roofline contract figure)
ALGO_BYTES = {"cfg2": 526, "cfg3": 630, "cfg3_radar": 630, "cfg4": 630, "cfg1": 630}
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback


def layout_bytes(workload, precision="fp32"):
    """Bytes per env-step the kernel's OWN layout moves (DESIGN.md section 2): state planes read + written, one delay-ring
    slot read + written per sensor, actions in, obs / reward / terminated / truncated out."""
    r = 4 if precision == "fp32" else 8
    v2 = workload in ("cfg1", "cfg3", "cfg3_radar", "cfg4")
    dr = workload in ("cfg3", "cfg3_radar")
    r_planes = 7 if v2 else 6                  # r0-r5 (+ r6 thrust / T0 with thrust lag or DR)
    f_planes = 3 + (1 if (dr and precision != "fp32") else 0)   # quaternion, wind + base Cd, Kalman P block (+ DR peak: in i0.y in the fp32 build)
    compact = workload == "cfg4" and precision == "fp32"   # counters ride in r6.w / f1.w: no i0 plane (hlynr_device.cuh load_env)
    state = r_planes * 4 * r + f_planes * 16 + (0 if compact else 16)   # + the counter plane i0
    rings = 2 * 4 * r + (16 if v2 else 0)                  # ground slot {rel, q}, {vel, flag}; onboard slot (sensor delay, v2.0)
    io = 24 + 104 + 4 + 1 + 1
    return 2 * state + 2 * rings + io


def measured_traffic(workload, n):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the step kernel, from the committed ncu capture of >= 10
    back-to-back steady-state launches (profiles/traffic.json, which names the capture), scaled to n envs; None if absent."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        t = json.load(open(p))[workload]
        return t["dram_bytes_per_launch"] * n / t["n_envs"]
    except Exception:
        return None


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def policy_roofline(flop, us):
    """The fused policy forward against the measured dense bf16 throughput of this pool's B200s (cuBLAS 8192^3, MEASURED_PEAKS.json:
    the burst figure, the kernel is timed alone); the nominal 2250 TFLOP/s if the file is absent."""
    peak, src = 2250.0, "nominal dense bf16"
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            peak, src = float(json.load(open(p))["bf16_tflops"]), "measured (MEASURED_PEAKS.json bf16_tflops)"
        except Exception:
            pass
    ach = flop / (us * 1e-6) / 1e12
    return {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "peak_source": src,
            "note": "per 128-row tile the GEMM phases run at tensor-pipe speed (9.9 us) and do not overlap the LayerNorm epilogues (16.2 us): "
                    "one tile's accumulators fill the 512 TMEM columns (DESIGN.md section 12)"}


class ClockSampler:
    """Samples nvidia-smi SM clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def count_between(self, t0, t1):
        return sum(1 for t, _ in self.rows if t0 <= t <= t1)

    def stop(self, windows=None):
        """windows: [(t0, t1), ...] perf_counter intervals whose samples count (None = all)."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        for t, r in self.rows:
            if windows is not None and not any(a <= t <= b for a, b in windows):
                continue
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------------------
# CPU legs
# ----------------------------------------------------------------------------------------------------------
def port_steps(workload, n_envs, steps, warmup, threads, seconds=None):
    """The oracle port (C restatement of the reference step) on `threads` host threads: K steps of n_envs envs, or as many as
    fit into `seconds`.  Returns (env-steps/s, steps, seconds)."""
    from hlynr_intercept_b200 import config
    from oracle import oracle

    P, cur = config.resolve_config(config.baseline_config(workload), warn_dead=False)
    sim = oracle.OracleBatch(P, cur, n_envs, seed=1234, threads=threads)
    sim.reset()
    rng = np.random.default_rng(0)
    acts = [rng.uniform(-1, 1, (n_envs, 6)).astype(np.float32) for _ in range(2)]
    for k in range(warmup):
        sim.step(acts[k % 2], want_info=False)
    t0 = time.perf_counter()
    done = 0
    while (done < steps) if seconds is None else (time.perf_counter() - t0 < seconds):
        sim.step(acts[done % 2], want_info=False)
        done += 1
    dt = time.perf_counter() - t0
    sim.close()
    return n_envs * done / dt, done, dt


def reference_python(workload, seconds):
    """The unmodified Python reference under the Pipe clone of SubprocVecEnv (baseline/ref_vecenv.py); None if not staged."""
    try:
        from baseline import ref_vecenv
        from hlynr_intercept_b200 import config

        if not ref_vecenv.available():
            return {"unavailable": "baseline/_ref/ is not staged (run __graft_entry__.build() where /root/reference exists)"}
        return ref_vecenv.measure(config.baseline_config(workload), seconds=seconds)
    except Exception as e:  # the baseline must never take the GPU measurement down with it
        return {"unavailable": f"{type(e).__name__}: {e}"}


def cpu_baseline(workload, seconds=12.0, n_envs=65536, threads=None, ref_seconds=10.0):
    threads = threads or os.cpu_count() or 1
    v, steps, dt = port_steps(workload, n_envs, 0, 3, threads, seconds=seconds)
    out = {"value": v, "unit": "env-steps/s", "cores": threads, "kind": "port",
           "sample": f"{n_envs} envs x {steps} ticks of {workload} ({dt:.1f} s), C oracle port of the reference step on {threads} threads"}
    if ref_seconds > 0:
        out["reference_python"] = reference_python(workload, ref_seconds)
    return out


def run_reference_arm(args):
    """--impl reference: the reference's CPU implementation of the step on all host threads, K steps of the FULL workload
    (the C port: the Python reference cannot hold 2^20 envs), and the unmodified Python reference as `reference_python`."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n_envs = args.ref_envs if args.ref_envs > 0 else args.envs_per_gpu
    v, steps, dt = port_steps(args.workload, n_envs, args.steps, args.warmup, threads)
    refpy = reference_python(args.workload, args.ref_python_seconds) if args.ref_python_seconds > 0 else None
    line = {"impl": "reference", "metric": "env-steps/s", "value": v, "unit": "env-steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args.workload), "envs_per_gpu": n_envs, "total_envs": n_envs,
                       "actions": "U(-1,1)^6 float32", "timed_region_s": dt},
            "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": threads, "kind": "port",
                             "sample": f"{n_envs} envs per step x {steps} steps ({dt:.1f} s): C oracle port of the reference step, "
                                       f"{threads} threads", "reference_python": refpy},
            "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def workload_name(w):
    return {"cfg4": "cfg4: medium scenario, physics v2.0 on, in-kernel auto-reset",
            "cfg2": "cfg2: medium scenario, physics v2.0 off",
            "cfg3": "cfg3: hard scenario, physics v2.0 on + domain randomization",
            "cfg1": "cfg1: easy scenario"}.get(w, w)


# ----------------------------------------------------------------------------------------------------------
# device legs
# ----------------------------------------------------------------------------------------------------------
class Ctx:
    def __init__(self):
        import torch
        import torch.distributed as dist

        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())


# Fused random-policy ticks before the warm-up.  Episodes last 800-1600 ticks and all start together, so the rate of finished episodes
# (= in-kernel auto-resets) oscillates for several episode lengths before it settles: 0 until tick 750, 1441 per tick at 1500, 349 at
# 1750, 740 at 2000-2025 (where a 2000-tick ageing put a 20-step timed region: a trough), 1280 at 2500 ... 871-895 from tick 8000 on
# (tools/done_rate_series.py, profiles/r02_n_done_rate_series.log).  8000 ticks cost 0.6 s and make a 20-step run and a 2000-step run
# time the same stationary workload.
AGE_TICKS = 8000


def make_aged_sim(ctx, workload, n, first, precision, seed=1234):
    from hlynr_intercept_b200 import config
    from hlynr_intercept_b200.sim import HlynrSim

    torch = ctx.torch
    sim = HlynrSim(config.baseline_config(workload), n_envs=n, device=ctx.local_rank, seed=seed, env_id_offset=first,
                   precision=precision, warn_dead=False)
    sim.reset()
    sim.rollout(AGE_TICKS, None, want_obs=False)
    g = torch.Generator(device=ctx.dev)
    g.manual_seed(seed + first)
    pool = [(torch.rand(n, 6, device=ctx.dev, generator=g) * 2 - 1).contiguous() for _ in range(4)]  # U(-1,1)^6 in HBM
    return sim, pool


def timed_ticks(ctx, sim, pool, K, W, collective=True, graph=False):
    """W warm-up ticks, then K timed ticks bracketed by barrier + synchronize, CUDA events on the launching stream; the
    rollout's one statistics all-reduce is inside the timed region.  Returns a dict (times are this rank's; max over ranks too)."""
    torch, dist = ctx.torch, ctx.dist
    sg = None
    T = 0
    if graph:
        T = math.lcm(sim.ring_period(), len(pool))
        while sim.tick_count() % sim.ring_period():     # captures start on a ring-period boundary
            sim.step(pool[0], want_terminal_obs=False)
        sg = sim.capture_steps([pool[k % len(pool)] for k in range(T)])
    for k in range(W):
        sim.step(pool[k % 4], want_terminal_obs=False)
    if sg is not None:
        while sim.tick_count() % sim.ring_period() != sg.phase:
            sim.step(pool[0], want_terminal_obs=False)
        sg.replay()
    stats_t = sim.stats_tensor()
    if ctx.world > 1 and collective:
        dist.all_reduce(stats_t)  # warm NCCL
    sim.stats(zero_after=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = sim.launch_count()
    sync = ctx.barrier if collective else torch.cuda.synchronize   # single-rank legs must not enter a collective barrier
    sync()
    t0 = time.perf_counter()
    e0.record()
    done = 0
    last = None
    if sg is not None:
        while done + T <= K:
            last = sg.replay()
            done += T
    for k in range(done, K):
        last = sim.step(pool[k % 4], want_terminal_obs=False)
    t_issue = time.perf_counter() - t0
    stats_t = sim.stats_tensor()  # one stats all-reduce per rollout (NVLink); tiny, latency-bound
    if ctx.world > 1 and collective:
        dist.all_reduce(stats_t)
    e1.record()
    sync()
    t1 = time.perf_counter()
    ms = e0.elapsed_time(e1)
    return {"ms": ms, "ms_max": ctx.max_over_ranks(ms) if collective else ms, "launches": sim.launch_count() - launches0,
            "stats": stats_t.cpu().numpy().tolist(), "window": (t0, t1), "host_issue_ms": t_issue * 1e3,
            "graph_ticks": T if sg is not None else 0, "last_outputs": last}


DUMP_MAX_ROWS = 1 << 18   # 2^18 envs x 124 B = 32.5 MB of .npy files


def dump_outputs(out_dir, outputs, first_env):
    """Writes what the last timed step returned to its caller (obs, reward, terminated, truncated of every env of this rank) as
    float32 .npy files, plus the global env id of every row.  Above DUMP_MAX_ROWS envs, a fixed seeded sample of the rows
    (the same rows in every run with the same --envs-per-gpu) keeps the files under 64 MB."""
    obs, reward, terminated, truncated = (t.cpu().numpy() for t in outputs[:4])
    n = obs.shape[0]
    rows = np.arange(n) if n <= DUMP_MAX_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_ROWS, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"obs": obs, "reward": reward, "terminated": terminated, "truncated": truncated}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a[rows].astype(np.float32))
    np.save(os.path.join(out_dir, "env_id.npy"), (rows + first_env).astype(np.float64))


def config_line(ctx, workload, n, K, W, precision, peak):
    """One BASELINE configuration at its own size on this rank's GPU (no collective): eager launches and CUDA-graph replay."""
    sim, pool = make_aged_sim(ctx, workload, n, 0, precision, seed=777)
    r = timed_ticks(ctx, sim, pool, K, W, collective=False)
    rg = timed_ticks(ctx, sim, pool, K, W, collective=False, graph=True)
    # the same ticks as ONE launch per 48 (hlynr_rollout with caller actions [k, N, 6]: state in registers, one observation at the
    # end): what a caller that knows its actions in advance -- the only case a step graph can serve too -- pays per tick
    import torch
    kf = 48
    acts = (torch.rand(kf, n, 6, device=sim.device) * 2 - 1).contiguous()
    sim.rollout(kf, acts)
    torch.cuda.synchronize(sim.device)
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = max(2, min(10, K // kf))
    f0.record()
    for _ in range(reps):
        sim.rollout(kf, acts)
    f1.record()
    torch.cuda.synchronize(sim.device)
    us_f = f0.elapsed_time(f1) / (reps * kf) * 1e3
    del acts
    sim.close()
    us, us_g = r["ms"] / K * 1e3, rg["ms"] / K * 1e3
    best = min(us, us_g)
    lb = layout_bytes(workload, precision)
    ws_mb = n * lb / 1e6
    return {"workload": workload_name(workload), "envs": n, "steps": K, "us_per_tick_eager": us, "us_per_tick_graph": us_g,
            "graph_ticks_per_replay": rg["graph_ticks"], "host_issue_us_per_tick_eager": r["host_issue_ms"] / K * 1e3,
            "us_per_tick_fused_rollout": us_f, "fused_ticks_per_launch": kf,
            "value": n / (best * 1e-6), "unit": "env-steps/s", "done_episodes_per_step": r["stats"][0] / K,
            "roofline_frac_contract": n * ALGO_BYTES[workload] / (best * 1e-6) / 1e9 / peak,
            "roofline_frac_layout": n * lb / (best * 1e-6) / 1e9 / peak,
            "note": (f"per-tick working set {ws_mb:.1f} MB " + ("fits the 126 MB L2: the tick is latency-bound, the HBM roofline is not the binding one"
                                                               if ws_mb < 100 else "exceeds the 126 MB L2"))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg4")
    ap.add_argument("--envs-per-gpu", type=int, default=1 << 20)
    ap.add_argument("--precision", default="fp32", choices=["fp32", "fp64"])
    ap.add_argument("--e2e-steps", type=int, default=30)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--ref-python-seconds", type=float, default=10.0, help="Python-reference SubprocVecEnv sample (0 = skip)")
    ap.add_argument("--ref-envs", type=int, default=0, help="--impl reference: envs per step (0 = the workload's --envs-per-gpu)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cfg5-cpu-seconds", type=float, default=8.0, help="CPU counterpart of the rollout collection (0 = skip)")
    ap.add_argument("--no-configs", action="store_true", help="skip the cfg2@4096 / cfg3@262144 block")
    ap.add_argument("--strong-total", type=int, default=1 << 20, help="total envs of the strong-scaling block (0 = skip)")
    ap.add_argument("--fused", type=int, default=64, help="k of the extra fused-rollout measurement (0 = skip)")
    ap.add_argument("--rollout-steps", type=int, default=24, help="n_steps of the extra on-device PPO rollout-collection measurement (0 = skip)")
    ap.add_argument("--rollout-envs", type=int, default=131072)
    ap.add_argument("--post-steps", type=int, default=200, help="steps of the extra step + frame-stack/normalise measurement (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the headline's last timed step (rank 0) as DIR/<name>.npy, to compare two builds")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; --impl reference has none to write")
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference_arm(args)
        return

    ctx = Ctx()
    torch, dist = ctx.torch, ctx.dist
    from hlynr_intercept_b200 import config, dist as hdist
    from hlynr_intercept_b200.sim import HlynrSim
    from hlynr_intercept_b200.vec_env import HlynrVecEnv

    world, rank, local_rank, dev = ctx.world, ctx.rank, ctx.local_rank, ctx.dev
    barrier = ctx.barrier
    n = args.envs_per_gpu
    K, W = args.steps, max(args.warmup, 3)
    env_cfg = config.baseline_config(args.workload)
    peak, peak_src = measured_peak()

    # ---- headline: weak scaling, n envs per GPU, steady state ---------------------------------------------------------------
    sim, pool = make_aged_sim(ctx, args.workload, n, rank * n, args.precision)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    head = timed_ticks(ctx, sim, pool, K, W)
    if args.dump_outputs and rank == 0:   # before any further step overwrites the output buffers
        dump_outputs(args.dump_outputs, head["last_outputs"], rank * n)
    total_ms = head["ms_max"]
    clock_windows, clock_note = [head["window"]], None
    if rank == 0 and sampler.proc and sampler.count_between(*head["window"]) < 3:
        # a timed region shorter than a few 20 ms sampler periods: sample over an UNTIMED repeat of the same launches as well
        t_probe0 = time.perf_counter()
        while time.perf_counter() - t_probe0 < 0.4:
            for k in range(50):
                sim.step(pool[k % 4], want_terminal_obs=False)
            torch.cuda.synchronize()
        clock_windows.append((t_probe0, time.perf_counter()))
        clock_note = "timed region shorter than the sampler period: sampled over an untimed repeat of the same launches as well"
    clocks = sampler.stop(clock_windows) if rank == 0 else None
    if clocks is not None and clock_note:
        clocks["note"] = clock_note
    value = world * n * K / (total_ms * 1e-3)
    stats_host = head["stats"]   # all-reduced over the ranks

    # extra: fused k-step rollout with the in-kernel random policy (state in registers between ticks)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fused = None
    if args.fused > 0:
        sim.rollout(args.fused, None, want_obs=False)
        barrier()
        e0.record()
        reps = 3
        for _ in range(reps):
            sim.rollout(args.fused, None, want_obs=False)
        e1.record()
        barrier()
        tf = ctx.max_over_ranks(e0.elapsed_time(e1))
        fused = {"k": args.fused, "value": world * n * args.fused * reps / (tf * 1e-3), "unit": "env-steps/s",
                 "note": "hlynr_rollout: k ticks per launch, in-kernel Philox random policy, obs written once"}

    # extra: step + on-device VecFrameStack(4) + VecNormalize (SURVEY 8f rank 1), the tensor a policy on the same GPU consumes
    post = None
    if args.post_steps > 0:
        from hlynr_intercept_b200.post import HlynrObsPipeline

        pipe = HlynrObsPipeline(sim, n_stack=4, training=True)
        pipe.reset()
        for k in range(5):
            pipe.step(pool[k % 4])
        barrier()
        e0.record()
        for k in range(args.post_steps):
            pipe.step(pool[k % 4])
        e1.record()
        barrier()
        ms_post = ctx.max_over_ranks(e0.elapsed_time(e1)) / args.post_steps
        post = {"value": world * n / (ms_post * 1e-3), "unit": "env-steps/s", "ms_per_step": ms_post, "n_stack": 4,
                "note": "hlynr_step writing into the frame ring + hlynr_post_step (stacked, normalised [N,104] output, running "
                        "mean/var updated every step, stacked terminal observations); SB3 parity of this pipeline is UNPINNED "
                        "(stable_baselines3 is not importable here; checked against a numpy restatement only)",
                "algorithmic_bytes_per_env_step_post": 104 + 416 + 416 + 25}
        pipe.close()
    sim.close()
    del pool

    # ---- strong scaling: BASELINE cfg4's 2^20 envs IN TOTAL, sharded by global id --------------------------------------------
    strong = None
    if args.strong_total > 0:
        first, count = hdist.shard_range(args.strong_total, rank, world)
        if world == 1 and count == n:
            strong = {"total_envs": args.strong_total, "envs_per_gpu": count, "value": value, "us_per_launch": total_ms / K * 1e3,
                      "note": "one GPU: identical to the headline measurement"}
        else:
            # a rollout of at least 600 ticks: at 131072 envs per GPU a tick is ~19 us, so the rollout's one NCCL all-reduce and the
            # graph upload would be a tenth of a 20-tick timed region and say nothing about the ticks
            Ks, Ws = max(K, 600), max(W, 50)
            ssim, spool = make_aged_sim(ctx, args.workload, count, first, args.precision)
            se = timed_ticks(ctx, ssim, spool, Ks, Ws)
            sg = timed_ticks(ctx, ssim, spool, Ks, Ws, graph=True)
            ssim.close()
            best = min(se["ms_max"], sg["ms_max"])
            strong = {"total_envs": args.strong_total, "envs_per_gpu": count, "value": args.strong_total * Ks / (best * 1e-3),
                      "unit": "env-steps/s", "steps": Ks, "warmup": Ws,
                      "us_per_launch_eager": se["ms_max"] / Ks * 1e3, "us_per_launch_graph": sg["ms_max"] / Ks * 1e3,
                      "host_issue_us_per_launch_eager": se["host_issue_ms"] / Ks * 1e3, "graph_ticks_per_replay": sg["graph_ticks"],
                      "done_episodes_per_step": se["stats"][0] / Ks,
                      "note": "2^20 envs in total through dist.shard_range, max over ranks, the rollout's stats all-reduce inside the "
                              "timed region; eager = one hlynr_step call per tick from Python, graph = ring-period ticks per CUDA-graph replay"}
            del spool

    # ---- BASELINE cfg2 at 4096 envs and cfg3 at 262144 envs (rank 0's GPU, no collective) --------------------------------------
    configs = None
    if not args.no_configs and rank == 0:
        kc = max(K, 600)
        configs = {"cfg2@4096": config_line(ctx, "cfg2", 4096, kc, W, args.precision, peak),
                   "cfg3@262144": config_line(ctx, "cfg3", 262144, max(K, 200), W, args.precision, peak)}
    barrier()

    # extra: PPO rollout collection fully on the device (SURVEY 8f rank 4 / BASELINE config 5)
    roll = None
    if args.rollout_steps > 0:
        roll = rollout_leg(ctx, args, env_cfg)

    # ---- e2e: the numpy VecEnv API a Stable-Baselines3 user calls (host buffers, H2D + D2H inside the timed region) ------------
    e2e = e2e_leg(ctx, args, env_cfg, n)

    if rank == 0:
        bytes_per_step = ALGO_BYTES.get(args.workload, 630) if args.precision == "fp32" else layout_bytes(args.workload, "fp64")
        lb = layout_bytes(args.workload, args.precision)
        per_launch_ms = head["ms"] / K  # rank-0 kernel time per launch, CUDA events on the launching stream
        achieved = n * bytes_per_step / (per_launch_ms * 1e-3) / 1e9
        traffic = measured_traffic(args.workload, n) if args.precision == "fp32" else None
        episodes = stats_host[0]
        line = {
            "metric": "env-steps/s", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if args.precision == "fp32" else "f64", "data": "synthetic",
            "config": {"workload": workload_name(args.workload), "envs_per_gpu": n, "total_envs": n * world,
                       "mode": "API: one hlynr_step launch per tick, actions U(-1,1)^6 float32 resident in HBM",
                       "state": f"steady state: episodes desynchronised by {AGE_TICKS} fused random-policy ticks before the warm-up",
                       "parallelism": f"env-sharded x{world}, no per-step communication, 1 NCCL stats all-reduce per rollout (inside the timed region)",
                       "l2": "per-tick working set (~0.6 GB state + I/O) exceeds the 126 MB L2, no flush needed",
                       "seed": 1234},
            "clocks": clocks,
            "e2e": e2e,
            "gpu_launches": int(head["launches"]),
            "done_episodes_per_step": episodes / K,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src, "kernel": "hlynr::step_kernel<float,false,F>",
                         "algorithmic_bytes_per_env_step": bytes_per_step, "units_per_launch": n,
                         "kernel_us_per_launch": per_launch_ms * 1e3,
                         "layout_bytes_per_env_step": lb, "frac_layout": n * lb / (per_launch_ms * 1e-3) / 1e9 / peak,
                         "frac_traffic": (traffic / (per_launch_ms * 1e-3) / 1e9 / peak) if traffic else None,
                         "note": "achieved/frac use SURVEY 8(d)'s contract bytes (630 B counts 40 state words and whole ring slots; the compact "
                                 "layout moves 550 B, so the contract fraction can exceed 1 -- frac_layout / frac_traffic are the ones to judge "
                                 "the kernel by); frac_layout uses the bytes the kernel's own SoA layout "
                                 "moves (DESIGN.md section 2); frac_traffic uses the ncu-measured DRAM bytes of profiles/traffic.json"},
            "strong": strong,
            "configs": configs,
            "fused_rollout": fused,
            "obs_pipeline": post,
            "rollout_collection": roll,
            "episode_stats": dict(zip(["episodes", "successes", "return_sum", "length_sum"], stats_host[:4])),
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args.workload, seconds=args.cpu_seconds, ref_seconds=args.ref_python_seconds)
        else:
            line["cpu_baseline"] = None
        if not args.no_cpu_baseline and args.rollout_steps > 0 and args.cfg5_cpu_seconds > 0:
            # BASELINE cfg5's CPU side: the same collection loop on the host cores (reference env + torch policy on the CPU), bounded
            try:
                from baseline import ref_collector

                c5 = ref_collector.collect(env_cfg, seconds=args.cfg5_cpu_seconds)
            except Exception as e:
                c5 = {"unavailable": f"{type(e).__name__}: {e}"}
            if line["cpu_baseline"] is None:
                line["cpu_baseline"] = {"value": None, "unit": "env-steps/s", "cores": os.cpu_count(), "kind": "reference",
                                        "sample": "N > 1: only the cfg5 CPU collector is timed (rank 0)"}
            line["cpu_baseline"]["cfg5_collector"] = c5
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def e2e_leg(ctx, args, env_cfg, n):
    from hlynr_intercept_b200.vec_env import HlynrVecEnv

    torch, world, rank = ctx.torch, ctx.world, ctx.rank
    out = None
    for obs_dim in (26, 17):
        venv = HlynrVecEnv(env_cfg, n_envs=n, device=ctx.local_rank, seed=99, env_id_offset=rank * n, precision=args.precision,
                           warn_dead=False, lazy_infos=True, obs_dim=obs_dim)
        venv.reset()
        venv.sim.rollout(AGE_TICKS, None, want_obs=False)  # age the episodes: the timed steps see the stationary done rate
        rng = np.random.default_rng(rank)
        host_actions = [rng.uniform(-1, 1, (n, 6)).astype(np.float32) for _ in range(2)]  # ordinary (unpinned) numpy arrays
        for k in range(3):
            venv.step(host_actions[k % 2])
        ctx.barrier()
        n_done = 0
        t0 = time.perf_counter()
        for k in range(args.e2e_steps):
            _, rew_h, _, infos_h = venv.step(host_actions[k % 2])
            n_done += len(infos_h.records)  # finished episodes (terminal observation + info) arrive as compact records
        torch.cuda.synchronize()
        sec = ctx.max_over_ranks(time.perf_counter() - t0)
        venv.close()
        blk = {"value": world * n * args.e2e_steps / sec, "unit": "env-steps/s", "obs_dim": obs_dim,
               "h2d_bytes_per_step": n * 6 * 4, "d2h_bytes_per_step": n * (obs_dim * 4 + 4 + 1 + 1 + 1) + 4 + 200 * min(n, 4096),
               "steps": args.e2e_steps, "done_episodes_per_step": n_done / max(args.e2e_steps, 1), "ms_per_step": sec / args.e2e_steps * 1e3}
        if obs_dim == 26:
            out = blk
            out["api"] = ("HlynrVecEnv.step(ordinary numpy actions) -> numpy obs, rewards, dones, infos (hlynr_step_host: chunks pipelined "
                          "over 3 streams; actions staged with streaming stores; obs by copy engine into alternating page-locked sets; "
                          "reward/terminated/truncated/dones written by the kernel straight into host memory; done episodes as compact records)")
        else:
            out["obs17"] = blk
            out["obs17"]["note"] = "HlynrVecEnv(obs_dim=17): the 17-D radar layout obs[0:17] of the 26-D vector, 36 B per env less to download"
    return out


def rollout_leg(ctx, args, env_cfg):
    """PPO rollout collection fully on the device: policy forward, env step, frame-stack/normalise, TimeLimit bootstrap, GAE;
    no host synchronisation inside collect().  The policy is the reference's network (train_flat_ppo.py:37-85 CustomMLP
    104 -> 512 -> 512 -> 256 + LayerNorm + ReLU, action_net / value_net / log_std): once as the fused sm_100a kernel
    (include/hlynr_policy.h: tcgen05 GEMMs, LayerNorm epilogues, heads and sampling in one launch) and once as the torch module
    on cuBLAS TF32."""
    from hlynr_intercept_b200.policy import FusedActorCritic, ReferenceActorCritic
    from hlynr_intercept_b200.post import HlynrObsPipeline
    from hlynr_intercept_b200.rollout import DeviceRolloutCollector
    from hlynr_intercept_b200.sim import HlynrSim

    torch, world, rank, dev = ctx.torch, ctx.world, ctx.rank, ctx.dev
    barrier = ctx.barrier
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_roll = min(args.envs_per_gpu, args.rollout_envs)
    T = args.rollout_steps
    rsim = HlynrSim(env_cfg, n_envs=n_roll, device=ctx.local_rank, seed=4321, env_id_offset=rank * n_roll, precision=args.precision,
                    warn_dead=False)
    rpipe = HlynrObsPipeline(rsim, n_stack=4, training=True)
    torch.manual_seed(rank)
    torch.backends.cuda.matmul.allow_tf32 = True   # the torch comparison runs its GEMMs on TF32 tensor cores, as PPO users do
    torch.backends.cudnn.allow_tf32 = True
    net = ReferenceActorCritic(device=dev)
    fused = FusedActorCritic(net, device=ctx.local_rank, seed=rank)

    def timed_collect(col, graph):
        col.collect()
        barrier()
        e0.record()
        col.collect()
        e1.record()
        barrier()
        eager = ctx.max_over_ranks(e0.elapsed_time(e1))
        if not graph:
            return eager, eager
        col.capture()   # the whole collect() as ONE CUDA-graph launch (launch-bound otherwise: ~25 kernels per step)
        col.replay()
        barrier()
        e0.record()
        col.replay()
        e1.record()
        barrier()
        return eager, ctx.max_over_ranks(e0.elapsed_time(e1))

    col = DeviceRolloutCollector(rpipe, fused, T)
    graphed = T % col.graph_period() == 0
    te_, tr_ = timed_collect(col, graphed)
    # the forward alone (policy step of one tick) at this batch size
    o = col.obs[0]
    fused(o); barrier(); e0.record()
    for _ in range(10):
        fused(o)
    e1.record(); barrier()
    fwd_us = e0.elapsed_time(e1) / 10 * 1e3
    flop = 2 * (104 * 512 + 512 * 512 + 512 * 256 + 256 * 7) * n_roll
    colt = DeviceRolloutCollector(rpipe, net, T)
    colt._started = True
    colt.obs[colt.T].copy_(col.obs[col.T])
    tte_, ttr_ = timed_collect(colt, graphed)

    class _NoPolicy(torch.nn.Module):   # the same loop without the policy network (random actions): what the simulator side costs
        def __init__(self):
            super().__init__()
            self.dummy = torch.nn.Parameter(torch.zeros(1, device=dev))

        def value(self, obs):
            return obs[:, 0].contiguous()

        def forward(self, obs):
            a = torch.rand(obs.shape[0], 6, device=obs.device) * 2 - 1
            return a, obs[:, 0], obs[:, 1]

    col2 = DeviceRolloutCollector(rpipe, _NoPolicy(), T, bootstrap_rows=max(256, n_roll // 32))
    col2._started = True
    col2.obs[col2.T].copy_(col.obs[col.T])
    tn_, _ = timed_collect(col2, False)
    rate = lambda ms: world * n_roll * T / (ms * 1e-3)  # noqa: E731
    # BASELINE configuration 5: >= 5 M env-steps of PPO rollout collection end to end (wall clock around the collect() calls of all
    # ranks, host-side launch work and the final synchronisation included), fused policy, graph replay when n_steps allows it
    reps = max(1, -(-5_000_000 // (world * n_roll * T)))
    barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        col.replay() if graphed else col.collect()
    torch.cuda.synchronize()
    cfg5_s = ctx.max_over_ranks(time.perf_counter() - t0)
    cfg5 = {"env_steps": world * n_roll * T * reps, "seconds": cfg5_s, "value": world * n_roll * T * reps / cfg5_s, "unit": "env-steps/s",
            "collects": reps, "n_steps": T, "envs_per_gpu": n_roll, "n_gpus": world,
            "note": "BASELINE cfg5: end-to-end PPO rollout collection (policy forward, env step, frame stack + normalisation, TimeLimit "
                    "bootstrap, GAE), >= 5 M env-steps, wall clock; the CPU counterpart of the same loop is cpu_baseline.cfg5_collector"}
    roll = {"value": rate(tr_), "unit": "env-steps/s", "envs_per_gpu": n_roll, "n_steps": T,
            "policy": "reference network 104->512->512->256 (LayerNorm, ReLU) + action_net/value_net, fused sm_100a forward "
                      "(hlynr_policy_forward: tcgen05 bf16 GEMMs, fp32 TMEM accumulators, TMA weight ring, LayerNorm/ReLU epilogues, "
                      "heads + Gaussian sampling in ONE kernel)",
            "cuda_graph": bool(graphed), "eager": rate(te_), "us_per_step": tr_ / T * 1e3,
            "policy_forward_us": fwd_us, "policy_forward_tflops": flop / (fwd_us * 1e-6) / 1e12,
            "policy_roofline": policy_roofline(flop, fwd_us),
            "with_torch_policy_tf32": rate(ttr_), "with_torch_policy_tf32_eager": rate(tte_),
            "without_policy_network": rate(tn_),
            "timeout_bootstrap_overflow": int(col.overflow.item()),
            "cfg5": cfg5,
            "note": "DeviceRolloutCollector.collect(): policy forward + hlynr_step + hlynr_post_step + value net on the finished "
                    "episodes (device-side row count) + hlynr_bootstrap_timeouts per step, hlynr_gae at the end; buffers [T,N,*] "
                    "resident in HBM; SB3 parity of the GAE / bootstrap restatement is UNPINNED (stable_baselines3 not importable here)"}
    fused.close()
    rpipe.close()
    rsim.close()
    return roll


if __name__ == "__main__":
    main()

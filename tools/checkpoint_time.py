"""Cost of checkpoints (DESIGN.md section 17): device time of the snapshot pack and unpack (CUDA events around
hlynr_snapshot_save / _load and hlynr_post_snapshot_save / _load, median of REPS) and wall time of the file round trip
(checkpoint.save + checkpoint.load, state_dict copies through pinned memory included), with the image bytes per env, for
  - cfg4 at 2^20 envs (the simulator alone), and
  - the 131 072-env DeviceRolloutCollector with frame_stack 4 (sim + observation pipeline + collector + fused policy counter).
Prints one JSON document with the card's name and power limit, and writes it to the file `--out` names, if given."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from hlynr_intercept_b200 import _lib, abi, checkpoint, config  # noqa: E402
from hlynr_intercept_b200.policy import FusedActorCritic, ReferenceActorCritic  # noqa: E402
from hlynr_intercept_b200.post import HlynrObsPipeline  # noqa: E402
from hlynr_intercept_b200.rollout import DeviceRolloutCollector  # noqa: E402
from hlynr_intercept_b200.sim import HlynrSim  # noqa: E402

REPS = 10


def _events(fn):
    """Median device time (ms) of fn() between two events on the current stream."""
    times = []
    for _ in range(REPS + 1):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times[1:]))


def _pack_unpack(h, L, prefix, info_cls):
    info, nb = info_cls(), C.c_size_t()
    getattr(L, prefix + "_layout")(h, C.byref(info), C.byref(nb))
    buf = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    ptr = C.c_void_p(buf.data_ptr())
    pack = _events(lambda: _lib.check(getattr(L, prefix + "_save")(h, ptr, C.byref(info), st)))
    unpack = _events(lambda: _lib.check(getattr(L, prefix + "_load")(h, C.byref(info), ptr, st)))
    return nb.value, pack, unpack


def _round_trip(parts, reps=3):
    times_save, times_load = [], []
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "ckpt.npz")
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            checkpoint.save(path, **parts)
            t1 = time.perf_counter()
            checkpoint.load(path, **parts)
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            times_save.append(t1 - t0)
            times_load.append(t2 - t1)
        size = os.path.getsize(path)
    return dict(file_bytes=size, save_s=float(np.median(times_save)), load_s=float(np.median(times_load)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON document to this file")
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    out = {"gpu": gpu.strip().splitlines()[0] if gpu.strip() else "unknown", "reps": REPS}
    # cfg4 at 2^20 envs, after a reset and 50 ticks of random actions
    n = 1 << 20
    sim = HlynrSim(config.baseline_config("cfg4"), n_envs=n, seed=1, warn_dead=False)
    sim.reset()
    g = torch.Generator(device="cuda")
    g.manual_seed(0)
    for _ in range(50):
        sim.step(torch.rand(n, 6, device="cuda", generator=g) * 2 - 1)
    nb, pack, unpack = _pack_unpack(sim.h, sim.L, "hlynr_snapshot", abi.HlynrSnapshotInfo)
    out["cfg4_2^20"] = dict(n_envs=n, image_bytes=nb, bytes_per_env=nb / n, pack_ms=pack, unpack_ms=unpack,
                            file=_round_trip(dict(sim=sim)))
    sim.close()
    del sim
    torch.cuda.empty_cache()
    # the 131 072-env collector, frame_stack 4, 104-wide fused policy, after one graph-replayed rollout
    n = 1 << 17
    sim = HlynrSim(config.baseline_config("cfg4"), n_envs=n, seed=2, warn_dead=False)
    pipe = HlynrObsPipeline(sim, n_stack=4, training=True)
    torch.manual_seed(0)
    fused = FusedActorCritic(ReferenceActorCritic(obs_dim=104), device=0, seed=3)
    col = DeviceRolloutCollector(pipe, fused, DeviceRolloutCollector(pipe, None, 1).graph_period() * 2)
    col.capture()
    col.replay()
    torch.cuda.synchronize()
    snb, spack, sunpack = _pack_unpack(sim.h, sim.L, "hlynr_snapshot", abi.HlynrSnapshotInfo)
    pnb, ppack, punpack = _pack_unpack(pipe.h, sim.L, "hlynr_post_snapshot", abi.HlynrPostSnapshotInfo)
    out["collector_131072_stack4"] = dict(
        n_envs=n, sim=dict(image_bytes=snb, bytes_per_env=snb / n, pack_ms=spack, unpack_ms=sunpack),
        pipe=dict(image_bytes=pnb, bytes_per_env=pnb / n, pack_ms=ppack, unpack_ms=punpack),
        file=_round_trip(dict(sim=sim, pipe=pipe, collector=col, policy=fused)))
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s)


if __name__ == "__main__":
    main()

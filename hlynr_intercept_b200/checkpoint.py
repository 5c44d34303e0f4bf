"""Checkpoint and resume a device training run bit for bit (DESIGN.md section 17).

    checkpoint.save("run/ckpt.npz", sim=sim, pipe=pipe, collector=collector, policy=fused)
    ...  # a new process: the same constructors, then
    checkpoint.load("run/ckpt.npz", sim=sim, pipe=pipe, collector=collector, policy=fused)

One uncompressed `.npz` holds a JSON descriptor (every part's non-array state, each array's dtype, shape and CRC32), the arrays
(the snapshot images of the sim and the observation pipeline, the collector's next observation row, ...) and the descriptor's
own CRC32.  `load` reads and checks the whole file before it changes anything, and refuses a file with a wrong format version,
a failed checksum, a missing part or a truncated or otherwise unreadable archive.  The policy's weights and the optimiser are
torch's own state_dict; `policy=` saves the fused policy's noise counter only.
"""
import json
import zipfile
import zlib

import numpy as np

FORMAT_VERSION = 1
PARTS = ("sim", "pipe", "collector", "policy")


class CheckpointError(ValueError):
    pass


def _crc(a):
    return zlib.crc32(np.ascontiguousarray(a).view(np.uint8).reshape(-1)) & 0xFFFFFFFF


def save(path, sim=None, pipe=None, collector=None, policy=None):
    """Writes the state_dict() of every given object to `path` (an .npz; numpy appends the suffix if it is missing)."""
    objs = dict(sim=sim, pipe=pipe, collector=collector, policy=policy)
    desc = {"format_version": FORMAT_VERSION, "parts": {}, "arrays": {}}
    arrays = {}
    for part in PARTS:
        if objs[part] is None:
            continue
        state = {}
        for key, value in objs[part].state_dict().items():
            if hasattr(value, "cpu"):   # a tensor
                value = value.cpu().numpy()
            if isinstance(value, np.ndarray):
                name = f"{part}.{key}"
                arrays[name] = np.ascontiguousarray(value)
                desc["arrays"][name] = {"dtype": value.dtype.str, "shape": list(value.shape), "crc32": _crc(value)}
                state[key] = {"array": name}
            else:
                state[key] = value
        desc["parts"][part] = state
    blob = np.frombuffer(json.dumps(desc).encode(), dtype=np.uint8)
    np.savez(path, descriptor=blob, descriptor_crc32=np.array([_crc(blob)], dtype=np.uint32), **arrays)


def read(path):
    """{part: state dict} of a checkpoint, every checksum verified (CheckpointError otherwise)."""
    try:
        with np.load(path, allow_pickle=False) as z:
            files = {k: z[k] for k in z.files}
    except (OSError, ValueError, EOFError, zipfile.BadZipFile, zlib.error) as e:
        raise CheckpointError(f"{path}: not a readable checkpoint ({type(e).__name__}: {e})") from e
    if "descriptor" not in files or "descriptor_crc32" not in files:
        raise CheckpointError(f"{path}: no checkpoint descriptor")
    blob = files["descriptor"]
    if blob.dtype != np.uint8 or files["descriptor_crc32"].shape != (1,) or _crc(blob) != int(files["descriptor_crc32"][0]):
        raise CheckpointError(f"{path}: the descriptor fails its checksum")
    desc = json.loads(blob.tobytes().decode())
    if desc.get("format_version") != FORMAT_VERSION:
        raise CheckpointError(f"{path}: checkpoint format version {desc.get('format_version')}, this build reads {FORMAT_VERSION}")
    for name, meta in desc["arrays"].items():
        a = files.get(name)
        if a is None or a.dtype.str != meta["dtype"] or list(a.shape) != meta["shape"] or _crc(a) != meta["crc32"]:
            raise CheckpointError(f"{path}: section {name!r} is missing or fails its checksum")
    return {part: {k: files[v["array"]] if isinstance(v, dict) and set(v) == {"array"} else v for k, v in state.items()}
            for part, state in desc["parts"].items()}


def load(path, sim=None, pipe=None, collector=None, policy=None):
    """Restores every given object from `path`, after the whole file has been checked.  The objects must have been built as the
    saved ones were (the same configuration, precision, n_envs, env_id_offset, observation width, frame_stack; refused otherwise).
    Returns the parts the file holds.  Captured graphs (DeviceRolloutCollector.capture, StepGraph) must be captured again."""
    parts = read(path)
    objs = dict(sim=sim, pipe=pipe, collector=collector, policy=policy)
    missing = [p for p in PARTS if objs[p] is not None and p not in parts]
    if missing:
        raise CheckpointError(f"{path}: holds no state for {missing}")
    for part in PARTS:   # the sim first: the pipeline and the collector continue from its state
        if objs[part] is not None:
            objs[part].load_state_dict(parts[part])
    return sorted(parts)

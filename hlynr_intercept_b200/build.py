"""Builds the C-ABI CUDA library in-tree for sm_100a:  hlynr_intercept_b200/libhlynr_b200.so"""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "libhlynr_b200.so")
SOURCES = [os.path.join(HERE, "csrc", "hlynr_capi.cu"), os.path.join(HERE, "csrc", "hlynr_post.cu"),
           os.path.join(HERE, "csrc", "hlynr_rollout.cu"), os.path.join(HERE, "csrc", "hlynr_policy.cu")]
DEPS = SOURCES + [os.path.join(HERE, "csrc", "hlynr_device.cuh"), os.path.join(HERE, "csrc", "hlynr_host.cuh"),
                  os.path.join(os.path.dirname(HERE), "include", "hlynr.h"),
                  os.path.join(os.path.dirname(HERE), "include", "hlynr_post.h"),
                  os.path.join(os.path.dirname(HERE), "include", "hlynr_rollout.h"),
                  os.path.join(os.path.dirname(HERE), "include", "hlynr_policy.h"),
                  os.path.join(os.path.dirname(HERE), "include", "hlynr_rng.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "--shared",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v", "--expt-relaxed-constexpr"]


def needs_build():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    return any(os.path.getmtime(d) > t for d in DEPS)


def build(force=False, verbose=False, report=False):
    """report=True (`python -m hlynr_intercept_b200.build --report`) rewrites csrc/ptxas_report.txt: registers / spills / smem
    per kernel, kept in git.  Off by default: nvcc's output depends on where the checkout sits (anonymous-namespace kernel names
    carry a hash of the source path), so an ordinary build that wrote it would modify a committed file."""
    if not force and not needs_build():
        return SO
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    cmd = [nvcc] + NVCC_FLAGS + ["-o", SO] + SOURCES
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout)
    if report:   # source paths relative to the checkout
        out = res.stdout.replace(os.path.dirname(HERE) + os.sep, "")
        with open(os.path.join(HERE, "csrc", "ptxas_report.txt"), "w") as f:
            f.write("".join(l for l in out.splitlines(True) if "Compile time" not in l))
    if verbose:
        print(res.stdout)
    return SO


if __name__ == "__main__":
    import sys

    build(force=True, verbose=True, report="--report" in sys.argv[1:])

"""Compile the native library in-tree: nvcc, sm_100a only, -fmad=false (bit-exact f64 bookkeeping).

    python -m gym_td_b200.build [--force] [--verbose]
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libtd_b200.so")
SOURCES = ["td_engine.cu", "td_mapgen.cpp"]
DEPS = SOURCES + ["td_kernels.cuh", "td_common.cuh", "td_rng.cuh", "td_rules.cuh", "td_obs.cuh", "td_rollout.cuh",
                  os.path.join("..", "..", "include", "td_b200.h")]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-fmad=false", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC,-pthread"]


def nvcc_path():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def up_to_date():
    if not os.path.exists(OUT):
        return False
    t = os.path.getmtime(OUT)
    return all(os.path.getmtime(os.path.join(CSRC, d)) <= t for d in DEPS)


def build(force=False, verbose=False):
    if not force and up_to_date():
        return OUT
    extra = os.environ.get("TD_NVCC_EXTRA", "").split()      # extra nvcc flags, e.g. -DTD_DEBUG_BOUNDS
    out = os.environ.get("TD_BUILD_OUT", OUT)                # experiments: a variant library next to the default
    cmd = [nvcc_path()] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", out] + \
          [os.path.join(CSRC, s) for s in SOURCES]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed (%d): %s" % (res.returncode, " ".join(cmd)))
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))

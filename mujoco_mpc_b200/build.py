"""Build the CUDA engine in-tree: nvcc -> mujoco_mpc_b200/csrc/libmjpc_b200.so (sm_100a only)."""
from __future__ import annotations

import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.environ.get("MJPC_B200_SO") or os.path.join(CSRC, "libmjpc_b200.so")  # override: perf experiments only
# -use_fast_math (approximate division / sqrt / sincos, flush-to-zero): the parity ablation with and without it is
# profiles/parity_ablation.py -> profiles/r02_fast_math_ablation.txt; MJPC_B200_NO_FAST_MATH=1 builds the IEEE variant
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17"] + \
             ([] if os.environ.get("MJPC_B200_NO_FAST_MATH") == "1" else ["-use_fast_math"]) + \
             os.environ.get("MJPC_B200_NVCC_EXTRA", "").split() + ["-Xcompiler", "-fPIC", "-shared"]


def sources():
    host = os.path.join(CSRC, "host")
    return [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh", ".h"))] + \
        [os.path.join(host, f) for f in sorted(os.listdir(host)) if f.endswith((".cc", ".h"))] + \
        [os.path.join(HERE, "..", "include", "mjpc_b200.h")]


def needs_build():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    return any(os.path.getmtime(s) > t for s in sources())


def _compile(verbose):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", SO, os.path.join(CSRC, "engine.cu"), os.path.join(CSRC, "host", "sampling_planner.cc"),
                                                                           os.path.join(CSRC, "host", "batch_sampling_planner.cc"),
                                                                           os.path.join(CSRC, "host", "cross_entropy_planner.cc"),
                                                                           os.path.join(CSRC, "host", "ilqg_planner.cc"),
                                                                           os.path.join(CSRC, "host", "robust_planner.cc"),
                                                                           os.path.join(CSRC, "host", "gradient_planner.cc"),
                                                                           os.path.join(CSRC, "host", "agent.cc"),
                                                                           os.path.join(CSRC, "host", "task_transition.cc")]
    subprocess.check_call(cmd, cwd=CSRC)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return SO
    _compile(verbose)
    # the static kernel tables (csrc/spec_*.h) are a function of the model compiler + the header/layout structs:
    # regenerate them from the library just built and compile once more if one changed
    from . import gen_spec
    if gen_spec.generate(SO):
        _compile(verbose)
    return SO


if __name__ == "__main__":
    print(build(force=True, verbose=True))

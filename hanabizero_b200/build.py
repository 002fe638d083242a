"""Builds hanabizero_b200/csrc/libhzb200.so (the C-ABI library of include/hzb200.h) with nvcc for
sm_100a.  In-tree on purpose: the built .so travels with the repo snapshot to the GPU box.

    python -m hanabizero_b200.build [--force]
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libhzb200.so")
SOURCES = ["hz_tree.cu", "hz_env.cu", "hz_nn.cu", "hz_gemm.cu", "hz_rowchain.cu", "hz_selfplay.cu", "hz_traj.cu", "hz_noise.cu", "hz_wave.cu", "hz_obs.cu", "hz_host.cpp"]
HEADERS = ["hz_common.cuh", "hz_math.cuh", "hz_decode.cuh", "hz_detmath.cuh", "../../include/hzb200.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    # bit-exact float semantics: no FMA contraction, IEEE div/sqrt, no flush-to-zero
    "-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-ffp-contract=off", "-Xcompiler", "-fvisibility=hidden",
    "-shared", "-cudart", "static",
    "-lcublasLt", "-Xlinker", "-rpath=/usr/local/cuda/lib64",
]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False, trace=False):
    """trace=True builds csrc/libhzb200_trace.so with -DHZ_TRACE (per-warp cycle stamps in the fused tree step,
    read by scripts/exp_trace.py); a debug artefact, never loaded by the product."""
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    if trace:
        out = LIB.replace(".so", "_trace.so")
    elif not force and not _stale():
        return LIB
    else:
        out = LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-DHZ_TRACE"] if trace else []) + (["-Xptxas", "-v"] if verbose else []) + ["-o", out] + srcs
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stderr)
    return out


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv, trace="--trace" in sys.argv))

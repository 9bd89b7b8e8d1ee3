"""Build libpyascore_b200.so in-tree for sm_100a (nvcc cross-compiles without a GPU).

    python pyascore_b200/csrc/build.py [--force]

-fmad=false: the reference is x86-64 -O2 code with no FMA contraction (SURVEY.md section 7.3); every
float/double operation must round separately.  Explicit fma() calls (glibc expf/logf restatement)
stay fused.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(os.path.dirname(HERE), "libpyascore_b200.so")
SRCS = ["pa_lib.cu", "pa_host.cpp", "pa_decode.cu", "pa_mzml.cpp"]
DEPS = sorted(f for f in os.listdir(HERE) if f.endswith((".cu", ".cuh", ".cpp"))) + ["../../include/pyascore_b200.h"]


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(os.path.join(HERE, d)) > t for d in DEPS)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
           "-fmad=false", "-Xcompiler", "-fPIC,-pthread", "-shared", "-o", OUT] + [os.path.join(HERE, s) for s in SRCS]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))

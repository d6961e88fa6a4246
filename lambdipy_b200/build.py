"""Build liblambdipy_b200.so (sm_100a) in-tree with nvcc.  `python -m lambdipy_b200.build`."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "liblambdipy_b200.so")
SOURCES = ["plan.cu", "compact.cu", "compact_tma.cu", "corpus.cu", "deflate.cu", "api.cu"]
HEADERS = ["lb2_common.cuh", "copy_device.cuh", os.path.join("..", "..", "include", "lambdipy_b200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-Wall,-Wno-unused-function", "--shared", "-cudart", "shared",
]


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


TIMING_OUT = os.path.join(HERE, "liblambdipy_b200_timing.so")  # -DLB2_PLAN_TIMING: per-phase clock64() printf of the plan kernel


def build(force=False, verbose=False, timing=False):
    """timing=True builds the diagnostic variant next to the product library (load it with
    LAMBDIPY_B200_LIB=<path>); it is never loaded by default."""
    out = TIMING_OUT if timing else OUT
    if not timing and not force and not needs_build():
        return OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-DLB2_PLAN_TIMING"] if timing else []) + (["-Xptxas", "-v"] if verbose else []) + \
        ["-o", out] + [os.path.join(CSRC, s) for s in SOURCES]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed building liblambdipy_b200.so")
    if verbose:
        sys.stderr.write(r.stdout + r.stderr)
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, timing="--timing" in sys.argv))

"""In-tree build of libhw1f.so (the C-ABI shared library) for sm_100a.

`python build.py` or `build()` runs one nvcc command; nvcc cross-compiles without a GPU.
The .so is git-ignored but travels to the GPU box with the repo snapshot.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libhw1f.so")
SOURCES = ["hw1f_api.cu", "hw1f_multi.cu", "hw1f_comm.cu", "xorwow_jump.cpp"]
HEADERS = ["hw1f_kernels.cuh", "hw1f_device.cuh", "hw1f_probe.cuh", "hw1f_kernels_extra.cuh", "hw1f_kernels_fast.cuh", "hw1f_kernels_swaption.cuh", "hw1f_kernels_book_vega.cuh", "hw1f_tail.cuh", "hw1f_comm.cuh", "xorwow_jump.hpp", os.path.join("..", "..", "include", "hw1f.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    # numerics of the reference build (--use_fast_math) that matter here: flush-to-zero.  Every
    # other fast-math effect is spelled out with intrinsics / PTX in hw1f_device.cuh, and FMA
    # contraction is disabled so that nothing fuses behind our back.
    "-ftz=true", "-fmad=false",
    "-Xcompiler", "-fPIC", "-shared",
    "-I/usr/include",          # nccl.h (types only; NCCL itself is dlopen'ed by hw1f_multi_create)
    "-ldl",
]


def nvcc_path():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the HW1F engine is CUDA-only and has no CPU fallback")


def is_stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, extra_flags=()):
    if not force and not is_stale():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    cmd = [nvcc_path()] + NVCC_FLAGS + list(extra_flags) + ["-o", LIB_PATH] + SOURCES
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
        print(" ".join(cmd), file=sys.stderr)
    res = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr, file=sys.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))

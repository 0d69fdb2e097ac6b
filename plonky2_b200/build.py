"""Build the in-tree CUDA library (sm_100a) with nvcc. No torch dependency: the product is a plain
C-ABI shared object (include/plonky2_b200.h)."""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libplonky2_b200.so")
SOURCES = ["plonky2_b200.cu"]
DEPS = ["plonky2_b200.cu", "gl_field.cuh", "gl_logup.cuh", "gl_lazy.cuh", "gl_ntt.cuh", "gl_ntt_host.cuh", "gl_poseidon.cuh", "gl_poseidon_constants.h",
        os.path.join("..", "..", "include", "plonky2_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def nvcc_path():
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found; cannot build libplonky2_b200.so")
    return p


def is_stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS)


def build(force=False, verbose=False):
    """Compile plonky2_b200/csrc/*.cu -> plonky2_b200/libplonky2_b200.so (cross-compiles without a GPU)."""
    if not force and not is_stale():
        return LIB
    cmd = [nvcc_path()] + NVCC_FLAGS + ["-o", LIB] + SOURCES
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    subprocess.check_call(cmd, cwd=CSRC)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))

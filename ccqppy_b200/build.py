"""Build the CUDA library in-tree: ccqppy_b200/csrc/libccqp_b200.so (sm_100a only).

nvcc cross-compiles without a GPU, so this also is the "does it build" check
(`__graft_entry__.build()`).  The .so is git-ignored but travels with the source tree."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libccqp_b200.so")
SOURCES = ["capi.cu", "dense_f64.cu", "batched.cu", "batched_f32.cu", "batched_sym.cu", "upload.cu", "emu.cu", "csr.cu", "dense_f32.cu"]      # see csrc/internal.h
HEADERS = ["common.cuh", "proj.cuh", "dense.cuh", "kernel_build.cuh", "batched.cuh", "microbench.cuh", "internal.h", "symcheck.h",
           os.path.join("..", "..", "include", "ccqp_b200.h")]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              # the reference computes every scalar with separately rounded * and +; fused
              # multiply-adds are written explicitly (fma()) where they are wanted
              "-fmad=false",
              "-Xcompiler", "-fPIC"]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, extra_flags=(), lib=None, defines=()):
    """Compile if the library is missing or older than its sources.  Returns the library path.
    `lib` / `defines`: build a tuning variant next to the product library (tools/sweep_*.py)."""
    from concurrent.futures import ThreadPoolExecutor
    target = lib or LIB
    if not force and lib is None and not _stale():
        return target
    nvcc = os.environ.get("NVCC", "nvcc")
    objdir = os.path.join(CSRC, "variants", os.path.splitext(os.path.basename(target))[0] + "_obj")
    os.makedirs(objdir, exist_ok=True)
    flags = NVCC_FLAGS + list(extra_flags) + ["-D" + d for d in defines]

    def compile_one(src):
        obj = os.path.join(objdir, os.path.splitext(src)[0] + ".o")
        cmd = [nvcc] + flags + ["-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        subprocess.run(cmd, check=True, cwd=CSRC)
        return obj
    with ThreadPoolExecutor(len(SOURCES)) as pool:
        objs = list(pool.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a"] + objs + ["-o", target]
    if verbose:
        print(" ".join(cmd), file=sys.stderr)
    subprocess.run(cmd, check=True, cwd=CSRC)
    return target


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))

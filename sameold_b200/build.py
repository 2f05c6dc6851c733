"""Builds the native library IN-TREE: sameold_b200/_build/libsame_b200.so (sm_100a only, no other arch, no fallback).

nvcc cross-compiles without a GPU.  Flags that matter for bit-exactness against the reference's f32 arithmetic:
-fmad=false (Rust never contracts a*b+c), -prec-div/-prec-sqrt=true, -ftz=false (subnormals are live in the squelch
power tracker, SURVEY.md §8c), host code with -ffp-contract=off.
"""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_build")
LIB = os.path.join(OUT_DIR, "libsame_b200.so")
SOURCES = ["same_kernels.cu", "same_long.cu", "same_engine.cu", "same_multi.cu", "same_synth.cu", "same_state.cu"]
HEADERS = ["same_params.h", "same_internal.h", "same_transport.cuh", "same_lane.cuh", "same_fast.cuh", os.path.join("..", "..", "include", "same_engine.h"),
           os.path.join("..", "..", "include", "same_synth.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math", "-Xptxas", "-v",
]


def _nvcc():
    for c in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found: cannot build libsame_b200.so (there is no CPU fallback)")


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS if os.path.exists(os.path.join(CSRC, f)))


def build_variant(name, defines):
    """Diagnostic: an extra in-tree build of the same ABI with -D switches (A/B timing via SAME_B200_LIB, tools/ab.sh)."""
    os.makedirs(OUT_DIR, exist_ok=True)
    out = os.path.join(OUT_DIR, name)
    srcs = [os.path.join(CSRC, f) for f in SOURCES]
    cmd = [_nvcc()] + [f for f in NVCC_FLAGS if f not in ("-Xptxas", "-v")] + ["-D" + d for d in defines] + ["-shared", "-o", out] + srcs
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + (r.stdout + r.stderr)[-4000:])
    return out


def build_native(force=False, verbose=False):
    """Compile every CUDA source for sm_100a into one shared library.  Returns the library path."""
    if not force and not needs_build():
        return LIB
    os.makedirs(OUT_DIR, exist_ok=True)
    srcs = [os.path.join(CSRC, f) for f in SOURCES if os.path.exists(os.path.join(CSRC, f))]
    cmd = [_nvcc()] + NVCC_FLAGS + ["-shared", "-o", LIB] + srcs
    r = subprocess.run(cmd, capture_output=True, text=True)
    log = r.stdout + r.stderr
    with open(os.path.join(OUT_DIR, "build.log"), "w") as f:
        f.write(" ".join(cmd) + "\n" + log)
    if verbose:
        print(log)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + log[-4000:])
    return LIB


if __name__ == "__main__":
    print(build_native(force=True, verbose=True))

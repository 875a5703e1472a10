"""Builds lib/libf1l.so (the C-ABI library, include/f1l.h) with nvcc for sm_100a, in-tree."""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
SRC_DIR = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "lib")
OUT = os.path.join(OUT_DIR, "libf1l.so")
SOURCES = ["f1l_api.cu"]
DEPS = ["f1l_api.cu", "f1l_common.cuh", "f1l_lattice.cuh", "f1l_pp.cuh", "f1l_peaks.cuh", "f1l_rollout.cuh",
        os.path.join("..", "..", "include", "f1l.h")]


def nvcc_path():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def is_stale():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(os.path.join(SRC_DIR, d)) > t for d in DEPS)


def build(force=False, verbose=False, out=None, defs=()):
    """`out` / `defs`: an A/B build of a kernel variant (-D switches) next to the product library."""
    if out is None and not force and not is_stale():
        return OUT
    os.makedirs(OUT_DIR, exist_ok=True)
    return _compile(out or OUT, verbose, defs)


def _compile(OUT, verbose, defs):
    cmd = [nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo",
           "-std=c++17", "-Xcompiler", "-fPIC", "-shared", "-diag-suppress", "177",
           "-o", OUT] + [os.path.join(SRC_DIR, s) for s in SOURCES]
    for d in list(defs) + os.environ.get("F1L_NVCC_DEFS", "").split():
        cmd.insert(1, "-D" + d)   # e.g. F1L_NVCC_DEFS="PP_UNROLL=4" for build-time experiments
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    env = dict(os.environ)
    # $CC/$CXX in this image point at a gcc that nvcc does not need; use the distro host compiler
    if os.path.exists("/usr/bin/g++"):
        cmd[1:1] = ["-ccbin", "/usr/bin/g++"]
    subprocess.run(cmd, check=True, env=env)
    return OUT


if __name__ == "__main__":
    import sys
    print(build(force=True, verbose="-v" in sys.argv))

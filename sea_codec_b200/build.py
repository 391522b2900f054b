"""Builds libsea_b200.so in-tree with nvcc for sm_100a (B200).  No torch extension machinery: the product is a plain
C-ABI shared library (include/sea_b200.h) that Python, C++ or a Rust `extern "C"` block can bind."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libsea_b200.so")
SOURCES = ["capi.cu", "capi_ext.cu", "capi_multi.cpp", "decode_kernels.cu", "decode_fast.cu", "decode_fast_mono.cu", "decode_vbr.cu", "decode_mc.cu", "decode_mc_odd.cu", "decode_latency.cu", "encode_kernels.cu", "misc_kernels.cu", "window_kernels.cu", "corpus_kernels.cu", "pool_kernels.cu", "sea_format.cpp"]
HEADERS = ["sea_common.cuh", "sea_device.cuh", "decode_chain.cuh", "decode_mc.cuh", "decode_fast.cuh", "sea_format.h", "sea_kernels.h", os.path.join("..", "..", "include", "sea_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math,-Wall,-Wno-unused-function",
    "--fmad=false",
    "-cudart", "static",
]


def nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libsea_b200.so cannot be built (there is no CPU build of this library)")


def is_stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False, extra_flags=(), lib_path: str = LIB, build_dir: str | None = None) -> str:
    """extra_flags / lib_path / build_dir: tuning builds (tools/build_variant.py) next to the product library."""
    if not force and not is_stale() and lib_path == LIB:
        return LIB
    build_dir = build_dir or os.path.join(HERE, "build")
    os.makedirs(build_dir, exist_ok=True)
    # one builder at a time (several ranks of a torchrun job may find the library stale at once); whoever waited re-checks
    import fcntl

    with open(os.path.join(build_dir, ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        if not force and not is_stale() and lib_path == LIB:
            return LIB
        return _build_locked(verbose, extra_flags, lib_path, build_dir)


def _build_locked(verbose, extra_flags, lib_path, build_dir) -> str:
    objs = []
    procs = []
    for s in SOURCES:
        obj = os.path.join(build_dir, os.path.splitext(s)[0] + ".o")
        cmd = [nvcc(), *NVCC_FLAGS, *extra_flags, "-x", "cu", "-c", os.path.join(CSRC, s), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- nvcc {s}\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    # the arch flag only keeps nvcc from assuming (and warning about) its default target at link time: the objects are sm_100a
    tmp = f"{lib_path}.tmp{os.getpid()}"  # link beside the target, then rename: a concurrent loader never sees a half-written file
    subprocess.run([nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", tmp, *objs, "-cudart", "static"], check=True)
    os.replace(tmp, lib_path)
    return lib_path


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))

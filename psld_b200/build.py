"""Builds libpsld_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.environ.get("PSLD_B200_LIB") or os.path.join(HERE, "libpsld_b200.so")
SOURCES = ["capi.cu", "phase_space.cu", "net_simt.cu", "conv_simt.cu", "conv_tc.cu", "conv_gn_tc.cu", "attn_tc.cu",
           "attn_stream_tc.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr",
]


def _nvcc():
    cand = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    return cand if os.path.exists(cand) else "nvcc"


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(os.path.dirname(HERE), "include", "psld_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compiles and links the library.  Safe with one process per GPU on a cold tree (torchrun /
    Lightning start every rank at once): the whole build runs under an exclusive file lock, objects
    go to a per-process directory, and the shared object is linked under a temporary name and moved
    into place atomically, so no rank can dlopen a half-written file."""
    if not force and not needs_build():
        return LIB
    import fcntl
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    with open(os.path.join(HERE, "build", ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not needs_build():     # another rank built it while we waited
                return LIB
            return _build_locked(verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(verbose: bool) -> str:
    objs = []
    odir = os.path.join(HERE, "build", f"obj.{os.getpid()}")
    os.makedirs(odir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(odir, src.replace(".cu", ".o"))
        cmd = [_nvcc(), *NVCC_FLAGS, *os.environ.get("PSLD_NVCC_EXTRA", "").split(), "-c",
               os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out.decode())
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}")
    tmp = LIB + f".tmp.{os.getpid()}"
    cmd = [_nvcc(), "-shared", "-o", tmp, *objs, "-gencode", "arch=compute_100a,code=sm_100a"]
    subprocess.check_call(cmd)
    os.replace(tmp, LIB)                       # atomic on the same filesystem
    import shutil
    shutil.rmtree(odir, ignore_errors=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))

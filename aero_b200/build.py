"""Build libaero_b200.so for sm_100a with nvcc (in-tree; the .so travels to the GPU box)."""
from __future__ import annotations

import glob
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libaero_b200.so")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-O3"]


def _sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def _digest():
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    for f in _sources() + sorted(glob.glob(os.path.join(CSRC, "*.cuh"))) + \
            [os.path.join(os.path.dirname(HERE), "include", "aero_b200.h")]:
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Compile every .cu in csrc/ into one shared library.  No-op when up to date."""
    stamp = LIB + ".stamp"
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == dig:
        return LIB
    # NVCC, else nvcc on PATH, else the toolkit at CUDA_HOME: the CUDA bin directory is often missing from a plain user's PATH
    nvcc = os.environ.get("NVCC") or shutil.which("nvcc") or \
        os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    objs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    procs = []
    for src in _sources():
        obj = os.path.join(HERE, "build", os.path.basename(src) + ".o")
        objs.append(obj)
        cmd = [nvcc, *NVCC_FLAGS, "-c", src, "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas")
            cmd.insert(2, "-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0 or verbose:
            sys.stderr.write(f"--- {os.path.basename(src)}\n{out}\n")
        failed |= pr.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    subprocess.check_call([nvcc, "-shared", "-o", LIB, *objs, "-lcudart", "-lcuda"])
    with open(stamp, "w") as fh:
        fh.write(dig)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))

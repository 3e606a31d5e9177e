"""Build recipe for the sm_100a kernel library (``fragnet_b200/_lib/libfragnet_b200.so``).

Plain ``nvcc -shared``: the library has a C ABI (``include/fragnet_b200.h``) and no torch / pybind
dependency, so it is built in-tree with one command and travels with the source snapshot.
"""
from __future__ import annotations

import glob
import os
import shutil
import subprocess

ROOT = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(ROOT, "csrc")
INCLUDE = os.path.join(os.path.dirname(ROOT), "include")
LIB_DIR = os.path.join(ROOT, "_lib")
LIB_PATH = os.path.join(LIB_DIR, "libfragnet_b200.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC", "-shared",
]


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def _stale() -> bool:
    if not os.path.isfile(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    deps = sources() + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(INCLUDE, "*.h"))
    return any(os.path.getmtime(p) > built for p in deps)


def nvcc_path():
    return shutil.which("nvcc") or ("/usr/local/cuda/bin/nvcc" if os.path.isfile("/usr/local/cuda/bin/nvcc") else None)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every ``csrc/*.cu`` for sm_100a into one shared library; returns its path."""
    if not force and not _stale():
        return LIB_PATH
    nvcc = nvcc_path()
    if nvcc is None:
        raise RuntimeError("nvcc not found: cannot build libfragnet_b200.so")
    os.makedirs(LIB_DIR, exist_ok=True)
    tmp = f"{LIB_PATH}.{os.getpid()}.tmp"      # several ranks may build at once: private output, atomic rename
    extra = os.environ.get("FNB_EXTRA_NVCC", "").split()      # experiments only (extra nvcc flags)
    cmd = [nvcc, *NVCC_FLAGS, *extra, "-I", INCLUDE, "-I", CSRC, "-o", tmp, *sources()]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    os.replace(tmp, LIB_PATH)
    if verbose:
        print(res.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force=True, verbose=True))

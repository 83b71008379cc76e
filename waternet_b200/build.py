"""Build libwaternet_b200.so in-tree with nvcc for sm_100a (no network, no pip).

``python -m waternet_b200.build`` or ``waternet_b200.build.build()``.  The shared
library lands next to this file so that it travels with a repository snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
OBJ_DIR = os.path.join(PKG_DIR, "csrc", "build")
LIB_NAME = "libwaternet_b200.so"
LIB_PATH = os.path.join(PKG_DIR, LIB_NAME)

ARCH_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xptxas", "-v",
              "--expt-relaxed-constexpr"]


def _nvcc() -> str:
    cand = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(cand):
        raise RuntimeError("nvcc not found; waternet_b200 needs the CUDA 12.9 toolchain to build")
    return cand


def _sources():
    return sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, lib_name: str = LIB_NAME) -> str:
    """Compile every .cu under csrc/ for sm_100a and link the shared library.

    ``lib_name`` links the library under another name next to the product library, e.g. a build of another
    revision for a same-box A/B run (``WATERNET_B200_LIB=<path>`` makes ``_lib.load()`` pick it up).
    """
    nvcc = _nvcc()
    lib_path = os.path.join(PKG_DIR, lib_name)
    os.makedirs(OBJ_DIR, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(PKG_DIR), "include", "waternet_b200.h"))
    objs = []
    for src in _sources():
        src_path = os.path.join(CSRC, src)
        obj = os.path.join(OBJ_DIR, src[:-3] + ".o")
        objs.append(obj)
        if force or _stale(obj, [src_path] + headers):
            cmd = [nvcc] + ARCH_FLAGS + NVCC_FLAGS + ["-c", src_path, "-o", obj]
            res = subprocess.run(cmd, capture_output=True, text=True)
            log = res.stdout + res.stderr
            with open(obj + ".log", "w") as f:
                f.write(" ".join(cmd) + "\n" + log)
            if verbose or res.returncode != 0:
                sys.stderr.write(log)
            if res.returncode != 0:
                raise RuntimeError(f"nvcc failed for {src} (see {obj}.log)")
    if force or _stale(lib_path, objs):
        cmd = [nvcc] + ARCH_FLAGS + ["-shared", "-o", lib_path] + objs
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            sys.stderr.write(res.stdout + res.stderr)
            raise RuntimeError("link failed")
    return lib_path


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))

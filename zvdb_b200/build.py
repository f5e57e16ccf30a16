"""Build libzvdb_b200.so in-tree with nvcc for sm_100a (explicit -gencode, -lineinfo).

    python -m zvdb_b200.build [--force] [--verbose] [--define NAME=VALUE ...] [--out PATH]

--define / --out build a variant of the library for an A/B run (e.g. --define ZVDB_F16_UNROLL=2 --out build/u2/libzvdb_b200.so,
then ZVDB_B200_LIB=build/u2/libzvdb_b200.so points the binding at it); without them the in-tree library is built.

The library is plain CUDA C++ behind a C ABI (include/zvdb_b200.h); it does not link torch.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_DIR = os.path.join(_HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libzvdb_b200.so")
SOURCES = ["capi.cu"]

NVCC_FLAGS = [
    "-O3", "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-fvisibility=hidden,-fno-fast-math",
    "-shared",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libzvdb_b200.so cannot be built")


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(_HERE, "..", "include", "zvdb_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, defines=(), out: str = "") -> str:
    out = os.path.abspath(out) if out else LIB_PATH
    if out == LIB_PATH and not defines and not force and not _stale():
        return LIB_PATH
    os.makedirs(os.path.dirname(out), exist_ok=True)
    cmd = [_nvcc(), *NVCC_FLAGS] + [f"-D{d}" for d in defines]
    if verbose:
        cmd += ["-Xptxas", "-v"]
    # the image's CC/CXX point at a wrapper; let nvcc use the system g++
    if os.path.exists("/usr/bin/g++"):
        cmd += ["-ccbin", "/usr/bin/g++"]
    cmd += ["-o", out] + [os.path.join(CSRC, s) for s in SOURCES]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode:
        raise RuntimeError("nvcc failed building libzvdb_b200.so")
    return out


if __name__ == "__main__":
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--define", action="append", default=[], metavar="NAME=VALUE", help="preprocessor definition (variant builds)")
    ap.add_argument("--out", default="", help="where to write the library (default: the in-tree zvdb_b200/lib/libzvdb_b200.so)")
    a = ap.parse_args()
    print(build(force=a.force, verbose=a.verbose, defines=a.define, out=a.out))

"""Build ``csrc/libsdnet_decode.so`` in-tree with nvcc for sm_100a.

    python structuredetector_b200/build.py [--force]

Run as a file, not with ``-m``: importing the package needs the extensions built here.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent
REPO = ROOT.parent
SOURCES = [ROOT / "csrc" / "sdnet_decode.cu"]
HEADERS = [REPO / "include" / "sdnet_decode.h", *sorted((ROOT / "csrc").glob("*.cuh"))]
OUTPUT = ROOT / "csrc" / "libsdnet_decode.so"

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    # numerics: IEEE division/sqrt, no flush-to-zero, no fast-math (the sigmoid must match
    # ATen's CUDA kernel bit for bit); FMA contraction is left on like ATen's build and the
    # grouping arithmetic uses explicitly rounded intrinsics instead.
    "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-Xcompiler", "-fPIC", "-shared",
]


def nvcc_path() -> str:
    found = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(found):
        raise RuntimeError("nvcc not found; cannot build the sm_100a extension")
    return found


def is_stale() -> bool:
    if not OUTPUT.exists():
        return True
    built = OUTPUT.stat().st_mtime
    return any(src.stat().st_mtime > built for src in SOURCES + HEADERS)


FASTOBJ_SRC = ROOT / "csrc" / "fastobj.c"


def fastobj_output() -> Path:
    import sysconfig

    return ROOT / ("_fastobj" + (sysconfig.get_config_var("EXT_SUFFIX") or ".so"))


def build_fastobj(force: bool = False, verbose: bool = False) -> Path:
    """The host-side object-assembly extension (CPython C API, plain gcc)."""
    import sysconfig

    out = fastobj_output()
    if not force and out.exists() and out.stat().st_mtime >= FASTOBJ_SRC.stat().st_mtime:
        return out
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        raise RuntimeError("gcc not found; cannot build the object-assembly extension")
    cmd = [cc, "-O2", "-fPIC", "-shared", "-Wall", f"-I{sysconfig.get_paths()['include']}", "-o", str(out), str(FASTOBJ_SRC)]
    if verbose:
        print(" ".join(cmd))
    subprocess.run(cmd, check=True)
    return out


def build(force: bool = False, verbose: bool = False) -> Path:
    build_fastobj(force, verbose)
    if not force and not is_stale():
        return OUTPUT
    cmd = [nvcc_path(), *NVCC_FLAGS, f"-I{REPO / 'include'}", f"-I{ROOT / 'csrc'}", "-o", str(OUTPUT), *map(str, SOURCES)]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd))
    subprocess.run(cmd, check=True)
    return OUTPUT


if __name__ == "__main__":
    out = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(out)

"""Builds liblatok_b200.so in-tree (nvcc cross-compiles sm_100a without a GPU).

    python -m latok_b200.build [--verbose]

The built library is git-ignored but travels with the working tree to the GPU box.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
LIB = PKG / "liblatok_b200.so"
# compiled in parallel, each once; latok_tok5.cu and latok_tok5_short.cu hold the tokenize kernel's two geometries
SOURCES = [CSRC / "latok_kernels.cu", CSRC / "latok_tok5.cu", CSRC / "latok_tok5_short.cu", CSRC / "latok_tokbytes.cu",
           CSRC / "latok_vocab.cu", CSRC / "latok_capi.cu", CSRC / "latok_reader.cpp"]
HEADERS = [CSRC / "latok_internal.h", CSRC / "latok_bits.h", CSRC / "latok_device.cuh", CSRC / "latok_tok5.cuh",
           ROOT / "include" / "latok_b200.h"]
GEN = CSRC / "_gen" / "latok_tables.h"
RANGES = PKG / "data" / "ucd11_latok_classes.txt"

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
    "-shared", "-cudart", "static",
]


def find_nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found; liblatok_b200.so cannot be built (there is no CPU fallback)")


PYPACK_SRC = CSRC / "latok_pypack.c"


def pypack_path() -> Path:
    import sysconfig
    return PKG / ("_pypack" + (sysconfig.get_config_var("EXT_SUFFIX") or ".so"))


def build_pypack(force: bool = False, verbose: bool = False) -> Path:
    """The CPython shim that packs list[str] into UTF-8 + offsets (host code, gcc)."""
    import sysconfig
    out = pypack_path()
    if not force and out.exists() and out.stat().st_mtime >= PYPACK_SRC.stat().st_mtime:
        return out
    cc = shutil.which("gcc") or shutil.which("cc")
    if not cc:
        raise RuntimeError("gcc not found; _pypack cannot be built")
    cmd = [cc, "-O3", "-shared", "-fPIC", "-I" + sysconfig.get_paths()["include"], str(PYPACK_SRC), "-o", str(out)]
    if verbose:
        print(" ".join(cmd))
    subprocess.run(cmd, check=True)
    return out


def _stale() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    deps = SOURCES + HEADERS + [RANGES, ROOT / "tools" / "gen_tables.py", Path(__file__)]
    return any(d.stat().st_mtime > t for d in deps)


def build_library(force: bool = False, verbose: bool = False) -> Path:
    if not force and not _stale():
        return LIB
    import tempfile
    from concurrent.futures import ThreadPoolExecutor
    subprocess.run([sys.executable, str(ROOT / "tools" / "gen_tables.py")], check=True,
                   stdout=None if verbose else subprocess.DEVNULL)
    flags = [f for f in NVCC_FLAGS if f != "-shared"]
    extra = []
    if os.environ.get("LATOK_PROFILE"):
        extra += ["-DLATOK_PROFILE"]
    if os.environ.get("LATOK_DEFS"):
        extra += os.environ["LATOK_DEFS"].split()
    if verbose:
        extra += ["-Xptxas", "-v"]
    # LATOK_B200_LIB_OUT: build somewhere else (e.g. a library for a newer UCD: LATOK_CLASSES / LATOK_LOW_LIMIT are read
    # by tools/gen_tables.py; the next default build regenerates the UCD-11 tables)
    out = Path(os.environ.get("LATOK_B200_LIB_OUT") or LIB)
    nvcc = find_nvcc()
    with tempfile.TemporaryDirectory() as tmp:
        jobs = [(src, Path(tmp) / (src.stem + ".o")) for src in SOURCES]

        def compile_one(job):
            src, obj = job
            cmd = [nvcc, *flags, *extra, "-c", str(src), "-o", str(obj)]
            if verbose:
                print(" ".join(cmd))
            r = subprocess.run(cmd, capture_output=True, text=True)
            return r.returncode, r.stdout + r.stderr

        with ThreadPoolExecutor(len(jobs)) as pool:
            results = list(pool.map(compile_one, jobs))
        for rc, log in results:
            if verbose or rc:
                sys.stderr.write(log)
        if any(rc for rc, _ in results):
            raise subprocess.CalledProcessError(1, "nvcc -c")
        cmd = [nvcc, *NVCC_FLAGS, *[str(o) for _, o in jobs], "-lz", "-o", str(out)]      # zlib: the csv.gz reader
        if verbose:
            print(" ".join(cmd))
        subprocess.run(cmd, check=True)
    return out


if __name__ == "__main__":
    path = build_library(force=True, verbose="--verbose" in sys.argv or "-v" in sys.argv)
    print(path)
    print(build_pypack(force=True, verbose="--verbose" in sys.argv or "-v" in sys.argv))

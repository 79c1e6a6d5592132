"""In-tree build of libraytracer.so (the C-ABI library) for sm_100a.

    python rust-swift-raytracer_b200/build.py [--force] [--verbose]

nvcc cross-compiles without a GPU.  The exact kernel TU is compiled with --fmad=false (see
csrc/rt_kernels_exact.cu), and so is the denoiser's (csrc/rt_denoise.cu); host code with
-ffp-contract=off.  The .so stays in-tree (git-ignored) so it travels to the GPU box with the snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
CSRC = HERE / "csrc"
# Tuning experiments only: RT_BUILD_VARIANT=name builds lib_<name>/ with extra -D flags from
# RT_BUILD_DEFINES ("A=1,B=2"); the package loads it when RT_LIB_VARIANT=name.  The shipped
# library is always lib/libraytracer.so.
_VARIANT = os.environ.get("RT_BUILD_VARIANT", "")
_DEFINES = ["-D" + d for d in os.environ.get("RT_BUILD_DEFINES", "").split(",") if d]
OUT_DIR = HERE / ("lib_" + _VARIANT if _VARIANT else "lib")
OBJ_DIR = OUT_DIR / "obj"
LIB = OUT_DIR / "libraytracer.so"

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_COMMON = ["-std=c++17", "-O3", "-lineinfo", "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math",
               "-Xptxas", "-v"]
CXX_FLAGS = ["-std=c++17", "-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra"]

UNITS = [
    # (source, extra flags, compiler)
    ("rt_kernels_exact.cu", ["--fmad=false"], "nvcc"),
    ("rt_kernels_fast.cu", ["--fmad=true"], "nvcc"),
    ("rt_denoise.cu", ["--fmad=false"], "nvcc"),
    ("rt_device.cu", [], "nvcc"),
    ("rt_scene.cpp", [], "cxx"),
    ("rt_capi.cpp", [], "cxx"),
]
HEADERS = ["rt_types.h", "rt_trace.cuh", "rt_kernels.cuh", "rt_denoise.cuh", "rt_host.hpp", "rt_unicode_alnum.h",
           "../../include/raytracer.h", "../../include/raytracer_b200.h"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found")


def _cxx() -> str:
    for cand in ("/usr/bin/g++", shutil.which("g++")):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("g++ not found")


def _stale(target: Path, deps) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(Path(d).stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    OBJ_DIR.mkdir(parents=True, exist_ok=True)
    hdrs = [CSRC / h for h in HEADERS] + [Path(__file__)]
    objs = []
    log = []
    for src, extra, comp in UNITS:
        s = CSRC / src
        o = OBJ_DIR / (s.stem + ".o")
        objs.append(o)
        if not force and not _stale(o, [s] + hdrs):
            continue
        if comp == "nvcc":
            cmd = [_nvcc(), "-ccbin", _cxx()] + ARCH + NVCC_COMMON + extra + _DEFINES + ["-c", str(s), "-o", str(o)]
        else:
            cmd = [_cxx()] + CXX_FLAGS + extra + _DEFINES + ["-c", str(s), "-o", str(o)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log.append("$ " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode:
            raise RuntimeError("build failed:\n" + log[-1])
    if force or _stale(LIB, objs):
        cmd = [_nvcc(), "-ccbin", _cxx(), "-shared"] + ARCH + ["-o", str(LIB)] + [str(o) for o in objs]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log.append("$ " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode:
            raise RuntimeError("link failed:\n" + log[-1])
    (OUT_DIR / "build.log").write_text("\n".join(log)) if log else None
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    p = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(p)

"""Build the native pieces in-tree for sm_100a (no JIT cache: the .so files travel with the repo).

  csrc/librtz.so        the product: CUDA kernels + the C ABI of include/rtz.h
  host/librtz_host.so   C++ mirror of the reference's Scene/Camera/... API above the C ABI
  host/rtz_main         the `main` of reference src/main.zig:14-36 on top of it
"""
from __future__ import annotations

import os
import shutil
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
HOST = PKG / "host"

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-fmad=false",          # arithmetic contract: only the explicit fmaf()/__ffma2_rn are fused
    "-Xcompiler", "-fPIC", "-shared",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found: librtz.so cannot be built")


def _stale(target: Path, sources) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(Path(s).stat().st_mtime > t for s in sources)


def _librtz_sources():
    return sorted(CSRC.glob("*.cu")) + sorted(CSRC.glob("*.cuh")) + [ROOT / "include" / "rtz.h"]


def _host_sources():
    return sorted(HOST.glob("*.cpp")) + sorted(HOST.glob("*.hpp")) + [ROOT / "include" / "rtz.h", CSRC / "librtz.so"]


def build_librtz(force: bool = False, verbose: bool = False) -> Path:
    so = CSRC / "librtz.so"
    if force or _stale(so, _librtz_sources()):
        cmd = [_nvcc(), *NVCC_FLAGS, "-o", str(so), str(CSRC / "rtz_api.cu")]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
        if verbose:
            print(r.stderr)
    return so


def build_host(force: bool = False) -> Path:
    so = HOST / "librtz_host.so"
    if not (HOST / "rtz_host_c.cpp").exists():
        return so
    srcs = _host_sources()
    cxx = os.environ.get("CXX", "g++")
    common = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-Wall", "-Wextra", f"-I{ROOT / 'include'}"]
    rpath = ["-Wl,-rpath,$ORIGIN/../csrc", f"-L{CSRC}", "-lrtz"]
    if force or _stale(so, srcs):
        r = subprocess.run([cxx, *common, "-shared", "-o", str(so), str(HOST / "rtz_host_c.cpp"), *rpath],
                           capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("host library build failed:\n" + r.stdout + r.stderr)
    exe = HOST / "rtz_main"
    if force or _stale(exe, srcs):
        r = subprocess.run([cxx, *common, "-o", str(exe), str(HOST / "main.cpp"), *rpath], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("rtz_main build failed:\n" + r.stdout + r.stderr)
    return so


def build_all(force: bool = False, verbose: bool = False) -> None:
    """Build everything; serialised with a file lock so that N torchrun ranks can all call it.  Writes nothing
    when every product is up to date, so a built tree may be read-only."""
    import fcntl
    if not force and not any(_stale(t, s) for t, s in ((CSRC / "librtz.so", _librtz_sources()),
                                                        (HOST / "librtz_host.so", _host_sources()),
                                                        (HOST / "rtz_main", _host_sources()))):
        return
    with open(PKG / ".build.lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            build_librtz(force, verbose)
            build_host(force)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


if __name__ == "__main__":
    import sys
    build_all(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print("built", CSRC / "librtz.so")

"""Build the native libraries in-tree with nvcc for sm_100a (no JIT cache: the .so files travel
to the GPU box with the repo snapshot).

  acarsdec_b200/libacars_b200.so         context API (include/acars_b200.h): CUDA kernels + host runtime
  acarsdec_b200/libacarsdec_compat.so    the reference's own symbols (include/acarsdec_compat.h)
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

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
# -fmad=false: the numerics contract forbids contracting separate mul/add (SURVEY.md §8a);
# the kernels also spell rounding-sensitive steps with __f*_rn intrinsics.
NVCC_FLAGS = ["-O3", "-lineinfo", "-std=c++17", "-fmad=false", "-Xcompiler", "-fPIC,-ffp-contract=off,-Wall",
              "-Xptxas", "-v"]

LIB = PKG / "libacars_b200.so"
COMPAT = PKG / "libacarsdec_compat.so"
COMPAT_AIR = PKG / "libacarsdec_compat_air.so"      # same shim built for -DWITH_AIR hosts (channel_t differs)
COMPAT_VARIANTS = [("WITH_RTL", COMPAT), ("WITH_AIR", COMPAT_AIR),
                   ("WITH_SOAPY", PKG / "libacarsdec_compat_soapy.so"),
                   ("WITH_SDRPLAY", PKG / "libacarsdec_compat_sdrplay.so")]
LIB_SRC = [CSRC / "kernels.cu", CSRC / "context.cu", CSRC / "hostmath.cpp", CSRC / "multi.cpp", CSRC / "outfmt.c"]
COMPAT_SRC = [CSRC / "compat.c"]
HEADERS = [CSRC / "acb_internal.h", CSRC / "frame_sm.h", CSRC / "demod_core.h", ROOT / "include" / "acars_b200.h",
           ROOT / "include" / "acarsdec_compat.h"]


def nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found: the CUDA extension cannot be built (there is no CPU fallback)")


def _stale(target: Path, deps) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(Path(d).exists() and Path(d).stat().st_mtime > t for d in deps)


def _run(cmd, log: Path) -> None:
    r = subprocess.run([str(c) for c in cmd], capture_output=True, text=True)
    log.write_text(r.stdout + r.stderr)
    if r.returncode:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("build failed: " + " ".join(str(c) for c in cmd))


def build(force: bool = False, verbose: bool = False) -> Path:
    """Build what is stale.  Several processes may call this at once (one rank per GPU under torchrun): an
    exclusive file lock serialises them, each link goes to a temporary name and is renamed into place, and
    whoever gets the lock second finds everything up to date.  A tree that is up to date is only read (it may be
    read-only)."""
    import fcntl
    if not force and not _lib_stale() and not _compat_stale():
        return LIB
    (PKG / "build").mkdir(exist_ok=True)
    with open(PKG / "build" / ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            return _build_locked(force, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _link(cmd, target: Path, log: Path) -> None:
    """Run a link command whose output is `target`, via a temporary file so a reader never sees a
    half-written library."""
    tmp = target.with_name(target.name + f".tmp{os.getpid()}")
    _run([tmp if c is target else c for c in cmd], log)
    os.replace(tmp, target)


def _lib_stale() -> bool:
    return _stale(LIB, LIB_SRC + HEADERS + [Path(__file__)])


def _compat_stale() -> bool:
    return all(p.exists() for p in COMPAT_SRC) and any(_stale(t, COMPAT_SRC + HEADERS + [LIB]) for _, t in COMPAT_VARIANTS)


def _build_locked(force: bool, verbose: bool) -> Path:
    if force or _lib_stale():
        cmd = [nvcc(), *ARCH, *NVCC_FLAGS, "-shared", "-o", LIB, *LIB_SRC, "-I", ROOT / "include"]
        _link(cmd, LIB, PKG / "build" / "libacars_b200.log")
        if verbose:
            print((PKG / "build" / "libacars_b200.log").read_text())
    if all(p.exists() for p in COMPAT_SRC) and (force or _compat_stale()):
        # plain C, the reference's language; the host's WITH_* macro selects channel_t's layout
        # (acarsdec.h:62-74) and the front-end symbols, so there is one shim per front-end
        for macro, target in COMPAT_VARIANTS:
            cmd = [os.environ.get("CC", "gcc"), "-O2", "-std=gnu11", "-fPIC", "-shared", "-Wall", "-D" + macro,
                   "-ffp-contract=off", "-o", target, *COMPAT_SRC, "-I", ROOT / "include", "-L", PKG, "-lacars_b200",
                   "-Wl,-rpath,$ORIGIN", "-lpthread", "-lm"]
            _link(cmd, target, PKG / "build" / (target.stem + ".log"))
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
    print("built", LIB)

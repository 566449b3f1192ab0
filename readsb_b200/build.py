"""In-tree builds: the CUDA/C-ABI library (nvcc, sm_100a) and the synthetic generator (gcc).

Everything is built next to its sources so the artefacts travel with a repo snapshot
(.so files are git-ignored, not gpurun-ignored).
"""
from __future__ import annotations

import os
import shutil
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
LIB_DEMOD = PKG / "libb200demod.so"
LIB_SYNTH = PKG / "libmodes_synth.so"

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC,-O2,-Wall,-fvisibility=hidden",
    "--fmad=false",            # the LUT arithmetic must not contract mul+add (convert.c:49-56)
    "-shared", "-cudart", "shared",
]


def _newer(target: Path, sources) -> bool:
    if not target.exists():
        return False
    t = target.stat().st_mtime
    return all(Path(s).stat().st_mtime <= t for s in sources)


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA library cannot be built")


def build_demod(force: bool = False, verbose: bool = False, defines=(), out: Path | None = None) -> Path:
    """defines / out: an experimental variant of the library (-D macros of csrc/*.cu) next to the product one; selected at
    run time with B200_DEMOD_LIB=<path> (readsb_b200/demod.py), used by tools/ for A/B timing on the GPU."""
    srcs = sorted(CSRC.glob("*.cu")) + sorted(CSRC.glob("*.cuh")) + sorted(CSRC.glob("*.h")) \
        + [ROOT / "include" / "b200_demod.h"]
    target = out or LIB_DEMOD
    if not force and _newer(target, srcs):
        return target
    cmd = [_nvcc(), *NVCC_FLAGS, "-I", str(ROOT / "include"), "-I", str(CSRC)] + [f"-D{d}" for d in defines]
    if verbose:
        cmd += ["-Xptxas", "-v"]
    cmd += [str(s) for s in sorted(CSRC.glob("*.cu"))] + ["-o", str(target)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return target


def build_synth(force: bool = False) -> Path:
    src = PKG / "synth" / "modes_synth.c"
    if not force and _newer(LIB_SYNTH, [src, PKG / "synth" / "modes_synth.h"]):
        return LIB_SYNTH
    cc = shutil.which("gcc") or "gcc"
    cmd = [cc, "-O2", "-std=c11", "-ffp-contract=off", "-fPIC", "-shared", "-Wall",
           str(src), "-o", str(LIB_SYNTH), "-lm"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("gcc failed:\n" + res.stdout + res.stderr)
    return LIB_SYNTH


def build_probe(force: bool = False) -> Path:
    """tools/liblatency_probe.so: bench.py's C stopwatch around the public C ABI (per-call latency of the drop-in's call shape)."""
    src = ROOT / "tools" / "latency_probe.c"
    out = ROOT / "tools" / "liblatency_probe.so"
    if not force and _newer(out, [src, ROOT / "include" / "b200_demod.h"]):
        return out
    cc = shutil.which("gcc") or "gcc"
    res = subprocess.run([cc, "-O2", "-std=c11", "-fPIC", "-shared", "-Wall", "-I", str(ROOT / "include"), str(src), "-o", str(out)],
                         capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("gcc failed:\n" + res.stdout + res.stderr)
    return out


def build_oracle() -> None:
    """Builds oracle/libmodes_oracle.so and, if /root/reference exists, oracle/_ref/libreadsb_ref.so.
    (Building the checker is not using it: nothing in this package loads those libraries.)"""
    res = subprocess.run(["make", "-C", str(ROOT / "oracle"), "CC=gcc"], capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + res.stdout + res.stderr)


def build_readsb_pair() -> None:
    """Where the reference tree is present (oracle/Makefile decides, REF=<dir>): the whole reference program, stock
    (oracle/_ref/readsb_cpu) and linked with integration/readsb_shim.c against libb200demod.so (oracle/_ref/readsb_b200),
    for tests/test_gpu_shim.py; without it the target builds nothing.  Needs build_demod() first.  Test infrastructure,
    like the rest of oracle/."""
    if not LIB_DEMOD.exists():
        return
    res = subprocess.run(["make", "-C", str(ROOT / "oracle"), "CC=gcc", "readsb-pair"], capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("readsb-pair build failed:\n" + res.stdout + res.stderr)


if __name__ == "__main__":
    import sys
    build_synth(force=True)
    build_oracle()
    print(build_demod(force=True, verbose="-v" in sys.argv))
    build_readsb_pair()

"""Builds libuyd.so in-tree with nvcc for sm_100a (no torch involved)."""
from __future__ import annotations

import os
import subprocess
from pathlib import Path

HERE = Path(__file__).resolve().parent
CSRC = HERE / "csrc"
LIB = HERE / "libuyd.so"
COMPAT_LIB = HERE / "libuyd_compat.so"   # the reference's own extern "C" symbols (include/uyd_compat.h) on top of libuyd.so
SOURCES = ["api.cu", "conv_direct.cu", "stem_fused.cu", "conv_tc.cu", "conv_chain.cu", "c3k_fused.cu", "c3k_flat.cu", "c3k_tc.cu", "pool_upsample.cu", "decode.cu", "nms.cu", "preprocess.cu", "evalmatch.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-Xptxas", "-v",
] + os.environ.get("UYD_NVCC_EXTRA", "").split()   # debug builds only, e.g. -DUYD_C3K_TIMELINE_BUILD (tools/c3k_timeline.py)


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.sep not in c or Path(c).exists()):
            return c
    raise RuntimeError("nvcc not found")


def build(force: bool = False, verbose: bool = False) -> Path:
    srcs = [CSRC / s for s in SOURCES]
    deps = srcs + [CSRC / "stem_v2.cuh", CSRC / "c3k_flat.cuh", CSRC / "tc_ptx.cuh", CSRC / "tlbr.cuh", CSRC / "camera.cuh", CSRC / "common.cuh", HERE.parent / "include" / "uyd.h"]
    if not force and LIB.exists() and all(d.stat().st_mtime <= LIB.stat().st_mtime for d in deps):
        build_compat(force)
        return LIB
    objs = []
    (HERE / "build").mkdir(exist_ok=True)
    logs = []
    for s in srcs:
        o = HERE / "build" / (s.stem + ".o")
        if force or not o.exists() or any(d.stat().st_mtime > o.stat().st_mtime for d in (s, *deps[len(srcs):])):
            r = subprocess.run([_nvcc(), *NVCC_FLAGS, "-c", str(s), "-o", str(o)], capture_output=True, text=True)
            logs.append(r.stderr)
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed on {s.name}:\n{r.stdout}\n{r.stderr}")
        objs.append(str(o))
    r = subprocess.run([_nvcc(), "-shared", "-o", str(LIB), *objs, "-cudart", "static"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    (HERE / "build" / "ptxas.log").write_text("\n".join(logs))
    if verbose:
        print("\n".join(logs))
    build_compat(True)
    return LIB


def build_compat(force: bool = False) -> Path:
    src = CSRC / "compat.cu"
    deps = [src, HERE.parent / "include" / "uyd.h", HERE.parent / "include" / "uyd_compat.h", LIB]
    if not force and COMPAT_LIB.exists() and all(d.stat().st_mtime <= COMPAT_LIB.stat().st_mtime for d in deps):
        return COMPAT_LIB
    r = subprocess.run([_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "-std=c++17", "-Xcompiler", "-fPIC", "-shared",
                        str(src), "-o", str(COMPAT_LIB), f"-L{HERE}", "-luyd", "-Xlinker", "-rpath=$ORIGIN", "-cudart", "static"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed on compat.cu:\n{r.stdout}\n{r.stderr}")
    return COMPAT_LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))

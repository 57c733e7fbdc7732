"""In-tree build of libpnr.so (the C-ABI CUDA library) with nvcc for sm_100a only.

No torch extension machinery: the library has no torch types in its ABI (include/pnr.h), so it is a
plain ``nvcc -shared`` of csrc/*.cu.  The .so is git-ignored but travels to the GPU box with gpurun.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB = PKG / "libpnr.so"
SOURCES = ["pnr_api.cu", "ray_kernels.cu", "stream_kernels.cu", "mlp_tc05.cu", "render.cu", "comm.cu", "panoptic_kernels.cu", "wgrad_tc05.cu", "linear_tc05.cu",
           "eval_kernels.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC"] + os.environ.get("PNR_NVCC_FLAGS", "").split()   # e.g. -DPNR_TIMELINE


def _nvcc() -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: libpnr cannot be built (there is no non-CUDA fallback)")
    return nvcc


def _digest() -> str:
    h = hashlib.sha256()
    for f in sorted(list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + list(CSRC.glob("*.h"))
                    + [PKG.parent / "include" / "pnr.h"]):
        h.update(f.name.encode())
        h.update(f.read_bytes())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def is_fresh() -> bool:
    stamp = PKG / "libpnr.stamp"
    return LIB.exists() and stamp.exists() and stamp.read_text().strip() == _digest()


def build(force: bool = False, verbose: bool = False, out: Path = None, extra_flags=()) -> Path:
    """Compile csrc/*.cu -> panopticnerf_b200/libpnr.so.  Cross-compiles without a GPU.
    `out` + `extra_flags`: a development variant next to the product library (e.g. the -DPNR_TIMELINE build that
    tools/timeline.py loads through PNR_LIB); the product library and its stamp are left alone."""
    if out is not None:
        return _compile(Path(out), list(extra_flags), verbose, PKG.parent / "build" / Path(out).stem)
    if not force and is_fresh():
        return LIB
    _compile(LIB, [], verbose, PKG.parent / "build" / "libpnr")
    (PKG / "libpnr.stamp").write_text(_digest())
    return LIB


def _compile(lib: Path, extra_flags, verbose: bool, objdir: Path) -> Path:
    nvcc = _nvcc()
    objdir.mkdir(parents=True, exist_ok=True)
    procs = []
    objs = []
    for src in SOURCES:
        obj = objdir / (src[:-3] + ".o")
        objs.append(str(obj))
        cmd = [nvcc, *NVCC_FLAGS, *extra_flags, "-c", str(CSRC / src), "-o", str(obj)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
        if verbose and out:
            print(out)
    link = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(lib), *objs,
            "-cudart", "shared", "-ldl"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    return lib


if __name__ == "__main__":
    import sys
    if "--timeline" in sys.argv:
        print(build(out=PKG / "libpnr_timeline.so", extra_flags=["-DPNR_TIMELINE"]))
    else:
        print(build(force=True, verbose=True))

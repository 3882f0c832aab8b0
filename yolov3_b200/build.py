"""In-tree build of the C-ABI shared library (nvcc, sm_100a only).  The .so lands next to this file so that it
travels with the repo snapshot to the GPU box; it is git-ignored."""
from __future__ import annotations

import os
import shutil
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB = PKG / "libyolov3_b200.so"
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-diag-suppress", "177",
              "--use_fast_math", "-shared"]
# kernels whose arithmetic must match the reference bit for bit are compiled without fast-math / FMA contraction
EXACT_SOURCES = {"y3_nms.cu", "y3_detect.cu", "y3_loss.cu", "y3_iou.cu", "y3_val.cu", "y3_metrics.cu", "y3_pre.cu", "y3_tta.cu"}


def nvcc_path() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found: the CUDA toolkit is required to build yolov3_b200")


def sources():
    return sorted(CSRC.glob("*.cu"))


def needs_build() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    deps = list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + list(CSRC.glob("*.h")) + [PKG.parent / "include" / "yolov3_b200.h"]
    return any(p.stat().st_mtime > t for p in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    if not force and not needs_build():
        return LIB
    nvcc = nvcc_path()
    objdir = PKG / "build"
    objdir.mkdir(exist_ok=True)
    objs = []
    procs = []
    for src in sources():
        obj = objdir / (src.stem + ".o")
        flags = [f for f in NVCC_FLAGS if f != "-shared"]
        if src.name in EXACT_SOURCES:
            flags = [f for f in flags if f != "--use_fast_math"] + ["-fmad=false"]
        cmd = [nvcc, *flags, "-c", str(src), "-o", str(obj)]
        if verbose:
            print(" ".join(cmd))
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(str(obj))
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src.name}:\n{out}")
        if verbose and out.strip():
            print(out)
    tmp = LIB.with_suffix(".so.tmp")
    link = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", str(tmp), *objs]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    os.replace(tmp, LIB)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))

"""Builds ``libagx_b200.so`` (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python -m anemoi_graphs_b200._build [--force]

The library is git-ignored but travels to the GPU box with the snapshot; there is no JIT at import
time and no CPU fallback - if the file is missing the package refuses to compute.
"""

from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB_DIR = PKG / "lib"
LIB_PATH = LIB_DIR / "libagx_b200.so"
OBJ_DIR = LIB_DIR / "obj"
SOURCES = ["agx_util.cu", "agx_index.cu", "agx_knn.cu", "agx_radius.cu", "agx_attrs.cu", "agx_mesh.cu", "agx_hex.cu", "agx_voronoi.cu", "agx_concat.cu", "agx_postprocess.cu", "agx_sparse.cu", "agx_group_norm.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "-Xcompiler", "-fvisibility=default",
]  # fmt: skip
LINK_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "--shared", "-cudart", "static"]


def find_nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def is_stale() -> bool:
    if not LIB_PATH.exists():
        return True
    built = LIB_PATH.stat().st_mtime
    deps = [CSRC / s for s in SOURCES] + list(CSRC.glob("*.cuh")) + [PKG.parent / "include" / "agx_b200.h"]
    return any(d.stat().st_mtime > built for d in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    if not force and not is_stale():
        return LIB_PATH
    LIB_DIR.mkdir(exist_ok=True)
    OBJ_DIR.mkdir(exist_ok=True)
    nvcc = find_nvcc()
    headers = list(CSRC.glob("*.cuh")) + [PKG.parent / "include" / "agx_b200.h"]
    newest_header = max(h.stat().st_mtime for h in headers)
    # one translation unit per source, compiled in parallel; an object is reused while it is newer than its
    # source and every header
    jobs = []
    for src in SOURCES:
        obj = OBJ_DIR / (src + ".o")
        if not force and obj.exists() and obj.stat().st_mtime > max((CSRC / src).stat().st_mtime, newest_header):
            continue
        cmd = [nvcc, *NVCC_FLAGS, "-c", "-o", str(obj), str(CSRC / src)]
        if verbose:
            cmd[1:1] = ["-Xptxas", "-v"]
            print(" ".join(cmd))
        jobs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)))
    for src, proc in jobs:
        out, err = proc.communicate()
        if proc.returncode != 0:
            for _, other in jobs:
                if other.poll() is None:
                    other.kill()
            raise RuntimeError(f"nvcc failed on {src}:\n{out}\n{err}")
        if verbose:
            print(err)
    tmp = LIB_PATH.with_suffix(".so.tmp")
    cmd = [nvcc, *LINK_FLAGS, "-o", str(tmp), *[str(OBJ_DIR / (s + ".o")) for s in SOURCES]]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"link failed:\n{res.stdout}\n{res.stderr}")
    os.replace(tmp, LIB_PATH)
    return LIB_PATH


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(path)

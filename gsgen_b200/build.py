"""Build libgsb200.so in-tree with nvcc for sm_100a (no torch dependency in the library itself).

    python -m gsgen_b200.build [--force] [--ptxas-v]

The .so lands next to this file (git-ignored, shipped to the GPU box by gpurun).
"""
from __future__ import annotations

import concurrent.futures as cf
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
BUILD = os.path.join(HERE, "_build")
LIB = os.path.join(HERE, "libgsb200.so")
SOURCES = ["api.cu", "preprocess.cu", "binning.cu", "composite_fwd.cu", "composite_bwd.cu", "composite_bwd_sh.cu",
           "optimizer.cu", "store.cu", "knn.cu", "normals.cu"]
NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "--expt-relaxed-constexpr",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "-DGSB200_BUILD",
]
# per-file flags: the normal estimate evaluates normals.cuh without FMA contraction, exactly as the g++ host build
# (-ffp-contract=off) of the test-suite does
FILE_FLAGS = {"normals.cu": ["-fmad=false"]}


def _deps_mtime() -> float:
    m = 0.0
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for f in os.listdir(root):
            if f.endswith((".cu", ".cuh", ".h")):
                m = max(m, os.path.getmtime(os.path.join(root, f)))
    return m


def build(force: bool = False, ptxas_v: bool = False, verbose: bool = True, defines=(), out: str = LIB) -> str:
    """defines: extra -D flags (tuning experiments); out: output .so (default: the in-tree library)."""
    if not force and os.path.exists(out) and os.path.getmtime(out) >= _deps_mtime():
        return out
    os.makedirs(BUILD, exist_ok=True)
    flags = list(NVCC_FLAGS) + (["-Xptxas", "-v"] if ptxas_v else []) + [f"-D{d}" for d in defines]
    tag = ("_" + "_".join(d.replace("=", "") for d in defines)) if defines else ""

    def compile_one(src):
        obj = os.path.join(BUILD, src.replace(".cu", tag + ".o"))
        cmd = ["nvcc", *flags, *FILE_FLAGS.get(src, []), "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        return src, obj, r

    objs = []
    with cf.ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        for src, obj, r in ex.map(compile_one, SOURCES):
            if verbose and (r.stderr.strip() or r.returncode):
                sys.stderr.write(f"--- nvcc {src} ---\n{r.stderr}\n")
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed on {src}")
            objs.append(obj)
    cmd = ["nvcc", "-shared", "-o", out, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    subprocess.check_call(cmd)
    return out


if __name__ == "__main__":
    _defs = [a[2:] for a in sys.argv[1:] if a.startswith("-D")]
    _out = next((a.split("=", 1)[1] for a in sys.argv[1:] if a.startswith("--out=")), LIB)
    print(build(force="--force" in sys.argv or bool(_defs), ptxas_v="--ptxas-v" in sys.argv, defines=_defs, out=_out))

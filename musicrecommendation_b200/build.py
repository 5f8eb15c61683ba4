"""Build libmrscore.so (the C-ABI of include/mrscore.h) in-tree with nvcc for sm_100a."""
from __future__ import annotations

import os
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
SO = PKG / "libmrscore.so"
SOURCES = ["mrscore.cu", "k1_count_gemm.cu", "k1_sparse_count.cu", "k2_aggregate.cu", "k3_topk.cu", "k4_itemspace.cu", "k5_evaluate.cu", "k6_ingest.cu", "k7_testlists.cu", "k8_similar.cu", "k9_audience.cu", "k10_filter.cu", "modelio.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--fmad=false",
              "-Xcompiler", "-fPIC,-fvisibility=hidden", "-cudart", "static"]


def build(force: bool = False, verbose: bool = False) -> Path:
    srcs = [CSRC / s for s in SOURCES]
    deps = srcs + list(CSRC.glob("*.cuh")) + list(CSRC.glob("*.h")) + [PKG.parent / "include" / "mrscore.h"]
    if not force and SO.exists() and all(SO.stat().st_mtime >= d.stat().st_mtime for d in deps):
        return SO
    def compile_one(s: Path) -> str:
        o = CSRC / (s.stem + ".o")
        if not force and o.exists() and all(o.stat().st_mtime >= d.stat().st_mtime for d in [s] + headers):
            return str(o)                     # unchanged translation unit
        cmd = ["nvcc", *NVCC_FLAGS, "-c", str(s), "-o", str(o)] + (["-Xptxas", "-v"] if verbose else [])
        subprocess.run(cmd, check=True)
        return str(o)

    headers = list(CSRC.glob("*.cuh")) + list(CSRC.glob("*.h")) + [PKG.parent / "include" / "mrscore.h"]
    if verbose:
        objs = [compile_one(s) for s in srcs]     # keep the ptxas output readable
    else:
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=min(len(srcs), os.cpu_count() or 4)) as pool:
            objs = list(pool.map(compile_one, srcs))
    subprocess.run(["nvcc", "-shared", "-cudart", "static", "-o", str(SO), *objs], check=True)
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))

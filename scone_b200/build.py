"""Compile libscone_b200.so in-tree for sm_100a (nvcc cross-compiles without a GPU).

    python -m scone_b200.build [--force]

The built library is git-ignored but travels to the GPU box with the repo snapshot.
"""

from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIB_DIR = os.path.join(PKG, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libscone_b200.so")
SOURCES = ["api.cu", "index.cu", "table.cu", "embed.cu", "pipeline.cu", "fold.cu", "fit.cu"]
# the fused path's kernels are compiled once per (table format, output type): eight translation units, in parallel
INST_SOURCE = "embed_inst.cu"
INSTANCES = [(q, o) for o in (0, 1) for q in (0, 1, 2, 3)]
HEADERS = ["common.cuh", "match.cuh", "embed_plan.h", "fold_plan.h", "row_format.cuh", "embed_kernels.cuh", "embed_pipe.cuh", os.path.join("..", "..", "include", "scone_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "-Xfatbin", "-compress-all",        # -lineinfo quadruples the cubins; compressed the library is ~10 MB instead of 42 MB
]
LINK_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-cudart", "static"]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libscone_b200.so cannot be built")


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES + [INST_SOURCE] + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > built for d in deps)


def _run(cmd) -> str:
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + proc.stdout + proc.stderr)
    return proc.stderr


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB_PATH
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(LIB_DIR, exist_ok=True)
    obj_dir = os.path.join(LIB_DIR, "obj")
    os.makedirs(obj_dir, exist_ok=True)
    nvcc = nvcc_path()
    common = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else [])
    jobs = []
    for q, o in INSTANCES:                                                 # the long ones first
        obj = os.path.join(obj_dir, f"embed_inst_q{q}_{o}.o")
        jobs.append((obj, common + [f"-DSCONE_INST_QUANT={q}", f"-DSCONE_INST_OUT={o}", "-c", os.path.join(CSRC, INST_SOURCE), "-o", obj]))
    for src in SOURCES:
        obj = os.path.join(obj_dir, src.replace(".cu", ".o"))
        jobs.append((obj, common + ["-c", os.path.join(CSRC, src), "-o", obj]))
    with ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 1))) as pool:
        logs = list(pool.map(lambda j: _run(j[1]), jobs))
    _run([nvcc] + LINK_FLAGS + ["-o", LIB_PATH] + [obj for obj, _ in jobs])
    if verbose:
        print("\n".join(logs))
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))

"""Ahead-of-time build of the CUDA library (sm_100a only), in-tree.

    python -m tensorized_rnn_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU, so this also runs in the CPU-only build container.
The product is `tensorized_rnn_b200/csrc/libttrnn_b200.so` (git-ignored; it travels
to the GPU box with the working tree).
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libttrnn_b200.so")
SOURCES = ["ttrnn_capi.cu", "tt_static_inst.cu"]
HEADERS = ["tt_plan.h", "tt_stage.cuh", "tt_kernels.cuh", "tt_proj.cuh", "tt_cell.cuh", "tt_gemm.cuh", "tt_umma.cuh", "tt_tc.cuh", "tt_ge2e.cuh", "tt_dense.cuh", "tt_bidir.cuh", "tt_dropout.cuh", "tt_utter.cuh", "tt_varlen.cuh", "tt_static.cuh", "tt_static_api.h",
           os.path.join("..", "..", "include", "ttrnn_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo", "--expt-relaxed-constexpr",
    "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


# headers each translation unit includes (an up-to-date object file is not recompiled)
TU_DEPS = {
    "ttrnn_capi.cu": HEADERS,
    "tt_static_inst.cu": ["tt_plan.h", "tt_umma.cuh", "tt_static.cuh", "tt_static_api.h", os.path.join("..", "..", "include", "ttrnn_b200.h")],
}


def _obj_stale(src: str, obj: str) -> bool:
    if not os.path.exists(obj):
        return True
    t = os.path.getmtime(obj)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in [src] + TU_DEPS[src])


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    # one nvcc per translation unit, in parallel; then link
    procs, objs, log = [], [], ""
    for src in SOURCES:
        obj = os.path.join(CSRC, os.path.splitext(src)[0] + ".o")
        objs.append(obj)
        if not force and os.environ.get("TTRNN_NVCC_EXTRA") is None and not _obj_stale(src, obj):
            continue
        extra = os.environ.get("TTRNN_NVCC_EXTRA", "").split()
        cmd = [_nvcc()] + NVCC_FLAGS + extra + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for cmd, pr in procs:
        out, _ = pr.communicate()
        log += " ".join(cmd) + "\n" + out + "\n"
        failed = failed or pr.returncode != 0
    if not failed:
        cmd = [_nvcc(), "-shared", "-o", LIB] + objs
        res = subprocess.run(cmd, capture_output=True, text=True)
        log += " ".join(cmd) + "\n" + res.stdout + res.stderr
        failed = res.returncode != 0
    with open(os.path.join(CSRC, "build.log"), "w") as f:
        f.write(log)
    if failed:
        raise RuntimeError("nvcc failed:\n" + log[-8000:])
    if verbose:
        print(log)
    return LIB


if __name__ == "__main__":
    path = build_library(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)

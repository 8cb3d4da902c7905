"""Builds libgbxq.so (the C-ABI CUDA library, include/gbxq.h) in-tree with nvcc for sm_100a.

    python -m gbx_lm_b200.build [--force] [--verbose]

Each .cu becomes an object under csrc/_obj (parallel), then one shared library next to this file.
The built .so is git-ignored but travels to the GPU box with the gpurun snapshot."""
from __future__ import annotations

import concurrent.futures as cf
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "_obj")
LIB = os.path.join(HERE, "libgbxq.so")
SOURCES = [
    "gbxq_api.cu",
    "gbxq_dequant.cu",
    "gbxq_quantize.cu",
    "gbxq_generic.cu",
    "gbxq_gemv.cu",
    "gbxq_skinny.cu",
    "gbxq_mmv.cu",
    "gbxq_mmv8.cu",
    "gbxq_mmv8_grouped.cu",
    "gbxq_stream.cu",
    "gbxq_glue.cu",
    "gbxq_qattn.cu",
    "gbxq_head.cu",
    "gbxq_gather.cu",
    "gbxq_gemm_sm100.cu",
    "gbxq_gemm_ts_sm100.cu",
    "gbxq_gemm_ts_direct_sm100.cu",
    "gbxq_gemm_ts_grouped_sm100.cu",
    "gbxq_allreduce.cu",
]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"] + ARCH


def nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; libgbxq.so cannot be built")
    return exe


def _deps_mtime() -> float:
    paths = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h"))]
    paths.append(os.path.join(HERE, "..", "include", "gbxq.h"))
    paths.append(os.path.abspath(__file__))
    return max(os.path.getmtime(p) for p in paths)


def needs_build() -> bool:
    return not os.path.exists(LIB) or os.path.getmtime(LIB) < _deps_mtime()


def build(force: bool = False, verbose: bool = False, variant: str = "", extra_flags=()) -> str:
    """variant / extra_flags: an A/B build with other -D flags into libgbxq_<variant>.so (objects kept apart)."""
    global OBJ, LIB
    if variant:
        OBJ = os.path.join(CSRC, "_obj_" + variant)
        LIB = os.path.join(HERE, f"libgbxq_{variant}.so")
        force = True
    if not force and not needs_build():
        return LIB
    os.makedirs(OBJ, exist_ok=True)
    exe = nvcc()
    env = dict(os.environ)
    env.pop("CC", None)  # the image exports CC=/opt/gcc/bin/gcc, which lacks libgomp spec files
    env.pop("CXX", None)
    hdr_time = max(
        os.path.getmtime(os.path.join(CSRC, f)) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))
    )
    hdr_time = max(hdr_time, os.path.getmtime(os.path.join(HERE, "..", "include", "gbxq.h")), os.path.getmtime(__file__))

    def compile_one(src: str) -> str:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src.replace(".cu", ".o"))
        if force or not os.path.exists(o) or os.path.getmtime(o) < max(os.path.getmtime(s), hdr_time):
            cmd = [exe, *NVCC_FLAGS, *extra_flags, "-c", s, "-o", o]
            if verbose:
                cmd.insert(1, "-Xptxas")
                cmd.insert(2, "-v")
                print(" ".join(cmd), flush=True)
            r = subprocess.run(cmd, env=env, capture_output=True, text=True)
            if verbose or r.returncode:
                sys.stderr.write(r.stdout + r.stderr)
            if r.returncode:
                raise RuntimeError(f"nvcc failed on {src}")
        return o

    with cf.ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [exe, "-shared", *ARCH, "-o", LIB + ".tmp", *objs]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True)
    if r.returncode:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link of libgbxq.so failed")
    os.replace(LIB + ".tmp", LIB)
    return LIB


if __name__ == "__main__":
    var = [a.split("=", 1)[1] for a in sys.argv if a.startswith("--variant=")]
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv, variant=var[0] if var else "",
                extra_flags=[a for a in sys.argv[1:] if a.startswith("-D")]))

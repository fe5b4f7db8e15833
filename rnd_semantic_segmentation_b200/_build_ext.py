"""Build libb200seg.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m rnd_semantic_segmentation_b200._build_ext [--force] [--verbose]

The library has no torch / python dependency: it is a plain C-ABI shared object
(include/b200seg.h) with the CUDA runtime linked statically, loaded with ctypes.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
ROOT = os.path.dirname(PKG_DIR)
LIB_PATH = os.path.join(PKG_DIR, "libb200seg.so")
OBJ_DIR = os.path.join(PKG_DIR, "_obj")
SOURCES = ["api.cu", "eval_kernels.cu", "ce_kernels.cu", "ce_v2_kernels.cu", "softce_kernels.cu",
           "gemm_sm100.cu", "aspp_head.cu", "conv_sm100.cu", "tta_kernels.cu", "optim_kernels.cu", "p2p_allreduce.cu",
           "seam_tail_kernels.cu"]
HEADERS = ["common.cuh", "ce_geom.cuh", "gemm_sm100.cuh", os.path.join(ROOT, "include", "b200seg.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _digest(paths) -> str:
    h = hashlib.sha256()
    h.update(" ".join(NVCC_FLAGS).encode())
    for p in paths:
        with open(p, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def build(force: bool = False, verbose: bool = False) -> str:
    srcs = sources()
    hdrs = [h if os.path.isabs(h) else os.path.join(CSRC, h) for h in HEADERS]
    os.makedirs(OBJ_DIR, exist_ok=True)
    stamp = os.path.join(OBJ_DIR, "stamp")
    want = _digest(srcs + hdrs)
    if not force and os.path.exists(LIB_PATH) and os.path.exists(stamp) and open(stamp).read() == want:
        return LIB_PATH
    nvcc = _nvcc()
    hdr_digest = _digest(hdrs)

    def compile_one(src):
        obj = os.path.join(OBJ_DIR, os.path.basename(src) + ".o")
        ostamp = obj + ".stamp"
        d = _digest([src]) + hdr_digest
        if not force and os.path.exists(obj) and os.path.exists(ostamp) and open(ostamp).read() == d:
            return obj
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        with open(ostamp, "w") as f:
            f.write(d)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        objs = list(ex.map(compile_one, srcs))
    link = [nvcc, "-shared", "-o", LIB_PATH] + objs + ["-gencode", "arch=compute_100a,code=sm_100a",
                                                       "-cudart", "static", "-Xcompiler", "-fPIC"]
    r = subprocess.run(link, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp, "w") as f:
        f.write(want)
    return LIB_PATH


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)

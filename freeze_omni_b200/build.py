"""Build freeze_omni_b200/libfo_b200.so (the C-ABI library of include/fo_b200.h) with nvcc for sm_100a.

The library is built IN-TREE so it travels to the GPU box with the repo snapshot; it is git-ignored.
nvcc cross-compiles without a GPU.  `python -m freeze_omni_b200.build [--force]`.
"""
from __future__ import annotations

import concurrent.futures
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "csrc", "build")
LIB = os.path.join(HERE, "libfo_b200.so")
SOURCES = ["fo_api.cu", "fo_gemm_simt.cu", "fo_gemm_tc.cu", "fo_elementwise.cu", "fo_attention.cu", "fo_fbank.cu", "fo_stack.cu",
           "fo_session.cu", "fo_partition.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]
if os.environ.get("FO_TC_TRACE_BUILD") == "1":        # in-kernel timeline stamps for tools/gemm_trace.py
    NVCC_FLAGS.append("-DFO_TC_TRACE_BUILD")
if os.environ.get("FO_TRACE_BUILD") == "1":           # whole-step CTA timeline (tools/step_timeline.py): a SEPARATE library
    NVCC_FLAGS.append("-DFO_TRACE_BUILD")
    OBJ = os.path.join(HERE, "csrc", "build_trace")
    LIB = os.path.join(HERE, "libfo_b200_trace.so")


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _digest(paths) -> str:
    h = hashlib.sha256()
    for p in sorted(paths):
        with open(p, "rb") as f:
            h.update(p.encode())
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "fo_b200.h"))
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    stamp = os.path.join(OBJ, "stamp")
    digest = _digest(srcs + headers)
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == digest:
        return LIB
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(OBJ, os.path.basename(src)[:-3] + ".o")
        cmd = [nvcc] + NVCC_FLAGS + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (src, r.stdout + r.stderr))
        if verbose and r.stderr:
            sys.stderr.write(r.stderr)
        return obj

    with concurrent.futures.ThreadPoolExecutor(max_workers=len(srcs)) as ex:
        objs = list(ex.map(compile_one, srcs))
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s" % (r.stdout + r.stderr))
    with open(stamp, "w") as f:
        f.write(digest)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))

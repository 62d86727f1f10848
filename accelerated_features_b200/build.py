"""Build libxfeat_sm100.so in-tree with nvcc (sm_100a only).  `python -m accelerated_features_b200.build`"""
from __future__ import annotations

import concurrent.futures as cf
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libxfeat_sm100.so")
OBJ = os.path.join(HERE, "build")
SOURCES = ["api.cu", "prep.cu", "stem.cu", "conv_simt.cu", "conv_tc.cu", "conv_tc_halo.cu", "block1_tc.cu", "head_chain_tc.cu", "heads.cu", "sparse.cu", "dense.cu", "mnn.cu", "mnn_tc.cu", "mnn_fast.cu", "refine.cu", "mlp_tc.cu", "helpers.cu", "ransac.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "--expt-relaxed-constexpr",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "-Xptxas", "-v"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stamp(paths) -> str:
    h = hashlib.sha1(" ".join(NVCC_FLAGS).encode())
    for p in sorted(paths):
        with open(p, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def build_library(force: bool = False, verbose: bool = False) -> str:
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    headers.append(os.path.join(HERE, "..", "include", "xfeat_b200.h"))
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    stamp = _stamp(headers + srcs)
    stamp_file = os.path.join(OBJ, "stamp")
    if not force and os.path.exists(LIB) and os.path.exists(stamp_file) and open(stamp_file).read() == stamp:
        return LIB
    os.makedirs(OBJ, exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(OBJ, os.path.basename(src)[:-3] + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log = r.stdout + r.stderr
        with open(obj + ".log", "w") as f:
            f.write(" ".join(cmd) + "\n" + log)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{log}")
        return obj, log

    with cf.ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        results = list(ex.map(compile_one, srcs))
    objs = [o for o, _ in results]
    if verbose:
        for _, log in results:
            sys.stderr.write(log)
    cmd = [nvcc, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    with open(stamp_file, "w") as f:
        f.write(stamp)
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))

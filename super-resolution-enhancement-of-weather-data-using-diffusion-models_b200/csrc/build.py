"""Builds libwsr.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python <pkg>/csrc/build.py [--force]

Output: <pkg>/_lib/libwsr.so (git-ignored, travels to the GPU box with the repo snapshot).
"""
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
OUT_DIR = os.path.join(PKG, "_lib")
LIB = os.path.join(OUT_DIR, "libwsr.so")
SOURCES = ["common.cu", "elementwise.cu", "simt.cu", "fd.cu", "gemm_tc.cu", "attn_tc.cu", "attn_small_tc.cu", "head.cu", "backward.cu", "wgrad_tc.cu", "edge.cu", "pretrain.cu", "ensemble.cu", "spectra.cu"]
HEADERS = ["common.cuh", "tc_common.cuh", "philox.cuh", os.path.join("..", "..", "include", "wsr.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--use_fast_math",
              "-Xcompiler", "-fPIC"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _digest():
    h = hashlib.sha256()
    for f in SOURCES + HEADERS + ["build.py"]:
        with open(os.path.join(HERE, f), "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=True):
    os.makedirs(OUT_DIR, exist_ok=True)
    stamp = os.path.join(OUT_DIR, "libwsr.sha256")
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read().strip() == dig:
        return LIB
    nvcc = _nvcc()
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(OUT_DIR, src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc] + NVCC_FLAGS + ["-c", os.path.join(HERE, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError("nvcc failed on %s:\n%s" % (src, out))
        if verbose and out.strip():
            print(out)
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-cudart", "static"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout)
    with open(stamp, "w") as fh:
        fh.write(dig)
    if verbose:
        print("built", LIB)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv)

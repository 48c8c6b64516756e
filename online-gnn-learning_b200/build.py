"""Build libogl_b200.so in-tree with nvcc for sm_100a (no torch headers, plain C ABI).

    python online-gnn-learning_b200/build.py [--force]
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "csrc", "_obj")
LIB = os.path.join(HERE, "libogl_b200.so")
SOURCES = ["common.cu", "graph.cu", "sample.cu", "replay.cu", "gemm_simt.cu", "gemm_tc.cu", "sage_kernels.cu", "peer.cu", "infer.cu", "full_infer.cu", "plan.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
         "-Xcompiler", "-fvisibility=hidden", "-Xptxas", "-v"]


def _newer(target, deps):
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(d) <= t for d in deps)


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(HERE, "..", "include", "ogl_b200.h"))

    def compile_one(src):
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src.replace(".cu", ".o"))
        if not force and _newer(o, [s] + headers):
            return o, ""
        r = subprocess.run([NVCC] + FLAGS + ["-c", s, "-o", o], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (src, r.stderr))
        return o, r.stderr

    with ThreadPoolExecutor(max_workers=8) as ex:
        results = list(ex.map(compile_one, SOURCES))
    objs = [o for o, _ in results]
    if verbose:
        for _, log in results:
            sys.stderr.write(log)
    if force or not _newer(LIB, objs):
        r = subprocess.run([NVCC, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"],
                           capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n" + r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))

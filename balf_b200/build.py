"""Build ``balf_b200/libbalf_b200.so`` in-tree with nvcc for sm_100a (no JIT cache, no torch
extension machinery: the library is a plain C-ABI shared object, see include/balf_b200.h)."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
OBJ = os.environ.get("BALF_OBJ_DIR") or os.path.join(ROOT, "build", "obj")
LIB = os.environ.get("BALF_LIB_OUT") or os.path.join(PKG, "libbalf_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O3", "-lineinfo",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"] + os.environ.get("NVCC_FLAGS", "").split()


# per-source flags: the float64 metric kernels follow the reference's unfused Python / NumPy arithmetic
EXTRA = {"metrics.cu": ["-fmad=false"], "homography.cu": ["-fmad=false"], "fundamental.cu": ["-fmad=false"]}


def sources():
    return sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(ROOT, "include", "balf_b200.h"))
    jobs = []
    for src in sources():
        obj = os.path.join(OBJ, src[:-3] + ".o")
        if force or _stale(obj, [os.path.join(CSRC, src)] + headers):
            jobs.append([NVCC] + FLAGS + EXTRA.get(src, []) + (["-Xptxas", "-v"] if verbose else []) +
                        ["-c", os.path.join(CSRC, src), "-o", obj])

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed: %s\n%s\n%s" % (" ".join(cmd), r.stdout, r.stderr))
        return r.stderr

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        logs = list(ex.map(run, jobs))
    if verbose:
        sys.stderr.write("".join(logs))
    objs = [os.path.join(OBJ, s[:-3] + ".o") for s in sources()]
    if force or jobs or _stale(LIB, objs):
        run([NVCC, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a",
                                                   "-Xcompiler", "-fPIC", "-ldl"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))

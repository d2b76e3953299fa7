"""Build libalabi_b200.so (sm_100a only) in-tree with nvcc.

    python -m alabi_b200.build [--force]

The shared library is written next to this file so that it travels with the
repo snapshot to the GPU box; objects go to build/ (git-ignored).
"""
import concurrent.futures
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(ROOT, "build", "obj")
LIB = os.path.join(HERE, "libalabi_b200.so")
SOURCES = ["api.cu", "cov.cu", "chol.cu", "chol_dataflow.cu", "trsv_dataflow.cu", "append.cu", "grad.cu", "predict.cu", "ensemble.cu", "ensemble_k0.cu", "ensemble_k1.cu", "ensemble_k2.cu", "ensemble_k3.cu", "nested.cu", "cv_batch.cu", "mvn.cu", "nccl_helpers.cu", "peak.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC", "-I", os.path.join(ROOT, "include"), "-I", CSRC]


def _deps():
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(ROOT, "include", "alabi_b200.h"))
    return max(os.path.getmtime(h) for h in hdrs)


def _compile(src):
    obj = os.path.join(OBJ, src.replace(".cu", ".o"))
    path = os.path.join(CSRC, src)
    if os.path.exists(obj) and os.path.getmtime(obj) > max(os.path.getmtime(path), _deps()):
        return obj, ""
    cmd = [NVCC] + FLAGS + ["-Xptxas", "-v", "-c", path, "-o", obj]
    p = subprocess.run(cmd, capture_output=True, text=True)
    if p.returncode != 0:
        raise RuntimeError(f"nvcc failed for {src}:\n{p.stdout}\n{p.stderr}")
    return obj, p.stderr


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    if force:
        for f in os.listdir(OBJ):
            os.remove(os.path.join(OBJ, f))
    with concurrent.futures.ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        results = list(ex.map(_compile, SOURCES))
    objs = [r[0] for r in results]
    log = "".join(r[1] for r in results)
    if verbose:
        print(log)
    if any("bytes spill stores" in ln and not ln.strip().startswith("0 bytes stack frame, 0 bytes spill stores")
           for ln in log.splitlines() if "spill" in ln):
        print("warning: register spills reported by ptxas", file=sys.stderr)
    if (not os.path.exists(LIB)) or any(os.path.getmtime(o) > os.path.getmtime(LIB) for o in objs):
        cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-ldl"]
        p = subprocess.run(cmd, capture_output=True, text=True)
        if p.returncode != 0:
            raise RuntimeError(f"link failed:\n{p.stdout}\n{p.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))

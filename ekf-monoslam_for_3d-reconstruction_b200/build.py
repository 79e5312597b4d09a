"""Builds libekf_b200.so (the CUDA kernels + C ABI) in-tree with nvcc for sm_100a.

nvcc cross-compiles without a GPU, so this runs in the CPU container as the "does it build" check
and the resulting .so travels to the GPU box with the repo snapshot.
"""
import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libekf_b200.so")
SOURCES = ["ekf_api.cu", "ekf_predict.cu", "ekf_match.cu", "ekf_update.cu", "ekf_gemm.cu", "ekf_batch.cu", "ekf_batch_detect.cu", "ekf_dist.cu", "ekf_detect.cu", "ekf_export.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "--fmad=false", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "-diag-suppress", "550"]


def _nvcc():
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found: the product cannot be built (there is no CPU fallback)")


def _stamp():
    hsh = hashlib.sha256()
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for name in sorted(os.listdir(root)):
            if name.endswith((".cu", ".cuh", ".h")):
                with open(os.path.join(root, name), "rb") as f:
                    hsh.update(name.encode()); hsh.update(f.read())
    hsh.update(" ".join(NVCC_FLAGS).encode())
    return hsh.hexdigest()


def build(force=False, verbose=False):
    """Compile every .cu for sm_100a and link libekf_b200.so.  No-op when sources are unchanged."""
    stamp_file = os.path.join(HERE, "build", "stamp")
    stamp = _stamp()
    if not force and os.path.exists(OUT) and os.path.exists(stamp_file) and open(stamp_file).read() == stamp:
        return OUT
    nvcc = _nvcc()
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]

    def one(src):
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
        return obj

    with ThreadPoolExecutor(max_workers=6) as ex:
        objs = list(ex.map(one, srcs))
    cmd = [nvcc, "-shared", "-o", OUT] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp_file, "w") as f:
        f.write(stamp)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))

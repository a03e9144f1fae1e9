"""Builds libtnn_b200.so (sm_100a only) in-tree with nvcc.

    python tinynn-autograd_b200/build.py [--force]

The shared library carries every CUDA kernel and the C ABI declared in include/tnn_b200.h.
Objects are rebuilt only when their source (or a shared header) is newer.
"""
import concurrent.futures
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libtnn_b200.so")

SOURCES = ["runtime.cu", "elementwise.cu", "reduce.cu", "layout.cu", "gemm_simt.cu",
           "gemm_tc.cu", "gemm_f16.cu", "fused.cu", "mlp_fused.cu", "comm.cu", "conv.cu",
           "batchnorm.cu", "loss.cu"]
HEADERS = [os.path.join(CSRC, "common.cuh"), os.path.join(CSRC, "math.cuh"), os.path.join(CSRC, "tc_ptx.cuh"),
           os.path.join(ROOT, "include", "tnn_b200.h")]

# -split-compile 0: the per-kernel optimisation phase runs on all host cores (gemm_tc.cu instantiates
# the tcgen05 kernel 16 times: 5.5 min -> 1.5 min)
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-diag-suppress", "550", "-split-compile", "0"]
# bit-faithful elementwise arithmetic (numpy does not contract a*b+c): no FMA contraction outside
# the GEMMs
NO_FMAD = {"elementwise.cu", "fused.cu", "reduce.cu", "loss.cu"}


def _nvcc():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _compile(src, force):
    obj = os.path.join(OBJ, src.replace(".cu", ".o"))
    path = os.path.join(CSRC, src)
    if not force and not _stale(obj, [path] + HEADERS):
        return obj, False
    cmd = [_nvcc()] + NVCC_FLAGS + (["-fmad=false"] if src in NO_FMAD else []) + ["-c", path, "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout[-4000:], r.stderr[-4000:]))
    return obj, True


def build(force=False, verbose=True):
    os.makedirs(OBJ, exist_ok=True)
    with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        results = list(ex.map(lambda s: _compile(s, force), SOURCES))
    objs = [o for o, _ in results]
    rebuilt = any(changed for _, changed in results)
    if rebuilt or _stale(LIB, objs):
        # nvcc links the static CUDA runtime by default; NCCL and the driver API are bound at
        # run time (dlopen / cudaGetDriverEntryPoint), so there is no other link dependency
        cmd = [_nvcc(), "-shared", "-o", LIB] + objs + ["-ldl"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (r.stdout[-4000:], r.stderr[-4000:]))
        if verbose:
            print("built", LIB)
    elif verbose:
        print("up to date:", LIB)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv)

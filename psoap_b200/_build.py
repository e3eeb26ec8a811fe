"""Build psoap_b200/csrc/libpsoap_b200.so with nvcc for sm_100a (in-tree, so it travels to the GPU box)."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libpsoap_b200.so")
SOURCES = ["api.cu"]
HEADERS = ["common.cuh", "fill.cuh", "chain.cuh", "chol.cuh", "gemm.cuh", "orbit.cuh", "predict.cuh", "grad.cuh", os.path.join("..", "..", "include", "psoap_b200.h")]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-shared", "-Xptxas", "-v"]


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build_library(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    extra = os.environ.get("PSOAP_NVCC_EXTRA", "").split()
    cmd = [nvcc] + NVCC_FLAGS + extra + [os.path.join(CSRC, f) for f in SOURCES] + ["-o", LIB]
    res = subprocess.run(cmd, capture_output=True, text=True)
    log = res.stdout + res.stderr
    with open(os.path.join(CSRC, "build.log"), "w") as fh:
        fh.write(" ".join(cmd) + "\n" + log)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + log[-4000:])
    if verbose:
        print(log)
    return LIB


if __name__ == "__main__":
    print(build_library(force=True, verbose=True))

"""Builds libgbnf_b200.so (hand-written sm_100a CUDA + the C ABI of include/gbnf.h) in-tree with nvcc."""
import os
import shutil
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libgbnf_b200.so")
SOURCES = ["gbnf_api.cu"]
HEADERS = ["common.cuh", "pack.cuh", "mixture.cuh", "actnorm_init.cuh", "coupling_fp32.cuh", "coupling_tc.cuh", "coupling_tc2.cuh", "coupling_tc3.cuh", "coupling_tc4.cuh", "coupling_tc5.cuh", "train_bwd.cuh",
           "tc_ptx.cuh"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def _nvcc():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def is_stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.join(PKG_DIR, "..", "include", "gbnf.h")]
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every CUDA source for sm_100a.  Returns the path of the shared library."""
    if not force and not is_stale():
        return LIB_PATH
    cmd = [_nvcc()] + NVCC_FLAGS + [os.path.join(CSRC, s) for s in SOURCES] + ["-o", LIB_PATH]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force=True, verbose=True))

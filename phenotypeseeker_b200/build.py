"""Build libpskmer.so (hand-written sm_100a CUDA + C-ABI) in-tree with nvcc."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libpskmer.so")
SOURCES = ["ps_api.cu"]
HEADERS = ["ps_common.cuh", "ps_decode.cuh", "ps_decode_bits.h", "ps_extract.cuh", "ps_sort.cuh", "ps_paged.cuh", "ps_rows.cuh",
           "ps_test.cuh", "ps_chi2_reach.h", "ps_mash.cuh", "ps_mash_bits.h", "ps_count.cuh", os.path.join("..", "..", "include", "pskmer.h")]

NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-shared", "--use_fast_math=false"]


def _nvcc():
    for p in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if p and (os.path.sep not in p or os.path.exists(p)):
            return p
    return "nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    flags = [f for f in NVCC_FLAGS if not f.startswith("--use_fast_math")]
    cmd = [_nvcc()] + flags + (["-Xptxas", "-v"] if verbose else []) + \
          ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed building libpskmer.so")
    if verbose:
        sys.stderr.write(res.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose="-v" in sys.argv))

"""Builds libc3r_b200.so in-tree with nvcc for sm_100a (no JIT cache, no fallback)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libc3r_b200.so")
SOURCES = ["c3r_abi.cu", "bam_io.cpp", "decode.cpp", "fasta_io.cpp"]
HEADERS = ["scan.cuh", "pileup.cuh", "call.cuh", "vcf_row.cuh", "bam_rec.cuh", "bgzf.cuh", "nn_fp32.cuh", "nn_tc.cuh", "nn_lstm2f.cuh", "nn_sched.h", "tc_ptx.cuh", os.path.join("..", "..", "include", "c3r_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared", "-lcuda", "-lz", "-lpthread"]


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + SOURCES
    out = subprocess.run(cmd, cwd=CSRC, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if out.returncode != 0:
        sys.stderr.write(out.stdout)
        raise RuntimeError("nvcc failed building libc3r_b200.so")
    if verbose:
        print(out.stdout)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))

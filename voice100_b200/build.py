"""Build libv100.so in-tree with nvcc for sm_100a (no JIT cache, no torch headers).

    python -m voice100_b200.build [--force]

The shared library is plain C ABI (include/v100.h) with the CUDA runtime linked statically, so it
loads on a machine without a GPU (symbol checks) and travels to the GPU box inside the repo snapshot.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libv100.so")
SOURCES = ["api.cu", "conv_gemm.cu", "dwconv.cu", "logmel.cu", "misc.cu", "seq.cu", "lstm.cu", "tts_align.cu",
           "world.cu", "resample.cu", "world_analysis.cu", "ctc_eval.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "--compiler-options", "-fPIC", "-shared"]


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "v100.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + SOURCES
    r = subprocess.run(cmd, cwd=CSRC, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout)
    if verbose:
        print(r.stdout)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))

"""Build liblirec_b200.so in-tree with nvcc for sm_100a (no torch, no pybind inside the .so).

Usage: python -m lirec_b200.build [--force]
The shared library lands next to this file so it travels to the GPU box with the repo
snapshot (it is git-ignored, not gpurun-ignored).
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "liblirec_b200.so")
STAMP = os.path.join(HERE, ".liblirec_b200.stamp")
SOURCES = ["abi.cu", "gemm_tcgen05.cu", "rows.cu", "softpool.cu", "loss.cu", "model.cu", "dp.cu", "collate.cu"]
NVCC_FLAGS = [
    "-std=c++17", "-O3", "-lineinfo",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=default",
    "--shared",
]
# Extra -D flags for instrumented builds (tools/build_variants.sh): LIREC_NVCC_DEFINES="-DLIREC_GEMM_TRACE=1"
NVCC_FLAGS += [f for f in os.environ.get("LIREC_NVCC_DEFINES", "").split() if f.startswith("-D")]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _digest():
    h = hashlib.sha256()
    root = os.path.dirname(HERE)
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))]
    files.append(os.path.join(root, "include", "lirec_b200.h"))
    for path in files:
        with open(path, "rb") as f:
            h.update(path.encode())
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Compile csrc/*.cu into liblirec_b200.so if sources changed. Returns the library path."""
    digest = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(STAMP):
        with open(STAMP) as f:
            if f.read().strip() == digest:
                return LIB
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    cmd = [_nvcc()] + NVCC_FLAGS + ["-o", LIB] + srcs
    if verbose:
        print(" ".join(cmd), file=sys.stderr)
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n%s\n%s" % (res.stdout, res.stderr))
    with open(STAMP, "w") as f:
        f.write(digest)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))

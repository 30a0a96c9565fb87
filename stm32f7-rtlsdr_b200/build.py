"""Build libb200sdr.so (hand-written CUDA, sm_100a only) in-tree with nvcc.

The shared library is the product: a plain C ABI (include/b200sdr.h).  It is built next to this
file so it travels with the repo snapshot to the GPU box; there is no JIT and no CPU fallback.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libb200sdr.so")
SOURCES = [os.path.join(CSRC, "api.cu"), os.path.join(CSRC, "frontend.cpp")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "--shared", "-Xcompiler", "-fPIC,-fvisibility=hidden,-O2",
    "-Xptxas", "-v",
    "-diag-suppress", "550",
]


def _newest_source_mtime():
    newest = 0.0
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for dirpath, _, files in os.walk(root):
            for f in files:
                newest = max(newest, os.path.getmtime(os.path.join(dirpath, f)))
    return newest


def build(force=False, verbose=False):
    if not force and os.path.exists(OUT) and os.path.getmtime(OUT) >= _newest_source_mtime():
        return OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + ["-o", OUT] + SOURCES
    res = subprocess.run(cmd, capture_output=True, text=True)
    log = res.stdout + res.stderr
    with open(os.path.join(HERE, "build.log"), "w") as fh:
        fh.write(" ".join(cmd) + "\n" + log)
    if res.returncode != 0:
        sys.stderr.write(log)
        raise RuntimeError("nvcc failed building libb200sdr.so")
    if verbose:
        print(log)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))

"""Build ``libhsv.so`` in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m megatts2_hierspeechpp_b200.build [--force]
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(_HERE), "include")
OUT = os.path.join(_HERE, "libhsv.so")
SOURCES = ["common.cu", "act1d.cu", "act1d_mma.cu", "conv_direct.cu", "conv_umma.cu", "pcm.cu", "sinegen.cu", "frame_ops.cu", "mha_mma.cu", "noise.cu", "sr_stream.cu", "resample.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.isfile(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "hsv.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return OUT
    cmd = [_nvcc(), *NVCC_FLAGS, "-I", INCLUDE, "-I", CSRC, *[os.path.join(CSRC, s) for s in SOURCES], "-o", OUT]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
        print(" ".join(cmd))
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed:\n{r.stdout}\n{r.stderr}")
    if verbose:
        print(r.stderr)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))

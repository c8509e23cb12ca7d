"""Build recipe for libwca_b200.so: nvcc, sm_100a only, in-tree output.

The shared library is plain CUDA runtime + extern "C" (include/wca_b200.h); it does not
link against torch.  `python -m whisper_char_alignment_b200.build` rebuilds it.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libwca_b200.so")
SOURCES = ["cabi.cu", "capture_simt.cu", "capture_tc.cu", "enc_attn.cu", "decode_attn.cu", "layernorm.cu", "medfilt_softmax.cu", "scores.cu", "token_probs.cu", "dtw.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "--shared", "-Xcompiler", "-fPIC",
    "-Xcompiler", "-fvisibility=hidden",
    # bit-exact DTW and fp32 parity: no fast-math, no implicit FMA contraction
    "--fmad=false", "--ftz=false", "--prec-div=true", "--prec-sqrt=true",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the sm_100a extension cannot be built")


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(PKG_DIR, "..", "include", "wca_b200.h"))
    return any(os.path.getmtime(d) > built for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB_PATH
    cmd = [_nvcc(), *NVCC_FLAGS]
    if verbose:
        cmd += ["-Xptxas", "-v"]
    cmd += [os.path.join(CSRC, s) for s in SOURCES] + ["-o", LIB_PATH]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + proc.stdout + proc.stderr)
    if verbose:
        print(proc.stdout + proc.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))

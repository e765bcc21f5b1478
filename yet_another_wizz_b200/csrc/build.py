"""Build libyawb.so in-tree with nvcc for sm_100a (no torch needed).

    python yet_another_wizz_b200/csrc/build.py [--force]
"""

from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
SOURCES = ["yawb_api.cu", "yawb_alloc.cu", "yawb_index.cu", "yawb_count.cu", "yawb_kmeans.cu"]
HEADERS = ["yawb_internal.cuh", "yawb_count_stream.cuh", os.path.join(ROOT, "include", "yawb.h")]
OUT = os.environ.get("YAWB_BUILD_OUT") or os.path.join(HERE, "libyawb.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
    "-Xptxas", "-v",
    "--fmad=true",  # the exact FP64 path uses __dmul_rn/__dadd_rn intrinsics, never contracted
    "-I", os.path.join(ROOT, "include"),
    "-I", HERE,
]


def needs_build() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(HERE, s) for s in SOURCES] + [h if os.path.isabs(h) else os.path.join(HERE, h) for h in HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return OUT
    extra = os.environ.get("YAWB_NVCC_EXTRA", "").split()
    cmd = [NVCC, *FLAGS, *extra, "-o", OUT, *[os.path.join(HERE, s) for s in SOURCES]]
    res = subprocess.run(cmd, capture_output=True, text=True)
    log = os.path.join(HERE, "build.log")
    with open(log, "w") as f:
        f.write(" ".join(cmd) + "\n" + res.stdout + res.stderr)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError(f"nvcc failed (see {log})")
    if verbose:
        print(res.stderr)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))

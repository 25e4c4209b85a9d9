"""In-tree build of libmodin_b200.so (sm_100a only) with plain nvcc.

``python -m modin_b200.build`` or ``__graft_entry__.build()``.  The shared library lands in
``modin_b200/_native/`` (git-ignored, like the build stamp next to it).  There is a
single code target -- ``-gencode arch=compute_100a,code=sm_100a`` -- and no fallback build.
"""

from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_native")
LIB_PATH = os.path.join(OUT_DIR, "libmodin_b200.so")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")

NVCC_FLAGS = [
    "-gencode",
    "arch=compute_100a,code=sm_100a",
    "-O3",
    "-std=c++17",
    "-lineinfo",
    "-Xcompiler",
    "-fPIC",
    "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libmodin_b200 cannot be built (there is no non-CUDA build)")


def sources() -> list[str]:
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def _digest() -> str:
    h = hashlib.sha256()
    files = sources() + sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh"))
    files.append(os.path.join(INCLUDE, "modin_b200.h"))
    for f in files:  # names relative to the checkout: the same tree gives the same stamp wherever it lives
        h.update(os.path.relpath(f, os.path.dirname(HERE)).encode())
        with open(f, "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu under csrc/ and link libmodin_b200.so; returns its path."""
    os.makedirs(OUT_DIR, exist_ok=True)
    stamp = os.path.join(OUT_DIR, "build.sha256")
    digest = _digest()
    if not force and os.path.exists(LIB_PATH) and os.path.exists(stamp):
        with open(stamp) as fh:
            if fh.read().strip() == digest:
                return LIB_PATH
    nvcc = _nvcc()
    objs = []

    def compile_one(src: str) -> str:
        obj = os.path.join(OUT_DIR, os.path.basename(src)[:-3] + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-I", INCLUDE, "-c", src, "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas")
            cmd.insert(2, "-v")
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{res.stdout}\n{res.stderr}")
        if verbose:
            sys.stderr.write(res.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        objs = list(ex.map(compile_one, sources()))
    link = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB_PATH, *objs, "-ldl"]
    res = subprocess.run(link, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"link failed:\n{res.stdout}\n{res.stderr}")
    with open(stamp, "w") as fh:
        fh.write(digest)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))

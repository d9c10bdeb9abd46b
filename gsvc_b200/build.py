"""In-tree build of libgsvc_rast.so with nvcc for sm_100a (no torch headers, no JIT cache).

The built library sits next to this file (git-ignored, but it travels to the GPU box with the
repo snapshot).  `python -m gsvc_b200.build` or `__graft_entry__.build()` runs it.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ_DIR = os.path.join(HERE, "_obj")
LIB_PATH = os.path.join(HERE, "libgsvc_rast.so")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
          "-Xptxas", "-v"]
# preprocess.cu must round every product/sum separately (bit-exact radii / tile rects / depth keys)
SOURCES = {
    "preprocess.cu": ["-fmad=false"],
    "binning.cu": [],
    "render.cu": [],
    "preprocess_bwd.cu": [],
    "epilogue.cu": [],
    "loss.cu": [],
    "quality.cu": [],
    "export.cu": [],
    "collective.cu": [],
    "api.cu": [],
}


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libgsvc_rast.so cannot be built (there is no CPU fallback)")


def _digest() -> str:
    h = hashlib.sha256()
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for name in sorted(os.listdir(root)):
            with open(os.path.join(root, name), "rb") as f:
                h.update(name.encode())
                h.update(f.read())
    h.update(repr((ARCH, COMMON, SOURCES)).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    stamp = os.path.join(OBJ_DIR, "digest.txt")
    digest = _digest()
    if not force and os.path.exists(LIB_PATH) and os.path.exists(stamp) and open(stamp).read() == digest:
        return LIB_PATH
    nvcc = _nvcc()
    os.makedirs(OBJ_DIR, exist_ok=True)
    objs = []
    log = []
    for src, extra in SOURCES.items():
        obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        cmd = [nvcc, *ARCH, *COMMON, *extra, "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log.append("$ " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            sys.stderr.write(log[-1])
            raise RuntimeError(f"nvcc failed on {src}")
        objs.append(obj)
    cmd = [nvcc, *ARCH, "-shared", "-o", LIB_PATH, *objs]
    r = subprocess.run(cmd, capture_output=True, text=True)
    log.append("$ " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if r.returncode != 0:
        sys.stderr.write(log[-1])
        raise RuntimeError("link failed")
    with open(os.path.join(OBJ_DIR, "build.log"), "w") as f:
        f.write("\n".join(log))
    with open(stamp, "w") as f:
        f.write(digest)
    if verbose:
        print("\n".join(log))
    return LIB_PATH


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
    print(LIB_PATH)

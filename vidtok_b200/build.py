"""In-tree build of libvidtok_b200.so (nvcc, sm_100a only).  No JIT cache: the .so sits next to this file so it
travels to the GPU box with the repo snapshot."""
from __future__ import annotations

import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libvidtok_b200.so")
SOURCES = ["conv_simt.cu", "conv_tc.cu", "conv_stem.cu", "tblock_tc.cu", "elementwise.cu", "model.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def _newest(paths) -> float:
    return max(os.path.getmtime(p) for p in paths)


def _inputs():
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "vidtok_b200.h"))
    return [os.path.join(CSRC, s) for s in SOURCES], headers


def is_stale() -> bool:
    """True when the in-tree library is missing or older than a source or header it is built from.  Writes nothing."""
    srcs, headers = _inputs()
    return not os.path.exists(LIB) or os.path.getmtime(LIB) < _newest(srcs + headers)


def build(force: bool = False, verbose: bool = False, out_dir: str | None = None) -> str:
    """Builds the library in the tree (or, with `out_dir`, the objects and the library in that directory) unless it is up
    to date; returns the library's path."""
    srcs, headers = _inputs()
    obj_dir = out_dir or OBJ
    lib = os.path.join(out_dir, os.path.basename(LIB)) if out_dir else LIB
    if not force and os.path.exists(lib) and os.path.getmtime(lib) >= _newest(srcs + headers):
        return lib
    os.makedirs(obj_dir, exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(obj_dir, os.path.basename(src).replace(".cu", ".o"))
        if not force and os.path.exists(obj) and os.path.getmtime(obj) >= _newest([src] + headers):
            return obj
        cmd = [nvcc] + NVCC_FLAGS + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose and r.stderr:
            print(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(srcs)) as ex:
        objs = list(ex.map(compile_one, srcs))
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib] + objs
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return lib


if __name__ == "__main__":
    print(build(force="--force" in os.sys.argv, verbose=True))

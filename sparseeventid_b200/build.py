"""In-tree build of libscn_b200.so (hand-written CUDA for sm_100a, C ABI in include/scn_b200.h).

``python -m sparseeventid_b200.build`` builds it and the thin PyTorch C++ layer (build_torch_ext below); ``build()``
builds the library alone.  nvcc cross-compiles without a GPU.
The .so stays in the tree (git-ignored) so it travels to the GPU box with the snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
TAG = os.environ.get("SCN_B200_BUILD_TAG", "")          # e.g. "dbg" with SCN_B200_NVCC_FLAGS=-DSCN_TC_TIMELINE: a second library
OBJ = os.path.join(HERE, "build" + ("_" + TAG if TAG else ""))
LIB_DIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIB_DIR, "libscn_b200" + ("_" + TAG if TAG else "") + ".so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Wno-deprecated-declarations",
         "--expt-relaxed-constexpr"] + os.environ.get("SCN_B200_NVCC_FLAGS", "").split()   # e.g. -DSCN_TC_TIMELINE


def _sources():
    return sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))


def _headers_mtime():
    m = 0.0
    for d in (CSRC, os.path.join(os.path.dirname(HERE), "include")):
        for f in os.listdir(d):
            if f.endswith((".cuh", ".h")):
                m = max(m, os.path.getmtime(os.path.join(d, f)))
    return m


def _compile(src, verbose):
    obj = os.path.join(OBJ, src[:-3] + ".o")
    spath = os.path.join(CSRC, src)
    if os.path.exists(obj) and os.path.getmtime(obj) >= max(os.path.getmtime(spath), _headers_mtime()):
        return obj, False
    cmd = [NVCC] + ARCH + FLAGS + ["-c", spath, "-o", obj]
    if verbose:
        print(" ".join(cmd), flush=True)
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
    return obj, True


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(LIB_DIR, exist_ok=True)
    if force:
        for f in os.listdir(OBJ):
            os.remove(os.path.join(OBJ, f))
    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        results = list(ex.map(lambda s: _compile(s, verbose), _sources()))
    objs = [o for o, _ in results]
    changed = any(c for _, c in results)
    if changed or not os.path.exists(LIB):
        cmd = [NVCC] + ARCH + ["-shared", "-Xlinker", "-soname=libscn_b200.so", "-o", LIB] + objs
        if verbose:
            print(" ".join(cmd), flush=True)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


TORCH_EXT_NAME = "scn_b200_torch"
TORCH_EXT_DIR = os.path.join(HERE, "build_torch")
TORCH_EXT_SO = os.path.join(TORCH_EXT_DIR, TORCH_EXT_NAME + ".so")


def build_torch_ext(verbose: bool = False) -> str:
    """In-tree build of the thin PyTorch C++ layer (csrc_torch/scn_torch.cpp -> build_torch/scn_b200_torch.so).
    Host C++ only: the kernels stay in libscn_b200.so, which the loader (scn/_ext.py) maps first."""
    import ctypes

    from torch.utils import cpp_extension
    # the extension NEEDs libscn_b200.so by soname: have it loaded (globally) before the import at the end of load()
    ctypes.CDLL(build(), mode=ctypes.RTLD_GLOBAL)
    os.makedirs(TORCH_EXT_DIR, exist_ok=True)
    cpp_extension.load(
        name=TORCH_EXT_NAME, sources=[os.path.join(HERE, "csrc_torch", "scn_torch.cpp")],
        extra_cflags=["-O2", "-std=c++17"], extra_include_paths=["/usr/local/cuda/include"],
        extra_ldflags=[f"-L{LIB_DIR}", "-lscn_b200", "-L/usr/local/cuda/lib64", "-lcudart"],
        build_directory=TORCH_EXT_DIR, verbose=verbose, is_python_module=True, with_cuda=True)
    return TORCH_EXT_SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
    print(build_torch_ext(verbose=True))

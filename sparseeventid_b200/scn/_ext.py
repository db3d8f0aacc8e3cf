"""Loader of the thin PyTorch C++ layer (build_torch/scn_b200_torch.so, built in-tree by
``python -m sparseeventid_b200.build`` / ``__graft_entry__.build()``).

It holds the autograd functions of the hot modules in C++ (csrc_torch/scn_torch.cpp) so a module forward/backward
costs one native call.  Like libscn_b200.so (_lib.load) it is required: if it is missing or does not load, the first
module that needs it raises.  It is loaded on first use, so importing the package, building networks and loading
checkpoints need neither library.
"""
from __future__ import annotations

import ctypes
import importlib.machinery
import importlib.util
import os

from .. import _lib
from ..build import TORCH_EXT_NAME, TORCH_EXT_SO

_mod = None


def get():
    """The extension module; raises RuntimeError if it is missing or cannot be loaded."""
    global _mod
    if _mod is not None:
        return _mod
    if not os.path.exists(TORCH_EXT_SO):
        raise RuntimeError(f"scn_b200_torch.so not found at {TORCH_EXT_SO}: build it with "
                           "`python -m sparseeventid_b200.build` (there is no Python fallback for the hot modules)")
    import torch  # noqa: F401  (libtorch must be mapped before the extension)
    _lib.load()
    try:
        ctypes.CDLL(_lib.LIB_PATH, mode=ctypes.RTLD_GLOBAL)   # resolves the extension's NEEDED libscn_b200.so
        loader = importlib.machinery.ExtensionFileLoader(TORCH_EXT_NAME, TORCH_EXT_SO)
        spec = importlib.util.spec_from_loader(TORCH_EXT_NAME, loader)
        mod = importlib.util.module_from_spec(spec)
        loader.exec_module(mod)
    except (ImportError, OSError) as e:       # e.g. built against another torch
        raise RuntimeError(f"{TORCH_EXT_SO} could not be loaded ({e}): rebuild it with "
                           "`python -m sparseeventid_b200.build`") from e
    _mod = mod
    return mod

"""Numerics mode of the sparse-convolution path.

The DEFAULT is "fp32": SparseConvNet computes in fp32, so unmodified reference code that imports this package gets the
reference's numerics (whole-network parity within 2e-3 of the float64 oracle, tests/test_bench_scale_parity.py).
The tensor-core modes are an explicit opt-in -- `scn.set_precision("bf16")` or SCN_B200_PRECISION=bf16 -- which is
what bench.py and BASELINE.json config 3 ("bf16 tensor-core convs") select.

  "fp32"  : fp32 features, exact fp32 FMA convolutions (parity mode; SCN itself is fp32,
            SURVEY.md App. C).
  "mixed" : fp32 features in HBM, bf16 tensor-core operands, fp32 accumulate.
  "tf32"  : fp32 features in HBM, TF32 operands (10-bit mantissa) on the tcgen05 tensor cores, fp32
            accumulate -- what PyTorch's dense fp32 convolutions use by default (cudnn.allow_tf32).
            Shapes outside the tcgen05 kernels keep the exact fp32 kernels; the one-channel stem runs
            its ~fp32-accurate hi/lo bf16 split.  BatchNorm, elementwise layers, parameters and
            gradients are exactly as in "fp32".
  "bf16"  : bf16 features in HBM, bf16 tensor-core operands, fp32 accumulate; BatchNorm
            statistics, parameters and parameter gradients stay fp32 (BASELINE.json config 3).
"""
from __future__ import annotations

import os

import torch

from .._lib import PREC_BF16, PREC_FP32, PREC_TF32

_MODES = ("fp32", "mixed", "tf32", "bf16")
_state = {"mode": os.environ.get("SCN_B200_PRECISION", "fp32"),
          "fusion": os.environ.get("SCN_B200_FUSION", "1") not in ("0", "false", "False")}
if _state["mode"] not in _MODES:
    raise ValueError(f"SCN_B200_PRECISION must be one of {_MODES}")


def set_precision(mode: str) -> None:
    if mode not in _MODES:
        raise ValueError(f"precision must be one of {_MODES}, got {mode!r}")
    _state["mode"] = mode


def get_precision() -> str:
    return _state["mode"]


def feature_dtype() -> torch.dtype:
    return torch.bfloat16 if _state["mode"] == "bf16" else torch.float32


def precision_code() -> int:
    return {"fp32": PREC_FP32, "tf32": PREC_TF32}.get(_state["mode"], PREC_BF16)


def set_fusion(flag: bool) -> None:
    """Cross-module fusion of BatchNormalization/AddTable with a following LeakyReLU/ReLU (one kernel instead of two)."""
    _state["fusion"] = bool(flag)


def fusion_enabled() -> bool:
    return _state["fusion"]

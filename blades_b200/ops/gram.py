"""Gram matrix ``G = [U;extra][U;extra]^T`` (K5 of SURVEY 2.7): tcgen05 split-K kernel
(csrc/cuda/gram_tcgen05.cu) with fp32 TMEM accumulation; returns float64 numpy ``[n, n]``."""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

__all__ = ["gram"]

import os

#: 'tf32' | 'tf32x3' (tcgen05 kernel) | 'fp32' (cuBLAS fp32 reference path); env BLADES_GRAM overrides
PRECISION = os.environ.get("BLADES_GRAM", "tf32x3")


def gram(data: torch.Tensor, extra: Optional[torch.Tensor] = None, precision: Optional[str] = None) -> np.ndarray:
    assert data.is_cuda
    precision = precision or PRECISION
    from . import _loader
    lib = _loader.cuda_lib()
    if precision != "fp32" and hasattr(lib, "bl_gram_tcgen05") and data.dtype == torch.float32 \
            and data.stride(1) == 1:
        from ._gram_impl import gram_pass, symmetrised
        n, d = data.shape
        r = gram_pass([(data.data_ptr(), data.stride(0), n)], d, 0, d, data.device, extra, precision == "tf32x3")
        if r is not None:
            return symmetrised(*r).double().cpu().numpy()
    full = data if extra is None else torch.cat([data, extra.reshape(-1, data.shape[1])], 0)
    full = torch.nan_to_num(full)
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        G = full @ full.T
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    return G.double().cpu().numpy()

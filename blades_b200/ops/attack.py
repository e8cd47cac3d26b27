"""Launchers for the on-device attacker kernels (csrc/cuda/attack.cu)."""
from __future__ import annotations

import ctypes as C
from typing import Sequence

import torch

from . import _loader, _structs

__all__ = ["fill_normal_", "attack_rows", "deviation", "KIND", "DEV_TYPE"]

#: kernel form of a virtual row: ALIE ``mean - p*std``, IPM ``-p*mean``, sign ``mean - p*sign(mean)``
KIND = {"alie": 1, "ipm": 2, "sign": 3}
#: deviation vector of the Min-Max / Min-Sum attacks
DEV_TYPE = {"unit_vec": 0, "std": 1, "sign": 2}

_counter = [0]


def fill_normal_(row: torch.Tensor, mean: float, std: float, seed: int = None, offset: int = None) -> torch.Tensor:
    """In-place N(mean, std) fill with the in-kernel Philox generator.  ``offset``: position in the Philox stream
    (in 128-bit blocks); default = a process-wide running counter."""
    assert row.is_cuda and row.dtype == torch.float32 and row.is_contiguous()
    lib = _loader.cuda_lib()
    if seed is None:
        seed = int(torch.initial_seed()) & 0xFFFFFFFFFFFFFFFF
    if offset is None:
        offset = _counter[0]
        _counter[0] += (row.numel() + 3) // 4
    lib.bl_fill_normal.argtypes = [C.c_void_p, C.c_longlong, C.c_float, C.c_float, C.c_ulonglong,
                                   C.c_ulonglong, C.c_void_p]
    _loader.check(lib.bl_fill_normal(row.data_ptr(), row.numel(), float(mean), float(std), seed, offset,
                                     _loader.stream_ptr(row.device)), "fill_normal")
    _loader.count_launch()
    return row


def attack_rows(honest_rows: Sequence[int], out_rows: Sequence[int], kind: str, param: float,
                c0: int, c1: int, device=None, param_ptr: int = 0) -> None:
    """Write the ALIE / IPM / sign malicious value into every row of ``out_rows`` for coords [c0,c1).
    ``param_ptr``: address of a device float32 that replaces ``param`` (written by the scale solver)."""
    lib = _loader.cuda_lib()
    p = _structs.AttackRowParams()
    assert len(honest_rows) <= _structs.MAX_ROWS and len(out_rows) <= _structs.MAX_ROWS
    for i, r in enumerate(honest_rows):
        p.rows[i] = r
    for i, r in enumerate(out_rows):
        p.out[i] = r
    p.n_stat, p.kind, p.param = len(honest_rows), KIND[kind], float(param)
    p.c0, p.c1, p.n_out = c0, c1, len(out_rows)
    p.param_ptr = param_ptr or None
    _loader.check(lib.bl_attack_rows(C.byref(p), _loader.stream_ptr(device)), "attack_rows")
    _loader.count_launch()


def deviation(honest_rows: Sequence[int], dev_type: str, c0: int, c1: int, out: torch.Tensor, device=None) -> None:
    """``out[c]`` for c in [c0, c1): the Min-Max / Min-Sum deviation vector over the honest rows -- their mean
    (``unit_vec``), unbiased std (``std``) or sign of the mean (``sign``), with the statistics of ``attack_rows``."""
    assert out.is_cuda and out.dtype == torch.float32 and out.is_contiguous() and c1 <= out.numel()
    assert 1 <= len(honest_rows) <= _structs.MAX_ROWS
    lib = _loader.cuda_lib()
    p = _structs.DeviationParams()
    for i, r in enumerate(honest_rows):
        p.rows[i] = r
    p.n_stat, p.dev_type, p.c0, p.c1, p.q = len(honest_rows), DEV_TYPE[dev_type], c0, c1, out.data_ptr()
    _loader.check(lib.bl_agr_deviation(C.byref(p), _loader.stream_ptr(device)), "agr_deviation")
    _loader.count_launch()

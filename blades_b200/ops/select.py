"""Launchers for the coordinate-select kernels (csrc/cuda/coord_select.cu):
trimmed mean / median over client rows with optional fused ALIE/IPM/sign virtual rows and the
replicated-store + server-step epilogue.  Rows are given as raw device pointers so the same
launcher serves one dense matrix and NVLink peer shards."""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import torch

from . import _loader, _structs

__all__ = ["trimmed_mean", "median", "launch_select", "row_pointers", "make_epilogue"]

_KIND = {None: 0, "alie": 1, "ipm": 2, "sign": 3}


def row_pointers(data: torch.Tensor, rows: Optional[Sequence[int]] = None) -> List[int]:
    assert data.dim() == 2 and data.stride(1) == 1 and data.dtype == torch.float32
    base, step = data.data_ptr(), data.stride(0) * 4
    rows = range(data.shape[0]) if rows is None else rows
    return [base + r * step for r in rows]


def make_epilogue(outs: Sequence[int], thetas: Sequence[int] = (), theta_src: int = 0,
                  lr: float = 0.0, mc_out: int = 0, mc_theta: int = 0) -> _structs.Epilogue:
    """``mc_out`` / ``mc_theta``: NVLS multicast addresses of the replicated ``agg`` / ``theta`` (one ``multimem.st``
    per value instead of one store per peer pointer); 0 keeps the per-peer stores."""
    ep = _structs.Epilogue()
    ep.mc_out = mc_out or None
    ep.mc_theta = (mc_theta or None) if len(thetas) else None
    assert len(outs) <= _structs.MAX_PEERS and len(thetas) <= _structs.MAX_PEERS
    for i, p in enumerate(outs):
        ep.out[i] = p
    for i, p in enumerate(thetas):
        ep.theta[i] = p
    ep.theta_src = theta_src
    ep.lr = lr
    ep.n_out = len(outs)
    ep.n_theta = len(thetas)
    return ep


def launch_select(stat_rows: Sequence[int], other_rows: Sequence[int], n_virtual: int, kind: Optional[str],
                  param: float, mode: int, trim_b: int, c0: int, c1: int, ep: _structs.Epilogue,
                  device=None, param_ptr: int = 0) -> None:
    """``stat_rows`` (pointers) enter the attack statistics; ``other_rows`` are real rows that do not.
    ``param_ptr``: address of a device float32 the kernel reads instead of ``param`` (the scale solver's output)."""
    lib = _loader.cuda_lib()
    p, fn = _select_params(lib, stat_rows, other_rows, n_virtual, kind, param, mode, trim_b, c0, c1, ep)
    p.virt_param_ptr = (param_ptr or None) if n_virtual else None
    _loader.check(fn(C.byref(p), _loader.stream_ptr(device)), "coord_select")
    _loader.count_launch()


def kernel_choice(n_stat: int, n_other: int, n_virtual: int, kind: Optional[str], mode: int, trim_b: int) -> str:
    """Which kernel a launch with these row counts takes: ``"partition"`` (two half sorts + bitonic splits),
    ``"network"`` (full sorting network) or ``"large"`` (shared-memory bitonic sort, > 128 real rows).  Pure host
    logic (asks the library's own dispatch predicate, no CUDA call)."""
    lib = _loader.cuda_lib()
    n_real = n_stat + n_other
    if n_real > 128:
        return "large"
    p, _ = _select_params(lib, [0] * n_stat, [0] * n_other, n_virtual, kind, 0.5, mode, trim_b, 0, 1, _structs.Epilogue())
    return {1: "network", 2: "partition"}[lib.bl_coord_select_choice(C.byref(p))]


def _select_params(lib, stat_rows, other_rows, n_virtual, kind, param, mode, trim_b, c0, c1, ep):
    rows = list(stat_rows) + list(other_rows)
    n_real = len(rows)
    total = n_real + n_virtual
    if n_real <= 128:
        p = _structs.SelectParams()
        for i in range(128):          # unused slots alias row 0: the kernel loads them unpredicated
            p.rows[i] = rows[i] if i < n_real else rows[0]
        fn = lib.bl_coord_select
    else:
        assert total <= _structs.MAX_ROWS, f"at most {_structs.MAX_ROWS} rows"
        p = _structs.SelectLargeParams()
        for i, r in enumerate(rows):
            p.rows[i] = r
        fn = lib.bl_coord_select_large
    p.n_real, p.n_stat, p.n_virtual = n_real, len(stat_rows), n_virtual
    p.virt_kind, p.virt_param = _KIND[kind if n_virtual else None], float(param)
    p.mode, p.trim_b, p.c0, p.c1, p.ep = mode, trim_b, c0, c1, ep
    return p, fn


def _dense(data: torch.Tensor, mode: int, b: int, virtual) -> torch.Tensor:
    assert data.is_cuda and data.dtype == torch.float32 and data.stride(1) == 1
    n, d = data.shape
    out = torch.empty(d, device=data.device, dtype=torch.float32)
    if virtual is not None and virtual.count:
        honest, other = virtual.partition(n)
        launch_select(row_pointers(data, honest), row_pointers(data, other), virtual.count, virtual.kind,
                      virtual.param, mode, b, 0, d, make_epilogue([out.data_ptr()]), data.device,
                      param_ptr=virtual.param_ptr())
    else:
        launch_select(row_pointers(data), [], 0, None, 0.0, mode, b, 0, d,
                      make_epilogue([out.data_ptr()]), data.device)
    return out


def trimmed_mean(data: torch.Tensor, b: int, virtual=None) -> torch.Tensor:
    return _dense(data, 0, b, virtual)


def median(data: torch.Tensor, virtual=None) -> torch.Tensor:
    return _dense(data, 1, 0, virtual)

"""Launchers of the on-device Gram solvers (csrc/cuda/gram_solve.cu): Krum / Multi-Krum scoring, Weiszfeld iterations
and centered clipping run on the N x N Gram matrix where the tcgen05 pass left it and write the combine weights to
device memory -- no D2H copy, no host sync between the Gram pass and the weighted row-combine."""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import List, Optional, Tuple

import torch

from . import _loader

__all__ = ["DeviceGram", "enabled", "krum_weights", "weiszfeld_weights", "centered_clip_coeffs", "fltrust_weights",
           "autogm_weights", "agr_scale"]


def enabled() -> bool:
    """``BLADES_DEVICE_SOLVE=0`` sends the Gram matrix to the host solvers (numpy / C++) instead (A/B, debugging)."""
    return os.environ.get("BLADES_DEVICE_SOLVE", "1") != "0"


@dataclass
class DeviceGram:
    """The padded Gram accumulators as the kernel wrote them + the logical -> padded row map, all on the device."""
    G: torch.Tensor            # [tile_rows, ld] fp32
    idx: torch.Tensor          # [n] int32
    n: int

    def dense(self) -> torch.Tensor:
        """``[n, n]`` symmetrised fp32 (what the host path converts to float64)."""
        i = self.idx.long()
        g = self.G[i][:, i]
        return 0.5 * (g + g.T)


class KrumParams(C.Structure):
    _fields_ = [("G", C.c_void_p), ("idx", C.c_void_p), ("ld", C.c_int), ("n", C.c_int), ("n_out", C.c_int),
                ("f", C.c_int), ("m", C.c_int), ("squared_twice", C.c_int), ("value", C.c_float),
                ("scores", C.c_void_p), ("counter", C.c_void_p), ("w", C.c_void_p)]


class IterParams(C.Structure):
    _fields_ = [("G", C.c_void_p), ("idx", C.c_void_p), ("ld", C.c_int), ("n", C.c_int), ("kind", C.c_int),
                ("maxiter", C.c_int), ("compounding", C.c_int), ("eps", C.c_double), ("ftol", C.c_double),
                ("tau", C.c_double), ("alphas", C.c_void_p), ("gs", C.c_void_p), ("use_smem", C.c_int),
                ("w", C.c_void_p), ("iters", C.c_void_p), ("lamb", C.c_double), ("sort_by_index", C.c_int),
                ("pad_", C.c_int)]


class AgrScaleParams(C.Structure):
    _fields_ = [("G", C.c_void_p), ("idx", C.c_void_p), ("ld", C.c_int), ("honest", C.c_void_p), ("n_h", C.c_int),
                ("q_row", C.c_int), ("minsum", C.c_int), ("dev_type", C.c_int), ("gamma_init", C.c_double),
                ("tol", C.c_double), ("gamma", C.c_void_p), ("param", C.c_void_p)]


class TrustParams(C.Structure):
    _fields_ = [("G", C.c_void_p), ("idx", C.c_void_p), ("ld", C.c_int), ("n", C.c_int), ("trusted", C.c_int),
                ("eps", C.c_double), ("w", C.c_void_p)]


_SCRATCH = {}
_IDX = {}


def index_tensor(idx, device) -> torch.Tensor:
    """Device int32 tensor of a logical -> padded row list, cached per (device, list): the list is the same every
    round, and an H2D copy from pageable memory is not allowed while a CUDA graph is being captured."""
    key = (torch.device(device).index or 0, tuple(idx))
    t = _IDX.get(key)
    if t is None:
        if len(_IDX) > 64:
            _IDX.clear()
        t = _IDX[key] = torch.tensor(list(idx), dtype=torch.int32, device=device)
    return t


def _scratch(device) -> dict:
    key = torch.device(device).index or 0
    if key not in _SCRATCH:
        _SCRATCH[key] = {"scores": torch.zeros(512, dtype=torch.float64, device=device),
                         "counter": torch.zeros(1, dtype=torch.int32, device=device),
                         "gs": None}
    return _SCRATCH[key]


def _lib():
    lib = _loader.cuda_lib()
    assert lib.bl_sizeof_krum_params() == C.sizeof(KrumParams), (lib.bl_sizeof_krum_params(), C.sizeof(KrumParams))
    assert lib.bl_sizeof_iter_params() == C.sizeof(IterParams), (lib.bl_sizeof_iter_params(), C.sizeof(IterParams))
    return lib


def krum_weights(dg: DeviceGram, n: int, f: int, m: int, squared_twice: bool, value: float) -> torch.Tensor:
    """Weights of ``combine``: ``value`` on the ``m`` best-scoring of the first ``n`` rows, 0 elsewhere."""
    lib = _lib()
    dev = dg.G.device
    sc = _scratch(dev)
    w = torch.empty(dg.n, dtype=torch.float32, device=dev)
    p = KrumParams()
    p.G, p.idx, p.ld = dg.G.data_ptr(), dg.idx.data_ptr(), dg.G.stride(0)
    p.n, p.n_out, p.f, p.m = n, dg.n, f, m
    p.squared_twice, p.value = int(bool(squared_twice)), float(value)
    p.scores, p.counter, p.w = sc["scores"].data_ptr(), sc["counter"].data_ptr(), w.data_ptr()
    _loader.check(lib.bl_gram_krum(C.byref(p), _loader.stream_ptr(dev)), "gram_krum")
    _loader.count_launch()
    return w


def _iter(dg: DeviceGram, kind: int, maxiter: int, compounding: bool, eps: float, ftol: float, tau: float,
          alphas: Optional[torch.Tensor], lamb: float = 0.0, sort_by_index: bool = True
          ) -> Tuple[torch.Tensor, torch.Tensor]:
    lib = _lib()
    dev = dg.G.device
    sc = _scratch(dev)
    n = dg.n
    w = torch.empty(n, dtype=torch.float32, device=dev)
    iters = torch.zeros(1, dtype=torch.int32, device=dev)
    p = IterParams()
    p.G, p.idx, p.ld, p.n, p.kind = dg.G.data_ptr(), dg.idx.data_ptr(), dg.G.stride(0), n, kind
    p.maxiter, p.compounding = int(maxiter), int(bool(compounding))
    p.eps, p.ftol, p.tau = float(eps), float(ftol), float(tau)
    p.lamb, p.sort_by_index = float(lamb), int(bool(sort_by_index))
    p.alphas = alphas.data_ptr() if alphas is not None else None
    if n * n * 4 > 200 * 1024:
        if sc["gs"] is None or sc["gs"].numel() < n * n:
            sc["gs"] = torch.empty(512 * 512, dtype=torch.float32, device=dev)
        p.gs = sc["gs"].data_ptr()
    p.w, p.iters = w.data_ptr(), iters.data_ptr()
    _loader.check(lib.bl_gram_iter(C.byref(p), _loader.stream_ptr(dev)), "gram_iter")
    _loader.count_launch()
    return w, iters


def weiszfeld_weights(dg: DeviceGram, alphas, maxiter: int, eps: float, ftol: float, compounding: bool
                      ) -> Tuple[torch.Tensor, torch.Tensor]:
    """(weights [n] fp32 on the device, iterations taken as a 1-element int32 device tensor)."""
    a = None
    if alphas is not None:
        a = torch.as_tensor(alphas, dtype=torch.float32).to(dg.G.device).contiguous()
        assert a.numel() == dg.n
    return _iter(dg, 0, maxiter, compounding, eps, ftol, 0.0, a)


def autogm_weights(dg: DeviceGram, lamb: Optional[float], maxiter: int, eps: float, ftol: float, sort_by_index: bool,
                   compounding: bool) -> torch.Tensor:
    """AutoGM weights (Weiszfeld inside the water-filling loop), one launch; ``lamb`` defaults to the row count."""
    return _iter(dg, 2, maxiter, compounding, eps, ftol, 0.0, None, lamb=float(dg.n if lamb is None else lamb),
                 sort_by_index=sort_by_index)[0]


def centered_clip_coeffs(dg: DeviceGram, tau: float, n_iter: int) -> torch.Tensor:
    """Coefficients over ``[u_0 .. u_{n-2}, m_prev]`` (the last Gram row is the previous momentum)."""
    return _iter(dg, 1, n_iter, False, 0.0, 0.0, tau, None)[0]


def fltrust_weights(dg: DeviceGram, trusted: int, eps: float = 1e-6) -> torch.Tensor:
    """Trust-score weights of every row against row ``trusted`` (its own weight is 0)."""
    lib = _lib()
    assert lib.bl_sizeof_trust_params() == C.sizeof(TrustParams)
    dev = dg.G.device
    w = torch.empty(dg.n, dtype=torch.float32, device=dev)
    p = TrustParams()
    p.G, p.idx, p.ld, p.n, p.trusted = dg.G.data_ptr(), dg.idx.data_ptr(), dg.G.stride(0), dg.n, int(trusted)
    p.eps, p.w = float(eps), w.data_ptr()
    _loader.check(lib.bl_gram_fltrust(C.byref(p), _loader.stream_ptr(dev)), "gram_fltrust")
    _loader.count_launch()
    return w


def agr_scale(dg: DeviceGram, honest: torch.Tensor, q_row: int, minsum: bool, dev_type: str, gamma_init: float,
              tol: float) -> Tuple[torch.Tensor, torch.Tensor]:
    """Min-Max / Min-Sum scale search on the Gram matrix of ``[U; q]`` (``honest``: int32 device tensor of the honest
    logical rows; ``q_row``: logical row of q, -1 for ``unit_vec``).  Returns ``(gamma, param)``: a float64 and a
    float32 one-element device tensor, ``param`` being the parameter of the virtual row's kernel form."""
    from .attack import DEV_TYPE
    lib = _lib()
    assert lib.bl_sizeof_agr_scale_params() == C.sizeof(AgrScaleParams)
    dev = dg.G.device
    gamma = torch.empty(1, dtype=torch.float64, device=dev)
    param = torch.empty(1, dtype=torch.float32, device=dev)
    p = AgrScaleParams()
    p.G, p.idx, p.ld = dg.G.data_ptr(), dg.idx.data_ptr(), dg.G.stride(0)
    p.honest, p.n_h, p.q_row = honest.data_ptr(), honest.numel(), int(q_row)
    p.minsum, p.dev_type = int(bool(minsum)), DEV_TYPE[dev_type]
    p.gamma_init, p.tol = float(gamma_init), float(tol)
    p.gamma, p.param = gamma.data_ptr(), param.data_ptr()
    _loader.check(lib.bl_gram_agr_scale(C.byref(p), _loader.stream_ptr(dev)), "gram_agr_scale")
    _loader.count_launch()
    return gamma, param

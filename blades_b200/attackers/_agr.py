"""Shared core of the Min-Max and Min-Sum attacks (Shejwalkar & Houmansadr, "Manipulating the Byzantine: Optimizing
Model Poisoning Attacks and Defenses for Federated Learning", NDSS 2021) -- the two "AGR-agnostic" attacks, which need
no knowledge of the aggregator.

Every Byzantine client uploads ``m(g) = mu - g * p``: ``mu`` is the mean of the honest updates ``u_i`` and ``p`` a
deviation vector (``unit_vec``: ``mu / ||mu||``; ``std``: coordinate-wise unbiased std; ``sign``: ``sign(mu)``).  The
scale ``g`` is the largest that passes the attack's test on squared L2 distances over the honest clients:

* Min-Max: ``max_i ||m - u_i||^2 <= max_{i,j} ||u_i - u_j||^2``
* Min-Sum: ``sum_i ||m - u_i||^2 <= max_i sum_j ||u_i - u_j||^2``

found by the authors' bisection (``search``).  Three evaluations of it live here:

* ``direct_scale`` -- fp64 distances on the rows themselves: the attackers' callbacks and ``VirtualRows.value()``;
* ``gram_scale``   -- the same search on the Gram matrix of ``[U; q]`` (numpy, fp64): the host twin of the device
  solver ``gram_agr_scale_kernel`` (csrc/cuda/gram_solve.cu), used when the Gram stays on the host;
* the device solver itself, reached through ``parallel.matrix.resolve_scaled_rows``.
"""
from __future__ import annotations

from typing import Callable, Optional, Sequence, Tuple

import numpy as np
import torch

from ..client import ByzantineClient

__all__ = ["DEV_TYPES", "KINDS", "MAX_ITER", "KERNEL_FORM", "check_args", "search", "deviation", "direct_scale",
           "gram_scale", "ScaledDeviationClient"]

DEV_TYPES = ("unit_vec", "std", "sign")
KINDS = ("minmax", "minsum")
#: iteration cap of the Gram-domain search (host twin and device solver); the loop itself ends after about
#: log2(gamma_init / tol) + 2 steps
MAX_ITER = 128
#: the closed form the aggregation kernels evaluate for each deviation type: ``unit_vec`` is the IPM form
#: ``-param * mu`` with ``param = g / ||mu|| - 1``, ``std`` the ALIE form ``mu - g * std``, ``sign``
#: ``mu - g * sign(mu)``
KERNEL_FORM = {"unit_vec": "ipm", "std": "alie", "sign": "sign"}


def check_args(kind: str, dev_type: str, gamma_init: float, tol: float) -> None:
    if kind not in KINDS:
        raise ValueError(f"unknown attack kind {kind!r}; expected one of {KINDS}")
    if dev_type not in DEV_TYPES:
        raise ValueError(f"dev_type must be one of {DEV_TYPES}, got {dev_type!r}")
    if not gamma_init > 0:
        raise ValueError(f"gamma_init must be > 0, got {gamma_init!r}")
    if not tol > 0:
        raise ValueError(f"tol must be > 0, got {tol!r}")


def check_honest(n_h: int, dev_type: str) -> None:
    if n_h < 1 or (dev_type == "std" and n_h < 2):
        raise ValueError(f"dev_type={dev_type!r} needs at least {2 if dev_type == 'std' else 1} honest clients, "
                         f"got {n_h}")


def search(test: Callable[[float], bool], gamma_init: float, tol: float, max_iter: Optional[int] = None) -> float:
    """The authors' bisection: the largest tested scale that passed (0.0 when none did)."""
    gamma, step, ok = float(gamma_init), float(gamma_init), 0.0
    it = 0
    while abs(ok - gamma) > tol and (max_iter is None or it < max_iter):
        if test(gamma):
            ok = gamma
            gamma += step / 2
        else:
            gamma -= step / 2
        step /= 2
        it += 1
    return ok


def deviation(honest: torch.Tensor, dev_type: str) -> torch.Tensor:
    """``p`` for the rows ``honest`` (any float dtype; computed in that dtype)."""
    mu = honest.mean(0)
    if dev_type == "unit_vec":
        nrm = torch.linalg.vector_norm(mu)
        return mu / nrm if nrm > 0 else torch.zeros_like(mu)
    if dev_type == "std":
        return honest.std(0, unbiased=True)
    return torch.sign(mu)


def _sq_dists_to(rows: torch.Tensor, v: torch.Tensor, chunk: int = 16) -> torch.Tensor:
    """``||rows[i] - v||^2`` for every i, without an [n, d] temporary for large d."""
    return torch.cat([((rows[a:a + chunk] - v) ** 2).sum(1) for a in range(0, rows.shape[0], chunk)])


def direct_scale(honest: torch.Tensor, kind: str, dev_type: str, gamma_init: float, tol: float
                 ) -> Tuple[float, torch.Tensor]:
    """``(g, m(g))`` with every distance computed directly on the rows in fp64 (``honest``: ``[n_h, d]``, already
    ``nan_to_num``-ed).  ``m`` is float64."""
    check_args(kind, dev_type, gamma_init, tol)
    check_honest(honest.shape[0], dev_type)
    u = honest.double()
    mu = u.mean(0)
    p = deviation(u, dev_type)
    per_row = torch.stack([_sq_dists_to(u, u[i]) for i in range(u.shape[0])])       # [n_h, n_h]
    thr = float(per_row.max() if kind == "minmax" else per_row.sum(1).max())

    def test(g: float) -> bool:
        d = _sq_dists_to(u, mu - g * p)
        return float(d.max() if kind == "minmax" else d.sum()) <= thr
    g = search(test, gamma_init, tol)
    return g, mu - g * p


def gram_scale(G: np.ndarray, honest: Sequence[int], q_row: int, kind: str, dev_type: str, gamma_init: float,
               tol: float) -> Tuple[float, float]:
    """The search on the Gram matrix of ``[U; q]`` (``q_row``: its row of q, -1 for ``unit_vec``), statement for
    statement what ``gram_agr_scale_kernel`` computes.  Returns ``(g, param)``, ``param`` being the parameter of the
    virtual row's kernel form (``KERNEL_FORM``)."""
    check_args(kind, dev_type, gamma_init, tol)
    check_honest(len(honest), dev_type)
    G = np.asarray(G, dtype=np.float64)
    h = np.asarray(honest, dtype=np.int64)
    Gh = G[np.ix_(h, h)]
    gii = np.diag(Gh).copy()
    mui = Gh.mean(1)
    mumu = float(mui.mean())
    D = np.maximum(gii[:, None] + gii[None, :] - 2.0 * Gh, 0.0)
    thr = float(D.max() if kind == "minmax" else D.sum(1).max())
    nrm = 0.0
    if dev_type == "unit_vec":
        nrm = float(np.sqrt(max(mumu, 0.0)))
        up, mup, pp = (mui / nrm, nrm, 1.0) if nrm > 0 else (np.zeros_like(mui), 0.0, 0.0)
    else:
        up = G[h, q_row]
        mup = float(up.mean())
        pp = float(G[q_row, q_row])
    d0 = np.maximum(mumu - 2.0 * mui + gii, 0.0)
    a = mup - up

    def test(g: float) -> bool:
        d = np.maximum(d0 - 2.0 * g * a + g * g * pp, 0.0)
        return float(d.max() if kind == "minmax" else d.sum()) <= thr
    g = search(test, gamma_init, tol, MAX_ITER)
    if dev_type == "unit_vec":
        return g, (g / nrm - 1.0 if nrm > 0 else -1.0)
    return g, g


class ScaledDeviationClient(ByzantineClient):
    """Base of ``MinmaxClient`` / ``MinsumClient``: every such client uploads the same ``m(g)``.

    ``dev_type``: ``"unit_vec"`` (default), ``"std"`` or ``"sign"``; ``gamma_init``: first (and half the largest)
    scale tried; ``tol``: the search stops when the step falls below it.
    """
    kind = ""

    def __init__(self, dev_type: str = "unit_vec", gamma_init: float = 10.0, tol: float = 1e-5, *args, **kwargs):
        super().__init__(*args, **kwargs)
        check_args(self.kind, dev_type, gamma_init, tol)
        self.dev_type = dev_type
        self.gamma_init = float(gamma_init)
        self.tol = float(tol)
        self._gamma = None          # float, or a 1-element float64 device tensor written by the scale solver

    @property
    def gamma(self) -> Optional[float]:
        """The scale of the last round (``None`` before the first).  When the search ran on the device, reading it
        waits for that kernel."""
        g = self._gamma
        return float(g) if g is not None else None

    def _set_gamma(self, g) -> None:
        self._gamma = g

    def fused_spec(self):
        return {"kind": self.kind, "param": 0.0, "dev_type": self.dev_type, "gamma_init": self.gamma_init,
                "tol": self.tol}

    def omniscient_callback(self, simulator):
        honest = [c.get_update() for c in simulator.get_clients() if not c.is_byzantine()]
        stacked = torch.stack(honest, 0)
        g, m = direct_scale(stacked, self.kind, self.dev_type, self.gamma_init, self.tol)
        self._gamma = g
        self.save_update(m.to(stacked.dtype))

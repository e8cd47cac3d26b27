"""``UpdateMatrix``: the logical ``U[N, d]`` stack of client updates.

The reference materialises ``U`` on the driver CPU with ``torch.stack``
(/root/reference/src/blades/aggregators/mean.py:21-28) and every aggregator is
written against that dense tensor.  Here aggregators are written against a
small set of *matrix primitives* instead, so the same aggregator code runs on

* ``LocalMatrix``    -- one dense tensor (CPU oracle, or one GPU with our kernels)
* ``ShardedMatrix``  -- rows spread over G trainer shards in NVLink-addressable
  symmetric memory (``comm.symm``); primitives run as pull-mode fused kernels
  and ``U`` is never gathered on one device (SURVEY 5.8 / 7.2.1).

Primitives (everything the 11 reference aggregators need, SURVEY 2.7 K2-K6):

=================  =========================================================
``mean()``          column mean                                  (K2)
``combine(w)``      ``sum_i w_i U[i]``                            (K2)
``trimmed_mean(b)`` coordinate-wise trimmed mean                 (K3)
``median()``        coordinate-wise median (avg of middle two)   (K4)
``gram(extra)``     ``[U;extra][U;extra]^T`` as float64 ``[N+e,N+e]`` (K5)
``rows()``          dense ``[N,d]`` (gathers; escape hatch for custom aggs)
=================  =========================================================

*Virtual rows* (SURVEY 7.2.3): a ``VirtualRows`` spec replaces the first ``f``
rows by a coordinate-wise closed form of the honest rows (ALIE / IPM), so the
fused kernels never store f identical malicious rows.  Min-Max / Min-Sum rows are
such a closed form with a scale found by a search over pairwise distances; the
search runs on the Gram matrix of ``[U; q]`` before the first primitive
(``resolve_scaled_rows``).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Callable, Optional, Sequence

import numpy as np
import torch

__all__ = ["VirtualRows", "UpdateMatrix", "LocalMatrix", "as_matrix", "resolve_scaled_rows", "SCALED_KINDS"]

#: virtual-row kinds whose value needs a scale search over the whole vector (attackers/_agr.py)
SCALED_KINDS = ("minmax", "minsum")


@dataclass
class VirtualRows:
    """``count`` identical rows ``value(honest rows)`` replacing rows ``replaced``.

    kind='alie'  : value = mean - z * std_unbiased   (reference alieclient.py:32-36)
    kind='ipm'   : value = -eps * mean               (reference ipmclient.py:16)
    kind='sign'  : value = mean - param * sign(mean)
    kind='minmax' / 'minsum': value = mean - gamma * p, ``p`` given by ``dev_type`` and ``gamma`` found by the
                   Min-Max / Min-Sum search (attackers/_agr.py; ``param`` is unused)
    Honest rows = all rows whose index is not in ``byzantine`` (all Byzantine rows,
    not only the replaced ones, are excluded from the statistics).
    """
    kind: str
    param: float
    replaced: Sequence[int]
    byzantine: Sequence[int] = field(default_factory=list)
    dev_type: str = "unit_vec"
    gamma_init: float = 10.0
    tol: float = 1e-5
    #: float32 one-element device tensor the kernels read instead of ``param`` (left there by the scale solver)
    param_dev: Optional[torch.Tensor] = field(default=None, repr=False)
    #: minmax / minsum: called with the scale of every evaluation (a float, or a float64 one-element device tensor)
    report: Optional[Callable] = field(default=None, repr=False, compare=False)

    def __post_init__(self):
        if self.kind not in ("alie", "ipm", "sign") + SCALED_KINDS:
            raise ValueError(self.kind)
        if self.kind in SCALED_KINDS:
            from ..attackers import _agr
            _agr.check_args(self.kind, self.dev_type, self.gamma_init, self.tol)
        if not self.byzantine:
            self.byzantine = list(self.replaced)

    @property
    def count(self) -> int:
        return len(self.replaced)

    def param_ptr(self) -> int:
        return self.param_dev.data_ptr() if self.param_dev is not None else 0

    def partition(self, n: int):
        """``(honest, other)`` of ``n`` rows: the rows that enter the attack statistics (not Byzantine), and the
        Byzantine rows that are not replaced (real rows that enter no statistic)."""
        byz, rep = set(self.byzantine), set(self.replaced)
        return [i for i in range(n) if i not in byz], [i for i in range(n) if i in byz and i not in rep]

    def value(self, honest: torch.Tensor) -> torch.Tensor:
        if self.kind in SCALED_KINDS:
            from ..attackers import _agr
            gamma, m = _agr.direct_scale(honest, self.kind, self.dev_type, self.gamma_init, self.tol)
            if self.report is not None:
                self.report(gamma)
            return m.to(honest.dtype)
        param = self.param if self.param_dev is None else float(self.param_dev)
        mu = honest.mean(dim=0)
        if self.kind == "alie":
            return mu - param * honest.std(dim=0, unbiased=True)
        if self.kind == "sign":
            return mu - param * torch.sign(mu)
        return -param * mu


def resolve_scaled_rows(matrix: "UpdateMatrix") -> None:
    """Min-Max / Min-Sum virtual rows -> the closed form the kernels evaluate, before the first primitive reads them.

    The scale depends on every coordinate, so it is found once for the whole vector: the deviation pass writes
    ``q`` (std or sign(mean) of the honest rows; ``unit_vec`` needs no pass, ``mean . u_i`` is a row mean of the
    Gram), one Gram pass covers ``[U; q]`` and the scale solver turns it into the parameter of an ALIE (std), IPM
    (unit_vec) or sign form (``attackers._agr.KERNEL_FORM``), left in device memory.  When the Gram cannot stay on
    the device (CPU, fp32 Gram precision, solvers disabled) the same search runs on the host on ``gram()``.
    ``matrix.virtual`` is replaced by the resolved form; other kinds are left alone."""
    v = matrix.virtual
    if v is None or not v.count or v.kind not in SCALED_KINDS:
        return
    from ..attackers import _agr
    from ..ops import _gram_impl
    if matrix.window is not None:
        raise ValueError(f"{v.kind} virtual rows depend on every coordinate and cannot be aggregated window by window")
    n = matrix.n_rows
    honest, _ = v.partition(n)
    _agr.check_honest(len(honest), v.dev_type)
    use_q = v.dev_type != "unit_vec"
    blocks = matrix.gram_block_rows() + ([1] if use_q else [])
    padded = _gram_impl.padded_rows(blocks)
    if padded > _gram_impl.MAX_PADDED_ROWS or len(blocks) > _gram_impl.MAX_BLOCKS:
        raise ValueError(f"{v.kind} with dev_type={v.dev_type!r} needs one Gram pass over the {n} client rows"
                         f"{' plus the deviation row' if use_q else ''}: {padded} padded rows in {len(blocks)} blocks, "
                         f"but the Gram pass takes at most {_gram_impl.MAX_PADDED_ROWS} padded rows in "
                         f"{_gram_impl.MAX_BLOCKS} blocks")
    matrix.virtual = None                    # the Gram below is of the clients' own rows
    q = matrix.deviation_row(honest, v.dev_type) if use_q else None
    q_row = n if use_q else -1
    dg = matrix.gram_device(extra=q)
    form = _agr.KERNEL_FORM[v.dev_type]
    if dg is not None:
        from ..ops import gram_solve
        gamma, param = gram_solve.agr_scale(dg, gram_solve.index_tensor(honest, matrix.device), q_row,
                                            v.kind == "minsum", v.dev_type, v.gamma_init, v.tol)
        resolved = VirtualRows(form, 0.0, v.replaced, v.byzantine, param_dev=param)
    else:
        gamma, param = _agr.gram_scale(matrix.gram(extra=q), honest, q_row, v.kind, v.dev_type, v.gamma_init, v.tol)
        resolved = VirtualRows(form, param, v.replaced, v.byzantine)
    if v.report is not None:
        v.report(gamma)
    matrix.virtual = resolved


class UpdateMatrix:
    """Interface; see module docstring.

    The kernel path of the primitives is written once here, over a few hooks each matrix supplies: ``_ptrs(rows)``
    (row pointers for a kernel reading coordinates ``_cols()``), ``_pre()`` (before the first launch), ``_epilogue()``
    (where the result is stored), ``_finish()`` (after the final launch), ``_rows_written()`` (after the virtual rows
    are written into the rows), ``_gram_blocks()`` and ``_gram_pass(extra)``."""

    n_rows: int
    n_cols: int
    device: torch.device
    virtual: Optional[VirtualRows] = None
    #: False: the primitives are the pure-torch oracle (``LocalMatrix`` only)
    use_kernels = True
    #: (lr,) -> the final primitive also applies ``theta += lr * agg`` on every replica (K8 fusion)
    server_step = None
    step_applied = False
    #: pipelined aggregation (engine/round.py): this matrix object only covers coordinates ``[window[0], window[1])``
    #: -- chunk number ``chunk`` of the round, ``last_chunk`` closes it.  Coordinate-wise primitives (mean / combine,
    #: trimmed mean, median, virtual-row materialisation) honour it; ``out_buffer`` is the round's shared result vector.
    window = None
    chunk = 0
    last_chunk = True
    out_buffer = None

    def _cols(self):
        return (0, self.n_cols) if self.window is None else (int(self.window[0]), int(self.window[1]))

    # -- hooks ------------------------------------------------------------------
    def _ptrs(self, rows) -> list: raise NotImplementedError
    def _pre(self) -> None: pass
    def _epilogue(self): raise NotImplementedError      # -> (epilogue, result tensor)
    def _finish(self) -> None: pass
    def _rows_written(self) -> None: pass
    def _gram_blocks(self) -> list: raise NotImplementedError  # -> [(base_ptr, ld_floats, rows)] in row order

    def _gram_pass(self, extra: Optional[torch.Tensor]):
        """``ops._gram_impl.gram_pass`` over ``_gram_blocks()`` (+ ``extra``), or ``None`` without a kernel path."""
        return None

    # coordinate-wise -----------------------------------------------------------
    def mean(self) -> torch.Tensor:
        w = torch.full((self.n_rows,), 1.0 / self.n_rows, dtype=torch.float64)
        return self.combine(w)

    def combine(self, weights, extra: Optional[torch.Tensor] = None, extra_weight: float = 0.0) -> torch.Tensor:
        """``sum_i w_i U[i] (+ extra_weight * extra)``."""
        from ..ops import combine as _k
        self.materialize_virtual()
        self._pre()
        rows = self._ptrs(range(self.n_rows))
        if torch.is_tensor(weights) and weights.is_cuda:
            # device-resident weights (on-device Gram solvers): no host copy; with ``extra`` the last weight is its.
            # ``extra`` is held past the launch: inside a graph capture the replay reads it
            if extra is not None:
                self._keep = extra.to(self.device, torch.float32).contiguous()
                rows = rows + [self._keep.data_ptr()]
            w = weights.to(torch.float32).contiguous()
        else:
            w = [float(x) for x in (weights.tolist() if hasattr(weights, "tolist") else weights)]
            if extra is not None and extra_weight != 0.0:
                extra = extra.contiguous()
                rows, w = rows + [extra.data_ptr()], w + [float(extra_weight)]
        c0, c1 = self._cols()
        ep, out = self._epilogue()
        _k.launch_combine(rows, w, c0, c1, ep, self.device)
        self._finish()
        return out

    def trimmed_mean(self, b: int) -> torch.Tensor:
        if self.n_rows - 2 * b <= 0:
            raise ValueError(f"trim {b} too large for {self.n_rows} rows")
        return self._select(0, b)

    def median(self) -> torch.Tensor:
        return self._select(1, 0)

    def _select(self, mode: int, b: int) -> torch.Tensor:
        from ..ops import select as _s
        resolve_scaled_rows(self)
        self._pre()
        v = self.virtual
        if v is not None and v.count:
            stat, other = v.partition(self.n_rows)
            count, kind, param, param_ptr = v.count, v.kind, v.param, v.param_ptr()
        else:
            stat, other, count, kind, param, param_ptr = range(self.n_rows), [], 0, None, 0.0, 0
        c0, c1 = self._cols()
        ep, out = self._epilogue()
        _s.launch_select(self._ptrs(stat), self._ptrs(other), count, kind, param, mode, b, c0, c1, ep, self.device,
                         param_ptr=param_ptr)
        self._finish()
        return out

    def materialize_virtual(self) -> None:
        """Write the virtual rows into the rows they replace (what the reference's callbacks do)."""
        v = self.virtual
        if v is not None and v.count:
            from ..ops import attack as _a
            resolve_scaled_rows(self)
            v = self.virtual
            self._pre()
            honest, _ = v.partition(self.n_rows)
            c0, c1 = self._cols()
            _a.attack_rows(self._ptrs(honest), self._ptrs(list(v.replaced)), v.kind, v.param, c0, c1, self.device,
                           param_ptr=v.param_ptr())
            self.virtual = None
            self._rows_written()

    # geometry ------------------------------------------------------------------
    def gram(self, extra: Optional[torch.Tensor] = None) -> np.ndarray: raise NotImplementedError

    def gram_device(self, extra: Optional[torch.Tensor] = None):
        """The Gram matrix left ON THE DEVICE (``ops.gram_solve.DeviceGram``) for the on-device solvers, or ``None``
        when this matrix has no kernel path (CPU oracle): callers then fall back to ``gram()`` + the host solvers."""
        from ..ops import gram_solve
        if not gram_solve.enabled():
            return None
        r = self._gram_pass(extra)
        if r is None:
            return None
        out, idx = r
        return gram_solve.DeviceGram(out, gram_solve.index_tensor(idx, self.device), len(idx))

    def gram_block_rows(self) -> list:
        """Row count of every block the Gram pass reads (each is padded to 8 rows)."""
        from ..ops._gram_impl import split_blocks
        return [b[2] for blk in self._gram_blocks() for b in split_blocks(*blk)]

    def deviation_row(self, honest: Sequence[int], dev_type: str) -> torch.Tensor:
        """The Min-Max / Min-Sum deviation vector q over the rows ``honest`` (``[n_cols]`` float32), over this
        matrix's coordinates ``_cols()`` (zero elsewhere)."""
        from ..ops import attack as _a
        self._pre()
        c0, c1 = self._cols()
        alloc = torch.empty if (c0, c1) == (0, self.n_cols) else torch.zeros
        q = alloc(self.n_cols, device=self.device, dtype=torch.float32)
        _a.deviation(self._ptrs(honest), dev_type, c0, c1, q, self.device)
        return q
    # escape hatch ----------------------------------------------------------------
    def rows(self) -> torch.Tensor: raise NotImplementedError

    def __len__(self) -> int:
        return self.n_rows


class LocalMatrix(UpdateMatrix):
    """Dense ``[N, d]`` tensor on one device.

    On CUDA the primitives dispatch to the hand-written sm_100a kernels in
    ``blades_b200.ops`` (coordinate-select, row-combine, tcgen05 Gram); on CPU they
    are the pure-torch oracle used by the tests.
    """

    def __init__(self, data: torch.Tensor, virtual: Optional[VirtualRows] = None,
                 use_kernels: Optional[bool] = None, theta: Optional[torch.Tensor] = None,
                 window=None, chunk: int = 0, last_chunk: bool = True, out_buffer: Optional[torch.Tensor] = None):
        assert data.dim() == 2, data.shape
        self.data = data
        self.theta = theta               # flat parameter vector for the fused server step
        self.n_rows, self.n_cols = data.shape
        self.device = data.device
        self.virtual = virtual
        if use_kernels is None:
            use_kernels = data.is_cuda and data.dtype == torch.float32
        self.use_kernels = use_kernels
        self.window, self.chunk, self.last_chunk, self.out_buffer = window, chunk, last_chunk, out_buffer

    # -- kernel hooks ---------------------------------------------------------------
    def _ptrs(self, rows) -> list:
        from ..ops import select as _s
        return _s.row_pointers(self.data, rows)

    def _epilogue(self):
        from ..ops import select as _s
        out = self.out_buffer
        if out is None:
            out = torch.empty(self.n_cols, device=self.device, dtype=torch.float32)
        if self.server_step is not None and self.theta is not None:
            self.step_applied = True
            return _s.make_epilogue([out.data_ptr()], [self.theta.data_ptr()], self.theta.data_ptr(),
                                    float(self.server_step[0])), out
        return _s.make_epilogue([out.data_ptr()]), out

    def _gram_blocks(self) -> list:
        return [(self.data.data_ptr(), self.data.stride(0), self.n_rows)]

    def _gram_pass(self, extra: Optional[torch.Tensor]):
        from ..ops import _gram_impl, gram as _k
        if not self.use_kernels or _k.PRECISION == "fp32" or self.rows().stride(1) != 1:
            return None
        return _gram_impl.gram_pass(self._gram_blocks(), self.n_cols, 0, self.n_cols, self.device, extra,
                                    _k.PRECISION == "tf32x3")

    # -- torch oracle (use_kernels=False) ---------------------------------------------
    def deviation_row(self, honest: Sequence[int], dev_type: str) -> torch.Tensor:
        if self.use_kernels:
            return super().deviation_row(honest, dev_type)
        from ..attackers import _agr
        return _agr.deviation(torch.nan_to_num(self.data[list(honest)]), dev_type).to(torch.float32)

    def materialize_virtual(self) -> torch.Tensor:
        """Write the virtual rows into ``data`` (what the reference's callbacks do)."""
        v = self.virtual
        if self.use_kernels:
            super().materialize_virtual()
        elif v is not None and v.count:
            val = v.value(self.data[v.partition(self.n_rows)[0]])
            self.data[list(v.replaced)] = val
            self.virtual = None
        return self.data

    def rows(self) -> torch.Tensor:
        return self.materialize_virtual()

    def _windowed(self, full: torch.Tensor) -> torch.Tensor:
        """CPU oracle of a windowed primitive: the full-width result restricted to this object's window, written into
        the round's shared result vector (coordinates outside the window are left to the other chunks)."""
        if self.window is None:
            return full
        c0, c1 = self._cols()
        if self.out_buffer is None:
            self.out_buffer = torch.zeros_like(full)
        self.out_buffer[c0:c1] = full[c0:c1]
        return self.out_buffer

    def combine(self, weights, extra: Optional[torch.Tensor] = None, extra_weight: float = 0.0) -> torch.Tensor:
        if self.use_kernels:
            return super().combine(weights, extra, extra_weight)
        w = torch.as_tensor(np.asarray(weights, dtype=np.float64) if not torch.is_tensor(weights) else weights)
        data = self.rows()
        res = (w.to(data.device, torch.float64)[:, None] * data.double()).sum(0)
        if extra is not None and extra_weight != 0.0:
            res = res + extra_weight * extra.to(res.device, torch.float64)
        return self._windowed(res.to(data.dtype))

    def mean(self) -> torch.Tensor:
        if self.use_kernels:
            return super().mean()
        return self._windowed(self.rows().mean(dim=0))

    def _select(self, mode: int, b: int) -> torch.Tensor:
        if self.use_kernels:
            return super()._select(mode, b)
        data, n = self.rows(), self.n_rows
        if mode == 0 and b == 0:
            return self._windowed(data.mean(0))
        srt = data.sort(dim=0).values
        if mode == 0:
            return self._windowed(srt[b: n - b].mean(dim=0))
        return self._windowed((srt[(n - 1) // 2] + srt[n // 2]) * 0.5)

    def gram(self, extra: Optional[torch.Tensor] = None) -> np.ndarray:
        data = self.rows()
        if extra is not None:
            extra = extra.reshape(-1, self.n_cols).to(data.device, data.dtype)
        if self.use_kernels:
            from ..ops import gram as _k
            return _k.gram(data, extra)
        full = data if extra is None else torch.cat([data, extra], 0)
        full = full.double()
        return (full @ full.T).cpu().numpy()


def as_matrix(inputs, virtual: Optional[VirtualRows] = None) -> UpdateMatrix:
    """Coerce the reference's three input conventions (mean.py:21-28) to a matrix."""
    from ..client import BladesClient
    if isinstance(inputs, UpdateMatrix):
        return inputs
    if torch.is_tensor(inputs):
        return LocalMatrix(inputs if inputs.dim() == 2 else inputs.reshape(1, -1), virtual)
    inputs = list(inputs)
    if len(inputs) and all(isinstance(e, BladesClient) for e in inputs):
        # virtual clients bound to consecutive rows of one matrix -> zero-copy
        slots = [c._slot for c in inputs]
        if all(s is not None for s in slots) and all(s.matrix is slots[0].matrix for s in slots) \
                and [s.row for s in slots] == list(range(len(slots))) \
                and slots[0].matrix.shape[0] == len(slots):
            mat = slots[0].matrix
            torch.nan_to_num_(mat)
            return LocalMatrix(mat, virtual)
        return LocalMatrix(torch.stack([c.get_update() for c in inputs]), virtual)
    if len(inputs) and all(torch.is_tensor(e) for e in inputs):
        return LocalMatrix(torch.stack(inputs, dim=0), virtual)
    if len(inputs) and all(callable(getattr(e, "get_update", None)) for e in inputs):
        # duck-typed clients (the reference only ever calls ``.get_update()``, mean.py:23)
        return LocalMatrix(torch.stack([e.get_update() for e in inputs]), virtual)
    raise TypeError("aggregator inputs must be clients, tensors or an UpdateMatrix")

"""``ShardedMatrix``: the update matrix spread over G trainer shards, rows in NVLink-addressable
symmetric memory, aggregation coordinate-sharded (SURVEY 5.8, 7.2.1).

Every primitive is ONE kernel per rank: rank g owns coordinates ``[c_g, c_{g+1})`` (of the whole
vector, or of the window of it this matrix object covers -- pipelined aggregation), its CTAs read
that coordinate range of EVERY row, reduce in registers / tensor cores, and store the result range
into every replica (``agg`` and, when the server step is fused, ``theta``; one ``multimem.st`` per
value when the fabric has a multicast object).  The rows reach the kernel in one of two ways:

* pull: local rows from HBM, peer rows with plain global loads / TMA on NVLink-mapped pointers;
* push (``push_plan``): every rank DMAs its rows' slice of the other ranks' ranges into their
  ``recv`` landing zones with copy-engine 2-D copies, the kernel then reads local memory only.

The reference's gather (Ray pickles -> torch.stack, simulator.py:235 + mean.py:23) and broadcast
(model pickled to every actor, simulator.py:222-233) therefore never exist as separate steps.
Gram partials are summed inside the NVSwitch (``SymmetricUpdates.reduce_scratch``) and handed to
the on-device solvers (``ops.gram_solve``) without leaving device memory.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch
import torch.distributed as dist

from ..ops import _gram_impl
from ..ops import gram as k_gram
from ..ops import select as k_select
from .matrix import UpdateMatrix, VirtualRows

__all__ = ["ShardedMatrix"]


def _push_enabled(world_size: int = 2) -> bool:
    """Push mode (copy-engine DMAs of finished windows + local reads) or pull mode (kernels read peer rows with loads
    over NVLink).  ``BLADES_AGG_PUSH`` = 1 / 0 forces one; the default follows the measurements on B200 NVSwitch nodes
    (profiles/README.md): push wins while the per-GPU NVLink volume is large next to the backward pass it hides behind
    (2 GPUs: 237 vs 199 rounds/s), pull wins at 8 GPUs (376 vs 344), where each DMA is small and the all-to-all of
    eight ranks x seven destinations tops out at the same ~470 GB/s per GPU either way."""
    import os
    v = os.environ.get("BLADES_AGG_PUSH", "auto")
    if v in ("0", "1"):
        return v == "1"
    return world_size <= 4


def push_plan(me: int, row0, n_local: int, ld: int, recv_ld: int, shards, recv_col: int, skip):
    """The 2-D copies rank ``me`` issues to ship its rows' slices of the other ranks' coordinate ranges (pure host
    logic, unit-tested without a GPU).  ``shards[g] = (d0, d1)``: coordinates rank g aggregates; ``skip``: global rows
    nobody reads (replaced by virtual attack rows).  Returns ``(dst_rank, first_global_row, dst_col, src_offset_floats,
    width_floats, n_rows)`` per copy: rows ``[first, first + n_rows)`` of the destination's landing zone, columns
    ``[dst_col, dst_col + width)``, read from ``U_local`` at float offset ``src_offset`` with row pitch ``ld``."""
    first = row0[me]
    runs, start = [], None                          # maximal runs of consecutive local rows that are needed
    for i in range(n_local + 1):
        need = i < n_local and (first + i) not in skip
        if need and start is None:
            start = i
        if not need and start is not None:
            runs.append((start, i))
            start = None
    plan = []
    for g, (d0, d1) in enumerate(shards):
        if g == me or d1 <= d0:
            continue
        assert recv_col + (d1 - d0) <= recv_ld, "landing zone too small for this window"
        for (a, b) in runs:
            plan.append((g, first + a, recv_col, a * ld + d0, d1 - d0, b - a))
    return plan


class ShardedMatrix(UpdateMatrix):
    def __init__(self, symm, virtual: Optional[VirtualRows] = None, window=None, chunk: int = 0,
                 last_chunk: bool = True, recv_col: int = 0):
        self.symm = symm
        self.n_rows = symm.n_total
        self.n_cols = symm.d
        self.device = symm.world.device
        self.virtual = virtual
        self.server_step = None          # (lr,) -> theta += lr*agg fused into the final primitive
        self.step_applied = False
        self._synced = False
        self.window, self.chunk, self.last_chunk = window, chunk, last_chunk
        self.recv_col = recv_col         # column of this window inside the recv rows (pipelined aggregation)
        self.push = _push_enabled(symm.world.size) and symm.world.size > 1 and symm.recv_ld > 0

    # ------------------------------------------------------------------ helpers
    def _shards(self):
        """Coordinate range of every rank for this matrix object (its window, or the whole vector)."""
        from ..comm.symm import coordinate_shards
        if self.window is None:
            return list(self.symm.col_ranges)
        lo, hi = int(self.window[0]), int(self.window[1])
        return [(lo + a, lo + b) for a, b in coordinate_shards(hi - lo, self.symm.world.size)]

    def _cols(self):
        """This rank's coordinate range: its shard of the whole vector, or -- pipelined aggregation -- its shard of the
        window this matrix object covers (every window is split evenly over the ranks)."""
        return self._shards()[self.symm.world.rank]

    # -- push mode: rows travel by copy-engine DMA, kernels read local memory ---------------------------------------
    def _push_rows(self) -> None:
        """DMA this rank's rows' slice of every OTHER rank's coordinate range into that rank's ``recv`` rows
        (cudaMemcpy2DAsync over the NVLink mapping: copy engines, no SM time).  Rows replaced by virtual attack rows are
        never read and stay home.  Stream ordered after the training kernels that wrote the rows; the device barrier
        that follows on every rank is what tells the aggregator that all pushes have landed."""
        from ..ops import nvls
        s = self.symm
        skip = set(self.virtual.replaced) if (self.virtual is not None and self.virtual.count) else set()
        plan = push_plan(s.world.rank, s.row0, s.n_local, s.ld, s.recv_ld, self._shards(), self.recv_col, skip)
        u0 = s.local_full.data_ptr()
        # one stream per destination: the copies to different peers are independent DMAs (separate copy engines /
        # NVLink ports); forked from and joined back into the calling stream, so they stay ordered after the training
        # kernels and before the barrier (inside a graph capture these become parallel memcpy nodes)
        cur = torch.cuda.current_stream(self.device)
        pool = s.push_streams()
        used = []
        for g in sorted({c[0] for c in plan}):
            st = pool[g % len(pool)]
            st.wait_stream(cur)
            used.append(st)
            with torch.cuda.stream(st):
                for (dst, grow, gcol, src_off, width, height) in plan:
                    if dst == g:
                        nvls.copy2d(s.recv_row_ptr(g, grow, gcol), s.recv_ld * 4, u0 + src_off * 4, s.ld * 4,
                                    width * 4, height, self.device)
        for st in used:
            cur.wait_stream(st)

    def _ptrs(self, rows):
        """Row pointers for a kernel that reads coordinates ``self._cols()``: NVLink peer pointers (pull mode), or --
        push mode -- local rows in ``U`` and remote rows in this rank's ``recv`` landing zone, pre-offset so that
        ``ptr + c`` addresses coordinate ``c``."""
        s = self.symm
        if not self.push:
            return s.row_ptrs(rows)
        me = s.world.rank
        c0, _ = self._cols()
        out = []
        for i in rows:
            r, _li = s.row_owner[i]
            out.append(s.row_ptr(i) if r == me else s.recv_row_ptr(me, i, self.recv_col) - c0 * 4)
        return out

    def _barrier(self):
        # chunks of a pipelined round run on a side stream while the main stream still trains: their flag exchanges
        # use their own signal-pad channel (1 + chunk); channel 0 closes the round
        self.symm.barrier(0 if self.window is None else 1 + self.chunk)

    def _pre(self):
        if not self._synced:             # all ranks finished writing (push mode: and shipping) their rows of this window
            if self.push:
                self._push_rows()
            self._barrier()
            self._synced = True

    def _rows_written(self):
        self._barrier()

    def _epilogue(self):
        s = self.symm
        if self.server_step is not None:
            self.step_applied = True
            return k_select.make_epilogue(s.agg_ptrs(), s.theta_ptrs(), s.theta.data_ptr(), float(self.server_step[0]),
                                          mc_out=s.mc_agg_ptr(), mc_theta=s.mc_theta_ptr()), s.agg
        return k_select.make_epilogue(s.agg_ptrs(), mc_out=s.mc_agg_ptr()), s.agg

    def _finish(self):
        if self.window is None or self.last_chunk:
            self.symm.barrier()          # every shard of agg/theta has landed everywhere

    def deviation_row(self, honest, dev_type: str) -> torch.Tensor:
        """q over this rank's coordinates only (the Gram pass of this rank reads no others); the rows are pulled from
        their owners, as the select kernels do."""
        self.push = False                # the Gram pass that follows pulls the rows of U itself
        return super().deviation_row(honest, dev_type)

    # ------------------------------------------------------------------ Gram
    def _gram_blocks(self) -> list:
        return self.symm.block_descs()

    def _gram_pass(self, extra: Optional[torch.Tensor]):
        """Summed Gram accumulators in every rank's symmetric scratch region + the logical -> padded row list."""
        self.push = False                # the Gram pass pulls the rows of U itself by TMA (peer descriptors)
        self.materialize_virtual()
        self._pre()
        s = self.symm
        c0, c1 = s.my_cols
        # partials accumulate in this rank's replica of the symmetric scratch region; the cross-GPU sum happens in the
        # NVSwitch (multimem.ld_reduce / multimem.st, csrc/cuda/nvls.cu) -- no NCCL call on the aggregation path.
        # When the 3xTF32 staging does not fit for this row count the pass runs in plain tf32
        r = _gram_impl.gram_pass(self._gram_blocks(), self.n_cols, c0, c1, self.device, extra,
                                 k_gram.PRECISION == "tf32x3", tf32_fallback=True, scratch=s.scratch)
        assert r is not None, "too many rows/blocks for one Gram pass"
        s.reduce_scratch(r[0].numel())
        return r

    def gram(self, extra: Optional[torch.Tensor] = None) -> np.ndarray:
        return _gram_impl.symmetrised(*self._gram_pass(extra)).double().cpu().numpy()

    def rows(self) -> torch.Tensor:
        self.push = False                # the gathered matrix must see materialised virtual rows in U itself
        self.materialize_virtual()
        self._pre()
        s = self.symm
        pad = s.local_full.contiguous()
        outs = [torch.empty_like(pad) for _ in range(s.world.size)]
        dist.all_gather(outs, pad)
        return torch.cat([o[:k, : self.n_cols] for o, k in zip(outs, s.shard_sizes)], 0)

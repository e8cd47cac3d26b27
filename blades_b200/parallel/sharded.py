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

from ..ops import attack as k_attack
from ..ops import combine as k_combine
from ..ops import select as k_select
from .matrix import UpdateMatrix, VirtualRows, resolve_scaled_rows

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
    def __init__(self, symm, virtual: Optional[VirtualRows] = None):
        self.symm = symm
        self.n_rows = symm.n_total
        self.n_cols = symm.d
        self.device = symm.world.device
        self.virtual = virtual
        self.server_step = None          # (lr,) -> theta += lr*agg fused into the final primitive
        self.step_applied = False
        self._synced = False
        self.recv_col = 0                # column of this window inside the recv rows (pipelined aggregation)
        self.push = _push_enabled(symm.world.size) and symm.world.size > 1 and symm.recv_ld > 0

    # ------------------------------------------------------------------ helpers
    def _cols(self):
        """This rank's coordinate range: its shard of the whole vector, or -- pipelined aggregation -- its shard of the
        window this matrix object covers (every window is split evenly over the ranks)."""
        if self.window is None:
            return self.symm.my_cols
        from ..comm.symm import coordinate_shards
        lo, hi = int(self.window[0]), int(self.window[1])
        c0, c1 = coordinate_shards(hi - lo, self.symm.world.size)[self.symm.world.rank]
        return lo + c0, lo + c1

    # -- push mode: rows travel by copy-engine DMA, kernels read local memory ---------------------------------------
    def _shards(self):
        """Coordinate range of every rank for this matrix object (its window, or the whole vector)."""
        from ..comm.symm import coordinate_shards
        if self.window is None:
            return list(self.symm.col_ranges)
        lo, hi = int(self.window[0]), int(self.window[1])
        return [(lo + a, lo + b) for a, b in coordinate_shards(hi - lo, self.symm.world.size)]

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

    def _epilogue(self, final: bool):
        s = self.symm
        if final and self.server_step is not None:
            self.step_applied = True
            return k_select.make_epilogue(s.agg_ptrs(), s.theta_ptrs(), s.theta.data_ptr(), float(self.server_step[0]),
                                          mc_out=s.mc_agg_ptr(), mc_theta=s.mc_theta_ptr())
        return k_select.make_epilogue(s.agg_ptrs(), mc_out=s.mc_agg_ptr())

    def _finish(self) -> torch.Tensor:
        if self.window is None or self.last_chunk:
            self.symm.barrier()          # every shard of agg/theta has landed everywhere
        return self.symm.agg

    def gram_block_rows(self) -> list:
        from ..ops import _gram_impl
        return [b[2] for (ptr, ld, rows) in self.symm.block_descs() for b in _gram_impl.split_blocks(ptr, ld, rows)]

    def deviation_row(self, honest, dev_type: str) -> torch.Tensor:
        """q over this rank's coordinates only (the Gram pass of this rank reads no others); the rows are pulled from
        their owners, as the select kernels do."""
        self.push = False                # the Gram pass that follows pulls the rows of U itself
        self._pre()
        q = torch.zeros(self.n_cols, device=self.device, dtype=torch.float32)
        c0, c1 = self._cols()
        k_attack.deviation(self._ptrs(honest), dev_type, c0, c1, q, self.device)
        return q

    def materialize_virtual(self):
        v = self.virtual
        if v is not None and v.count:
            resolve_scaled_rows(self)
            v = self.virtual
            self._pre()
            s = self.symm
            byz = set(v.byzantine)
            honest = [i for i in range(self.n_rows) if i not in byz]
            c0, c1 = self._cols()
            k_attack.attack_rows(self._ptrs(honest), self._ptrs(list(v.replaced)), v.kind, v.param, c0, c1,
                                 self.device, param_ptr=v.param_ptr())
            self.virtual = None
            self._barrier()

    # ------------------------------------------------------------------ primitives
    def _select(self, mode: int, b: int) -> torch.Tensor:
        resolve_scaled_rows(self)
        self._pre()
        s = self.symm
        c0, c1 = self._cols()
        v = self.virtual
        if v is not None and v.count:
            byz, rep = set(v.byzantine), set(v.replaced)
            stat = self._ptrs([i for i in range(self.n_rows) if i not in byz])
            other = self._ptrs([i for i in range(self.n_rows) if i in byz and i not in rep])
            k_select.launch_select(stat, other, v.count, v.kind, v.param, mode, b, c0, c1,
                                   self._epilogue(True), self.device, param_ptr=v.param_ptr())
        else:
            k_select.launch_select(self._ptrs(range(self.n_rows)), [], 0, None, 0.0, mode, b, c0, c1,
                                   self._epilogue(True), self.device)
        return self._finish()

    def trimmed_mean(self, b: int) -> torch.Tensor:
        if self.n_rows - 2 * b <= 0:
            raise ValueError(f"trim {b} too large for {self.n_rows} rows")
        return self._select(0, b)

    def median(self) -> torch.Tensor:
        return self._select(1, 0)

    def combine(self, weights, extra: Optional[torch.Tensor] = None, extra_weight: float = 0.0) -> torch.Tensor:
        self.materialize_virtual()
        self._pre()
        s = self.symm
        if torch.is_tensor(weights) and weights.is_cuda:
            # device-resident weights (on-device Gram solvers): no host copy; with ``extra`` the last weight is its
            rows = self._ptrs(range(self.n_rows))
            if extra is not None:
                self._keep = extra.to(self.device, torch.float32).contiguous()
                rows = rows + [self._keep.data_ptr()]
            c0, c1 = self._cols()
            k_combine.launch_combine(rows, weights.to(torch.float32).contiguous(), c0, c1, self._epilogue(True), self.device)
            return self._finish()
        w = [float(x) for x in (weights.tolist() if hasattr(weights, "tolist") else weights)]
        rows = self._ptrs(range(self.n_rows))
        if extra is not None and extra_weight != 0.0:
            rows = rows + [extra.contiguous().data_ptr()]
            w = w + [float(extra_weight)]
        c0, c1 = self._cols()
        k_combine.launch_combine(rows, w, c0, c1, self._epilogue(True), self.device)
        return self._finish()

    def gram(self, extra: Optional[torch.Tensor] = None) -> np.ndarray:
        out, idx = self._gram_scratch(extra)
        idx_t = torch.tensor(idx, device=self.device)
        G = out[idx_t][:, idx_t]
        return (0.5 * (G + G.T)).double().cpu().numpy()

    def gram_device(self, extra: Optional[torch.Tensor] = None):
        from ..ops import gram_solve
        if not gram_solve.enabled():
            return None
        out, idx = self._gram_scratch(extra)
        return gram_solve.DeviceGram(out, gram_solve.index_tensor(idx, self.device), len(idx))

    def _gram_scratch(self, extra: Optional[torch.Tensor] = None):
        """Summed Gram accumulators in every rank's symmetric scratch region + the logical -> padded row list."""
        from ..ops import _gram_impl, gram as k_gram
        self.push = False                # the Gram pass pulls the rows of U itself by TMA (peer descriptors)
        self.materialize_virtual()
        self._pre()
        s = self.symm
        blocks = []
        for (ptr, ld, rows) in s.block_descs():
            blocks += _gram_impl.split_blocks(ptr, ld, rows)
        e = 0
        if extra is not None:
            extra = extra.reshape(-1, self.n_cols)
            e = extra.shape[0]
            buf = torch.zeros(e, s.ld, device=self.device, dtype=torch.float32)
            buf[:, : self.n_cols] = extra
            blocks += _gram_impl.split_blocks(buf.data_ptr(), s.ld, e)
        total_pad = sum((b[2] + 7) // 8 * 8 for b in blocks)
        assert total_pad <= 512 and len(blocks) <= 9, "too many rows/blocks for one Gram pass"
        tile_rows = (total_pad + 127) // 128 * 128
        ldg = (total_pad + 31) // 32 * 32
        # partials accumulate in this rank's replica of the symmetric scratch region; the cross-GPU sum happens in the
        # NVSwitch (multimem.ld_reduce / multimem.st, csrc/cuda/nvls.cu) -- no NCCL call on the aggregation path
        out = s.scratch[: tile_rows * ldg].view(tile_rows, ldg)
        out.zero_()
        c0, c1 = s.my_cols
        starts = _gram_impl.launch_gram(blocks, self.n_cols, c0, c1, out, k_gram.PRECISION == "tf32x3", self.device)
        if starts is None:               # 3xTF32 staging does not fit for this row count: plain tf32
            starts = _gram_impl.launch_gram(blocks, self.n_cols, c0, c1, out, False, self.device)
        s.reduce_scratch(tile_rows * ldg)
        idx = []
        for (_, _, rows), st in zip(blocks, starts):
            idx += list(range(st, st + rows))
        return out, idx

    def rows(self) -> torch.Tensor:
        self.push = False                # the gathered matrix must see materialised virtual rows in U itself
        self.materialize_virtual()
        self._pre()
        s = self.symm
        pad = s.local_full.contiguous()
        outs = [torch.empty_like(pad) for _ in range(s.world.size)]
        dist.all_gather(outs, pad)
        return torch.cat([o[:k, : self.n_cols] for o, k in zip(outs, s.shard_sizes)], 0)

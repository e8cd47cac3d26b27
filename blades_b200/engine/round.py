"""The per-rank round engine: local training of this rank's virtual clients, attack
phase, robust aggregation, server step.  Replaces the reference's
``Simulator.train_actor`` + ``_RayActor.local_training`` pipeline
(/root/reference/src/blades/simulator.py:203-245, actor.py:23-33):

reference (per round)                          | here
-----------------------------------------------+------------------------------------------
pickle global model + N client objects to Ray   | nothing moves: theta[d] is device resident
actors                                          | and replicated on every rank
per client: load_state_dict, clone params,      | fedsgd: ONE batched fwd/bwd for all local
k SGD steps, 2x flat concat to CPU              | clients, wgrad epilogue writes the update
                                                | row; fedavg/custom: time-sliced on a shared
                                                | worker model, one fused diff kernel per client
gather N CPU vectors, torch.stack               | rows already sit in U_g[n_local, d]
                                                | (NVLink-addressable symmetric memory)
f attacker callbacks on CPU                     | virtual rows inside the aggregation kernel;
                                                | row-local attackers (Noise) on the owning rank
aggregator on CPU [N,d]                         | fused kernels per coordinate window, started on a
                                                | side stream while the backward pass still runs
                                                | (_AggPipeline); tcgen05 Gram + on-device solvers
per-param python loop + optimizer.step          | theta += lr*agg in the kernel epilogue
                                                | (multimem.st to every replica)
"""
from __future__ import annotations

import copy
import logging
import time
from typing import Callable, Dict, List, Optional, Sequence

import numpy as np
import torch
import torch.nn as nn

from ..client import BladesClient, ByzantineClient
from ..comm.group import World, split_clients
from ..datasets.dataset import RaggedBatches
from ..parallel.matrix import LocalMatrix, UpdateMatrix, VirtualRows
from ..server import BladesServer
from . import batched as cb
from .flat import FlatParams

#: stream-capture mode of every CUDA graph the engine records.  "thread_local": only the capturing thread is policed --
#: the input prefetcher's worker thread may allocate / copy / synchronise on its own stream while a chunk's graph is
#: being captured (the default "global" mode would fail the capture for that).
_CAPTURE_MODE = "thread_local"

__all__ = ["RoundEngine", "PhaseTimer"]


class PhaseTimer:
    """CUDA-event (or wall-clock on CPU) timing of the round phases (SURVEY 5.1)."""

    def __init__(self, device: torch.device, enabled: bool = True):
        self.cuda = device.type == "cuda"
        self.enabled = enabled
        self.records: List[Dict[str, float]] = []
        self._cur: Dict[str, tuple] = {}

    def start(self, name: str):
        if not self.enabled:
            return
        if self.cuda:
            torch.cuda.nvtx.range_push(name)
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self._cur[name] = (ev, None)
        else:
            self._cur[name] = (time.perf_counter(), None)

    def stop(self, name: str):
        if not self.enabled or name not in self._cur:
            return
        beg, _ = self._cur[name]
        if self.cuda:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            torch.cuda.nvtx.range_pop()
            self._cur[name] = (beg, ev)
        else:
            self._cur[name] = (beg, time.perf_counter())

    def flush(self) -> Dict[str, float]:
        out = {}
        if self.cuda and self._cur:
            torch.cuda.synchronize()
        for k, (b, e) in self._cur.items():
            if e is None:
                continue
            out[k] = b.elapsed_time(e) if self.cuda else (e - b) * 1e3
        self._cur = {}
        if out:
            self.records.append(out)
        return out


class _HostRead:
    """Pending pinned-memory copy: ``get()`` blocks until its event has completed and returns the host tensor."""
    __slots__ = ("buf", "event")

    def __init__(self, buf: torch.Tensor, event):
        self.buf, self.event = buf, event

    def get(self) -> torch.Tensor:
        self.event.synchronize()
        return self.buf


def _diff(after: torch.Tensor, before: torch.Tensor, out: torch.Tensor) -> None:
    """``out = nan_to_num(after - before)``: the time-sliced client update, sanitised where it is produced (reference
    client.py:195-198); our streaming kernel on CUDA, torch on the CPU."""
    if out.is_cuda and out.dtype == torch.float32 and after.is_contiguous() and before.is_contiguous() \
            and out.is_contiguous():
        from ..ops import fused as _kf
        _kf.diff_rows(after, before, out)
    else:
        torch.sub(after, before, out=out)
        torch.nan_to_num_(out)


class _AggPipeline:
    """Pipelined aggregation inside the whole-round graph.  ``progress(lo)`` (called by the backward pass) says that
    every update coordinate ``>= lo`` is final; once enough of them have accumulated, the aggregation of that window
    (pre-barrier across the GPUs on the window's own channel, fused attack + select / combine + server step over the
    rank's share of the window) is enqueued on a low-priority side stream that forks off the training stream, and
    joins it again after the last window.  Per-coordinate arithmetic is unchanged, so the result is bit-identical to
    the unpipelined round; what changes is that the pull over NVLink and the selection network overlap the rest of
    the backward pass instead of following it (reference: gather + aggregate strictly after training,
    simulator.py:235-245)."""

    MIN_FRACTION = 0.04          # smaller windows wait for the next stage

    def __init__(self, eng: "RoundEngine", aggregate_fn):
        self.eng, self.fn = eng, aggregate_fn
        self.hi = eng.d
        self.k = 0
        self.windows = []
        self.out = None if eng.symm is not None else torch.empty(eng.d, device=eng.device, dtype=torch.float32)
        self.agg = None
        self.col = 0                                   # next free column of the push-mode landing rows

    def _launch(self, lo: int, hi: int, last: bool) -> None:
        main = torch.cuda.current_stream(self.eng.device)
        side = self.eng._agg_stream
        side.wait_stream(main)
        with torch.cuda.stream(side):
            self.agg = self.fn(window=(lo, hi), chunk=self.k, last=last, out=self.out, recv_col=self.col)
        if self.eng.symm is not None:
            self.col += (self.eng.symm.window_span(lo, hi) + 127) // 128 * 128
        self.windows.append((lo, hi))
        self.k += 1
        self.hi = lo

    def progress(self, lo: int) -> None:
        lo = (int(lo) + 127) // 128 * 128              # whole 512 B row segments per window (round up: coordinates below ``lo`` are not final yet)
        if lo <= 0 or (self.hi - lo) < self.MIN_FRACTION * self.eng.d or self.k >= 6:
            return
        self._launch(lo, self.hi, False)

    def finish(self):
        self._launch(0, self.hi, True)
        torch.cuda.current_stream(self.eng.device).wait_stream(self.eng._agg_stream)
        return self.agg


def _overrides(obj, name: str, base=BladesClient) -> bool:
    return getattr(type(obj), name) is not getattr(base, name)


def _default_ce(fn) -> bool:
    return (type(fn) is nn.CrossEntropyLoss and fn.weight is None and fn.reduction == "mean"
            and fn.label_smoothing == 0.0 and fn.ignore_index == -100)


def _fusable_classes():
    from ..attackers.alieclient import AlieClient
    from ..attackers.ipmclient import IpmClient
    from ..attackers.minmaxclient import MinmaxClient
    from ..attackers.minsumclient import MinsumClient
    return (AlieClient, IpmClient, MinmaxClient, MinsumClient)


class RoundEngine:
    def __init__(self, world: World, dataset, clients: Sequence[BladesClient], device: torch.device,
                 use_kernels: Optional[bool] = None, profile: bool = False):
        self.world = world
        self.dataset = dataset
        self.clients = list(clients)
        self.device = torch.device(device)
        self.n_total = len(self.clients)
        parts = split_clients(self.n_total, world.size)
        self.local_idx = [int(i) for i in parts[world.rank]]
        self.row_of = {gi: r for r, gi in enumerate(self.local_idx)}
        self.shard_sizes = [len(p) for p in parts]
        self.use_kernels = (self.device.type == "cuda") if use_kernels is None else use_kernels
        self.timer = PhaseTimer(self.device, enabled=profile)
        self.debug_logger = logging.getLogger("debug")
        self.server: Optional[BladesServer] = None
        self.gflat: Optional[FlatParams] = None
        self.worker: Optional[nn.Module] = None
        self.wflat: Optional[FlatParams] = None
        self.U: Optional[torch.Tensor] = None
        self.matrix_factory: Optional[Callable] = None
        self.last_client_losses: Optional[torch.Tensor] = None
        self.kernel_launches = 0
        self._clamps = {}
        self._clamps_in_graphs = set()
        self._shape_votes = {}      # staged input shape -> how often it occurred (tail batches are the rare ones)
        self._pf_pool = None
        self._pf_stream = None
        self._zc_plans = {}
        self._pf_jobs = {}
        self._pf_deferred = None
        self._pf_slot_of = {}       # request key -> next slot (0/1)
        self._pf_keyidx = {}        # request key -> index (names the pinned staging buffers)
        self._pf_pre = {}           # request key -> {client id: cursor before its unconsumed prefetched batch}
        self._pf_copied = {}        # (request key, slot) -> event after the H2D copies out of its pinned staging
        self._stash = {}            # request key -> inputs (or RaggedBatches) handed back by a caller that could not use them
        self._ragged_data = {}      # local row -> pre-drawn host batches for the time-sliced path
        self.track_cursors = False
        import os
        #: exercise the worker-thread prefetcher without a GPU (tests)
        self.prefetch_on_cpu = os.environ.get("BLADES_PREFETCH_CPU", "0") == "1"
        self.prefetch = os.environ.get("BLADES_PREFETCH", "1") != "0"
        #: clients per fused forward/backward (0 = all local clients at once)
        self.max_batched_clients = int(os.environ.get("BLADES_MAX_BATCHED_CLIENTS", "0"))
        self._sliced_graphs = {}
        self._eager_slice_bufs = {}
        self._workers = []
        self._slice_copied = {}
        self._round_graphs = {}     # (client lr, server lr) -> captured whole-round graph state
        self.static_aggregate = None
        self._graphs = {}           # (rows, lr, shape) -> (CUDAGraph, static X, static y, losses)
        self._graph_seen = {}       # graph key -> how often it was requested (capture on the second request)
        self._graph_lr = {}         # captured graph key -> learning rate baked into it
        self.prestaged = None       # optional (X[n,1,B,...], y[n,1,B]) already on the device
        self.h2d_bytes = 0

    # ------------------------------------------------------------------ setup
    def setup(self, model: nn.Module, server_opt, aggregator, loss: str, client_lr: float,
              client_optimizer="SGD", server_lr: float = 0.1) -> BladesServer:
        model.to(self.device)
        from .flat import param_layout
        _, d = param_layout(model)
        self.d = d
        self._alloc_updates(len(self.local_idx), d)
        self.gflat = FlatParams(model, device=self.device,
                                storage=self.symm.theta if self.symm is not None else None)
        if server_opt == "SGD" or server_opt is None:
            server_opt = torch.optim.SGD(model.parameters(), lr=server_lr)
        self.server = BladesServer(optimizer=server_opt, model=model, aggregator=aggregator, flat=self.gflat)
        self.worker = copy.deepcopy(model)
        self.wflat = FlatParams(self.worker, device=self.device)
        # 'SGD' | optimizer class / factory ``f(params, lr=...)``.  An optimizer *instance* (what the
        # reference's scripts pass, scripts/cifar10.py:43-55) is ignored like in the reference (quirk
        # Q2: clients always run plain SGD; the instance only drives the lr scheduler).
        if isinstance(client_optimizer, torch.optim.Optimizer):
            client_optimizer = "SGD"
        self.client_opt_spec = client_optimizer
        self.worker_opt = torch.optim.SGD(self.worker.parameters(), lr=client_lr)
        for c in self.clients:
            c.set_loss(loss)
            c.device = self.device
        for gi in self.local_idx:
            self.clients[gi].bind_row(self.U, self.row_of[gi])
        self.batchable_model = cb.is_batchable(model)
        return self.server

    def _alloc_updates(self, n_local: int, d: int) -> None:
        if self.world.distributed and self.device.type == "cuda" and self._peer_access_everywhere():
            from ..comm import symm
            self.symm = symm.SymmetricUpdates(self.world, self.shard_sizes, d)
            self.U = self.symm.local
        else:
            self.symm = None
            ld = (d + 63) // 64 * 64          # 256 B aligned rows: 16 B vector loads + TMA strides
            if self.device.type == "cuda":
                from ..ops import nvls
                self.U = nvls.zero_(torch.empty(max(n_local, 1), ld, device=self.device, dtype=torch.float32))[:n_local, :d]
            else:
                self.U = torch.zeros(max(n_local, 1), ld, device=self.device, dtype=torch.float32)[:n_local, :d]

    def _peer_access_everywhere(self) -> bool:
        """``BLADES_SYMM=0`` (set identically on every rank) disables the NVLink symmetric-memory path: rows are then
        gathered with NCCL and every rank aggregates the dense matrix itself -- the slower baseline path, also what
        the CPU/gloo runs use.  By default symmetric memory is required on a multi-GPU run and a failing rendezvous
        (no peer access) raises."""
        import os
        if os.environ.get("BLADES_SYMM", "1") != "0":
            return True
        if self.world.rank == 0:
            import logging
            logging.getLogger("debug").warning("BLADES_SYMM=0: NCCL all_gather + per-rank aggregation")
        return False

    # ------------------------------------------------------------------ training
    def _stock_for_batching(self, c: BladesClient) -> bool:
        """The fused passes hard-wire mean cross-entropy (clamped per client): anything else -- a custom loss callable
        (``Simulator.run(loss=callable)``), class weights, label smoothing, another reduction -- trains on the
        time-sliced path, which calls ``client.loss_func``."""
        return _default_ce(c.loss_func) and not (
            _overrides(c, "local_training") or _overrides(c, "on_train_round_begin")
            or _overrides(c, "on_train_round_end") or _overrides(c, "set_para")
            or _overrides(c, "_post_backward") and not hasattr(c, "grad_sign"))

    def train_local(self, local_steps: int, lr: float) -> None:
        """Fill U[r] for every local client r."""
        local = [self.clients[gi] for gi in self.local_idx]
        plain = self.client_opt_spec in ("SGD", None, torch.optim.SGD)
        batch_rows, slice_rows = [], []
        for r, c in enumerate(local):
            if local_steps == 1 and plain and self.batchable_model and self._stock_for_batching(c):
                batch_rows.append(r)
            else:
                slice_rows.append(r)
        if batch_rows:
            try:
                # bound the activation footprint: at most ``max_batched_clients`` clients per fused pass
                step = self.max_batched_clients or len(batch_rows)
                for i in range(0, len(batch_rows), step):
                    self._train_batched(batch_rows[i: i + step], lr)
            except cb.BatchedUnsupported:
                slice_rows = sorted(slice_rows + batch_rows)
        if slice_rows:
            slice_rows = self._train_sliced_graphed(slice_rows, local_steps, lr)
        for r in slice_rows:
            self._train_timesliced(r, local_steps, lr)

    # -- batched fedsgd ------------------------------------------------------------
    def stage_batches(self, rows: Optional[Sequence[int]] = None, num_batches: int = 1):
        """This round's inputs on the device.  The inputs of round r+1 are produced WHILE round r computes, into
        per-request double buffers ordered by events: either the zero-copy gather kernel reads the selected
        samples straight from the pinned host shards (``_zero_copy_submit``), or a worker thread assembles the
        batches (multi-threaded C++ gather into pinned staging) and copies them H2D on a side stream.  The
        reference does one blocking ``.to(device)`` per batch per client inside the training loop (client.py:186).

        A "request" is one ``(rows, num_batches)`` key -- with ``max_batched_clients`` chunking there are several
        per round; every key owns its two slots, so the prefetch of one chunk can never land in a buffer another
        chunk has not consumed yet."""
        rows = list(range(len(self.local_idx))) if rows is None else list(rows)
        on_cuda = self.device.type == "cuda"
        back = self._stash.pop((tuple(rows), num_batches), None)
        if back is not None:                 # inputs staged earlier for a path that had to decline them
            if isinstance(back, RaggedBatches):
                raise back
            return back
        if not self.prefetch or not (on_cuda or self.prefetch_on_cpu):
            X, y = self._assemble(rows, num_batches, 0)
            self.h2d_bytes = X.numel() * X.element_size() + y.numel() * y.element_size()
            # synchronous fallback: blocking copies, because the pinned staging buffer is reused by the next call
            return X.to(self.device), y.to(self.device)
        key = (tuple(rows), num_batches)
        self.flush_prefetch()
        fut = self._pf_jobs.pop(key, None)
        if fut is None:
            fut = self._pf_submit(rows, num_batches)
        consumed = None
        try:
            X, y, ev, slot = fut.result()
        except RaggedBatches:
            # the batches of this round cannot be stacked (they travel with the exception); keep prefetching
            self._pf_pre.pop(key, None)
            if on_cuda:
                consumed = torch.cuda.Event()
                consumed.record(torch.cuda.current_stream(self.device))
            self._pf_deferred = (key, rows, num_batches, consumed)
            raise
        self._pf_pre.pop(key, None)                      # that batch is consumed now
        if on_cuda:
            torch.cuda.current_stream(self.device).wait_event(ev)
        self.h2d_bytes = X.numel() * X.element_size() + y.numel() * y.element_size()
        if self._zc_plans.get(key):
            self.h2d_bytes += y.numel() * 8              # zero-copy path: the index list is uploaded as well
        # The request for round r+1 is issued by flush_prefetch() AFTER this round's work has been launched (its
        # host part then overlaps the GPU).  It refills the key's OTHER slot, last read one round ago: everything
        # enqueued on the main stream up to here is a safe (conservative) ordering point for that refill.
        if on_cuda:
            consumed = torch.cuda.Event()
            consumed.record(torch.cuda.current_stream(self.device))
        self._pf_deferred = (key, rows, num_batches, consumed)
        return X, y

    def flush_prefetch(self) -> None:
        """Issue the deferred request for the next round's inputs (called right after a round is launched)."""
        d, self._pf_deferred = self._pf_deferred, None
        if d is not None:
            key, rows, num_batches, consumed = d
            self._pf_jobs[key] = self._pf_submit(rows, num_batches, consumed)

    def _assemble(self, rows, num_batches, slot):
        ids = [self.clients[self.local_idx[r]].id() for r in rows]
        return self.dataset.get_train_batches(ids, num_batches, slot=slot)

    def _next_slot(self, key) -> int:
        """Each request key alternates between its own two slots."""
        s = self._pf_slot_of.get(key, 0)
        self._pf_slot_of[key] = s ^ 1
        return s

    def _snapshot_cursors(self, key, rows) -> None:
        """Per-client stream cursors right BEFORE the batches of a prefetch are drawn: what a checkpoint must
        store for these clients while that prefetched batch is still unconsumed (``data_cursors``)."""
        if hasattr(self.dataset, "stream_state"):
            self._pf_pre[key] = {self.clients[self.local_idx[r]].id():
                                 self.dataset.stream_state(self.clients[self.local_idx[r]].id()) for r in rows}

    def _pf_submit(self, rows, num_batches, consumed=None):
        import concurrent.futures as cf
        on_cuda = self.device.type == "cuda"
        key = (tuple(rows), num_batches)
        if on_cuda:
            zc = self._zero_copy_submit(rows, num_batches, consumed)
            if zc is not None:
                return zc
        if self._pf_pool is None:
            self._pf_pool = cf.ThreadPoolExecutor(max_workers=1, thread_name_prefix="blades-prefetch")
            self._pf_dev = {}
        if on_cuda and self._pf_stream is None:
            self._pf_stream = torch.cuda.Stream(device=self.device)
        slot = self._next_slot(key)
        # pinned staging buffers of the dataset are keyed by an integer: unique per (key, slot); ids >= 100 belong
        # to the fedavg worker replicas
        staging = 2 * self._pf_keyidx.setdefault(key, len(self._pf_keyidx)) + slot
        if staging >= 100:
            raise RuntimeError("too many distinct prefetch requests per round; set BLADES_PREFETCH=0")
        if on_cuda and consumed is None:
            consumed = torch.cuda.Event()
            consumed.record(torch.cuda.current_stream(self.device))

        def job():
            if on_cuda:
                torch.cuda.set_device(self.device)
            prev = self._pf_copied.get((key, slot))
            if prev is not None:
                prev.synchronize()           # the H2D copy that last read this pinned staging buffer has finished
            self._snapshot_cursors(key, rows)
            X, y = self._assemble(rows, num_batches, staging)
            bufs = self._pf_dev.get((key, slot))
            if bufs is None or bufs[0].shape != X.shape:
                bufs = self._pf_dev[(key, slot)] = (torch.empty(X.shape, dtype=X.dtype, device=self.device),
                                                    torch.empty(y.shape, dtype=y.dtype, device=self.device))
            if not on_cuda:
                bufs[0].copy_(X)
                bufs[1].copy_(y)
                return bufs[0], bufs[1], None, slot
            with torch.cuda.stream(self._pf_stream):
                self._pf_stream.wait_event(consumed)
                bufs[0].copy_(X, non_blocking=True)
                bufs[1].copy_(y, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self._pf_stream)
            self._pf_copied[(key, slot)] = ev
            return bufs[0], bufs[1], ev, slot
        return self._pf_pool.submit(job)

    def _zero_copy_submit(self, rows, num_batches, consumed=None):
        """Next round's inputs via the zero-copy gather kernel: host work = drawing the index list."""
        import os
        if os.environ.get("BLADES_ZERO_COPY", "1") == "0":
            return None
        key = (tuple(rows), num_batches)
        plan = self._zc_plans.get(key)
        if plan is None:
            ids = [self.clients[self.local_idx[r]].id() for r in rows]
            got = self.dataset.device_gather_plan(ids) if hasattr(self.dataset, "device_gather_plan") else None
            if got is None:
                self._zc_plans[key] = False
                return None
            streams, shp, bs = got
            n, per = len(streams), num_batches * bs
            tab_x = torch.tensor([s.data.ctypes.data for s in streams], dtype=torch.int64).to(self.device)
            tab_y = torch.tensor([s.labels.ctypes.data for s in streams], dtype=torch.int64).to(self.device)
            sample_floats = int(np.prod(shp))
            plan = self._zc_plans[key] = dict(
                streams=streams, n=n, per=per, bs=bs, tab_x=tab_x, tab_y=tab_y, sample_floats=sample_floats,
                h_idx=[torch.empty(n * per, dtype=torch.int64).pin_memory() for _ in range(2)],
                d_idx=[torch.empty(n * per, dtype=torch.int64, device=self.device) for _ in range(2)],
                X=[torch.empty((n, num_batches, bs) + shp, dtype=torch.float32, device=self.device) for _ in range(2)],
                y=[torch.empty((n, num_batches, bs), dtype=torch.int64, device=self.device) for _ in range(2)],
                idx_done=[None, None])
            if self._pf_stream is None:
                self._pf_stream = torch.cuda.Stream(device=self.device)
        elif plan is False:
            return None
        from ..ops import gather as kg
        slot = self._next_slot(key)
        if plan["idx_done"][slot] is not None:
            plan["idx_done"][slot].synchronize()         # the pinned index buffer of this slot is free again
        self._snapshot_cursors(key, rows)
        h = plan["h_idx"][slot].numpy().reshape(plan["n"], plan["per"])
        bs = plan["bs"]
        for i, st in enumerate(plan["streams"]):
            for j in range(plan["per"] // bs):
                h[i, j * bs:(j + 1) * bs] = st.next_indices()
        if consumed is None:
            consumed = torch.cuda.Event()
            consumed.record(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(self._pf_stream):
            self._pf_stream.wait_event(consumed)
            plan["d_idx"][slot].copy_(plan["h_idx"][slot], non_blocking=True)
            done = torch.cuda.Event()
            done.record(self._pf_stream)
            plan["idx_done"][slot] = done
            kg.gather_samples(plan["tab_x"], plan["tab_y"], plan["d_idx"][slot], plan["X"][slot], plan["y"][slot],
                              plan["per"], plan["sample_floats"])
            ev = torch.cuda.Event()
            ev.record(self._pf_stream)

        class _Done:
            def __init__(self, v):
                self.v = v

            def result(self):
                return self.v
        return _Done((plan["X"][slot], plan["y"][slot], ev, slot))

    def finish(self) -> None:
        """End of a run: give back the batches the prefetcher drew for a round that will not happen (the streams are
        rewound to the cursors snapshotted before those draws), so a following ``run`` / evaluation / checkpoint sees
        the data streams exactly where the last trained round left them; stop the worker thread."""
        self._pf_deferred = None
        for fut in list(self._pf_jobs.values()):
            try:
                fut.result()
            except RaggedBatches:
                pass
        self._pf_jobs.clear()
        if hasattr(self.dataset, "load_state_dict"):
            for pre in self._pf_pre.values():
                self.dataset.load_state_dict(pre)
        self._pf_pre.clear()
        self._stash.clear()
        if self._pf_pool is not None:
            self._pf_pool.shutdown(wait=True)
            self._pf_pool = None

    def data_cursors(self):
        """Data-stream cursors as of the batches CONSUMED so far.  The prefetcher runs one round ahead: for every
        request whose prefetched batch is still unconsumed, its clients' cursors are the ones snapshotted right
        before that batch was drawn."""
        if not hasattr(self.dataset, "state_dict"):
            return {}
        for fut in list(self._pf_jobs.values()):
            fut.result()                                 # let in-flight draws finish before reading the streams
        cur = self.dataset.state_dict()
        for pre in list(self._pf_pre.values()):
            cur.update(pre)
        return cur

    def _graph_eligible(self, rows: List[int]) -> bool:
        """CUDA-graph replay of the batched step needs every hook to be a pure device-tensor function:
        true for the stock client classes; user subclasses run eagerly."""
        import os
        if self.device.type != "cuda" or os.environ.get("BLADES_GRAPH", "1") == "0":
            return False
        return self._stock_types(rows)

    def _stock_types(self, rows: List[int]) -> bool:
        from .. import attackers as A
        stock = (BladesClient, A.NoiseClient, A.LabelflippingClient, A.SignflippingClient, A.AlieClient, A.IpmClient,
                 A.MinmaxClient, A.MinsumClient)
        return all(type(self.clients[self.local_idx[r]]) in stock for r in rows)

    def _train_batched(self, rows: List[int], lr: float) -> None:
        """fedsgd for the listed local rows in one fused forward/backward.  On CUDA the whole step
        (forward, backward, per-client wgrad epilogues into U) is captured once in a CUDA graph and
        replayed every round: the ~700 kernel launches of a ResNet-18 step cost one graph launch."""
        if self.prestaged is not None:           # device-resident inputs (kernel-only benchmarking)
            X, y = self.prestaged
            if X.shape[0] != len(rows):
                X, y = X[rows[0]: rows[-1] + 1], y[rows[0]: rows[-1] + 1]
        else:
            try:
                X, y = self.stage_batches(rows, 1)
            except RaggedBatches as e:
                self._train_ragged(rows, lr, e.batches)
                return
        self._shape_votes[tuple(X.shape)] = self._shape_votes.get(tuple(X.shape), 0) + 1
        if not self._graph_eligible(rows):
            self.last_client_losses = self._batched_step(rows, lr, X.clone(), y.clone())
            return
        key = (tuple(rows), float(lr), tuple(X.shape))
        entry = self._graphs.get(key)
        if entry is None and not self._worth_capturing(self._graphs, key, lr):
            # first round with this (rows, lr, shape): run eagerly; a graph is captured when it comes back
            self.last_client_losses = self._batched_step(rows, lr, X.clone(), y.clone())
            return
        if entry is None:
            self._clamp_tensor(rows)
            self._clamps_in_graphs.add(tuple(rows))
            sx, sy = X.clone(), y.clone()        # static input buffers owned by the graph
            side = torch.cuda.Stream(device=self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(side):        # warm-up: autotuning, lazy inits, smem attributes
                for _ in range(2):
                    sx.copy_(X)
                    sy.copy_(y)
                    self._batched_step(rows, lr, sx, sy)
            torch.cuda.current_stream(self.device).wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            sx.copy_(X)
            sy.copy_(y)
            from ..ops import _loader
            before = _loader.LAUNCHES
            with torch.cuda.graph(graph, capture_error_mode=_CAPTURE_MODE):
                losses = self._batched_step(rows, lr, sx, sy)
            entry = self._graphs[key] = (graph, sx, sy, losses, _loader.LAUNCHES - before)
            _loader.count_launch(-entry[4])          # capture does not execute
        graph, sx, sy, losses, n_native = entry
        sx.copy_(X, non_blocking=True)
        sy.copy_(y, non_blocking=True)
        graph.replay()
        self.flush_prefetch()
        from ..ops import _loader
        _loader.count_launch(n_native)               # our kernels inside the replayed graph
        self.last_client_losses = losses

    def _worth_capturing(self, cache: dict, key, lr: float) -> bool:
        """Capture policy shared by the step graphs and the fedavg visit graphs.  The learning rate is baked into a
        captured graph (it is the epilogue scale of the wgrad / BatchNorm kernels), so a schedule that changes it
        every round would otherwise capture -- and keep -- a new graph per round.  A key is captured the SECOND time
        it is requested; graphs of at most two distinct learning rates are kept (piecewise-constant schedules such
        as the reference's MultiStepLR replay graphs almost always; continuously varying ones simply run eagerly)."""
        seen = self._graph_seen[key] = self._graph_seen.get(key, 0) + 1
        if len(self._graph_seen) > 512:
            self._graph_seen = {key: seen}
        if seen < 2:
            return False
        lrs = []
        for k in cache:
            if self._graph_lr[k] not in lrs:
                lrs.append(self._graph_lr[k])
        if float(lr) not in lrs and len(lrs) >= 2:
            for k in [k for k in cache if self._graph_lr[k] == lrs[0]]:
                del cache[k], self._graph_lr[k]
        self._graph_lr[key] = float(lr)
        return True

    def _train_ragged(self, rows: List[int], lr: float, batches) -> None:
        """fedsgd round whose batches have different sizes (tail batches of shards that are not a multiple of the
        batch size, out of phase across clients): one eager fused pass per size group.  The reference just trains
        each client on whatever its generator yields (client.py:178-193)."""
        groups = {}
        for r in rows:
            x, _ = batches[self.clients[self.local_idx[r]].id()][0]
            groups.setdefault(tuple(x.shape), []).append(r)
        losses = torch.zeros(len(rows), device=self.device)
        pos = {r: i for i, r in enumerate(rows)}
        for _, grp in sorted(groups.items(), key=lambda kv: kv[1][0]):
            xs = torch.stack([batches[self.clients[self.local_idx[r]].id()][0][0] for r in grp])
            ys = torch.stack([batches[self.clients[self.local_idx[r]].id()][0][1] for r in grp])
            X = xs.unsqueeze(1).to(self.device, torch.float32)
            y = ys.unsqueeze(1).to(self.device)
            losses[[pos[r] for r in grp]] = self._batched_step(grp, lr, X, y).to(losses.dtype)
        self.last_client_losses = losses

    # -- whole-round CUDA graph ------------------------------------------------------------
    def all_rows_static(self) -> bool:
        import os
        if os.environ.get("BLADES_ROUND_GRAPH", "1") == "0":
            return False
        rows = list(range(len(self.local_idx)))
        if not rows or not self.batchable_model or self.client_opt_spec not in ("SGD", None, torch.optim.SGD):
            return False
        if self.max_batched_clients and self.max_batched_clients < len(rows):
            return False
        return self._graph_eligible(rows) and all(
            self._stock_for_batching(self.clients[self.local_idx[r]]) for r in rows)

    def static_round(self, lr: float, aggregate_fn, matrix_fn) -> bool:
        """Run one complete round through a captured CUDA graph.  The first two rounds with a given
        (lr, server lr) run eagerly (they are real rounds and serve as warm-up); the third is captured and
        replayed.  Returns False when the caller must run the round eagerly."""
        rows = list(range(len(self.local_idx)))
        key = (float(lr), float(self.server.current_lr()))
        st = self._round_graphs.get(key)
        if st is None:
            if len(self._round_graphs) >= 2:           # bounded: each graph owns an activation pool
                self._round_graphs.pop(next(iter(self._round_graphs)))
            st = self._round_graphs[key] = {"seen": 0}
        st["seen"] += 1
        if st.get("disabled") or st["seen"] <= 2:
            return False
        from ..ops import _loader
        if self.prestaged is not None:
            X, y = self.prestaged
        else:
            try:
                X, y = self.stage_batches(rows, 1)
            except RaggedBatches as e:
                self._stash[(tuple(rows), 1)] = e        # the eager round picks these batches up again
                return False
        shape = tuple(X.shape)
        votes = self._shape_votes[shape] = self._shape_votes.get(shape, 0) + 1
        if ("graph" in st and shape != tuple(st["sx"].shape)) or ("graph" not in st and votes < 2):
            # the shorter tail batch of an epoch: neither replay the captured graph with it nor spend the one
            # whole-round capture on it -- hand the inputs to the per-step path
            self._stash[(tuple(rows), 1)] = (X, y)
            return False
        if "graph" not in st:
            sx, sy = X.clone(), y.clone()
            self._clamp_tensor(rows)
            self._clamps_in_graphs.add(tuple(rows))
            torch.cuda.synchronize(self.device)
            graph = torch.cuda.CUDAGraph()
            before = _loader.LAUNCHES
            try:
                pipe = _AggPipeline(self, aggregate_fn) if (self._pipeline_enabled() and getattr(self, "agg_windows_ok", True)) else None
                with torch.cuda.graph(graph, stream=self._capture_stream(), capture_error_mode=_CAPTURE_MODE):
                    if pipe is None:
                        losses = self._batched_step(rows, lr, sx, sy)
                        agg = aggregate_fn()
                    else:
                        # aggregation of the coordinates whose backward pass is done starts on a side stream while
                        # the rest of the backward pass still runs (fork / join inside the captured graph)
                        losses = self._batched_step(rows, lr, sx, sy, progress=pipe.progress)
                        agg = pipe.finish()
                        st["chunks"] = pipe.windows
                mat = matrix_fn()
                ok = mat is not None and mat.step_applied
            except Exception as e:     # capture is an optimisation: fall back to eager rounds, but say so
                ok = False
                torch.cuda.synchronize(self.device)
                import logging
                logging.getLogger("debug").warning(f"whole-round CUDA graph capture failed, running eagerly: {e!r}")
            n_native = _loader.LAUNCHES - before
            _loader.count_launch(-n_native)
            if not ok:
                st["disabled"] = True
                if self.prestaged is None:
                    self._stash[(tuple(rows), 1)] = (X, y)      # the eager round trains on these inputs
                return False
            st.update(graph=graph, sx=sx, sy=sy, losses=losses, agg=agg, n_native=n_native)
            import os
            if os.environ.get("BLADES_GC_FREEZE", "1") != "0":
                # the simulation's long-lived objects (clients, datasets, captured graph state) are in place: keep the
                # cyclic collector from rescanning them -- a full collection is a multi-10-ms host stall, which at
                # 8 GPUs (2.7 ms rounds, every rank waiting for the slowest at the device barrier) shows up as a
                # whole-job hiccup
                import gc
                gc.collect()
                gc.freeze()
        st["sx"].copy_(X, non_blocking=True)
        st["sy"].copy_(y, non_blocking=True)
        st["graph"].replay()
        self.flush_prefetch()
        _loader.count_launch(st["n_native"])
        self.last_client_losses = st["losses"]
        self.static_aggregate = st["agg"]
        return True

    def _clamp_tensor(self, rows: List[int]) -> torch.Tensor:
        """Per-client loss clamps as a device tensor (cached: no H2D copy inside a graph capture)."""
        key = tuple(rows)
        t = self._clamps.get(key)
        if t is None and len(self._clamps) > 256:        # ragged rounds request ever-changing row groups
            # captured graphs have the address of their clamp tensor baked in: those entries must stay alive
            self._clamps = {k: v for k, v in self._clamps.items() if k in self._clamps_in_graphs}
        if t is None:
            t = self._clamps[key] = torch.tensor(
                [float(self.clients[self.local_idx[r]].loss_clamp) for r in rows], device=self.device)
        return t

    def losses_to_host_async(self) -> Optional["_HostRead"]:
        """Start a device->host copy of this round's per-client losses into a pinned double buffer, stream ordered
        after the round, and return a handle whose ``get()`` waits for THAT copy only.  Lets a driver loop issue round
        r+1 (host indices, graph launch) before it reads the result of round r, so the host work of a round hides
        behind the previous round's GPU time instead of leaving the GPU idle between rounds (the reference reads every
        client's loss synchronously inside the training loop, client.py:190)."""
        t = self.last_client_losses
        if t is None or not t.is_cuda:
            return None
        slots = getattr(self, "_loss_slots", None)
        if slots is None or slots[0][0].numel() != t.numel():
            slots = self._loss_slots = [(torch.empty(t.numel(), dtype=t.dtype).pin_memory(), torch.cuda.Event())
                                        for _ in range(2)]
            self._loss_turn = 0
        buf, ev = slots[self._loss_turn]
        self._loss_turn ^= 1
        buf.copy_(t.reshape(-1), non_blocking=True)
        ev.record(torch.cuda.current_stream(self.device))
        return _HostRead(buf, ev)

    def _pipeline_enabled(self) -> bool:
        import os
        return os.environ.get("BLADES_AGG_PIPELINE", "1") != "0"

    def _capture_stream(self) -> torch.cuda.Stream:
        """Stream the whole-round graph is captured on: one priority level above the aggregation side stream, so the
        block scheduler serves the (latency-bound) training chain first and the streaming aggregation kernels fill
        the SMs it leaves idle."""
        if getattr(self, "_cap_stream", None) is None:
            self._cap_stream = torch.cuda.Stream(device=self.device, priority=-1)
            self._agg_stream = torch.cuda.Stream(device=self.device, priority=0)
        return self._cap_stream

    def _batched_step(self, rows: List[int], lr: float, X: torch.Tensor, y: torch.Tensor, progress=None) -> torch.Tensor:
        """X: [n, 1, B, ...], y: [n, 1, B] on the device (may be modified in place by client hooks).
        ``progress``: see ``resnet_fused.step`` (ignored when rows need a post-pass: sign flips, scattered rows)."""
        model = self.server.get_model()
        n = len(rows)
        X = X[:, 0]
        y = y[:, 0]
        B = X.shape[1]
        clamp = self._clamp_tensor(rows)
        signs = []
        for j, r in enumerate(rows):
            c = self.clients[self.local_idx[r]]
            if _overrides(c, "on_train_batch_begin"):
                xj, yj = c.on_train_batch_begin(data=X[j], target=y[j])
                if xj is not X[j]:
                    X[j] = xj
                y[j] = yj
            if getattr(c, "grad_sign", 1.0) != 1.0:
                signs.append((r, float(c.grad_sign)))
        contiguous_rows = rows == list(range(rows[0], rows[0] + n))
        out = self.U[rows[0]: rows[0] + n] if contiguous_rows else torch.empty(n, self.d, device=self.device)
        sink = cb.GradSink(out, self.gflat.specs, n, alpha=-lr)
        model.train()
        if signs or not contiguous_rows:
            progress = None
        per_client = cb.batched_step(model, sink, X.reshape((n * B,) + tuple(X.shape[2:])), y.reshape(-1), n, clamp,
                                     progress)
        missing = [s.name for s in self.gflat.specs if s.name not in sink.written]
        for name in missing:       # parameters unused in the forward pass: zero update
            sink.view(name).zero_()
        if not contiguous_rows:
            self.U[rows] = out
        for r, sgn in signs:
            self.U[r].mul_(sgn)
        return per_client

    # -- time-sliced (fedavg, custom clients) --------------------------------------------
    def _lend(self, c: BladesClient, lr: float):
        c.model = self.worker
        if self.client_opt_spec in ("SGD", None, torch.optim.SGD):
            c.optimizer = self.worker_opt
        else:
            c.optimizer = self.client_opt_spec(self.worker.parameters(), lr=lr)
        c.set_lr(lr)

    # -- fedavg for stock clients: one captured CUDA graph per client visit ---------------------------
    def _sliced_graph_key(self, c: BladesClient, local_steps: int, lr: float, shape):
        return (type(c), float(getattr(c, "grad_sign", 1.0)), float(c.loss_clamp), getattr(c, "num_classes", None),
                local_steps, float(lr), tuple(shape))

    def _sliced_body(self, c: BladesClient, local_steps: int, lr: float, sx: torch.Tensor, sy: torch.Tensor,
                     scratch: torch.Tensor, wk=None) -> torch.Tensor:
        """k local SGD steps of one client on the shared worker model, written as pure device work:
        theta_w <- theta; k x (forward, clamp(CE), backward into the flat grad, theta_w -= lr*g);
        scratch <- theta_w - theta.  Same math as reference client.py:178-193 + 127-131."""
        worker, w = wk if wk is not None else (self.worker, self.wflat)
        g = self.gflat
        with torch.no_grad():
            w.theta.copy_(g.theta)
            for (_, bw), (_, bg) in zip(worker.named_buffers(), self.server.get_model().named_buffers()):
                bw.copy_(bg)
        worker.train()
        sign = float(getattr(c, "grad_sign", 1.0))
        loss = None
        import contextlib
        if self.batchable_model:
            # same layer functions as the client-batched engine with n = 1: parameter gradients come from our
            # tcgen05 wgrad / BN kernels straight into the flat grad vector (cuDNN's fp32 NHWC wgrad picks a
            # 0.6 ms "grouped_direct" fallback per conv at batch 32 -- 45 % of the eager step)
            sink = cb.GradSink(w.grad.view(1, -1), w.specs, 1, alpha=1.0)
            ctx = cb.client_batched(worker, sink, sx.shape[1])
        else:
            ctx = contextlib.nullcontext()
        with ctx:
            for j in range(local_steps):
                data, target = c.on_train_batch_begin(data=sx[j], target=sy[j])
                w.grad.zero_()
                out = worker(data)
                loss = torch.clamp(torch.nn.functional.cross_entropy(out, target), 0, float(c.loss_clamp))
                loss.backward()
                with torch.no_grad():
                    w.theta.add_(w.grad, alpha=-lr * sign)
        with torch.no_grad():
            _diff(w.theta, g.theta, scratch)
        return loss.detach()

    def _slice_workers(self, k: int):
        """k independent worker replicas (model + flat params + stream): client visits are tiny kernels, so
        several clients run concurrently on separate streams to fill the 148 SMs."""
        while len(self._workers) < k:
            if not self._workers:
                m, f = self.worker, self.wflat
            else:
                m = copy.deepcopy(self.worker)
                f = FlatParams(m, device=self.device)
            if f.grad is None:
                f.attach_grad()
            self._workers.append((m, f, torch.cuda.Stream(device=self.device)))
        return self._workers[:k]

    def _train_sliced_graphed(self, rows: List[int], local_steps: int, lr: float) -> List[int]:
        """Graph-replayed time slices for the stock clients among ``rows`` (CUDA).  Returns the rows that
        still need the eager path."""
        import os
        if self.device.type != "cuda" or self.client_opt_spec not in ("SGD", None, torch.optim.SGD):
            return rows
        # BLADES_GRAPH=0 runs the SAME body eagerly: the result of a run must not depend on the capture policy
        # (the stock autograd loop computes weight gradients in fp32 cuBLAS, the body with the tf32 tcgen05 kernels)
        use_graph = os.environ.get("BLADES_GRAPH", "1") != "0"
        todo = [r for r in rows if self._stock_types([r]) and self._stock_for_batching(self.clients[self.local_idx[r]])
                ]
        rest = [r for r in rows if r not in set(todo)]
        if not todo:
            return rest
        n_streams = max(1, min(int(os.environ.get("BLADES_SLICE_STREAMS", "8")), len(todo)))
        workers = self._slice_workers(n_streams)
        main = torch.cuda.current_stream(self.device)
        ready = torch.cuda.Event()
        ready.record(main)
        for i, r in enumerate(todo):
            wi = i % n_streams
            model_w, flat_w, stream = workers[wi]
            c = self.clients[self.local_idx[r]]
            prev = self._slice_copied.get(wi)
            if prev is not None:
                prev.synchronize()                     # the pinned slot of this worker is free again
            try:
                X, y = self.dataset.get_train_batches([c.id()], local_steps, slot=100 + wi)   # pinned [1,k,B,..]
            except RaggedBatches as e:
                # this visit contains a short tail batch: it runs on the eager time-sliced path with these batches
                self._ragged_data[r] = e.batches[c.id()]
                rest.append(r)
                continue
            X, y = X[0], y[0]
            key = (wi,) + self._sliced_graph_key(c, local_steps, lr, X.shape)
            st = self._sliced_graphs.get(key)
            if st is None and not (use_graph and self._worth_capturing(self._sliced_graphs, key, lr)):
                # not (yet) captured: the same body, eagerly, on this worker's stream
                with torch.cuda.stream(stream):
                    stream.wait_event(ready)
                    ek = ("eager", wi, tuple(X.shape))
                    bufs = self._eager_slice_bufs.get(ek)
                    if bufs is None:
                        bufs = self._eager_slice_bufs[ek] = (
                            torch.empty(X.shape, device=self.device, dtype=torch.float32),
                            torch.empty(y.shape, device=self.device, dtype=torch.int64),
                            torch.empty(self.d, device=self.device, dtype=torch.float32))
                    sx, sy, scratch = bufs
                    sx.copy_(X, non_blocking=True)
                    sy.copy_(y, non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record(stream)
                    self._slice_copied[wi] = ev
                    self._sliced_body(c, local_steps, lr, sx, sy, scratch, (model_w, flat_w))
                    self.U[r].copy_(scratch)
                c._state["saved_update"] = self.U[r]
                continue
            with torch.cuda.stream(stream):
                stream.wait_event(ready)
                if st is None:
                    sx = torch.empty(X.shape, device=self.device, dtype=torch.float32)
                    sy = torch.empty(y.shape, device=self.device, dtype=torch.int64)
                    scratch = torch.empty(self.d, device=self.device, dtype=torch.float32)
                    sx.copy_(X)
                    sy.copy_(y)
                    for _ in range(2):                       # warm-up on this stream
                        self._sliced_body(c, local_steps, lr, sx, sy, scratch, (model_w, flat_w))
                    stream.synchronize()
                    graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(graph, stream=stream, capture_error_mode=_CAPTURE_MODE):
                        loss = self._sliced_body(c, local_steps, lr, sx, sy, scratch, (model_w, flat_w))
                    st = self._sliced_graphs[key] = (graph, sx, sy, scratch, loss)
                graph, sx, sy, scratch, loss = st
                sx.copy_(X, non_blocking=True)
                sy.copy_(y, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(stream)
                self._slice_copied[wi] = ev
                graph.replay()
                self.U[r].copy_(scratch)
            c._state["saved_update"] = self.U[r]
        for _, _, stream in workers:
            main.wait_stream(stream)
        return sorted(rest)

    def _train_timesliced(self, r: int, local_steps: int, lr: float) -> None:
        gi = self.local_idx[r]
        c = self.clients[gi]
        with torch.no_grad():
            self.wflat.theta.copy_(self.gflat.theta)
            for (_, bw), (_, bg) in zip(self.worker.named_buffers(), self.server.get_model().named_buffers()):
                bw.copy_(bg)
        self._lend(c, lr)
        custom_begin = _overrides(c, "on_train_round_begin")
        custom_end = _overrides(c, "on_train_round_end")
        if custom_begin or custom_end:
            c.on_train_round_begin()
        else:
            self.worker.train()
        data = self._ragged_data.pop(r, None)           # batches already drawn by a path that could not stack them
        if data is None:
            data = self.dataset.get_train_data(c.id(), local_steps)
        c.local_training(data_batches=data)
        if custom_end:
            c.on_train_round_end()          # client computes/saves its own update (lands in U via bind_row)
        else:
            with torch.no_grad():
                if not self.wflat.is_aliased():
                    self.wflat.realias()
                _diff(self.wflat.theta, self.gflat.theta, self.U[r])
                c._state["saved_update"] = self.U[r]
        c.model = None
        c.optimizer = None

    # ------------------------------------------------------------------ attack phase
    def fusable_attack(self, callbacks: Sequence[Callable]) -> Optional[VirtualRows]:
        """If every registered omniscient callback belongs to a stock ALIE / IPM / Min-Max / Min-Sum client with
        identical parameters, describe the attack as virtual rows."""
        if not callbacks:
            return None
        owners = []
        for fn in callbacks:
            owner = getattr(fn, "__self__", None)
            if not isinstance(owner, ByzantineClient):
                return None
            spec = owner.fused_spec()
            stock = any(type(owner).omniscient_callback is getattr(k, "omniscient_callback")
                        for k in _fusable_classes())
            if spec is None or not stock:
                return None
            owners.append((owner, spec))
        kinds = {(s["kind"], round(s["param"], 12), s.get("dev_type"), s.get("gamma_init"), s.get("tol"))
                 for _, s in owners}
        if len(kinds) != 1:
            return None
        idx_of = {id(c): i for i, c in enumerate(self.clients)}
        replaced = sorted(idx_of[id(o)] for o, _ in owners if id(o) in idx_of)
        if len(replaced) != len(owners):
            return None
        byz = [i for i, c in enumerate(self.clients) if c.is_byzantine()]
        spec = owners[0][1]
        if spec["kind"] in ("minmax", "minsum"):
            clients = [o for o, _ in owners]

            def report(gamma):              # every attacker's ``gamma`` property reads the last scale
                for o in clients:
                    o._set_gamma(gamma)
            return VirtualRows(spec["kind"], spec["param"], replaced, byz, dev_type=spec["dev_type"],
                               gamma_init=spec["gamma_init"], tol=spec["tol"], report=report)
        return VirtualRows(spec["kind"], spec["param"], replaced, byz)

    # ------------------------------------------------------------------ aggregation
    def make_matrix(self, virtual: Optional[VirtualRows] = None, window=None, chunk: int = 0, last: bool = True,
                    out: Optional[torch.Tensor] = None, recv_col: int = 0) -> UpdateMatrix:
        """``window`` / ``chunk`` / ``last`` / ``out`` / ``recv_col``: pipelined aggregation (``_AggPipeline``) -- the
        matrix covers coordinates ``[window[0], window[1])`` only; see ``UpdateMatrix.window``."""
        if self.symm is not None:
            from ..parallel.sharded import ShardedMatrix
            return ShardedMatrix(self.symm, virtual, window=window, chunk=chunk, last_chunk=last, recv_col=recv_col)
        # no symmetric memory (CPU / gloo): gather the rows; every rank aggregates identically
        U = self.gather_dense()
        return LocalMatrix(U, virtual, use_kernels=self.use_kernels and U.is_cuda, theta=self.gflat.theta,
                           window=window, chunk=chunk, last_chunk=last, out_buffer=out)

    def gather_dense(self) -> torch.Tensor:
        """Dense [N, d] on every rank (escape hatch for custom callbacks/aggregators)."""
        if not self.world.distributed:
            return self.U
        import os
        if os.environ.get("BLADES_FORBID_DENSE_GATHER", "0") == "1":
            raise RuntimeError("dense [N, d] gather requested while BLADES_FORBID_DENSE_GATHER=1")
        import torch.distributed as dist
        nmax = max(self.shard_sizes)
        pad = torch.zeros(nmax, self.d, device=self.U.device)
        pad[: self.U.shape[0]] = self.U
        out = [torch.empty_like(pad) for _ in range(self.world.size)]
        dist.all_gather(out, pad)
        return torch.cat([o[:k] for o, k in zip(out, self.shard_sizes)], 0)

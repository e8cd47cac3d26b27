"""``Simulator``: synchronous Byzantine-robust FL simulation, B200-native runtime.

Public surface = the reference's (/root/reference/src/blades/simulator.py:44-61,
364-378; SURVEY Appendix A): same constructor and ``run`` keyword arguments, same
name-based plugin lookup for aggregators (``aggregators.<name>.<Name>``) and
attackers (``attackers.<name>client.<Name>Client``), same hooks and log records.

What changed underneath (SURVEY 7.1/7.2): no Ray.  The program is SPMD -- launched
once (1 GPU / CPU) or under ``torchrun`` with one process per GPU.  Every rank holds a
replica of the global parameters as one flat device vector, hosts the virtual clients
``np.array_split`` assigns to it (the reference's client->actor split, simulator.py:223)
and keeps their update rows in NVLink-addressable memory.  A round is:
``engine.train_local`` -> attack phase (virtual rows or callbacks) -> aggregator on an
``UpdateMatrix`` (fused pull-mode kernels) -> server step (fused into the aggregation
epilogue when the optimizer is plain SGD).

Arguments that only made sense for Ray (``num_actors``, ``num_trainers``,
``gpu_per_actor``, ``mode``) are accepted and ignored; the world size decides the
number of trainer shards.
"""
from __future__ import annotations

import importlib
import logging
from time import time
from typing import Any, Callable, Dict, List, Optional, Union

import numpy as np
import torch

from .client import BladesClient, ByzantineClient
from .comm.group import World, get_world
from .datasets.dataset import FLDataset
from .engine.round import RoundEngine
from .parallel.matrix import SCALED_KINDS, VirtualRows
from .server import BladesServer
from .utils import initialize_logger, reset_model_weights, set_random_seed, top1_accuracy

__all__ = ["Simulator"]

BUILTIN_ATTACKS = ("noise", "labelflipping", "signflipping", "alie", "ipm", "minmax", "minsum")


class _NullBar:
    def __init__(self, it):
        self._it = it

    def __iter__(self):
        return iter(self._it)

    def set_postfix(self, **kw):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def _progress(total: int, enabled: bool):
    rng = range(1, total + 1)
    if enabled:
        try:
            from tqdm import trange
            return trange(1, total + 1)
        except Exception:  # pragma: no cover
            pass
    return _NullBar(rng)


class Simulator(object):
    """Synchronous and parallel training with specified aggregators.

    :param dataset: ``FLDataset`` or a ``BaseDataset`` (``.get_dls()`` is called).
    :param aggregator: name of a built-in scheme or a callable ``inputs -> Tensor[d]``.
    :param num_byzantine: number of Byzantine clients under a built-in attack (first ids).
    :param attack: ``None`` | ``noise`` | ``labelflipping`` | ``signflipping`` | ``alie`` | ``ipm``.
    :param log_path: directory of the ``stats`` / ``debug`` log files (wiped on construction).
    :param use_cuda: place clients/server on the GPU of this rank.
    :param seed: seed for python/numpy/torch (``None`` = do not seed).
    """

    def __init__(
            self,
            dataset: FLDataset,
            num_byzantine: Optional[int] = 0,
            attack: Optional[str] = None,
            attack_kws: Optional[Dict[str, float]] = None,
            aggregator: Union[Callable[[list], torch.Tensor], str] = 'mean',
            aggregator_kws: Optional[Dict[str, float]] = None,
            num_actors: Optional[int] = 1,
            num_trainers: Optional[int] = 1,
            gpu_per_actor: Optional[float] = 0,
            mode: Optional[str] = 'actor',
            log_path: str = "./outputs",
            metrics: Optional[dict] = None,
            use_cuda: Optional[bool] = False,
            seed: Optional[int] = None,
            **kwargs,
    ):
        # engine options are accepted through kwargs so the reference signature stays intact
        self._opts = {
            "world": kwargs.pop("world", None),
            "fuse_attack": kwargs.pop("fuse_attack", True),
            "fuse_server_step": kwargs.pop("fuse_server_step", True),
            "use_kernels": kwargs.pop("use_kernels", None),
            "progress": kwargs.pop("progress", True),
            "profile": kwargs.pop("profile", False),
            "wipe_logs": kwargs.pop("wipe_logs", True),
        }
        self.use_actor = mode == 'actor'
        want_cuda = bool(use_cuda) or (gpu_per_actor is not None and gpu_per_actor > 0.0)
        self.world: World = self._opts["world"] or get_world()
        if want_cuda:
            if not torch.cuda.is_available():
                raise RuntimeError("use_cuda=True but no CUDA device is visible")
            self.device = self.world.device if self.world.device.type == "cuda" else torch.device("cuda")
        else:
            self.device = torch.device("cpu")

        self._init_aggregator(aggregator=aggregator, aggregator_kws=aggregator_kws or {})

        self.log_path = log_path
        if self.world.rank == 0:
            initialize_logger(log_path, wipe=self._opts["wipe_logs"])
        self.world.barrier()
        self.metrics = {"top1": top1_accuracy} if metrics is None else metrics
        self.json_logger = logging.getLogger("stats")
        self.debug_logger = logging.getLogger("debug")
        self.debug_logger.info(str(self))

        self.random_states = {}
        self.omniscient_callbacks: List[Callable] = []

        if kwargs:
            unknown = ", ".join(kwargs)
            raise RuntimeError(f"Unknown keyword argument(s): {unknown}")

        if isinstance(dataset, FLDataset):
            self.dataset = dataset            # (the reference forgets this branch, Q10)
        else:
            traindls, testdls = dataset.get_dls()
            self.dataset = FLDataset(traindls, testdls)

        self._setup_clients(attack, num_byzantine=num_byzantine, attack_kws=attack_kws or {})
        self.seed = seed
        set_random_seed(seed, use_cuda=self.device.type == "cuda")

        self.engine: Optional[RoundEngine] = None
        self.server: Optional[BladesServer] = None
        self.round = 0
        self.client_lr = None
        self.last_aggregate: Optional[torch.Tensor] = None

    # ------------------------------------------------------------------ plugin lookup
    def _init_aggregator(self, aggregator, aggregator_kws):
        if isinstance(aggregator, str):
            mod = importlib.import_module(f'{__package__}.aggregators.{aggregator}')
            self.aggregator = getattr(mod, aggregator.capitalize())(**aggregator_kws)
        else:
            self.aggregator = aggregator

    def _setup_clients(self, attack: Optional[str], num_byzantine, attack_kws):
        if attack is None:
            num_byzantine = 0
        self._clients: Dict[Any, BladesClient] = {}
        for i, u in enumerate(self.dataset.get_clients()):
            if i < num_byzantine:
                mod = importlib.import_module(f'{__package__}.attackers.{attack}client')
                cls = getattr(mod, f'{attack.capitalize()}Client')
                client = cls(id=u, device=self.device, **attack_kws)
                self._register_omniscient_callback(client.omniscient_callback)
            else:
                client = BladesClient(id=u, device=self.device)
            self._clients[u] = client

    def _register_omniscient_callback(self, callback):
        self.omniscient_callbacks.append(callback)

    # ------------------------------------------------------------------ client management
    def get_clients(self) -> List[BladesClient]:
        """All clients, in id order."""
        return list(self._clients.values())

    def set_trusted_clients(self, ids: List) -> None:
        """Mark clients as trusted (used by trust-bootstrapped aggregators such as FLTrust)."""
        for i in ids:
            self._clients[i].trust()

    def register_attackers(self, clients: List[ByzantineClient], replace_indices=None) -> None:
        """Install custom Byzantine clients: ``clients[k]`` replaces the client at position
        ``replace_indices[k]`` (default: the first ``len(clients)`` positions) and inherits
        its id.  (The reference indexes ``clients`` by the *replace index* and asserts
        ``len(clients) < len(replace_indices)`` -- quirk Q11 -- which only works for the
        default; fixed here.)"""
        if replace_indices is None:
            replace_indices = list(range(len(clients)))
        assert len(clients) == len(replace_indices), "need one replace index per attacker"
        assert len(clients) < len(self._clients)
        current = self.get_clients()
        for k, pos in enumerate(replace_indices):
            cid = current[pos].id()
            clients[k].set_id(cid)
            clients[k].device = self.device
            self._clients[cid] = clients[k]
            self._register_omniscient_callback(clients[k].omniscient_callback)

    def reference_order(self, vec: torch.Tensor) -> torch.Tensor:
        """Convert an update / aggregate vector (or ``[.., d]`` matrix) from the engine's flat layout to the
        reference's coordinate order (``named_parameters()`` flattening, client.py:216-228).  On the GPU conv
        weights are stored channels_last ([Cout, kh, kw, Cin]) inside the flat vector, which permutes the
        coordinates *within* each conv weight; every built-in aggregator/attack is invariant to that."""
        return self.engine.gflat.to_reference_order(vec)

    # ------------------------------------------------------------------ RNG hygiene
    def cache_random_state(self) -> None:
        if self.device.type == "cuda":
            self.random_states["torch_cuda"] = torch.cuda.get_rng_state(self.device)
        self.random_states["torch"] = torch.get_rng_state()
        self.random_states["numpy"] = np.random.get_state()

    def restore_random_state(self) -> None:
        if self.device.type == "cuda":
            torch.cuda.set_rng_state(self.random_states["torch_cuda"], self.device)
        torch.set_rng_state(self.random_states["torch"])
        np.random.set_state(self.random_states["numpy"])

    def parallel_call(self, clients, f: Callable[[BladesClient], None]) -> None:
        self.cache_random_state()
        for c in clients:
            f(c)
        self.restore_random_state()

    def parallel_get(self, clients, f: Callable[[BladesClient], Any]) -> list:
        out = []
        for c in clients:
            self.cache_random_state()
            out.append(f(c))
            self.restore_random_state()
        return out

    # ------------------------------------------------------------------ one round
    def _aggregate(self, virtual: Optional[VirtualRows], window=None, chunk: int = 0, last: bool = True, out=None,
                   recv_col: int = 0):
        """``window`` / ``chunk`` / ``last`` / ``out``: pipelined aggregation (``RoundEngine.static_round``) -- aggregate
        only the coordinates ``[window[0], window[1])`` into the round's shared result vector."""
        eng = self.engine
        agg = self.aggregator
        from .aggregators.base import _BaseAggregator
        if isinstance(agg, _BaseAggregator) and type(agg).aggregate is _BaseAggregator.aggregate:
            # reference-style subclass: only ``__call__`` is overridden (it uses ``self._get_updates(inputs)``, e.g.
            # aggregators/byzantinesgd.py); no server-step fusion, no virtual rows (``_consumes_matrix``)
            self._last_matrix = None
            return agg(eng.make_matrix(None))
        if isinstance(agg, _BaseAggregator):
            from .aggregators.fltrust import Fltrust
            matrix = eng.make_matrix(virtual, window, chunk, last, out, recv_col)
            if self._opts["fuse_server_step"] and getattr(agg, "fusable_final", False) \
                    and self.server._flat_fast_path_ok() and matrix.use_kernels:
                matrix.server_step = (self.server.current_lr(),)
            self._last_matrix = matrix
            if isinstance(agg, Fltrust):
                trusted = [i for i, c in enumerate(self.get_clients()) if c.is_trusted()]
                assert len(trusted) == 1, "FLTrust needs exactly one trusted client"
                return agg.aggregate(matrix, trusted[0])
            return agg.aggregate(matrix)
        # custom callable: reference convention = list of clients (get_update() -> row view)
        if self.world.distributed:
            dense = eng.gather_dense()
            for i, c in enumerate(self.get_clients()):
                c._state["saved_update"] = dense[i]
        return agg(self.get_clients())

    def train_actor(self, global_round: int, num_rounds: int, clients: List[BladesClient], lr: float) -> None:
        """One communication round: local training of every client (``num_rounds`` local
        steps), attack callbacks, aggregation, server step."""
        eng = self.engine
        self.debug_logger.info(f"Train global round {global_round}")
        if self._static_round_possible(num_rounds):
            # whole round (train -> barrier -> fused attack+aggregate+server step -> barrier) as ONE CUDA
            # graph replay: no per-round Python/launch overhead (matters most when G GPUs split the work)
            virtual = self._cached_virtual()
            if eng.static_round(lr, lambda **kw: self._aggregate(virtual, **kw), lambda: self._last_matrix):
                self.last_aggregate = eng.static_aggregate
                return
        eng.timer.start("train")
        eng.train_local(num_rounds, lr)
        eng.timer.stop("train")

        eng.timer.start("aggregate")
        callbacks = self._active_callbacks()
        virtual = self._cached_virtual()
        self._round_index = int(global_round)
        if virtual is None and callbacks and self.world.distributed and \
                all(getattr(getattr(cb, "__self__", None), "row_local_attack", False) for cb in callbacks):
            # every attacker only rewrites ITS OWN row (NoiseClient): the rank that owns the client runs the callback
            # on the row where it lives -- no [N, d] gather over NCCL, no write-back (reference noiseclient.py:16-25)
            mine = set(eng.local_idx)
            index = {id(c): i for i, c in enumerate(self.get_clients())}
            for cb in callbacks:
                if index.get(id(cb.__self__)) in mine:
                    cb(self)
            callbacks = []
        if virtual is None and callbacks:
            if self.world.distributed:
                dense = eng.gather_dense()
                for i, c in enumerate(self.get_clients()):
                    c._state["saved_update"] = dense[i]
                    c._slot = None
            for cb in callbacks:
                cb(self)
            if self.world.distributed:
                # write the (possibly modified) local rows back into the shard matrix
                for gi in eng.local_idx:
                    c = self.get_clients()[gi]
                    eng.U[eng.row_of[gi]].copy_(c._state["saved_update"])
                    c.bind_row(eng.U, eng.row_of[gi])
        self._last_matrix = None
        aggregated = self._aggregate(virtual)
        self.last_aggregate = aggregated
        eng.timer.stop("aggregate")
        eng.timer.start("apply")
        if not (self._last_matrix is not None and self._last_matrix.step_applied):
            self.server.apply_update(aggregated)      # else: already done in the kernel epilogue
        eng.timer.stop("apply")
        eng.timer.flush()

    def _active_callbacks(self) -> List[Callable]:
        """Registered omniscient callbacks minus the inherited no-op (label/sign flipping clients register
        ``ByzantineClient.omniscient_callback``, which does nothing)."""
        noop = ByzantineClient.omniscient_callback
        return [cb for cb in self.omniscient_callbacks if getattr(cb, "__func__", None) is not noop]

    def _cached_virtual(self):
        cbs = self._active_callbacks()
        key = tuple(id(cb) for cb in cbs)
        if getattr(self, "_virt_key", None) != key:
            self._virt_key = key
            self._virt_val = self.engine.fusable_attack(cbs) if (self._opts["fuse_attack"] and cbs
                                                                 and self._consumes_matrix()) else None
        return self._virt_val

    def _consumes_matrix(self) -> bool:
        """Virtual (fused) attack rows exist only inside an ``UpdateMatrix``: they may replace the attacker callbacks
        only when the aggregator is a built-in style ``_BaseAggregator`` implementing ``aggregate(matrix)``.  A plain
        callable, or a reference-style subclass that overrides only ``__call__``, sees the clients' real rows, so
        the callbacks must run for it."""
        from .aggregators.base import _BaseAggregator
        agg = self.aggregator
        return isinstance(agg, _BaseAggregator) and type(agg).aggregate is not _BaseAggregator.aggregate

    def _static_round_possible(self, local_steps: int) -> bool:
        """The round is a fixed sequence of device work (no host decisions): fedsgd on the batched engine,
        attack fused as virtual rows (or none), coordinate-wise built-in aggregator, fused SGD server step."""
        from .aggregators import Autogm, Centeredclipping, Fltrust, Geomed, Krum, Mean, Median, Multikrum, Trimmedmean
        eng = self.engine
        if local_steps != 1 or eng.device.type != "cuda" or eng.timer.enabled or not self._opts["fuse_server_step"]:
            return False
        coordwise = type(self.aggregator) in (Mean, Median, Trimmedmean)
        # Gram-based aggregators whose solver runs on the device (ops/gram_solve) are a fixed sequence of launches too:
        # Gram pass -> (in-switch reduce) -> solver -> combine with device-resident weights
        from .ops import gram_solve
        devsolve = type(self.aggregator) in (Krum, Multikrum, Geomed, Autogm, Centeredclipping, Fltrust) and gram_solve.enabled() \
            and eng.use_kernels
        virtual = self._cached_virtual() if self._active_callbacks() else None
        # only coordinate-wise aggregators can be pipelined window by window, and only when the attack is
        # coordinate-wise as well: the Min-Max / Min-Sum scale depends on every coordinate
        scaled = virtual is not None and virtual.kind in SCALED_KINDS
        eng.agg_windows_ok = coordwise and not scaled
        if not (coordwise or devsolve) or not self.server._flat_fast_path_ok():
            return False
        if self._active_callbacks() and virtual is None:
            return False
        if scaled:
            # the scale search must stay on the device (a host solve syncs, and a capture fails on a sync)
            from .ops import gram as _gram
            if not (gram_solve.enabled() and eng.use_kernels and _gram.PRECISION != "fp32"):
                return False
        return eng.all_rows_static()

    def train_trainer(self, epoch, num_rounds, clients):
        """``mode='trainer'`` of the reference is non-functional (quirk Q1); it maps onto the
        same engine path here."""
        cl = list(clients.values()) if isinstance(clients, dict) else list(clients)
        self.train_actor(epoch, num_rounds, cl, self.client_lr)

    # ------------------------------------------------------------------ evaluation
    def test_actor(self, global_round, batch_size):
        """Evaluate the global model on every client's test shard (length-weighted)."""
        eng = self.engine
        model = self.server.get_model()
        records = self._test_fused(global_round, batch_size)
        if records is None:
            records = self._test_batched(global_round, batch_size)
        if records is None:
            records = []
            for gi in eng.local_idx:
                c = self.get_clients()[gi]
                data = self.dataset.get_all_test_data(c.id())
                records.append(c.evaluate(round_number=global_round, test_set=data, batch_size=batch_size,
                                          metrics=self.metrics, use_actor=True, model=model))
        if self.world.distributed:
            records = [r for part in self.world.all_gather_object(records) for r in part]
        loss, top1 = self.log_validate(records)
        self.debug_logger.info(f"Test global round {global_round}, loss: {loss}, top1: {top1}")
        return loss, top1

    def _eval_shards(self, clients):
        """Device-resident copies of the local test shards (cached): ``(X, y, lens)`` or None when a shard is not a
        deterministic tensor dataset."""
        from .datasets.customdataset import CustomTensorDataset
        cache = getattr(self, "_eval_cache", None)
        if cache is None:
            xs, ys, lens = [], [], []
            for c in clients:
                ds = self.dataset.get_all_test_data(c.id())
                if not isinstance(ds, CustomTensorDataset) or not ds.deterministic:
                    return None
                x, y = ds.tensors
                if ds.transforms is not None and len(x):
                    x = torch.stack([ds.transforms(xi) for xi in x])
                xs.append(x), ys.append(y), lens.append(len(y))
            if min(lens) == 0:
                return None
            dev = self.engine.device
            seg = torch.repeat_interleave(torch.arange(len(lens)), torch.tensor(lens))
            cache = self._eval_cache = (torch.cat(xs).to(dev), torch.cat(ys).to(dev), seg.to(dev), lens)
        return cache

    def _test_fused(self, global_round, batch_size):
        """Evaluation of the ResNet family through the own-kernel forward pass (``engine/resnet_fused.py``; SURVEY
        K10).  The reference evaluates client by client in batches of ``batch_size`` (client.py:144-176); these models
        normalise with the statistics of every forward batch, so the grouping matters: each evaluation batch of the
        reference becomes one statistics group of ONE fused forward over all local clients' test data (batches of the
        same size share a launch; the shorter tail batches of the shards form a second one).  Same per-client
        records, one host sync.  Returns None when the conditions do not hold."""
        import torch.nn as nn

        eng = self.engine
        clients = [self.get_clients()[gi] for gi in eng.local_idx]
        if not clients or eng.device.type != "cuda" or set(self.metrics) != {"top1"} \
                or self.metrics["top1"] is not top1_accuracy:
            return None
        from .engine.round import _default_ce
        if any(type(c).evaluate is not BladesClient.evaluate or not _default_ce(c.loss_func) for c in clients):
            return None
        model = self.server.get_model()
        from .engine import resnet_fused as rf
        shards = self._eval_shards(clients)
        if shards is None or not rf.supports_eval(model, shards[0]):
            return None
        X, y, _, lens = shards
        from .ops import fused as kf
        bs = int(batch_size)
        # contiguous runs of equally sized evaluation batches: (first sample, batch size, owners of the batches).  The
        # shards sit back to back in X, so the full batches of consecutive clients form ONE run (a slice, no gather)
        # unless a shorter tail batch interrupts it.
        runs, start = [], 0
        for j, n in enumerate(lens):
            for o in range(0, n, bs):
                size = min(bs, n - o)
                if runs and runs[-1][1] == size and runs[-1][0] + size * len(runs[-1][2]) == start + o:
                    runs[-1][2].append(j)
                else:
                    runs.append((start + o, size, [j]))
            start += n
        max_groups = max(1, 8192 // bs)                                    # bound the activation footprint
        pending = []
        for first, size, owners in runs:
            for g0 in range(0, len(owners), max_groups):
                part = owners[g0: g0 + max_groups]
                a = first + g0 * size
                b = a + len(part) * size
                logits = rf.forward_logits(model, X[a:b], len(part))
                gl, gh = kf.group_eval(logits, y[a:b], len(part))
                pending.append((part, size, gl, gh))
        stats = np.zeros((2, len(lens)))
        for part, size, gl, gh in pending:                           # host syncs only after everything is queued
            np.add.at(stats[0], part, gl.cpu().numpy().astype(np.float64) * size)
            np.add.at(stats[1], part, gh.cpu().numpy().astype(np.float64))
        records = []
        for j, c in enumerate(clients):
            rec = {"_meta": {"type": "client_validation"}, "E": global_round, "Length": lens[j],
                   "Loss": float(stats[0, j]) / lens[j], "top1": 100.0 * float(stats[1, j]) / lens[j]}
            c._json_logger.info(rec)
            records.append(rec)
        return records

    def _test_batched(self, global_round, batch_size):
        """Evaluation fast path (SURVEY K10): the reference evaluates client by client in batches of
        ``batch_size`` (client.py:144-176, ~2 small forwards + 2 host syncs per client).  When the result cannot
        depend on how samples are grouped -- default top-1 metric, cross-entropy, stock ``evaluate``, test shards
        without a random per-item transform, no batch-statistics BatchNorm in eval mode -- all local test shards
        are cached on the device once, pushed through the global model in large chunks, and per-sample loss /
        correctness are segment-reduced per client: same per-client records, one host sync.  Returns ``None`` when
        any condition fails (the caller then runs the per-client loop)."""
        import torch.nn as nn
        import torch.nn.functional as F

        from .datasets.customdataset import CustomTensorDataset
        eng = self.engine
        clients = [self.get_clients()[gi] for gi in eng.local_idx]
        if not clients or set(self.metrics) != {"top1"} or self.metrics["top1"] is not top1_accuracy:
            return None
        if any(type(c).evaluate is not BladesClient.evaluate or not isinstance(c.loss_func, nn.CrossEntropyLoss)
               for c in clients):
            return None
        model = self.server.get_model()
        if any(isinstance(m, nn.modules.batchnorm._BatchNorm) and not m.track_running_stats for m in model.modules()):
            return None
        cache = self._eval_shards(clients)
        if cache is None:
            return None
        X, y, seg, lens = cache
        was_training = model.training
        model.eval()
        chunk = max(int(batch_size), 4096)
        loss_sum = torch.zeros(len(lens), device=X.device, dtype=torch.float64)
        hit_sum = torch.zeros(len(lens), device=X.device, dtype=torch.float64)
        with torch.no_grad():
            for i in range(0, len(y), chunk):
                out = model(X[i:i + chunk])
                yy = y[i:i + chunk]
                loss_sum.index_add_(0, seg[i:i + chunk], F.cross_entropy(out, yy, reduction="none").double())
                hit_sum.index_add_(0, seg[i:i + chunk], (out.argmax(1) == yy).double())
        model.train(was_training)
        stats = torch.stack([loss_sum, hit_sum]).cpu()              # the one host sync
        records = []
        for j, c in enumerate(clients):
            rec = {"_meta": {"type": "client_validation"}, "E": global_round, "Length": lens[j],
                   "Loss": float(stats[0, j]) / lens[j], "top1": 100.0 * float(stats[1, j]) / lens[j]}
            c._json_logger.info(rec)
            records.append(rec)
        return records

    # ------------------------------------------------------------------ logging
    def log_variance(self, cur_round, update):
        stack = torch.vstack(list(update)) if not torch.is_tensor(update) else update
        var = torch.var(stack, dim=0, unbiased=False)
        rec = {"_meta": {"type": "variance"}, "Round": cur_round, "avg": var.mean().item(),
               "norm": var.norm().item(), "avg_norm": (var / (stack ** 2).mean(0)).mean().item()}
        if self.world.rank == 0:
            self.json_logger.info(rec)
        return rec

    def log_validate(self, metrics):
        lengths = [m['Length'] for m in metrics]
        top1 = float(np.average([m['top1'] for m in metrics], weights=lengths)) if 'top1' in metrics[0] else float('nan')
        loss = float(np.average([m['Loss'] for m in metrics], weights=lengths))
        rec = {"_meta": {"type": "test"}, "Round": metrics[0]['E'], "top1": top1,
               "Length": int(np.sum(lengths)), "Loss": loss}
        for name in self.metrics:
            if name != 'top1':
                rec[name] = float(np.average([m[name] for m in metrics], weights=lengths))
        if self.world.rank == 0:
            self.json_logger.info(rec)
        return loss, top1

    def log_train(self, progress, batch_idx, epoch, results):
        length = sum(r["length"] for r in results)
        rec = {"_meta": {"type": "train"}, "Round": epoch, "B": batch_idx, "Length": length,
               "Loss": sum(r["loss"] * r["length"] for r in results) / length}
        for name in self.metrics:
            rec[name] = sum(r["metrics"][name] * r["length"] for r in results) / length
        if self.world.rank == 0:
            self.json_logger.info(rec)
        return rec

    # ------------------------------------------------------------------ the loop
    def prepare(self, model: torch.nn.Module, server_optimizer='SGD', client_optimizer='SGD',
                loss='crossentropy', server_lr=0.1, client_lr=0.1, reset_weights: bool = True) -> None:
        """Build the engine/server for ``model`` (called by ``run``; separate so checkpoints
        can be restored before the first round)."""
        if reset_weights:
            reset_model_weights(model)
            if self.world.distributed:   # every rank must start from identical weights
                self._sync_model(model)
        self.engine = RoundEngine(self.world, self.dataset, self.get_clients(), self.device,
                                  use_kernels=self._opts["use_kernels"], profile=self._opts["profile"])
        self.client_opt = client_optimizer
        self.server = self.engine.setup(model, server_optimizer, self.aggregator, loss, client_lr,
                                        client_optimizer, server_lr)
        self.server_opt = self.server.get_opt()
        self.client_lr = client_lr

    def _sync_model(self, model):
        import torch.distributed as dist
        model.to(self.device)
        for t in list(model.parameters()) + list(model.buffers()):
            dist.broadcast(t.data, src=0)

    def run(
            self,
            model: torch.nn.Module,
            server_optimizer: Union[torch.optim.Optimizer, str] = 'SGD',
            client_optimizer: Union[torch.optim.Optimizer, str] = 'SGD',
            loss: Optional[str] = 'crossentropy',
            global_rounds: Optional[int] = 1,
            local_steps: Optional[int] = 1,
            validate_interval: Optional[int] = 1,
            test_batch_size: Optional[int] = 64,
            server_lr: Optional[float] = 0.1,
            client_lr: Optional[float] = 0.1,
            server_lr_scheduler=None,
            client_lr_scheduler=None,
            resume: Optional[str] = None,
            checkpoint_path: Optional[str] = None,
            checkpoint_interval: int = 0,
    ):
        """Run the adversarial training; returns the list of per-round seconds.  On CUDA the rounds are timed with CUDA
        events on the round stream (completion of round r-1 to completion of round r) and the host does NOT wait for
        the device after every round: it issues round r+1 (batch indices, graph launch) while round r still runs, so
        no launch gap opens between rounds (the reference reports host wall clock per round without any device
        synchronisation, simulator.py:330-360).  Validation rounds, checkpoints and the end of the run synchronise."""
        self.prepare(model, server_optimizer, client_optimizer, loss, server_lr, client_lr,
                     reset_weights=resume is None)
        self.engine.track_cursors = bool(checkpoint_path and checkpoint_interval)
        start_round = 1
        if resume is not None:
            from .checkpoint import load_checkpoint
            start_round = load_checkpoint(resume, self, server_lr_scheduler, client_lr_scheduler) + 1
            client_lr = self.client_lr
        global_start = time()
        ret = []
        on_cuda = self.device.type == "cuda"
        marks = []                      # CUDA events at round boundaries (on_cuda): marks[i] .. marks[i+1] = one round

        def _flush_marks():
            if len(marks) > 1:
                marks[-1].synchronize()
                ret.extend(marks[i].elapsed_time(marks[i + 1]) / 1e3 for i in range(len(marks) - 1))
                del marks[:-1]
        if on_cuda:
            marks.append(torch.cuda.Event(enable_timing=True))
            marks[0].record(torch.cuda.current_stream(self.device))
        show = self._opts["progress"] and self.world.rank == 0
        bar = _progress(global_rounds, show) if start_round == 1 else _NullBar(range(start_round, global_rounds + 1))
        with bar as t:
            for rnd in t:
                round_start = time()
                self.round = rnd
                self.client_lr = client_lr
                if self.use_actor:
                    self.train_actor(rnd, local_steps, self.get_clients(), client_lr)
                else:
                    self.train_trainer(rnd, local_steps, self._clients)
                if validate_interval and rnd % validate_interval == 0:
                    vloss, top1 = self.test_actor(global_round=rnd, batch_size=test_batch_size)
                    t.set_postfix(loss=vloss, top1=top1)
                if server_lr_scheduler:
                    server_lr_scheduler.step()
                if client_lr_scheduler:
                    import warnings
                    with warnings.catch_warnings():
                        # the client schedule is a user-owned scheduler on a dummy optimizer that never steps
                        # (reference scripts/cifar10.py:43-46): torch's ordering warning does not apply
                        warnings.filterwarnings("ignore", message="Detected call of `lr_scheduler.step\\(\\)` before")
                        client_lr_scheduler.step()
                    client_lr = client_lr_scheduler.get_last_lr()[0]
                if on_cuda:
                    marks.append(torch.cuda.Event(enable_timing=True))
                    marks[-1].record(torch.cuda.current_stream(self.device))
                    if len(marks) > 256:
                        _flush_marks()
                else:
                    ret.append(time() - round_start)
                self.debug_logger.info(
                    f"E={rnd}; Client learning rate = {client_lr:}; Time cost = {time() - global_start}")
                if checkpoint_path and checkpoint_interval and rnd % checkpoint_interval == 0:
                    _flush_marks()
                    from .checkpoint import save_checkpoint
                    self.client_lr = client_lr
                    save_checkpoint(checkpoint_path, self, server_lr_scheduler, client_lr_scheduler)
        self.client_lr = client_lr
        _flush_marks()
        if on_cuda:
            torch.cuda.synchronize(self.device)
        self.engine.finish()          # rewind batches prefetched for a round that will not happen
        return ret

    def __str__(self):
        return f"Simulator(world={self.world.size}, device={getattr(self, 'device', None)}, aggregator={getattr(self, 'aggregator', None)})"

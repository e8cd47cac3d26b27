"""FL participants: ``BladesClient`` (honest) and ``ByzantineClient`` (attack base).

API contract follows /root/reference/src/blades/client.py:12-253 (SURVEY Appendix A):
same method names, same hook order, same ``_state['saved_update']`` slot that
attackers poke directly.  The design differs:

* A client does NOT own a deep-copied model by default.  On the engine path
  (``blades_b200.engine``) a client is a *virtual* client: a row index into the
  trainer shard's device-resident update matrix ``U_g[n_local, d]`` plus its hook
  methods.  ``get_update()`` then returns a (device) view of that row and
  ``save_update`` writes into it; no per-client model/optimizer exists.
* The eager, object-per-client path of the reference (deepcopy + SGD per client,
  reference client.py:78-89,178-193) is kept as the CPU oracle and as the
  fallback for user subclasses that override ``local_training``.
"""
from __future__ import annotations

import copy
import logging
from collections import defaultdict
from typing import Callable, Dict, Iterable, Optional, Tuple

import torch
import torch.nn as nn
from torch.utils.data import DataLoader

__all__ = ["BladesClient", "ByzantineClient"]


class _RowSlot:
    """Binding of a virtual client to one row of a device update matrix."""
    __slots__ = ("matrix", "row")

    def __init__(self, matrix: torch.Tensor, row: int):
        self.matrix = matrix
        self.row = row

    def view(self) -> torch.Tensor:
        return self.matrix[self.row]


class BladesClient:
    """Base class of every client (honest clients subclass this too)."""

    _is_byzantine: bool = False
    _is_trusted: bool = False
    device = "cpu"
    #: loss clamp used in local training (reference client.py:191)
    loss_clamp: float = 1e6

    def __init__(self, id: Optional[str] = None, device: Optional[str] = "cpu"):
        self._state: Dict[str, dict] = defaultdict(dict)
        self.set_id(id)
        self.device = device
        self._running: dict = {}
        self._slot: Optional[_RowSlot] = None
        self.model: Optional[nn.Module] = None
        self.optimizer: Optional[torch.optim.Optimizer] = None
        self.loss_func: Optional[Callable] = None
        self._json_logger = logging.getLogger("stats")
        self.debug_logger = logging.getLogger("debug")

    # ------------------------------------------------------------------ identity
    def set_id(self, id) -> None:
        self._id = id

    def id(self):
        """Unique id of the client.

        >>> BladesClient(id='1').id()
        '1'
        """
        return self._id

    def getattr(self, attr):
        return getattr(self, attr)

    def is_byzantine(self) -> bool:
        return self._is_byzantine

    def is_trusted(self) -> bool:
        return self._is_trusted

    def trust(self, trusted: Optional[bool] = True) -> None:
        self._is_trusted = trusted

    def __str__(self) -> str:
        return type(self).__name__

    # ------------------------------------------------------------------ engine binding
    def bind_row(self, matrix: torch.Tensor, row: int) -> None:
        """Attach this (virtual) client to row ``row`` of a device update matrix."""
        self._slot = _RowSlot(matrix, row)
        self._state["saved_update"] = self._slot.view()

    def unbind_row(self) -> None:
        self._slot = None

    # ------------------------------------------------------------------ model / optim
    def set_model(self, model: nn.Module, opt, lr: float) -> None:
        """Give the client its own copy of ``model`` and a fresh optimizer ``opt(params, lr=lr)``."""
        self.model = copy.deepcopy(model)
        self.optimizer = opt(self.model.parameters(), lr=lr)

    def set_lr(self, lr: float) -> None:
        if self.optimizer is None:
            self._running["lr"] = lr
            return
        for g in self.optimizer.param_groups:
            g["lr"] = lr

    def set_loss(self, loss_func="crossentropy") -> None:
        if callable(loss_func):
            self.loss_func = loss_func
        elif loss_func == "crossentropy":
            self.loss_func = nn.CrossEntropyLoss()
        else:
            raise NotImplementedError(f"unsupported loss {loss_func!r}")

    def set_para(self, model: nn.Module) -> None:
        self.model.load_state_dict(model.state_dict())

    # ------------------------------------------------------------------ hooks
    def on_train_round_begin(self, use_actor: bool = True) -> None:
        """Snapshot parameters, move the model to the client device, enter train mode."""
        self._save_para()
        self.model = self.model.to(self.device)
        self.model.train()

    def on_train_round_end(self) -> None:
        """update = theta_after - theta_before (flat, ``named_parameters`` order)."""
        delta = self._get_para(current=True) - self._get_para(current=False)
        self.save_update(delta)

    def on_train_batch_begin(self, data, target, logs=None):
        """Per-batch hook; attackers (e.g. label flipping) override it."""
        return data, target

    # ------------------------------------------------------------------ training / eval
    def local_training(self, data_batches: Iterable[Tuple[torch.Tensor, torch.Tensor]]) -> None:
        """Plain SGD steps over ``data_batches`` (eager oracle path)."""
        for data, target in data_batches:
            data, target = data.to(self.device), target.to(self.device)
            data, target = self.on_train_batch_begin(data=data, target=target)
            self.optimizer.zero_grad()
            out = self.model(data)
            loss = torch.clamp(self.loss_func(out, target), 0, self.loss_clamp)
            loss.backward()
            self._post_backward()
            self.optimizer.step()

    def _post_backward(self) -> None:
        """Hook between backward and step (sign flipping negates grads here)."""
        return None

    @torch.no_grad()
    def evaluate(self, round_number, test_set, batch_size, metrics, use_actor: bool = True,
                 model: Optional[nn.Module] = None) -> dict:
        """Evaluate ``model`` (default: the client's own copy) on ``test_set``.

        Returns the same record schema as reference client.py:147-176.
        """
        net = self.model if model is None else model
        net.eval()
        rec = {"_meta": {"type": "client_validation"}, "E": round_number, "Length": 0, "Loss": 0.0}
        for name in metrics:
            rec[name] = 0.0
        loader = test_set if isinstance(test_set, DataLoader) else DataLoader(test_set, batch_size=batch_size)
        dev = next(net.parameters()).device if model is not None else self.device
        for data, target in loader:
            data, target = data.to(dev), target.to(dev)
            out = net(data)
            n = len(target)
            rec["Loss"] += self.loss_func(out, target).item() * n
            rec["Length"] += n
            for name, fn in metrics.items():
                rec[name] += fn(out, target) * n
        denom = max(rec["Length"], 1)
        for name in metrics:
            rec[name] /= denom
        rec["Loss"] /= denom
        self._json_logger.info(rec)
        return rec

    # ------------------------------------------------------------------ update storage
    def get_update(self) -> torch.Tensor:
        """Saved local update as a flat vector, NaN/inf sanitised (reference client.py:195-198)."""
        return torch.nan_to_num(self._get_saved_update())

    def save_update(self, update: torch.Tensor) -> None:
        if self._slot is not None:
            self._slot.view().copy_(update.detach().to(self._slot.matrix.device))
            self._state["saved_update"] = self._slot.view()
        else:
            self._state["saved_update"] = update.detach().clone()

    def _get_saved_update(self) -> torch.Tensor:
        upd = self._state["saved_update"]
        if isinstance(upd, dict):  # never set (defaultdict default)
            raise RuntimeError(f"client {self._id!r} has no saved update yet")
        return upd

    def _trainable(self):
        return [(n, p) for n, p in self.model.named_parameters() if p.requires_grad]

    def _save_para(self) -> None:
        self._state["saved_para"] = {n: p.detach().clone() for n, p in self._trainable()}

    def _get_para(self, current: bool = True) -> torch.Tensor:
        if current:
            parts = [p.detach().reshape(-1) for _, p in self._trainable()]
        else:
            saved = self._state["saved_para"]
            parts = [saved[n].reshape(-1) for n, _ in self._trainable()]
        return torch.cat(parts).to("cpu")


class ByzantineClient(BladesClient):
    """Base class of attackers.  Override ``on_train_batch_begin``, ``local_training``
    and/or ``omniscient_callback`` (reference client.py:231-253).

    ``fused_spec()`` is the B200 addition: an attacker may describe itself as a
    coordinate-wise closed form so the aggregation kernel can insert it as
    *virtual rows* instead of materialising f identical rows (SURVEY 7.2.3):
    ``{"kind": "alie" | "ipm", "param": p}``, or ``{"kind": "minmax" | "minsum", "param": 0.0,
    "dev_type": "unit_vec" | "std" | "sign", "gamma_init": g0, "tol": t}`` (the scale of the
    Min-Max / Min-Sum row is searched on the device, attackers/_agr.py).
    """
    _is_byzantine = True

    def omniscient_callback(self, simulator) -> None:
        """Runs on the driver after all updates were gathered; full-knowledge hook."""
        return None

    def fused_spec(self) -> Optional[dict]:
        return None

"""Reference arm of ``bench.py --impl reference``: drives the UNMODIFIED reference package installed under
``baseline/_ref`` through its own public API (``blades.simulator.Simulator(...).run(...)``, reference
``simulator.py:44-108,364-457``) on the headline configuration.  Nothing from ``blades_b200`` is imported here.

Three things the reference needs that this image does not have are supplied from OUTSIDE the reference tree:

* ``ray`` (not installed, no network).  ``_install_ray_shim`` registers a minimal stand-in for the four symbols the
  reference touches (``ray.remote``, ``Actor.options(...).remote(...)``, ``method.remote(...)``,
  ``ray.util.ActorPool.map``; ``ray.train.Trainer`` only has to be importable).  Every actor is a dedicated worker
  thread bound to one CUDA device; arguments are passed by reference instead of being pickled through an object
  store -- i.e. the shim is strictly *cheaper* than real Ray, so the measured reference time is a lower bound.
* ``torch._six`` (removed from torch 2.x; reference ``aggregators/torch_utils.py:7`` imports ``inf`` from it).
* data + model of the headline config: the reference ships no ResNet-18 and its CIFAR-10 generator downloads from
  the internet (and crashes, SURVEY quirk Q8).  ``SyntheticCIFAR10`` subclasses the reference's own ``BaseDataset``
  extension point (``basedataset.py:13-56``: implement ``generate_datasets``) with class-conditional Gaussian images
  of the CIFAR-10 shape; the model is torchvision's stock ``resnet18(num_classes=10)``.
"""
from __future__ import annotations

import concurrent.futures as cf
import math
import os
import sys
import tempfile
import time
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "baseline", "_ref")


# ------------------------------------------------------------------------------------------- dependency shims
def _install_ray_shim(num_devices: int) -> None:
    import torch

    class _Method:
        def __init__(self, handle, name):
            self._h, self._name = handle, name

        def remote(self, *a, **k):
            return self._h._pool.submit(self._h._call, self._name, a, k)

    class _Handle:
        _count = 0

        def __init__(self, cls, a, k):
            self._dev = _Handle._count % max(1, num_devices)
            _Handle._count += 1
            self._pool = cf.ThreadPoolExecutor(max_workers=1)
            self._obj = self._pool.submit(self._make, cls, a, k).result()

        def _bind(self):
            if torch.cuda.is_available() and num_devices:
                torch.cuda.set_device(self._dev)          # per-thread current device = the actor's GPU

        def _make(self, cls, a, k):
            self._bind()
            return cls(*a, **k)

        def _call(self, name, a, k):
            self._bind()
            return getattr(self._obj, name)(*a, **k)

        def __getattr__(self, name):
            return _Method(self, name)

    class _Factory:
        def __init__(self, cls):
            self._cls = cls

        def options(self, **kw):
            return self

        def remote(self, *a, **k):
            return _Handle(self._cls, a, k)

    def remote(*a, **k):
        if len(a) == 1 and isinstance(a[0], type) and not k:
            return _Factory(a[0])
        return lambda cls: _Factory(cls)

    def get(x):
        if isinstance(x, (list, tuple)):
            return [get(v) for v in x]
        return x.result() if isinstance(x, cf.Future) else x

    class ActorPool:
        def __init__(self, actors):
            self._actors = list(actors)

        def map(self, fn, values):
            futs = [fn(self._actors[i % len(self._actors)], v) for i, v in enumerate(values)]
            for f in futs:
                yield get(f)

    class Trainer:                                         # mode='trainer' is non-functional in the reference (Q1)
        def __init__(self, *a, **k):
            raise RuntimeError("ray.train.Trainer is not available in the ray shim")

    ray = types.ModuleType("ray")
    ray.remote, ray.get = remote, get
    ray.init = lambda *a, **k: None
    ray.shutdown = lambda *a, **k: None
    ray.is_initialized = lambda: True
    util = types.ModuleType("ray.util")
    util.ActorPool = ActorPool
    train = types.ModuleType("ray.train")
    train.Trainer = Trainer
    ray.util, ray.train = util, train
    sys.modules.update({"ray": ray, "ray.util": util, "ray.train": train})


def _install_torch_six_shim() -> None:
    import torch
    if "torch._six" not in sys.modules:
        six = types.ModuleType("torch._six")
        six.inf = math.inf
        six.string_classes = (str, bytes)
        sys.modules["torch._six"] = six
        torch._six = six


def import_reference(num_devices: int = 1):
    """Make ``import blades`` resolve to the unmodified tree under baseline/_ref."""
    if not os.path.isdir(os.path.join(REF, "blades")):
        raise ImportError("baseline/_ref/blades is missing (run baseline/install_ref.sh)")
    _install_ray_shim(num_devices)
    _install_torch_six_shim()
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import blades.simulator as rs
    if not os.path.abspath(rs.__file__).startswith(REF):
        raise ImportError(f"'blades' resolved to {rs.__file__}, not to baseline/_ref")
    return rs


# ------------------------------------------------------------------------------------------- headline workload
def synthetic_arrays(num_clients: int, batch: int, shape=(3, 32, 32), classes: int = 10, train_sizes=None, seed: int = 1):
    """Class-conditional Gaussian images, ``2*batch`` train / ``batch`` test per client (or ``train_sizes[u]`` train):
    the ``(train ids, train, test ids, test)`` tuple a ``generate_datasets`` returns.  Needs nothing but numpy, so
    tests can rebuild the exact arrays the reference was given."""
    import numpy as np
    rng = np.random.default_rng(seed)
    means = rng.standard_normal((classes,) + tuple(shape)).astype(np.float32)
    ids = list(range(num_clients))
    train, test = {}, {}
    for u in ids:
        for store, n in ((train, train_sizes[u] if train_sizes else 2 * batch), (test, batch)):
            y = rng.integers(0, classes, n)
            x = (means[y] + rng.standard_normal((n,) + tuple(shape))).astype(np.float32)
            store[u] = {"x": x, "y": y.astype(np.int64)}
    return ids, train, ids, test


def make_dataset(num_clients: int, batch: int, data_root: str, shape=(3, 32, 32), classes: int = 10, train_sizes=None):
    from blades.datasets.basedataset import BaseDataset

    class SyntheticCIFAR10(BaseDataset):
        """CIFAR-10-shaped class-conditional Gaussian images (``synthetic_arrays``)."""

        def generate_datasets(self, path="./data", iid=True, alpha=0.1, num_clients=20, seed=1):
            return synthetic_arrays(num_clients, batch, shape, classes, train_sizes, seed)

    os.makedirs(data_root, exist_ok=True)
    return SyntheticCIFAR10(data_root=data_root, train_bs=batch, num_clients=num_clients, seed=1)


def run(steps: int, warmup: int, gpus: int = 1, clients: int = 100, byzantine: int = 20, batch: int = 32,
        model_name: str = "resnet18", budget_s: float = 420.0, soft_deadline_s: float = 1300.0) -> dict:
    """Time the reference's own round loop.  ``Simulator.run`` returns its per-round wall times (reference
    ``simulator.py:452-457``; every round ends with the CPU-side aggregation + server step, so the wall clock is the
    round time).  The reference round is minutes long on this config (CPU aggregation of a 4.5 GB update matrix), so
    the number of rounds is bounded: one warm-up round, then at least three timed rounds (more while ``budget_s``
    lasts, at most ``steps``; only ``soft_deadline_s`` can cut the minimum short).  The counts actually run are
    reported."""
    import torch
    rs = import_reference(gpus)
    use_cuda = torch.cuda.is_available()
    tmp = tempfile.mkdtemp(prefix="blades_ref_")
    ds = make_dataset(clients, batch, os.path.join(tmp, "data"),
                      shape=(28, 28) if model_name == "mlp" else (3, 32, 32))
    sim = rs.Simulator(dataset=ds, num_byzantine=byzantine, attack="alie",
                       attack_kws={"num_clients": clients, "num_byzantine": byzantine},
                       aggregator="trimmedmean", aggregator_kws={"nb": byzantine},
                       num_actors=max(1, gpus), gpu_per_actor=1.0 if use_cuda else 0, use_cuda=use_cuda,
                       log_path=os.path.join(tmp, "log"), seed=1)

    def model():
        if model_name == "mlp":
            from blades.models.mnist import MLP
            return MLP()
        import torchvision
        return torchvision.models.resnet18(num_classes=10)

    kw = dict(server_optimizer="SGD", client_optimizer="SGD", loss="crossentropy", local_steps=1,
              validate_interval=10 ** 9, server_lr=1.0, client_lr=0.1)
    t0 = time.time()
    probe = sim.run(model(), global_rounds=1, **kw)               # warm-up / probe round
    per_round = max(probe[0], 1e-3)
    req = {"steps": steps, "warmup": warmup, "budget_s": budget_s, "soft_deadline_s": soft_deadline_s}
    # After the warm-up round: at least ``MIN_TIMED`` timed rounds whatever the budget says (a ratio against a single
    # un-warmed round is not a measurement), more while the budget lasts, never more than ``steps``.  Only the soft
    # deadline (the caller's hard limit minus a margin) can cut the minimum short.
    MIN_TIMED = 3
    left = budget_s - (time.time() - t0)
    k = max(MIN_TIMED, min(steps, int(left / per_round)))
    k = min(k, steps)
    room = int((soft_deadline_s - (time.time() - t0)) / (1.15 * per_round))
    note = ""
    if room < k:
        note = f"soft deadline: {max(room, 1)} timed round(s) instead of {k}"
        k = max(room, 1)
    times = sim.run(model(), global_rounds=k, **kw)
    sec = sum(times)
    return {"value": len(times) / sec, "ms_per_step": 1e3 * sec / len(times), "steps": len(times),
            "warmup": 1, "requested": req, "round_s": [round(t, 3) for t in [probe[0]] + list(times)], "note": note}


if __name__ == "__main__":
    import argparse
    import json
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--clients", type=int, default=100)
    ap.add_argument("--byzantine", type=int, default=20)
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--model", default="resnet18")
    ap.add_argument("--budget", type=float, default=420.0)
    ap.add_argument("--soft-deadline", type=float, default=1300.0)
    a = ap.parse_args()
    out = run(a.steps, a.warmup, a.gpus, a.clients, a.byzantine, a.batch, a.model, a.budget, a.soft_deadline)
    print("REF_RESULT " + json.dumps(out), flush=True)

#!/usr/bin/env python
"""Headline benchmark (BASELINE.json): FL rounds/sec, CIFAR-10-shaped synthetic data, ResNet-18,
fedsgd, 100 clients (20 ALIE attackers), Trimmedmean(nb=20), on N B200s of one node.

    python bench.py --gpus 1 --steps K --warmup W
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Prints ONE JSON line on rank 0.  ``value`` is device-timed (CUDA events, max over ranks) with the
round's inputs already resident on the device; ``e2e`` runs the same rounds through the public
``Simulator`` API including, per round, host batch assembly, the pinned H2D copy of the inputs and
a D2H read of the mean client loss.  ``--impl reference`` runs the UNMODIFIED reference from
baseline/_ref through its own ``Simulator.run`` (DESIGN.md section 6; ray / torch._six shimmed from
outside the tree); ``--impl baseline`` runs the reference round on stock torch + NCCL with the
aggregation on the GPU (baseline/nccl_torch.py: what a straightforward GPU port achieves).  All arms
print the same ``metric`` string; how the time was taken is in ``timing``.  ``vs_baseline`` of our
arm = value / the GPU port measured in the same invocation (BASELINE.md has no published number; the
GPU port is the baseline that document constructs), a few rounds after our own measurement.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "FL rounds/sec"

CONFIGS = {
    # name: (model, classes, clients, byzantine, attack, aggregator, agg_kws, local_steps)
    "headline": ("resnet18", 10, 100, 20, "alie", "trimmedmean", {"nb": 20}, 1),
    "fedavg_median": ("resnet18", 10, 100, 20, "ipm", "median", {}, 5),
    "multikrum": ("resnet18", 10, 200, 40, "labelflipping", "multikrum", {"num_byzantine": 40}, 1),
    "geomed_r50": ("resnet50", 100, 512, 100, "alie", "geomed", {}, 1),
    "mlp": ("mlp", 10, 4, 1, "noise", "mean", {}, 1),
}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int = 0):
        self.proc = None
        self.lines = []
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_model(name: str, classes: int):
    from blades_b200.models import MLP, resnet18, resnet50
    return {"mlp": lambda: MLP(), "resnet18": lambda: resnet18(num_classes=classes),
            "resnet50": lambda: resnet50(num_classes=classes)}[name]()


def dump_outputs(directory: str, arrays: dict, max_elems: int = 1 << 22) -> None:
    """``<directory>/<name>.npy`` in float32 for every tensor of ``arrays``.  A tensor longer than ``max_elems`` is
    stored as the same fixed, seeded sample of its coordinates in every run (at most 16 MB per array), so two builds
    can be compared output for output."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().reshape(-1).float().cpu().numpy()
        if a.size > max_elems:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, max_elems, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), a)


def run_ours(args) -> dict:
    import torch

    from blades_b200 import Simulator
    from blades_b200.comm.group import init_world
    from blades_b200.datasets import synthetic_fldataset
    from blades_b200.ops import _loader

    world = init_world(use_cuda=True)
    model_name, classes, n_clients, n_byz, attack, agg, agg_kws, local_steps = CONFIGS[args.config]
    if args.clients:
        n_byz = max(1, n_byz * args.clients // n_clients) if n_byz else 0
        n_clients = args.clients
        if "nb" in agg_kws:
            agg_kws = {"nb": n_byz}
    shape = (28, 28) if model_name == "mlp" else (3, 32, 32)
    ds = synthetic_fldataset(n_clients, shape=shape, num_classes=classes, train_bs=args.batch,
                             train_per_client=2 * args.batch, test_per_client=args.batch, seed=1)
    attack_kws = {"num_clients": n_clients, "num_byzantine": n_byz} if attack == "alie" else {}
    sim = Simulator(ds, num_byzantine=n_byz, attack=attack, attack_kws=attack_kws, aggregator=agg,
                    aggregator_kws=dict(agg_kws), use_cuda=True, seed=1, log_path=tempfile.mkdtemp(),
                    progress=False, wipe_logs=True)
    model = build_model(model_name, classes)
    sim.prepare(model, "SGD", "SGD", "crossentropy", server_lr=1.0, client_lr=0.1)
    eng = sim.engine
    if args.max_batched:
        eng.max_batched_clients = args.max_batched
    elif model_name == "resnet50":
        eng.max_batched_clients = 64          # bound the activation footprint of the fused pass
    dev = eng.device
    clients = sim.get_clients()

    def one_round(r):
        sim.train_actor(r, local_steps, clients, 0.1)

    # ---------------- device-timed: inputs resident on the device ----------------
    if local_steps == 1:
        eng.prestaged = eng.stage_batches(None, 1)
    for r in range(args.warmup):
        one_round(r)
    torch.cuda.synchronize()
    world.barrier()
    sampler = ClockSampler(dev.index or 0)
    if world.rank == 0:
        sampler.start()
    launches0 = _loader.LAUNCHES
    beg, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    beg.record()
    for r in range(args.steps):
        one_round(args.warmup + r)
    end.record()
    torch.cuda.synchronize()
    world.barrier()
    ms = world.all_reduce_max(beg.elapsed_time(end))
    launches = _loader.LAUNCHES - launches0
    clocks = sampler.stop() if world.rank == 0 else {}
    eng.prestaged = None
    if args.dump_outputs and world.rank == 0:
        # what the last timed round handed back: the new global model, the aggregate the server applied and the
        # per-client losses (rank 0's clients), parameters in the model's named_parameters() order
        outs = {"theta": eng.gflat.to_reference_order(eng.gflat.theta)}
        if sim.last_aggregate is not None and sim.last_aggregate.numel() == eng.d:
            outs["aggregate"] = eng.gflat.to_reference_order(sim.last_aggregate.reshape(-1))
        if eng.last_client_losses is not None:
            outs["client_losses"] = eng.last_client_losses
        dump_outputs(args.dump_outputs, outs)

    # ---------------- end-to-end through the public API ----------------
    h2d = d2h = 0
    e2e_ms, e2e_note, per_round = None, "", []
    issued = []                                            # host time of every round's issue part (diagnostic)

    def e2e_phase():
        nonlocal d2h
        rounds = []
        issued.clear()
        for r in range(max(args.warmup, 10)):       # untimed: also absorbs one-off host stalls after the phase switch
            one_round(r)
            float(eng.last_client_losses.mean()) if eng.last_client_losses is not None else None
        torch.cuda.synchronize()
        world.barrier()
        t0 = time.perf_counter()
        pending, tr = None, t0
        for r in range(args.steps):
            ti = time.perf_counter()
            one_round(r)                                   # host indices -> gather from pinned host memory -> round
            issued.append((time.perf_counter() - ti) * 1e3)
            # D2H read of EVERY round's result (per-client losses) through the engine's pinned double buffer; the read
            # of round r-1 completes here, after round r has been issued, so the host part of a round overlaps the
            # previous round's GPU time (depth-1 software pipeline of the driver loop)
            nxt = eng.losses_to_host_async()
            if nxt is None:                                # CPU fallback paths: plain synchronous read
                loss_host = sim.last_aggregate[:1].cpu()
                d2h = 4
            if pending is not None:
                loss_host = pending.get()
                d2h = loss_host.numel() * loss_host.element_size()
                now = time.perf_counter()
                rounds.append((now - tr) * 1e3)            # completion-to-completion time of one round
                tr = now
            pending = nxt
        if pending is not None:
            loss_host = pending.get()
            d2h = loss_host.numel() * loss_host.element_size()
            rounds.append((time.perf_counter() - tr) * 1e3)
        torch.cuda.synchronize()
        world.barrier()
        return world.all_reduce_max((time.perf_counter() - t0) * 1e3), rounds

    if not args.no_e2e:
        try:
            e2e_ms, per_round = e2e_phase()
        except Exception as e:      # keep the device-timed result; retry the input path without the prefetcher
            e2e_note = f"prefetching input path failed ({type(e).__name__}: {e}); measured with synchronous staging"
            try:
                eng.finish()
                eng.prefetch = False
                e2e_ms, per_round = e2e_phase()
            except Exception as e2:
                e2e_ms, e2e_note = None, f"end-to-end phase failed: {type(e2).__name__}: {e2}"
        h2d = eng.h2d_bytes

    value = args.steps / (ms / 1e3)
    out = {
        "metric": METRIC, "timing": "device (CUDA events around the K rounds, max over ranks)", "value": value,
        "unit": "rounds/s", "n_gpus": world.size, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "fp32 (tf32 tensor-core GEMMs)",
        "data": "synthetic (class-conditional Gaussian images of the named shape), random-init weights",
        "impl": "ours",
        "config": {"model": f"{model_name}({classes} classes)", "clients": n_clients, "byzantine": n_byz,
                   "attack": attack, "aggregator": f"{agg}{agg_kws}", "local_steps": local_steps,
                   "client_batch": args.batch, "global_batch": n_clients * args.batch,
                   "seq_len": None, "parallelism": f"client-shard x{world.size} + coordinate-sharded aggregation",
                   "l2_policy": "per-round working set (update matrix %.2f GB) >> 126 MB L2; no explicit flush"
                                % (n_clients * eng.d * 4 / 1e9)},
        "clocks": clocks, "gpu_launches": launches,
    }
    if e2e_ms is None and e2e_note:
        out["e2e"] = {"error": e2e_note}
    if e2e_ms is not None:
        out["e2e"] = {"value": args.steps / (e2e_ms / 1e3), "unit": "rounds/s", "ms_per_step": e2e_ms / args.steps,
                      "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                      "round_ms_median_rank0": sorted(per_round)[len(per_round) // 2], "round_ms_max_rank0": max(per_round),
                      "note": e2e_note,
                      # the slowest round of every rank: (round index, total ms, of which host issue ms) -- where a stall sits
                      "slowest_round_per_rank": world.all_gather_object(
                          (per_round.index(max(per_round)), round(max(per_round), 2),
                           round(issued[per_round.index(max(per_round))], 2)) if per_round and issued else None),
                      "h2d_mechanism": ("gather kernel reading the pinned host shards over PCIe (zero-copy) + index upload"
                                        if eng.prefetch and any(eng._zc_plans.values())
                                        else "pinned staging buffer + cudaMemcpyAsync")}
    if not args.no_port:
        # the constructed baseline of BASELINE.md section 2-3 (stock torch + NCCL GPU port of the reference round),
        # a few rounds in the same invocation on the same GPUs: vs_baseline = ours / port
        try:
            import copy
            from baseline.nccl_torch import run_baseline
            eng.finish()
            pa = copy.copy(args)
            pa.steps, pa.warmup = 3, 1
            port = run_baseline(pa, CONFIGS)
            if world.rank == 0 and port:
                out["vs_baseline"] = value / port["value"]
                out["baseline_port"] = {"impl": port["impl"], "value": port["value"], "unit": "rounds/s",
                                        "steps": port["steps"], "warmup": port["warmup"], "timing": port["timing"],
                                        "e2e_value": port["e2e"]["value"],
                                        "note": "reference round semantics on stock torch/cuDNN/NCCL, aggregation on "
                                                "the GPU, none of this repo's kernels (baseline/nccl_torch.py)"}
        except Exception as e:      # the comparison arm must never lose the measurement
            out["baseline_port"] = {"error": f"{type(e).__name__}: {e}"}
    return out if world.rank == 0 else {}


def run_reference(args) -> dict:
    """The UNMODIFIED reference (baseline/_ref, see baseline/install_ref.sh) through its own Simulator API on the
    headline config; ray / torch._six are shimmed from outside the tree (baseline/ref_arm.py).  Runs in a child
    process with a hard deadline: one reference round on this config is minutes of CPU-side aggregation."""
    import subprocess
    if not os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "blades")):
        return {"impl": "reference", "unavailable": "baseline/_ref/blades missing: the reference's sdist installs an "
                "empty distribution (no blades/__init__.py); run baseline/install_ref.sh -- see DESIGN.md section 6"}
    model_name, classes, n_clients, n_byz, attack, agg, agg_kws, local_steps = CONFIGS[args.config]
    if args.config != "headline":
        return {"impl": "reference", "unavailable": "the reference arm is wired for the headline config only"}
    if args.clients:
        n_byz = max(1, n_byz * args.clients // n_clients)
        n_clients = args.clients
    budget = float(os.environ.get("BLADES_REF_BUDGET_S", "420"))
    deadline = float(os.environ.get("BLADES_REF_DEADLINE_S", "1500"))
    cmd = [sys.executable, os.path.join(ROOT, "baseline", "ref_arm.py"), "--steps", str(args.steps), "--warmup",
           str(args.warmup), "--gpus", str(args.gpus), "--clients", str(n_clients), "--byzantine", str(n_byz),
           "--batch", str(args.batch), "--model", model_name, "--budget", str(budget),
           "--soft-deadline", str(max(60.0, deadline - 200.0))]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")}
    if "WORLD_SIZE" in os.environ:
        env.pop("OMP_NUM_THREADS", None)       # torchrun pins it to 1; the reference aggregates on the CPU
    proc = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, start_new_session=True,
                            env=env)
    try:
        out, err = proc.communicate(timeout=deadline)
    except subprocess.TimeoutExpired:
        os.killpg(proc.pid, 9)                      # the process group this function started, nothing else
        proc.wait()
        return {"impl": "reference", "unavailable": f"one reference round did not finish within {deadline:.0f} s "
                "(CPU-side ALIE + trimmed mean over a 4.5 GB update matrix)"}
    res = [ln for ln in out.splitlines() if ln.startswith("REF_RESULT ")]
    if proc.returncode != 0 or not res:
        tail = (err or out).strip().splitlines()[-1:] or ["no output"]
        return {"impl": "reference", "unavailable": f"reference run failed (rc={proc.returncode}): {tail[0][:300]}"}
    r = json.loads(res[-1][len("REF_RESULT "):])
    return {
        "impl": "reference", "metric": METRIC, "timing": "wall clock of the reference's own round loop "
        "(Simulator.run's per-round times; its only path is end to end)", "value": r["value"], "unit": "rounds/s", "n_gpus": args.gpus, "steps": r["steps"], "warmup": r["warmup"],
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "fp32 (torch defaults)", "data": "synthetic (class-conditional Gaussian images, CIFAR-10 shape), "
        "random-init torchvision resnet18", "config": {
            "model": f"{model_name}({classes} classes)", "clients": n_clients, "byzantine": n_byz, "attack": attack,
            "aggregator": f"{agg}{agg_kws}", "local_steps": local_steps, "client_batch": args.batch,
            "global_batch": n_clients * args.batch, "seq_len": None,
            "parallelism": f"{max(1, args.gpus)} actor(s), one per GPU (ray API shim: in-process actor threads, "
                           "no object-store pickling -- cheaper than real Ray)"},
        "e2e": {"value": r["value"], "unit": "rounds/s",
                # derived from the reference's code path, not instrumented: per client per round the batch and the
                # model go H2D (client.py:124,186) and the flat parameters come back twice (client.py:216-228)
                "h2d_bytes_per_step": n_clients * (args.batch * (3 * 32 * 32 * 4 + 8) + 11181642 * 4),
                "d2h_bytes_per_step": n_clients * 2 * 11181642 * 4,
                "note": "the reference has one path: host batches -> per-client .to(device) -> train -> updates "
                        "to CPU -> CPU aggregation; its wall clock IS end to end"},
        "gpu_launches": 0, "requested": r["requested"], "round_s": r["round_s"], "note": r.get("note", ""),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "baseline"])
    ap.add_argument("--config", default="headline", choices=sorted(CONFIGS))
    ap.add_argument("--clients", type=int, default=0, help="override the client count (debug)")
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-port", action="store_true", help="skip the GPU-port comparison rounds (vs_baseline stays null)")
    ap.add_argument("--max-batched", type=int, default=0, help="clients per fused training pass (0 = all local)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed round computed to DIR/<name>.npy (float32, <= 64 MB in all); "
                         "--impl ours only")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours only")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps(run_reference(args)), flush=True)
        return
    if args.impl == "baseline":
        from baseline.nccl_torch import run_baseline
        out = run_baseline(args, CONFIGS)
    else:
        out = run_ours(args)
    if out:
        print(json.dumps(out), flush=True)
    from blades_b200.comm.group import shutdown
    shutdown()


if __name__ == "__main__":
    main()

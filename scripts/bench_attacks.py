"""Cost of the fused Min-Max / Min-Sum attacks next to ALIE on the headline workload (ResNet-18, 100 clients, 20
attackers, Trimmedmean(nb=20), fedsgd, one GPU), and of each of their kernels at that shape.

    python scripts/bench_attacks.py [--steps 20] [--warmup 5] [--reps 3] [--out FILE]

* Rounds/s of each attack, device-timed (CUDA events around ``--steps`` rounds).  The attacks run in alternation,
  ``--reps`` times, each on its own simulator with the same data and seed; the median is reported.
* Kernel times at the headline shape (the update matrix of the last ALIE round, 80 honest rows): the deviation pass
  (``std``), the Gram pass of ``[U; q]`` (and of ``U`` alone, the ``unit_vec`` case), and the scale solve; CUDA
  events around ``--launches`` back-to-back launches after a warm-up.  U (4.5 GB) is far larger than the L2.

Prints one JSON object with the GPU name and power limit beside the numbers.  Needs a CUDA device.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench import CONFIGS, build_model  # noqa: E402

VARIANTS = [("alie", None), ("minmax", "unit_vec"), ("minmax", "std"), ("minsum", "std")]


def gpu_info() -> dict:
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = out
    except Exception as e:                                  # the numbers stay valid, only their label is thinner
        info["power_limit_and_max_sm_clock"] = f"unavailable ({type(e).__name__})"
    return info


def make_sim(attack: str, dev_type, batch: int):
    from blades_b200 import Simulator
    from blades_b200.datasets import synthetic_fldataset
    model_name, classes, n_clients, n_byz, _, agg, agg_kws, _ = CONFIGS["headline"]
    ds = synthetic_fldataset(n_clients, shape=(3, 32, 32), num_classes=classes, train_bs=batch,
                             train_per_client=2 * batch, test_per_client=batch, seed=1)
    kws = {"num_clients": n_clients, "num_byzantine": n_byz} if attack == "alie" else {"dev_type": dev_type}
    sim = Simulator(ds, num_byzantine=n_byz, attack=attack, attack_kws=kws, aggregator=agg,
                    aggregator_kws=dict(agg_kws), use_cuda=True, seed=1, log_path=tempfile.mkdtemp(),
                    progress=False, wipe_logs=True)
    sim.prepare(build_model(model_name, classes), "SGD", "SGD", "crossentropy", server_lr=1.0, client_lr=0.1)
    sim.engine.prestaged = sim.engine.stage_batches(None, 1)
    return sim


def time_rounds(sim, first: int, steps: int) -> float:
    """ms per round over ``steps`` rounds (device time)."""
    clients = sim.get_clients()
    beg, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    beg.record()
    for r in range(steps):
        sim.train_actor(first + r, 1, clients, 0.1)
    end.record()
    torch.cuda.synchronize()
    return beg.elapsed_time(end) / steps


def time_launches(fn, launches: int) -> float:
    """µs per call of ``fn`` over ``launches`` back-to-back calls, after a warm-up."""
    for _ in range(3):
        fn()
    beg, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    beg.record()
    for _ in range(launches):
        fn()
    end.record()
    torch.cuda.synchronize()
    return beg.elapsed_time(end) * 1e3 / launches


def kernel_times(U: torch.Tensor, byz, launches: int) -> dict:
    from blades_b200.ops import attack, gram_solve, select
    from blades_b200.parallel.matrix import LocalMatrix
    n, d = U.shape
    honest = [i for i in range(n) if i not in set(byz)]
    ptrs = select.row_pointers(U, honest)
    idx = gram_solve.index_tensor(honest, U.device)
    q = torch.empty(d, device=U.device)
    mat = LocalMatrix(U)
    attack.deviation(ptrs, "std", 0, d, q)
    dg_q, dg = mat.gram_device(q), mat.gram_device()
    assert dg_q is not None and dg is not None, "the Gram pass did not stay on the device"
    out = {"shape": {"rows": n, "honest": len(honest), "d": d}}
    out["deviation_std_us"] = time_launches(lambda: attack.deviation(ptrs, "std", 0, d, q), launches)
    out["deviation_sign_us"] = time_launches(lambda: attack.deviation(ptrs, "sign", 0, d, q), launches)
    out["gram_U_plus_q_us"] = time_launches(lambda: mat.gram_device(q), launches)
    out["gram_U_us"] = time_launches(lambda: mat.gram_device(), launches)
    for kind in ("minmax", "minsum"):
        out[f"solve_{kind}_std_us"] = time_launches(
            lambda: gram_solve.agr_scale(dg_q, idx, n, kind == "minsum", "std", 10.0, 1e-5), launches)
        out[f"solve_{kind}_unit_vec_us"] = time_launches(
            lambda: gram_solve.agr_scale(dg, idx, -1, kind == "minsum", "unit_vec", 10.0, 1e-5), launches)
    # bytes the deviation pass must read (honest rows) over its time: an achieved-bandwidth figure
    out["deviation_std_GBps"] = len(honest) * d * 4 / (out["deviation_std_us"] * 1e-6) / 1e9
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_attacks.py needs a CUDA device")
    import logging

    class Keep(logging.Handler):                             # why a round graph was not captured, if it was not
        def __init__(self):
            super().__init__(logging.WARNING)
            self.msgs = []

        def emit(self, record):
            self.msgs.append(record.getMessage()[:300])
    keep = Keep()
    logging.getLogger("debug").addHandler(keep)
    sims = {}
    for attack, dev_type in VARIANTS:
        sim = make_sim(attack, dev_type, args.batch)
        time_rounds(sim, 0, args.warmup)                     # eager warm-up rounds, then the captured round graph
        sims[(attack, dev_type)] = sim
    runs = {k: [] for k in sims}
    rounds = {k: args.warmup for k in sims}
    for _ in range(args.reps):
        for k, sim in sims.items():
            runs[k].append(time_rounds(sim, rounds[k], args.steps))
            rounds[k] += args.steps
    res = {"gpu": gpu_info(), "workload": "ResNet-18, 100 clients, 20 attackers, Trimmedmean(nb=20), fedsgd, 1 GPU",
           "timing": f"CUDA events around {args.steps} rounds, median of {args.reps} alternating repetitions",
           "rounds": {}}
    base = statistics.median(runs[("alie", None)])
    for (attack, dev_type), ms in runs.items():
        med = statistics.median(ms)
        sim = sims[(attack, dev_type)]
        name = attack if dev_type is None else f"{attack}/{dev_type}"
        entry = {"rounds_per_s": 1e3 / med, "ms_per_round": med, "ms_per_round_runs": ms,
                 "extra_ms_vs_alie": med - base,
                 "round_graph": any("graph" in st for st in sim.engine._round_graphs.values())}
        if dev_type is not None:
            entry["gamma"] = [c.gamma for c in sim.get_clients() if c.is_byzantine()][0]
        res["rounds"][name] = entry
    if keep.msgs:
        res["warnings"] = keep.msgs
    alie = sims[("alie", None)]
    byz = [i for i, c in enumerate(alie.get_clients()) if c.is_byzantine()]
    res["kernels"] = kernel_times(alie.engine.U, byz, args.launches)
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()

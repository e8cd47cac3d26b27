"""Multi-GPU (symmetric memory, pull-mode fused aggregation) must reproduce the single-GPU run."""
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = [pytest.mark.gpu, pytest.mark.multigpu]


def _launch(nproc, out_dir, agg, attack, model, n_clients, port):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "_mgpu_worker.py"),
           out_dir, agg, attack, model, str(n_clients)]
    env = dict(os.environ)
    if attack == "noise":
        env["BLADES_FORBID_DENSE_GATHER"] = "1"      # row-local attackers must not gather the [N, d] matrix
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    if r.returncode != 0:
        errs = ""
        for f in sorted(os.listdir(out_dir)):
            if f.startswith("error_rank"):
                errs += f"\n--- {f}\n" + open(os.path.join(out_dir, f)).read()[-2500:]
        raise AssertionError(errs or r.stderr[-3000:])


@pytest.mark.parametrize("agg,attack,model,n", [("trimmedmean", "alie", "mlp", 10), ("median", "ipm", "mlp", 9),
                                                ("mean", "none", "mlp", 7), ("krum", "noise", "mlp", 10),
                                                ("geomed", "labelflipping", "mlp", 10),
                                                ("centeredclipping", "signflipping", "mlp", 10),
                                                ("trimmedmean", "alie", "resnet18", 10)])
def test_sharded_equals_single(agg, attack, model, n, tmp_path):
    ngpu = torch.cuda.device_count()
    out = str(tmp_path)
    sizes = [1, 2] + ([ngpu] if ngpu > 2 else [])
    if os.environ.get("BLADES_MGPU_SIZES"):          # e.g. "1,8": skip the 2-GPU leg on an expensive 8-GPU lease
        sizes = [int(v) for v in os.environ["BLADES_MGPU_SIZES"].split(",")]
    for i, w in enumerate(sizes):
        _launch(w, out, agg, attack, model, n, 29610 + i)
    a = None if attack == "none" else attack
    base = torch.load(os.path.join(out, f"theta_{agg}_{a}_{model}_1_0.pt"))
    for w in sizes[1:]:
        vecs = [torch.load(os.path.join(out, f"theta_{agg}_{a}_{model}_{w}_{r}.pt")) for r in range(w)]
        for v in vecs[1:]:
            assert torch.equal(v, vecs[0]), "replicas diverged"
        # (noise rows: the Philox stream position depends on (round, client) only, so they match as well)
        if model == "resnet18":
            # different total batch per GPU -> cuDNN picks different TF32 algorithms; BN over 8-sample client
            # batches amplifies the rounding noise.  The communication path is checked exactly by the MLP cases.
            rel = ((vecs[0] - base).norm() / base.norm()).item()
            assert rel < 5e-2, (w, rel)
        else:
            assert torch.allclose(vecs[0], base, atol=5e-4, rtol=1e-2), (w, (vecs[0] - base).abs().max())

"""The reference's own example scripts run UNCHANGED on this package through ``blades_b200.compat`` (module alias
``blades`` -> ``blades_b200`` + a no-op ``ray``): only the hard-coded round counts are shortened, and torchvision's
MNIST download is replaced by a deterministic fake.  The reference's scripts cannot be stored here, so every test runs
test-owned scripts of the same two experiments written in the same style (``blades`` + ``ray`` APIs), and the
reference's own scripts as well when the reference is installed under baseline/_ref (baseline/install_ref.sh).  The
global model the reference ends with is stored under tests/golden/reference (tests/_golden.py), so the comparison of
the two packages runs without it."""
import os
import re
import subprocess
import sys

import pytest

from _golden import golden, key, params, params_max, params_mismatches

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXAMPLES = os.path.join(ROOT, "baseline", "_ref", "blades", "examples")
HAVE_EXAMPLES = os.path.isdir(EXAMPLES)


_RUNNER = r'''
import re, sys, torch, torchvision
sys.path.insert(0, {root!r})

class FakeMNIST:
    def __init__(self, train=True, download=True, root=None, **kw):
        g = torch.Generator().manual_seed(11 if train else 12)
        n = 1200 if train else 200
        self.data = torch.randint(0, 256, (n, 28, 28), generator=g, dtype=torch.uint8)
        self.targets = torch.randint(0, 10, (n,), generator=g)
torchvision.datasets.MNIST = FakeMNIST

import blades_b200.compat as compat
def shorten(src):
    src = re.sub(r'"global_rounds":\s*\d+', '"global_rounds": 3', src)
    return re.sub(r'"local_steps":\s*\d+', '"local_steps": 2', src)
g = compat.run_script({script!r}, patch=shorten)
sim = g["simulator"]
import blades, blades.simulator, blades_b200.simulator
assert blades.simulator.Simulator is blades_b200.simulator.Simulator and type(sim) is blades_b200.simulator.Simulator
print("RAN", type(sim).__module__, len(sim.get_clients()), sum(c.is_byzantine() for c in sim.get_clients()))
'''


# Reference-style scripts of the two experiments of the reference's examples, written against the ``blades`` and
# ``ray`` APIs: MNIST with 10 clients, MLP, SGD (client lr 0.1), seed 1.  mini_example: 4 ALIE attackers, mean
# aggregation.  customize_attack: five clients replaced by an attacker that trains on flipped labels (9 - y), ascends
# the loss (clamped to [0, 1e5]) instead of descending it, and finally submits -100 x the mean honest update; clipped
# clustering aggregation.  The round counts are those of ``patch``.
_OWN_SCRIPTS = {
    "mini_example.py": '''
import ray
from blades.datasets import MNIST
from blades.models.mnist import MLP
from blades.simulator import Simulator

ray.init(num_gpus=0, local_mode=False)
simulator = Simulator(dataset=MNIST(data_root="./data", train_bs=32, num_clients=10), aggregator="mean",
                      num_byzantine=4, attack="alie", attack_kws={"num_clients": 10, "num_byzantine": 4},
                      num_actors=1, use_cuda=False, gpu_per_actor=0.0, seed=1)
run_params = {"model": MLP(), "server_optimizer": "SGD", "client_optimizer": "SGD", "loss": "crossentropy",
              "global_rounds": 4, "local_steps": 3, "server_lr": 1.0, "client_lr": 0.1}
simulator.run(**run_params)
''',
    "customize_attack.py": '''
import ray
import torch
from blades.client import ByzantineClient
from blades.datasets import MNIST
from blades.models.mnist import MLP
from blades.simulator import Simulator


class FlippedLabelAscent(ByzantineClient):
    """Trains on labels 9 - y, ascends the loss, then reports -100 x the honest clients' mean update."""

    def on_train_batch_begin(self, data, target):
        return data, 9 - target

    def local_training(self, data_batches):
        opt, model = self.optimizer, self.model
        for x, y in data_batches:
            x, y = self.on_train_batch_begin(x.to(self.device), y.to(self.device))
            opt.zero_grad()
            ascent = -torch.clamp(self.loss_func(model(x), y), 0, 1e5)      # minimising -loss ascends the loss
            ascent.backward()
            opt.step()

    def omniscient_callback(self, simulator):
        honest = torch.stack([c.get_update() for c in simulator.get_clients() if not c.is_byzantine()])
        self.save_update(honest.mean(0) * -100)


ray.init(num_gpus=0, local_mode=True)
simulator = Simulator(dataset=MNIST(data_root="./data", train_bs=32, num_clients=10), aggregator="clippedclustering",
                      num_actors=1, seed=1)
simulator.register_attackers([FlippedLabelAscent() for _ in range(5)])
run_params = {"model": MLP(), "server_optimizer": "SGD", "client_optimizer": "SGD", "loss": "crossentropy",
              "global_rounds": 4, "local_steps": 3, "client_lr": 0.1}
simulator.run(**run_params)
''',
}


@pytest.mark.parametrize("script,clients,byz", [("mini_example.py", 10, 4), ("customize_attack.py", 10, 5)])
def test_reference_example_runs_unchanged(tmp_path, script, clients, byz):
    """The test-owned script of the experiment, and the reference's own example when it is installed, run unchanged
    on blades_b200 through ``blades_b200.compat``."""
    own = tmp_path / script
    own.write_text(_OWN_SCRIPTS[script])
    for path in [str(own)] + ([os.path.join(EXAMPLES, script)] if HAVE_EXAMPLES else []):
        code = _RUNNER.format(root=ROOT, script=path)
        out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=tmp_path)
        assert out.returncode == 0, (path, out.stderr[-3000:])
        m = re.search(r"RAN (\S+) (\d+) (\d+)", out.stdout)
        assert m and m.group(1) == "blades_b200.simulator" and int(m.group(2)) == clients and int(m.group(3)) == byz, \
            (path, out.stdout[-500:])


def test_alias_modules_are_the_same_objects():
    code = ("import sys; sys.path.insert(0, %r); import blades_b200.compat as c; c.install();"
            "import blades.aggregators.krum as a, blades_b200.aggregators.krum as b; assert a is b;"
            "from blades.attackers.alieclient import AlieClient; from blades.models.cifar10 import CCTNet;"
            "from blades.datasets import MNIST, CIFAR10; from blades.client import BladesClient, ByzantineClient;"
            "from blades.server import BladesServer; import ray; ray.init(num_gpus=0); print('ok')" % ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


_COMPARE = r'''
import re, sys, torch, torchvision
sys.path.insert(0, {root!r})

class FakeMNIST:
    def __init__(self, train=True, download=True, root=None, **kw):
        g = torch.Generator().manual_seed(11 if train else 12)
        n = 1200 if train else 200
        self.data = torch.randint(0, 256, (n, 28, 28), generator=g, dtype=torch.uint8)
        self.targets = torch.randint(0, 10, (n,), generator=g)
torchvision.datasets.MNIST = FakeMNIST

def patch(src):
    src = re.sub(r'"global_rounds":\s*\d+', '"global_rounds": 4', src)
    src = re.sub(r'"local_steps":\s*\d+', '"local_steps": 3', src)
    return re.sub(r'"num_actors":\s*\d+', '"num_actors": 1', src)      # one actor: deterministic call order

if {which!r} == "reference":
    import sklearn.cluster as skc                 # the reference passes sklearn's removed ``affinity=`` kwarg (Q7)
    _orig = skc.AgglomerativeClustering
    def _compat(*a, affinity=None, **k):
        if affinity is not None:
            k["metric"] = affinity
        return _orig(*a, **k)
    skc.AgglomerativeClustering = _compat
    from baseline import ref_arm
    ref_arm.import_reference(0)
    import os
    os.makedirs("data", exist_ok=True)                                # torchvision's download would create it
    glob = {{"__name__": "__main__", "__file__": {script!r}}}
    exec(compile(patch(open({script!r}).read()), {script!r}, "exec"), glob)
else:
    import blades_b200.compat as compat
    # same batch order as the reference for the comparison (the default streams use independent per-client RNGs)
    import blades_b200.datasets.basedataset as bd
    bd.BaseDataset.compat = True
    glob = compat.run_script({script!r}, patch=patch)
model = glob["run_params"]["model"]
torch.save([(n, p.detach()) for n, p in model.named_parameters()], {out!r})
'''

def _final_model(tmp_path, which, script):
    import torch
    wd = tmp_path / which
    wd.mkdir()
    out = str(wd / "theta.pt")
    code = _COMPARE.format(root=ROOT, script=script, which=which, out=out)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=wd)
    assert r.returncode == 0, r.stderr[-3000:]
    return torch.load(out)


@pytest.mark.parametrize("script", ["mini_example.py", "customize_attack.py"])
def test_reference_example_gives_the_same_model_on_both_packages(tmp_path, request, script):
    """The reference's example executed on the reference package, and the same experiment executed on blades_b200
    through ``blades_b200.compat``: the same global model at the end (every parameter tensor checked against the
    stored summary, ``params_mismatches``)."""
    want = golden(key(request), lambda: params(_final_model(tmp_path, "reference", os.path.join(EXAMPLES, script))))
    own = tmp_path / script
    own.write_text(_OWN_SCRIPTS[script])
    runs = [("own", str(own))] + ([("ours", os.path.join(EXAMPLES, script))] if HAVE_EXAMPLES else [])
    for which, path in runs:
        bad = params_mismatches(_final_model(tmp_path, which, path), want, 1e-5 * max(1.0, params_max(want)))
        assert not bad, (which, bad[:5])

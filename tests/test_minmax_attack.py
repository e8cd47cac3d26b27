"""Min-Max / Min-Sum attacks (Shejwalkar & Houmansadr, NDSS 2021) without a GPU: the attackers' callbacks, the
virtual-row oracle and the Gram-domain search all agree with an independent implementation of the paper's loop."""
import numpy as np
import pytest
import torch

from blades_b200.attackers import MinmaxClient, MinsumClient, _agr
from blades_b200.parallel.matrix import LocalMatrix, VirtualRows, resolve_scaled_rows


# ----------------------------------------------------------------------------- independent oracle (numpy, fp64)
def oracle_deviation(u, dev_type):
    mu = u.mean(0)
    if dev_type == "unit_vec":
        n = np.linalg.norm(mu)
        return mu / n if n > 0 else np.zeros_like(mu)
    if dev_type == "std":
        return u.std(0, ddof=1)
    return np.sign(mu)


def oracle_threshold(u, kind):
    D = np.array([[np.sum((a - b) ** 2) for b in u] for a in u])
    return D.max() if kind == "minmax" else D.sum(1).max()


def oracle_test(u, kind, m, thr):
    d = np.array([np.sum((m - x) ** 2) for x in u])
    return (d.max() if kind == "minmax" else d.sum()) <= thr


def oracle_gamma(u, kind, dev_type, gamma_init=10.0, tol=1e-5):
    mu, p = u.mean(0), oracle_deviation(u, dev_type)
    thr = oracle_threshold(u, kind)
    g, step, ok = gamma_init, gamma_init, 0.0
    while abs(ok - g) > tol:
        if oracle_test(u, kind, mu - g * p, thr):
            ok = g
            g += step / 2
        else:
            g -= step / 2
        step /= 2
    return ok


def _rows(n_h, d, seed):
    """float32-representable rows (the attackers see float32 updates) with a common component."""
    rng = np.random.default_rng(seed)
    shift = rng.normal(size=d) * 0.3
    return (rng.normal(size=(n_h, d)) + shift).astype(np.float32).astype(np.float64)


CASES = [(n_h, d) for n_h in (2, 3, 10, 80) for d in (1, 37, 5000)]


class _Sim:
    def __init__(self, clients):
        self._c = clients

    def get_clients(self):
        return self._c


class _Honest:
    def __init__(self, u):
        self.u = u

    def get_update(self):
        return self.u

    def is_byzantine(self):
        return False


@pytest.mark.parametrize("kind", ["minmax", "minsum"])
@pytest.mark.parametrize("dev_type", ["unit_vec", "std", "sign"])
@pytest.mark.parametrize("n_h,d", CASES)
def test_all_paths_match_the_paper_loop(kind, dev_type, n_h, d):
    u = _rows(n_h, d, seed=n_h * 1000 + d)
    want = oracle_gamma(u, kind, dev_type)
    ut = torch.from_numpy(u).float()
    # attacker callback (unfused path)
    cls = MinmaxClient if kind == "minmax" else MinsumClient
    atk = cls(dev_type=dev_type)
    atk.is_byzantine = lambda: True
    saved = []
    atk.save_update = saved.append
    atk.omniscient_callback(_Sim([_Honest(r) for r in ut] + [atk]))
    assert atk.gamma == pytest.approx(want, rel=1e-9, abs=1e-12)
    mu, p = ut.double().mean(0), oracle_deviation(ut.double().numpy(), dev_type)
    assert torch.allclose(saved[0].double(), mu - atk.gamma * torch.from_numpy(p), atol=1e-5, rtol=1e-5)
    # the virtual-row oracle
    got = []
    vr = VirtualRows(kind, 0.0, [n_h], dev_type=dev_type, report=got.append)
    val = vr.value(ut)
    assert got[0] == pytest.approx(want, rel=1e-9, abs=1e-12)
    assert torch.allclose(val, saved[0])
    # the Gram-domain search (host twin of the device solver), with the deviation as extra Gram row
    q = torch.from_numpy(p) if dev_type != "unit_vec" else None
    full = ut.double() if q is None else torch.cat([ut.double(), q[None]], 0)
    G = (full @ full.T).numpy()
    g, param = _agr.gram_scale(G, list(range(n_h)), n_h if q is not None else -1, kind, dev_type, 10.0, 1e-5)
    assert abs(g - want) <= 2e-5, (g, want)


def _check_property(u, kind, dev_type, g, gamma_init=10.0, tol=1e-5, slack=0.0):
    mu, p = u.mean(0), oracle_deviation(u, dev_type)
    thr = oracle_threshold(u, kind)
    assert oracle_test(u, kind, mu - g * p, thr * (1 + slack) + 1e-12)
    if g < 2 * gamma_init - 4 * tol:
        assert not oracle_test(u, kind, mu - (g + 4 * tol) * p, thr * (1 - slack))


@pytest.mark.parametrize("kind", ["minmax", "minsum"])
@pytest.mark.parametrize("dev_type", ["unit_vec", "std", "sign"])
@pytest.mark.parametrize("seed", range(4))
def test_returned_scale_is_the_largest_that_passes(kind, dev_type, seed):
    rng = np.random.default_rng(seed)
    n_h, d = int(rng.integers(2, 30)), int(rng.integers(1, 300))
    u = _rows(n_h, d, seed)
    gamma_init = float(rng.choice([0.5, 10.0, 100.0]))
    g, _ = _agr.direct_scale(torch.from_numpy(u), kind, dev_type, gamma_init, 1e-5)
    _check_property(u, kind, dev_type, g, gamma_init)


@pytest.mark.parametrize("kind", ["minmax", "minsum"])
def test_identical_honest_rows(kind):
    u = np.tile(np.array([0.5, -1.25, 2.0, 0.0]), (5, 1))       # threshold 0; every mean is exact
    for dev_type in ("unit_vec", "sign"):
        # any step along a non-zero p leaves the ball of radius 0
        g, m = _agr.direct_scale(torch.from_numpy(u), kind, dev_type, 10.0, 1e-5)
        assert g == oracle_gamma(u, kind, dev_type) == 0.0
        assert torch.equal(m, torch.from_numpy(u[0]))
    # std = 0: m = mu for every scale, the search runs to its ceiling
    g, m = _agr.direct_scale(torch.from_numpy(u), kind, "std", 10.0, 1e-5)
    assert g == oracle_gamma(u, kind, "std") and 20.0 - 2e-5 < g < 20.0
    G = u @ u.T
    assert _agr.gram_scale(G, range(5), -1, kind, "unit_vec", 10.0, 1e-5)[0] == 0.0


def test_zero_mean_unit_vec():
    u = np.array([[1.0, -2.0, 0.5], [-1.0, 2.0, -0.5]])
    for kind in ("minmax", "minsum"):
        g, m = _agr.direct_scale(torch.from_numpy(u), kind, "unit_vec", 10.0, 1e-5)
        assert g == oracle_gamma(u, kind, "unit_vec")
        assert torch.equal(m, torch.zeros(3, dtype=torch.float64))          # p = 0: m = mu
        gg, param = _agr.gram_scale(u @ u.T, [0, 1], -1, kind, "unit_vec", 10.0, 1e-5)
        assert gg == g and param == -1.0                                    # IPM form -(-1) * mu = mu


def test_bad_arguments():
    one = torch.ones(1, 4)
    with pytest.raises(ValueError):
        _agr.direct_scale(one, "minmax", "std", 10.0, 1e-5)
    with pytest.raises(ValueError):
        _agr.gram_scale(np.ones((2, 2)), [0], 1, "minsum", "std", 10.0, 1e-5)
    for kw in ({"gamma_init": 0.0}, {"gamma_init": -1.0}, {"tol": 0.0}, {"tol": -1e-5}, {"dev_type": "l2"}):
        with pytest.raises(ValueError):
            MinmaxClient(**kw)
        with pytest.raises(ValueError):
            MinsumClient(**kw)
        with pytest.raises(ValueError):
            VirtualRows("minmax", 0.0, [0], **kw)
    # too few honest rows for a std inside a matrix
    m = LocalMatrix(torch.randn(3, 8), VirtualRows("minsum", 0.0, [0, 1], dev_type="std"), use_kernels=False)
    with pytest.raises(ValueError):
        resolve_scaled_rows(m)


def test_gram_row_limit_is_a_value_error():
    m = LocalMatrix(torch.randn(512, 4), VirtualRows("minmax", 0.0, [0], dev_type="std"), use_kernels=False)
    with pytest.raises(ValueError, match="512"):
        resolve_scaled_rows(m)


@pytest.mark.parametrize("kind", ["minmax", "minsum"])
@pytest.mark.parametrize("dev_type", ["unit_vec", "std", "sign"])
def test_resolved_form_on_a_cpu_matrix(kind, dev_type):
    """The Gram-domain fallback of a matrix gives the kernel form whose value is the virtual-row oracle's."""
    torch.manual_seed(0)
    U = torch.randn(12, 257) * 0.1 + 0.05
    byz = [0, 5, 7]
    got = []
    vr = VirtualRows(kind, 0.0, byz, dev_type=dev_type, report=got.append)
    m = LocalMatrix(U.clone(), vr, use_kernels=False)
    resolve_scaled_rows(m)
    form = m.virtual
    assert form.kind == _agr.KERNEL_FORM[dev_type] and list(form.replaced) == byz
    honest = U[[i for i in range(12) if i not in byz]]
    want = vr.value(honest)
    assert abs(got[0] - got[1]) <= 2e-5
    assert torch.allclose(form.value(honest), want, atol=5e-5 * max(1.0, float(want.abs().max())))


def test_fusable_attack_needs_identical_parameters(tmp_path):
    from blades_b200 import Simulator
    from blades_b200.datasets import synthetic_fldataset
    ds = synthetic_fldataset(6, shape=(28, 28), train_bs=4, train_per_client=8, test_per_client=4, seed=3)
    sim = Simulator(ds, num_byzantine=2, attack="minsum", attack_kws={"dev_type": "sign", "tol": 1e-4},
                    aggregator="median", use_cuda=False, seed=1, log_path=str(tmp_path), progress=False)
    from blades_b200.models import MLP
    sim.prepare(MLP())
    cbs = sim._active_callbacks()
    v = sim.engine.fusable_attack(cbs)
    assert (v.kind, v.dev_type, v.gamma_init, v.tol) == ("minsum", "sign", 10.0, 1e-4)
    assert sorted(v.replaced) == sorted(v.byzantine) and len(v.replaced) == 2
    cbs[0].__self__.tol = 2e-4
    assert sim.engine.fusable_attack(cbs) is None


AGGS = {"mean": None, "median": None, "trimmedmean": {"nb": 2}, "krum": {"num_clients": 10, "num_byzantine": 2},
        "multikrum": {"num_byzantine": 2}, "geomed": None, "autogm": None, "centeredclipping": None,
        "clippedclustering": None, "clustering": None, "fltrust": None}


def _run(tmp_path, attack, agg, fuse, rounds=2, attack_kws=None):
    from blades_b200 import Simulator
    from blades_b200.datasets import synthetic_fldataset
    from blades_b200.models import MLP
    ds = synthetic_fldataset(10, shape=(28, 28), train_bs=4, train_per_client=8, test_per_client=4, seed=3,
                             separation=2.0)
    sim = Simulator(ds, num_byzantine=2, attack=attack, attack_kws=attack_kws, aggregator=agg,
                    aggregator_kws=AGGS[agg], use_cuda=False, seed=1, log_path=str(tmp_path / f"{agg}{fuse}"),
                    progress=False, fuse_attack=fuse)
    if agg == "fltrust":
        sim.set_trusted_clients([9])
    torch.manual_seed(5)
    m = MLP()
    sim.run(m, global_rounds=rounds, local_steps=1, server_lr=1.0, client_lr=0.1, validate_interval=rounds)
    return sim, torch.cat([p.detach().reshape(-1) for p in m.parameters()])


@pytest.mark.parametrize("attack", ["minmax", "minsum"])
@pytest.mark.parametrize("agg", sorted(AGGS))
def test_every_builtin_aggregator_runs(tmp_path, attack, agg):
    sim, theta = _run(tmp_path, attack, agg, True, rounds=1)
    assert torch.isfinite(theta).all()
    g = [c.gamma for c in sim.get_clients() if c.is_byzantine()]
    assert g[0] is not None and g[0] >= 0 and len(set(g)) == 1


@pytest.mark.parametrize("attack,dev_type", [("minmax", "unit_vec"), ("minsum", "std"), ("minmax", "sign")])
@pytest.mark.parametrize("agg", ["trimmedmean", "median", "krum"])
def test_fused_equals_callbacks(tmp_path, attack, dev_type, agg):
    a = _run(tmp_path, attack, agg, True, attack_kws={"dev_type": dev_type})[1]
    b = _run(tmp_path, attack, agg, False, attack_kws={"dev_type": dev_type})[1]
    assert torch.allclose(a, b, atol=1e-5, rtol=0), (a - b).abs().max()

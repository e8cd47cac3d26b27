"""Min-Max / Min-Sum attacks on the B200: the deviation kernel, the on-device scale solver, the device-resident
virtual-row parameter of the select / attack-row kernels, the fused aggregation paths and the whole-round graph."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from blades_b200.attackers import _agr

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _dev():
    return torch.device("cuda", 0)


@pytest.fixture(scope="module", autouse=True)
def _lib():
    from blades_b200.ops import _loader, _structs
    lib = _loader.cuda_lib()
    _structs.verify(lib)
    return lib


def _updates(n, d, seed, scale=0.01):
    """Rows with a common component, in a matrix whose rows are padded to 64 floats like the engine's."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    u = torch.randn(n, d, generator=g) * scale + torch.randn(d, generator=g) * scale * 0.5
    store = torch.zeros(n, (d + 63) // 64 * 64, device=_dev())
    store[:, :d] = u.to(_dev())
    return store[:, :d]


def _deviation_ref(honest, dev_type):
    h = honest.double()
    mu = h.mean(0)
    if dev_type == "std":
        return h.std(0, unbiased=True)
    return torch.sign(mu) if dev_type == "sign" else mu


# ----------------------------------------------------------------------------- deviation kernel
@pytest.mark.parametrize("dev_type", ["unit_vec", "std", "sign"])
@pytest.mark.parametrize("n,d", [(2, 1001), (17, 40003), (200, 5000)])
def test_deviation_kernel_matches_torch(dev_type, n, d):
    from blades_b200.ops import attack, select
    U = _updates(n + 2, d, n + d)
    U[n:] = float("nan")                      # rows outside the honest set are never read
    U[1, :5] = float("nan")                   # a non-finite honest row is sanitised like nan_to_num
    if dev_type != "std":                     # (inf -> FLT_MAX: its square overflows the fp32 std, as in ALIE)
        U[1, 5:9] = float("inf")
    honest = list(range(n))
    q = torch.full((d,), 7.0, device=_dev())
    attack.deviation(select.row_pointers(U, honest), dev_type, 0, d, q)
    ref = _deviation_ref(torch.nan_to_num(U[honest]), dev_type)
    if dev_type == "sign":
        mu = torch.nan_to_num(U[honest]).double().mean(0)
        clear = mu.abs() > 1e-6                                     # fp32 vs fp64 mean: only exact signs compared
        assert torch.equal(q.double()[clear], ref[clear])
    else:
        assert torch.allclose(q.double(), ref, rtol=1e-4, atol=1e-7)
    # a coordinate range is written, nothing outside it
    q2 = torch.full((d,), 7.0, device=_dev())
    attack.deviation(select.row_pointers(U, honest), dev_type, 128, d // 2, q2)
    assert torch.equal(q2[128: d // 2], q[128: d // 2])
    assert (q2[:128] == 7.0).all() and (q2[d // 2:] == 7.0).all()


# ----------------------------------------------------------------------------- scale solver
def _direct_test(u, kind, m, thr):
    d = ((u - m) ** 2).sum(1)
    return float(d.max() if kind == "minmax" else d.sum()) <= thr


def _direct_thr(u, kind):
    D = torch.stack([((u - u[i]) ** 2).sum(1) for i in range(u.shape[0])])
    return float(D.max() if kind == "minmax" else D.sum(1).max())


@pytest.mark.parametrize("kind", ["minmax", "minsum"])
@pytest.mark.parametrize("dev_type", ["unit_vec", "std", "sign"])
@pytest.mark.parametrize("n_h,f,d,gamma_init", [(2, 1, 3001, 10.0), (10, 3, 20000, 10.0), (80, 20, 50000, 10.0),
                                                (200, 50, 8000, 1.0), (30, 0, 777, 0.05)])
def test_device_solver_matches_host_search(kind, dev_type, n_h, f, d, gamma_init):
    from blades_b200.ops import attack, gram_solve, select
    from blades_b200.parallel.matrix import LocalMatrix
    tol = 1e-5 if gamma_init > 0.1 else 1e-7
    n = n_h + f
    U = _updates(n, d, n_h * 7 + f)
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(n)).tolist()
    byz = sorted(perm[:f])
    honest = [i for i in range(n) if i not in byz]
    q = None
    if dev_type != "unit_vec":
        q = torch.empty(d, device=_dev())
        attack.deviation(select.row_pointers(U, honest), dev_type, 0, d, q)
    dg = LocalMatrix(U).gram_device(q)
    assert dg is not None
    q_row = n if q is not None else -1
    gamma, param = gram_solve.agr_scale(dg, gram_solve.index_tensor(honest, _dev()), q_row, kind == "minsum",
                                        dev_type, gamma_init, tol)
    g = float(gamma)
    # host twin on the same Gram
    gh, ph = _agr.gram_scale(dg.dense().double().cpu().numpy(), honest, q_row, kind, dev_type, gamma_init, tol)
    assert abs(g - gh) <= 2 * tol, (g, gh)
    # property on fp64 direct distances (the Gram is 3xTF32: 1e-4 relative slack on the threshold)
    u = U[honest].double()
    mu = u.mean(0)
    p = _deviation_ref(U[honest], dev_type)
    if dev_type == "unit_vec":
        p = p / p.norm()
    thr = _direct_thr(u, kind)
    assert _direct_test(u, kind, mu - g * p, thr * (1 + 1e-4))
    if g < 2 * gamma_init - 4 * tol:
        assert not _direct_test(u, kind, mu - (g + 4 * tol) * p, thr * (1 - 1e-4))
    # the kernel parameter reproduces m(g): for unit_vec it is g / ||mu|| - 1 with ||mu|| taken from the same Gram
    # (mean of its honest block), which agrees with the direct norm to the Gram's precision
    if dev_type == "unit_vec":
        Gh = dg.dense().double()[honest][:, honest]
        nrm = float(Gh.mean().clamp_min(0).sqrt())
        assert float(param) == pytest.approx(g / nrm - 1.0, rel=1e-6, abs=1e-7)
        assert (float(param) + 1.0) * float(mu.norm()) == pytest.approx(g, rel=1e-4)
    else:
        assert float(param) == pytest.approx(g, rel=1e-6)


def test_device_solver_zero_mean_unit_vec():
    from blades_b200.ops import gram_solve
    from blades_b200.parallel.matrix import LocalMatrix
    u = _updates(1, 4096, 1)
    U = torch.cat([u, -u], 0)
    dg = LocalMatrix(U).gram_device()
    gamma, param = gram_solve.agr_scale(dg, gram_solve.index_tensor([0, 1], _dev()), -1, False, "unit_vec", 10.0, 1e-5)
    assert float(param) == -1.0
    gh, _ = _agr.gram_scale(dg.dense().double().cpu().numpy(), [0, 1], -1, "minmax", "unit_vec", 10.0, 1e-5)
    assert float(gamma) == gh


# ----------------------------------------------------------------------------- device-resident parameter
@pytest.mark.parametrize("kind,param", [("alie", 0.2858), ("ipm", 0.7131), ("sign", 0.00123)])
@pytest.mark.parametrize("n,f,b,d,expect", [(100, 20, 20, 30011, "partition"), (12, 3, 3, 20011, "network"),
                                            (230, 30, 40, 7001, "large")])
def test_select_reads_param_from_device(kind, param, n, f, b, d, expect):
    """With ``param_dev`` holding the same float the launch would pass, ALIE and IPM give bit-identical output on the
    partition, network and large kernels; the sign form matches torch."""
    from blades_b200.ops import attack, select
    from blades_b200.parallel.matrix import VirtualRows
    g = torch.Generator(device="cpu").manual_seed(n + d)
    U = (torch.randn(n, d, generator=g) * 0.1 + torch.sign(torch.randn(d, generator=g))).to(_dev())   # |mean| ~ 1
    host = VirtualRows(kind, param, list(range(f)))
    dev = VirtualRows(kind, 0.0, list(range(f)), param_dev=torch.tensor([param], device=_dev()))
    assert select.kernel_choice(n - f, 0, f, kind, 0, b) == expect
    for fn in (lambda v: select.trimmed_mean(U, b, virtual=v), lambda v: select.median(U, virtual=v)):
        assert torch.equal(fn(dev), fn(host))
    # against torch, sign form included
    honest = U[f:].double()
    mu = honest.mean(0)
    val = {"alie": mu - param * honest.std(0), "ipm": -param * mu, "sign": mu - param * torch.sign(mu)}[kind]
    Um = U.clone()
    Um[:f] = val.float()
    s = Um.double().sort(0).values
    assert torch.allclose(select.trimmed_mean(U, b, virtual=dev).double(), s[b: n - b].mean(0), atol=2e-5, rtol=1e-4)
    assert torch.allclose(select.median(U, virtual=dev).double(), (s[(n - 1) // 2] + s[n // 2]) / 2, atol=2e-5,
                          rtol=1e-4)
    # the attack-row kernel (Gram-based aggregators) reads the same pointer
    out_h, out_d = U.clone(), U.clone()
    rows_h = select.row_pointers(out_h, list(range(f, n)))
    rows_d = select.row_pointers(out_d, list(range(f, n)))
    attack.attack_rows(rows_h, select.row_pointers(out_h, list(range(f))), kind, param, 0, d)
    attack.attack_rows(rows_d, select.row_pointers(out_d, list(range(f))), kind, 0.0, 0, d,
                       param_ptr=dev.param_ptr())
    assert torch.equal(out_h, out_d)
    assert torch.allclose(out_d[:f].double(), val.expand(f, d), atol=1e-5, rtol=1e-5)


# ----------------------------------------------------------------------------- matrices with minmax / minsum rows
@pytest.mark.parametrize("attack,dev_type", [("minmax", "unit_vec"), ("minsum", "std"), ("minmax", "sign"),
                                             ("minsum", "unit_vec")])
@pytest.mark.parametrize("agg", ["trimmedmean", "median", "krum", "geomed"])
def test_local_matrix_matches_cpu_oracle(attack, dev_type, agg):
    from blades_b200.aggregators import Geomed, Krum, Median, Trimmedmean
    from blades_b200.parallel.matrix import LocalMatrix, VirtualRows
    n, f, d = 40, 8, 30000
    U = _updates(n, d, 11)
    byz = list(range(3, 3 + f))
    aggr = {"trimmedmean": lambda: Trimmedmean(nb=f), "median": Median, "krum": lambda: Krum(n, f, compat=False),
            "geomed": Geomed}[agg]
    res, gammas = [], []
    for use_kernels in (True, False):
        got = []
        v = VirtualRows(attack, 0.0, byz, dev_type=dev_type, report=got.append)
        data = U.clone() if use_kernels else U.cpu().clone()
        out = aggr().aggregate(LocalMatrix(data, v, use_kernels=use_kernels))
        res.append(out.detach().double().cpu().clone())
        gammas.append(float(got[0]))
        if use_kernels:
            assert torch.is_tensor(got[0]) and got[0].is_cuda, "the scale search did not stay on the device"
    assert abs(gammas[0] - gammas[1]) <= 1e-4 * max(1.0, gammas[1]), gammas
    scale = float(res[1].abs().max())
    assert torch.allclose(res[0], res[1], atol=1e-4 * scale, rtol=1e-3), (res[0] - res[1]).abs().max()


# ----------------------------------------------------------------------------- whole-round graph
@pytest.mark.parametrize("agg,attack,kws", [("trimmedmean", "minmax", None), ("median", "minsum", None),
                                            ("multikrum", "minmax", {"dev_type": "std"}),
                                            ("krum", "minsum", {"dev_type": "sign"})])
def test_whole_round_graph_equals_eager_minmax(agg, attack, kws, tmp_path, monkeypatch):
    """The round (train -> deviation pass -> Gram -> scale solve -> fused aggregation + server step) is one CUDA graph
    replay: a capture fails on any host sync, so a captured graph shows the round has none."""
    from blades_b200 import Simulator
    from blades_b200.datasets import synthetic_fldataset
    from blades_b200.models import MLP
    res, gammas = [], []
    for flag in ("1", "0"):
        monkeypatch.setenv("BLADES_ROUND_GRAPH", flag)
        monkeypatch.setenv("BLADES_GRAPH", flag)
        ds = synthetic_fldataset(10, shape=(28, 28), train_bs=8, seed=3, separation=2.0)
        sim = Simulator(ds, num_byzantine=3, attack=attack, attack_kws=kws, aggregator=agg,
                        aggregator_kws={"nb": 3} if agg == "trimmedmean" else (
                            {"num_clients": 10, "num_byzantine": 3} if agg == "krum" else (
                                {"num_byzantine": 3} if agg == "multikrum" else None)), use_cuda=True, seed=1,
                        log_path=str(tmp_path / f"l{flag}"), progress=False)
        torch.manual_seed(5)
        m = MLP()
        sim.run(m, global_rounds=6, local_steps=1, server_lr=1.0, client_lr=0.1, validate_interval=6)
        if flag == "1":
            assert any("graph" in st for st in sim.engine._round_graphs.values()), "round graph was not captured"
        res.append(torch.cat([p.detach().cpu().reshape(-1) for p in m.parameters()]))
        gammas.append([c.gamma for c in sim.get_clients() if c.is_byzantine()])
    assert len(set(gammas[0])) == 1 and gammas[0][0] > 0
    assert gammas[0][0] == pytest.approx(gammas[1][0], rel=1e-3, abs=1e-4)
    assert torch.allclose(res[0], res[1], atol=1e-5, rtol=1e-4), (res[0] - res[1]).abs().max()


# ----------------------------------------------------------------------------- multi-GPU
def _launch(nproc, out_dir, agg, attack, model, n_clients, port):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "_mgpu_worker.py"),
           out_dir, agg, attack, model, str(n_clients)]
    env = dict(os.environ, BLADES_FORBID_DENSE_GATHER="1")       # the fused attack never gathers [N, d]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    if r.returncode != 0:
        errs = ""
        for f in sorted(os.listdir(out_dir)):
            if f.startswith("error_rank"):
                errs += f"\n--- {f}\n" + open(os.path.join(out_dir, f)).read()[-2500:]
        raise AssertionError(errs or r.stderr[-3000:])


@pytest.mark.multigpu
@pytest.mark.parametrize("agg,attack", [("trimmedmean", "minmax"), ("krum", "minsum")])
def test_sharded_minmax_equals_single(agg, attack, tmp_path):
    ngpu = torch.cuda.device_count()
    out = str(tmp_path)
    sizes = [1, 2] + ([ngpu] if ngpu > 2 else [])
    for i, w in enumerate(sizes):
        _launch(w, out, agg, attack, "mlp", 10, 29710 + i)
    base = torch.load(os.path.join(out, f"theta_{agg}_{attack}_mlp_1_0.pt"))
    for w in sizes[1:]:
        vecs = [torch.load(os.path.join(out, f"theta_{agg}_{attack}_mlp_{w}_{r}.pt")) for r in range(w)]
        for v in vecs[1:]:
            assert torch.equal(v, vecs[0]), "replicas diverged"
        assert torch.allclose(vecs[0], base, atol=5e-4, rtol=1e-2), (w, (vecs[0] - base).abs().max())

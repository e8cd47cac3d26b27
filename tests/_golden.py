"""Stored outputs of the original package (bladesteam/blades) that the parity tests compare against.

The parity tests run this package and compare with what the unmodified original computed on the same inputs.  Those
outputs live under ``tests/golden/reference/`` (one ``.npz`` per test case), so the comparisons need nothing outside
the repository.  With the original installed under ``baseline/_ref`` (``baseline/install_ref.sh``),
``BLADES_RECORD_GOLDEN=1 pytest tests/test_reference_parity.py tests/test_compat_scripts.py`` recomputes every stored
value from it and rewrites the files.  Long vectors are stored as a fixed, seeded sample of their coordinates plus their
length and largest magnitude; a model's parameters as a fixed sample of every parameter tensor plus each tensor's sum,
L2 norm and largest magnitude, so that every tensor is checked."""
import json
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DIR = os.path.join(ROOT, "tests", "golden", "reference")
REF_INSTALLED = os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "blades"))
RECORD = os.environ.get("BLADES_RECORD_GOLDEN") == "1"
SAMPLE = 256
PER_TENSOR = 32


def key(request) -> str:
    return re.sub(r"[^\w.-]+", "_", request.node.name).strip("_")


def golden(name: str, compute) -> dict:
    """``compute()`` (which runs the original) when recording, else the stored result of an earlier recording."""
    path = os.path.join(DIR, name + ".npz")
    if RECORD:
        assert REF_INSTALLED, "recording needs the original package under baseline/_ref (baseline/install_ref.sh)"
        os.makedirs(DIR, exist_ok=True)
        np.savez_compressed(path, **{k: np.asarray(v) for k, v in compute().items()})
    with np.load(path, allow_pickle=False) as z:
        return {k: z[k] for k in z.files}


def js(obj):
    """A JSON-serialisable value as something ``golden`` can store."""
    return np.frombuffer(json.dumps(obj).encode(), dtype=np.uint8)


def unjs(a):
    return json.loads(a.tobytes().decode())


def _index(n: int, k: int = SAMPLE) -> np.ndarray:
    return np.sort(np.random.default_rng(n).choice(n, min(n, k), replace=False))


def sample(v, prefix: str = "v") -> dict:
    """A long vector as ``{prefix: sampled coordinates, prefix_n: length, prefix_max: largest |value|}``."""
    v = np.asarray(v.detach().cpu() if hasattr(v, "detach") else v).reshape(-1)
    return {prefix: v[_index(v.size)], prefix + "_n": v.size, prefix + "_max": np.abs(v).max()}


def sampled_err(got, want: dict, prefix: str = "v") -> float:
    """Largest |got - want| over the stored coordinates of a vector stored by ``sample``."""
    got = np.asarray(got.detach().cpu() if hasattr(got, "detach") else got, dtype=np.float64).reshape(-1)
    assert got.size == int(want[prefix + "_n"]), (got.size, int(want[prefix + "_n"]))
    return float(np.abs(got[_index(got.size)] - want[prefix].astype(np.float64)).max())


def _named(model_or_named):
    named = model_or_named.named_parameters() if hasattr(model_or_named, "named_parameters") else model_or_named
    return [(n, np.asarray(p.detach().cpu()).reshape(-1)) for n, p in named]


def params(model, prefix: str = "") -> dict:
    """A model's parameters (``named_parameters()`` order): per tensor ``PER_TENSOR`` seeded coordinates and
    ``[numel, sum, L2 norm, largest |value|]``."""
    named = _named(model)
    out = {prefix + "names": np.array([n for n, _ in named]),
           prefix + "stats": np.array([[v.size, v.astype(np.float64).sum(), np.linalg.norm(v.astype(np.float64)),
                                        np.abs(v).max()] for _, v in named])}
    out.update({f"{prefix}p{i}": v[_index(v.size, PER_TENSOR)] for i, (_, v) in enumerate(named)})
    return out


def params_max(want: dict, prefix: str = "") -> float:
    """Largest |value| over all parameters stored by ``params``."""
    return float(want[prefix + "stats"][:, 3].max())


def params_mismatches(model, want: dict, atol: float, prefix: str = "") -> list:
    """Every way ``model``'s parameters can be shown to differ from the stored ones by more than ``atol`` in some
    coordinate: names, sizes, the stored coordinates, and each tensor's sum, norm and largest magnitude (a sum can move
    by at most ``atol * numel`` and a norm by at most ``atol * sqrt(numel)`` when every coordinate is within ``atol``).
    Empty when they agree."""
    named = _named(model)
    names = [n for n, _ in named]
    if names != want[prefix + "names"].tolist():
        return [("names", names)]
    bad = []
    for i, ((name, v), (n, s, l2, mx)) in enumerate(zip(named, want[prefix + "stats"])):
        g = v.astype(np.float64)
        if g.size != int(n):
            bad.append((name, "numel", g.size, int(n)))
            continue
        err = float(np.abs(g[_index(g.size, PER_TENSOR)] - want[f"{prefix}p{i}"].astype(np.float64)).max())
        slack = 1e-9 * (1.0 + abs(s) + l2)                      # float64 rounding of the sums themselves
        checks = {"coords": (err, atol), "sum": (abs(g.sum() - s), atol * g.size + slack),
                  "norm": (abs(np.linalg.norm(g) - l2), atol * np.sqrt(g.size) + slack),
                  "max": (abs(np.abs(g).max() - mx), atol)}
        bad += [(name, what, d, tol) for what, (d, tol) in checks.items() if not d <= tol]
    return bad

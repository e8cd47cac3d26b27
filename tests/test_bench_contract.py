"""bench.py contract pieces that can be checked without a GPU."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ref_arm(*extra, env=None):
    e = dict(os.environ, **(env or {}))
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1",
                          "--steps", "1", "--warmup", "1", "--clients", "4", *extra],
                         capture_output=True, text=True, cwd=ROOT, env=e)
    assert out.returncode == 0, out.stderr
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_reference_arm_contract():
    """``--impl reference`` prints ONE json line and exits 0: a measured value when the unmodified reference is
    installed under baseline/_ref (baseline/install_ref.sh), otherwise ``unavailable`` with the reason."""
    rec = _ref_arm(env={"BLADES_REF_BUDGET_S": "1"})
    assert rec["impl"] == "reference"
    if os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "blades")):
        assert "unavailable" not in rec, rec
        assert rec["value"] > 0 and rec["unit"] == "rounds/s" and rec["steps"] >= 1
        assert rec["config"]["model"].startswith("resnet18") and rec["config"]["attack"] == "alie"
    else:
        assert "unavailable" in rec


def test_reference_arm_deadline_is_enforced():
    rec = _ref_arm(env={"BLADES_REF_DEADLINE_S": "0.5"})
    assert rec["impl"] == "reference" and "unavailable" in rec


def _tree_digest(top):
    import hashlib
    return {os.path.relpath(os.path.join(d, f), top): hashlib.sha256(open(os.path.join(d, f), "rb").read()).hexdigest()
            for d, dirs, files in os.walk(top) if "__pycache__" not in d.split(os.sep) for f in files}


def test_reference_arm_uses_unmodified_tree():
    """The installed reference is byte for byte the released tree: every file's SHA-256 as listed in
    tests/golden/reference_tree.json (recorded from the reference's src/blades)."""
    ref = os.path.join(ROOT, "baseline", "_ref", "blades")
    if not os.path.isdir(ref):
        import pytest
        pytest.skip("reference not installed under baseline/_ref")
    with open(os.path.join(ROOT, "tests", "golden", "reference_tree.json")) as fh:
        want = json.load(fh)
    got = _tree_digest(ref)
    assert got == want, sorted(set(got.items()) ^ set(want.items()))[:5]


def test_graft_entry_build_is_idempotent():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as g
    g.build()
    g.build()
    assert os.path.exists(os.path.join(ROOT, "blades_b200", "_cuda.so"))
    assert os.path.exists(os.path.join(ROOT, "blades_b200", "_host.so"))

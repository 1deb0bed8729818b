"""Acceptance on the reference's own callers (SURVEY section 2, rows 6 and 7): the UNMODIFIED reference test-suite
(43 cases) and examples/demo.py, run against this package on a B200.

The reference sources are not part of this repository: `oracle/make_ref.py` (called by `__graft_entry__.build()`) copies
them from the checkout that CGNN_REFERENCE names into the git-ignored oracle/_ref/; without that copy both tests skip.
Each run is a subprocess whose PYTHONPATH puts THIS package first, so `import connectome_gnn` inside the reference's
tests / demo resolves to the B200 build; the subprocess output is checked for that."""
import os
import re
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref", "callers")
PKG = os.path.join(ROOT, "connectome-gnn-suite_b200")


def _env():
    env = dict(os.environ)
    env["PYTHONPATH"] = PKG + os.pathsep + env.get("PYTHONPATH", "")
    env["PYTHONDONTWRITEBYTECODE"] = "1"
    return env


def _need_ref():
    if not os.path.isdir(os.path.join(REF, "tests")):
        pytest.skip("oracle/_ref is absent (run __graft_entry__.build() with CGNN_REFERENCE set to a checkout of the reference)")
    # the subprocesses share the device with this process: hand back what its caching allocator still holds from the
    # full-size tests, so that the reference's tests never compete with tens of cached GB
    import gc
    import torch
    gc.collect()
    if torch.cuda.is_available():
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


def _keep(path, out) -> str:
    """Tail of a subprocess's output for the assertion message; the whole of it goes to ``path`` for a post-mortem."""
    with open(path, "w") as f:
        f.write(out.stdout + "\n==== stderr ====\n" + out.stderr)
    return out.stdout[-2500:] + out.stderr[-1500:]


def test_reference_test_suite_passes_against_the_package(tmp_path):
    _need_ref()
    probe = "import connectome_gnn, sys; sys.stdout.write(connectome_gnn.__file__ + ' ' + getattr(connectome_gnn, 'BACKEND', 'reference'))"
    who = subprocess.run([sys.executable, "-c", probe], env=_env(), cwd=REF, capture_output=True, text=True, timeout=300)
    assert PKG in who.stdout and "cuda-sm_100a" in who.stdout, who.stdout + who.stderr
    out = subprocess.run([sys.executable, "-m", "pytest", os.path.join(REF, "tests"), "-q", "-p", "no:cacheprovider",
                          "--rootdir", REF, "-x"], env=_env(), cwd=REF, capture_output=True, text=True, timeout=1200)
    tail = _keep(tmp_path / "ref_suite.log", out)
    assert out.returncode == 0, tail
    m = re.search(r"(\d+) passed", out.stdout)
    assert m and int(m.group(1)) == 43, tail


def test_reference_demo_runs_unchanged(tmp_path):
    """examples/demo.py (BASELINE configs[0]: 300 subjects x 84 nodes, batch 16, hidden 64, 30 epochs, patience 8) end to
    end on the B200 package.  The trajectory depends on the dropout stream (SURVEY A.4-9), so the check is what the
    reference itself promises: both models train, stop early or finish, and report a test accuracy."""
    _need_ref()
    out = subprocess.run([sys.executable, os.path.join(REF, "examples", "demo.py")], env=_env(), cwd=REF, capture_output=True,
                         text=True, timeout=1200)
    text = out.stdout
    assert out.returncode == 0, _keep(tmp_path / "ref_demo.log", out)
    accs = [float(x) for x in re.findall(r"[Tt]est acc(?:uracy)?\s*[:=]\s*([0-9.]+)", text)]
    assert len(accs) >= 2, text[-1500:]
    assert all(0.3 <= a <= 1.0 for a in accs), accs

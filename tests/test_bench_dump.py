"""bench.py --dump-outputs: what the last timed step returned, as .npy files that two builds can compare entry for entry."""
import glob
import os
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

import helpers

BENCH = os.path.join(helpers.ROOT, "bench.py")


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_under_test", BENCH)
    mod = importlib.util.module_from_spec(spec)
    keep = sys.dont_write_bytecode            # bench.py turns bytecode caching off for its own process
    try:
        spec.loader.exec_module(mod)
    finally:
        sys.dont_write_bytecode = keep
    return mod


def _fake_step():
    """Host-side stand-ins for what run_b200 hands dump_outputs: trainers with a model and gradients, per-leg results."""
    from connectome_gnn.models import GCNConnectome, GraphSAGEConnectome
    torch.manual_seed(0)
    trainers = {}
    for kind, cls in (("gcn", GCNConnectome), ("sage", GraphSAGEConnectome)):
        model = cls(in_channels=5, hidden_dim=64, num_classes=2, num_layers=3)
        for p in model.parameters():
            p.grad = torch.randn_like(p)
        trainers[kind] = types.SimpleNamespace(model=model)
    last = {"gcn_train": (torch.tensor(0.69),), "sage_train": (torch.tensor(0.70),),
            "gcn_infer": (torch.tensor(0.68), torch.tensor(2100)), "sage_infer": (torch.tensor(0.67), torch.tensor(2000))}
    return last, trainers


def _load(d):
    return {os.path.basename(p)[:-4]: np.load(p) for p in sorted(glob.glob(os.path.join(d, "*.npy")))}


def test_dump_writes_every_result_as_float_arrays(tmp_path):
    bench = _bench_module()
    last, trainers = _fake_step()
    bench.dump_outputs(str(tmp_path), last, trainers)
    got = _load(tmp_path)
    assert all(v.dtype in (np.float32, np.float64) for v in got.values())
    assert float(got["gcn_infer.correct"]) == 2100.0 and float(got["sage_train.loss"]) == pytest.approx(0.70)
    for kind in ("gcn", "sage"):
        model = trainers[kind].model
        for k, v in model.state_dict().items():
            assert np.array_equal(got[f"{kind}_train.{k}"], v.double().numpy() if not v.is_floating_point() else v.numpy())
        for k, p in model.named_parameters():
            assert np.array_equal(got[f"{kind}_train.grad.{k}"], p.grad.numpy())
    assert not any(k.startswith(("gcn_infer.", "sage_infer.")) and not k.endswith(("loss", "correct")) for k in got)


def test_dump_over_budget_is_a_fixed_sample(tmp_path):
    bench = _bench_module()
    last, trainers = _fake_step()
    full = tmp_path / "full"
    bench.dump_outputs(str(full), last, trainers)
    budget = 20000
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), last, trainers, budget=budget)
    a, b, ref = _load(tmp_path / "a"), _load(tmp_path / "b"), _load(full)
    assert a.keys() == b.keys() == ref.keys()
    assert sum(v.nbytes for v in a.values()) <= budget + 8 * len(a)      # at least one entry per array
    for k in a:
        assert np.array_equal(a[k], b[k]), k
        assert np.isin(a[k], ref[k].reshape(-1)).all(), k                 # entries of the full array, not new values


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_two_runs_with_the_same_arguments_dump_the_same_outputs(tmp_path):
    """Inputs, weights and dropout streams are seeded: two runs of the timed path must agree to the parity tolerance."""
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")}
    dumps = []
    for run in ("a", "b"):
        out = tmp_path / run
        res = subprocess.run([sys.executable, BENCH, "--gpus", "1", "--steps", "2", "--warmup", "1", "--batch", "64",
                              "--pool", "64", "--regions", "84", "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(out)],
                             env=env, cwd=str(tmp_path), capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-2000:]
        assert res.stdout.strip().startswith("{"), res.stdout[-500:]
        dumps.append(_load(out))
    a, b = dumps
    assert a.keys() == b.keys() and {"gcn_train.loss", "sage_infer.correct", "gcn_train.grad.convs.0.linear.weight"} <= a.keys()
    for k in a:
        assert a[k].dtype == b[k].dtype and a[k].shape == b[k].shape, k
        assert np.isfinite(a[k]).all(), k
        helpers.assert_close(a[k], b[k], k)

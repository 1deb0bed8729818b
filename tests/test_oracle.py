"""The oracle is only worth something if it IS the reference: pin it.

Every function of ``oracle/port.py`` and ``oracle/csr_ref.c`` is checked against the fixtures
``tests/golden/make_golden.py`` produced by running the unmodified reference
(danieleschmidt/connectome-gnn-suite, connectome_gnn/{graph,models,train}.py).  Float results are
expected BIT-EXACT here: the port issues the same ATen CPU ops in the same order as the reference,
on the torch build the fixtures were made with (8 threads, see ref_meta.json); a different
torch/thread count falls back to the fp32 tolerance of helpers.REL_TOL.
"""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import helpers
from oracle import port

META = json.load(open(os.path.join(helpers.GOLDEN, "ref_meta.json")))
SAME_BUILD = torch.__version__ == META["made_with"]["torch"]
FIXTURES = ["ref_small.npz", "ref_ragged.npz", "ref_c1.npz", "ref_c3.npz", "ref_c5.npz"]
REFERENCE = os.environ.get("CGNN_REFERENCE", "")   # optional checkout of the reference, for the live comparison


@pytest.fixture(autouse=True)
def _threads():
    old = torch.get_num_threads()
    torch.set_num_threads(META["made_with"]["threads"])
    yield
    torch.set_num_threads(old)


GRAD_TOL = 5e-6   # the reference's own CPU backward is not run-to-run deterministic at 8 threads
                  # (index_put_(accumulate=True) behind x[src]); measured spread ~7e-7 on ref_c1


def _same(got, ref, what, noise_atol=0.0, grad=False):
    """Bit-identical on the fixture's torch build for everything computed by a deterministic op sequence
    (collate, degrees, every forward tensor, loss).  Gradients (`grad=True`) are held to GRAD_TOL instead;
    `noise_atol` admits tensors that are analytically zero (GCN conv biases feed BatchNorm, SURVEY 2.2)
    and therefore pure reduction-order round-off."""
    got, ref = torch.as_tensor(got), torch.as_tensor(np.array(ref))
    if noise_atol > 0.0:
        assert float((got.double() - ref.double()).abs().max()) <= noise_atol, what
        return
    if grad:
        helpers.assert_close(got, ref, what, tol=GRAD_TOL)
        return
    if SAME_BUILD and torch.get_num_threads() == META["made_with"]["threads"]:
        assert torch.equal(got, ref.to(got.dtype)), f"{what}: oracle is not bit-identical to the reference"
    else:
        helpers.assert_close(got, ref, what)


def _batch(a):
    graphs = helpers.graphs_from_store(a)
    return graphs, port.collate(graphs)


@pytest.mark.parametrize("fixture", FIXTURES)
def test_collate_matches_reference(fixture):
    a = helpers.golden(fixture)
    _, b = _batch(a)
    assert torch.equal(b["ptr"], torch.from_numpy(a["batch.ptr"]))
    assert torch.equal(b["labels"], torch.from_numpy(a["batch.labels"]))
    if "batch.edge_index" in a:
        for k in ("node_features", "edge_index", "edge_weight", "batch"):
            assert torch.equal(b[k], torch.from_numpy(a["batch." + k])), k


@pytest.mark.parametrize("fixture", FIXTURES)
def test_structure_matches_reference(fixture):
    a = helpers.golden(fixture)
    _, b = _batch(a)
    n = b["node_features"].shape[0]
    _, _, w_hat, deg, dinv = port.gcn_structure(b["edge_index"], b["edge_weight"], n)
    assert torch.equal(deg, torch.from_numpy(a["deg"]))        # bit-exact on any build: sequential fp32 adds
    assert torch.equal(port.sage_wsum(b["edge_index"], b["edge_weight"], n)[:, 0], torch.from_numpy(a["wsum"]))
    _same(dinv, a["dinv"], "dinv")
    if "w_norm" in a:
        _same(w_hat, a["w_norm"], "w_norm")


@pytest.mark.parametrize("fixture", FIXTURES)
@pytest.mark.parametrize("kind", ["gcn", "sage"])
def test_models_match_reference(fixture, kind):
    a = helpers.golden(fixture)
    _, b = _batch(a)
    params = helpers.state_dict_from(a, f"{kind}.init")
    layers = []
    with torch.no_grad():
        _same(port.encode(kind, dict(params), b, collect=layers), a[f"{kind}.eval.emb"], "eval emb")
        _same(port.forward(kind, dict(params), b), a[f"{kind}.eval.logits"], "eval logits")
    for l, z in enumerate(layers):
        if f"{kind}.eval.z{l}" in a:
            _same(z, a[f"{kind}.eval.z{l}"], f"eval z{l}")
    p = {k: v.clone() for k, v in params.items()}
    logits, loss, grads = port.loss_and_grads(kind, p, b, training=True, dropout=0.0)
    _same(logits, a[f"{kind}.train.logits"], "train logits")
    _same(loss, a[f"{kind}.train.loss"], "train loss")
    scale = max(float(np.abs(a[f"{kind}.train.grad.{k}"]).max()) for k in grads)
    for k, g in grads.items():
        zero_by_construction = kind == "gcn" and k.startswith("convs.") and k.endswith(".bias")
        _same(g, a[f"{kind}.train.grad.{k}"], f"grad {k}", noise_atol=5e-6 * scale if zero_by_construction else 0.0,   # pure round-off, not deterministic at 8 threads
              grad=True)
    for k in p:
        if "running" in k or "num_batches" in k:
            _same(p[k], a[f"{kind}.train.after.{k}"], f"after {k}")


@pytest.mark.parametrize("kind", ["gcn", "sage"])
def test_training_loop_matches_reference(kind):
    """Trainer.fit trajectory (reference train.py:76-127 with Adam, randperm shuffling) on the port's loop."""
    a = helpers.golden("ref_trainer.npz")
    graphs = helpers.graphs_from_store(a)
    module = port.Module(kind, helpers.state_dict_from(a, f"{kind}.init"), dropout=0.0)
    opt = torch.optim.Adam(module.parameters(), lr=1e-3, weight_decay=1e-4)
    torch.manual_seed(1)
    ref = META["trainer"][kind]
    for epoch in range(3):
        tl = port.train_epoch(module, opt, graphs[:30], 10, shuffle=True)
        ev = port.evaluate(module, graphs[30:], 10)
        assert tl == pytest.approx(ref["history"]["train_loss"][epoch], rel=1e-6)
        assert ev["loss"] == pytest.approx(ref["history"]["val_loss"][epoch], rel=1e-6)
        assert ev["accuracy"] == ref["history"]["val_acc"][epoch]
    final = helpers.state_dict_from(a, f"{kind}.final")
    for k, v in module.tensors().items():
        helpers.assert_close(v, final[k], f"final {k}", tol=1e-5)


# ---- C part: collate + stable CSR + degrees ---------------------------------------------------

def _run_c_oracle(a):
    lib = C.CDLL(helpers.build_oracle())
    lib.oracle_collate_csr.restype = C.c_int
    st = {k[6:]: np.ascontiguousarray(v) for k, v in a.items() if k.startswith("store.")}
    S = len(st["node_ptr"]) - 1
    ids = np.arange(S, dtype=np.int64)
    rows, edges, F = int(st["node_ptr"][-1]), int(st["edge_ptr"][-1]), st["x"].shape[1]
    out = dict(
        x=np.empty((rows, F), np.float32), edge_index=np.empty((2, edges), np.int64), edge_weight=np.empty(edges, np.float32),
        batch=np.empty(rows, np.int64), labels=np.empty(S, np.int64), ptr=np.empty(S + 1, np.int64), eptr=np.empty(S + 1, np.int64),
        in_rowptr=np.empty(rows + 1, np.int32), in_col=np.empty(edges, np.int32), in_w=np.empty(edges, np.float32),
        in_wn=np.empty(edges, np.float32), out_rowptr=np.empty(rows + 1, np.int32), out_col=np.empty(edges, np.int32),
        out_w=np.empty(edges, np.float32), out_wn=np.empty(edges, np.float32), deg=np.empty(rows, np.float32),
        dinv=np.empty(rows, np.float32), wsum=np.empty(rows, np.float32))
    p = lambda arr: arr.ctypes.data_as(C.c_void_p)
    rc = lib.oracle_collate_csr(p(st["x"]), p(st["src"]), p(st["dst"]), p(st["w"]), p(st["node_ptr"]), p(st["edge_ptr"]),
                                p(st["label"]), C.c_int32(F), p(ids), C.c_int64(S),
                                *[p(out[k]) for k in ("x", "edge_index", "edge_weight", "batch", "labels", "ptr", "eptr",
                                                      "in_rowptr", "in_col", "in_w", "in_wn", "out_rowptr", "out_col",
                                                      "out_w", "out_wn", "deg", "dinv", "wsum")])
    assert rc == 0
    return out


@pytest.mark.parametrize("fixture", FIXTURES)
def test_c_oracle_matches_reference(fixture):
    a = helpers.golden(fixture)
    out = _run_c_oracle(a)
    assert np.array_equal(out["ptr"], a["batch.ptr"])
    assert np.array_equal(out["labels"], a["batch.labels"])
    if "batch.edge_index" in a:
        assert np.array_equal(out["x"], a["batch.node_features"])
        assert np.array_equal(out["edge_index"], a["batch.edge_index"])
        assert np.array_equal(out["edge_weight"], a["batch.edge_weight"])
        assert np.array_equal(out["batch"], a["batch.batch"])
    assert np.array_equal(out["deg"], a["deg"]), "D^ must be bit-exact (sequential fp32 adds, self loop last)"
    assert np.array_equal(out["wsum"], a["wsum"])
    helpers.assert_close(out["dinv"], a["dinv"], "dinv", tol=2e-7)
    # the CSR is a stable sort of the COO: check against numpy's stable argsort
    src, dst = out["edge_index"]
    for key, col_of, rowptr, col, w in ((dst, src, out["in_rowptr"], out["in_col"], out["in_w"]),
                                        (src, dst, out["out_rowptr"], out["out_col"], out["out_w"])):
        order = np.argsort(key, kind="stable")
        assert np.array_equal(col, col_of[order].astype(np.int32))
        assert np.array_equal(w, out["edge_weight"][order])
        assert np.array_equal(rowptr, np.searchsorted(key[order], np.arange(len(out["deg"]) + 1)).astype(np.int32))
    if "w_norm" in a:   # reference w^ in COO order (real edges first), compare through the permutation
        order = np.argsort(dst, kind="stable")
        helpers.assert_close(out["in_wn"], a["w_norm"][: len(src)][order], "w_norm", tol=3e-7)


def test_c1_fingerprints():
    """SURVEY Appendix B fingerprints of collate_graphs(generate_dataset(16, 84, seed=42))."""
    import hashlib
    a = helpers.golden("ref_c1.npz")
    out = _run_c_oracle(a)
    h = lambda arr: hashlib.sha256(np.ascontiguousarray(arr).tobytes()).hexdigest()[:16]
    fp = META["fingerprints"]
    assert h(out["x"]) == fp["c1.x"] and h(out["edge_index"]) == fp["c1.edge_index"]
    assert h(out["edge_weight"]) == fp["c1.edge_weight"] and h(out["batch"]) == fp["c1.batch"]
    assert h(out["deg"]) == fp["c1.deg"] and h(out["wsum"]) == fp["c1.wsum"]
    assert out["labels"].tolist() == fp["c1.labels"]


# ---- generator: the package's restatement must emit the reference's subjects ---------------------

def test_generator_matches_reference_fingerprints():
    import hashlib
    from connectome_gnn.synthetic import REGION_NAMES, generate_connectome, generate_dataset
    gen = META["generator"]
    h = lambda t: hashlib.sha256(t.contiguous().numpy().tobytes()).hexdigest()[:16]
    assert len(REGION_NAMES) == gen["num_regions"]
    assert hashlib.sha256("|".join(REGION_NAMES).encode()).hexdigest()[:16] == gen["region_names"]
    for key, ref in gen.items():
        if not key.startswith("n"):
            continue
        if key in ("num_regions",):
            continue
        n, seed = (int(s[1:]) for s in key.split("."))
        g = generate_connectome(num_regions=n, seed=seed)
        assert (h(g.edge_index), h(g.edge_weight), h(g.node_features), int(g.label), g.subject_id, g.num_edges) == \
            (ref["edge_index"], ref["edge_weight"], ref["node_features"], ref["label"], ref["subject_id"], ref["num_edges"]), key
    ds = generate_dataset(num_subjects=6, num_regions=84, seed=42)
    for g, ref in zip(ds, gen["dataset.84.42"]):
        assert (h(g.edge_index), h(g.node_features), int(g.label), g.subject_id) == \
            (ref["edge_index"], ref["node_features"], ref["label"], ref["subject_id"])


@pytest.mark.skipif(not (REFERENCE and os.path.isdir(os.path.join(REFERENCE, "connectome_gnn"))),
                    reason="needs CGNN_REFERENCE: a checkout of the reference, which is not part of this repository")
def test_oracle_against_live_reference():
    """Run the reference itself (separate process: it shares the import name with the package) on a fresh
    random case and compare the port on the same inputs."""
    code = r'''
import sys, json, torch, numpy as np
sys.path.insert(0, sys.argv[1])
from connectome_gnn.synthetic import generate_dataset
from connectome_gnn.graph import collate_graphs
from connectome_gnn.models import GCNConnectome, GraphSAGEConnectome
torch.set_num_threads(8)
gs = generate_dataset(5, 30, seed=99); b = collate_graphs(gs)
out = {}
for kind, cls in (("gcn", GCNConnectome), ("sage", GraphSAGEConnectome)):
    torch.manual_seed(3); m = cls(5, 24, 2, 2, 0.0); m.train()
    lg = m(b); loss = torch.nn.functional.cross_entropy(lg, b.labels); loss.backward()
    out[kind] = {"sd": {k: v.tolist() for k, v in m.state_dict().items()}, "logits": lg.tolist(), "loss": float(loss),
                 "grads": {k: p.grad.tolist() for k, p in m.named_parameters()}}
print(json.dumps(out))
'''
    res = subprocess.run([sys.executable, "-c", code, REFERENCE], capture_output=True, text=True, check=True,
                         env={**os.environ, "PYTHONDONTWRITEBYTECODE": "1", "PYTHONPATH": ""})
    ref = json.loads(res.stdout)
    from connectome_gnn.synthetic import generate_dataset
    b = port.collate(generate_dataset(5, 30, seed=99))
    for kind in ("gcn", "sage"):
        # the freshly trained reference model's state_dict already contains the post-step running stats;
        # reset them to their initial values to replay the step
        sd = {k: torch.tensor(v) for k, v in ref[kind]["sd"].items()}
        for k in sd:
            if k.endswith("running_mean"): sd[k] = torch.zeros_like(sd[k])
            if k.endswith("running_var"): sd[k] = torch.ones_like(sd[k])
            if k.endswith("num_batches_tracked"): sd[k] = torch.tensor(0)
        logits, loss, grads = port.loss_and_grads(kind, sd, b, training=True, dropout=0.0)
        _same(logits, np.array(ref[kind]["logits"], dtype=np.float32), "live logits")
        scale = max(float(np.abs(np.array(v)).max()) for v in ref[kind]["grads"].values())
        for k, g in grads.items():
            zero_by_construction = kind == "gcn" and k.startswith("convs.") and k.endswith(".bias")
            _same(g, np.array(ref[kind]["grads"][k], dtype=np.float32), f"live grad {k}",
                  noise_atol=5e-6 * scale if zero_by_construction else 0.0, grad=True)

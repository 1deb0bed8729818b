#!/usr/bin/env python3
"""Generate the golden fixtures in this directory FROM THE UNMODIFIED REFERENCE.

Run with a checkout of the reference first on the import path:

    PYTHONDONTWRITEBYTECODE=1 PYTHONPATH=<reference checkout> python tests/golden/make_golden.py

It imports ``connectome_gnn`` from that checkout (never the package in this repo), runs the
reference's own collate / models / Trainer on seeded synthetic inputs and stores inputs + outputs
as small ``.npz`` / ``.json`` files.  The oracle (``oracle/``) is pinned against these files by
``tests/test_oracle.py``; the CUDA path is compared against them (and the oracle) by the
``-m gpu`` tests.  Environment the committed files were made with: torch 2.11.0+cu128 (CPU),
numpy 2.3.5, Python 3.12.3, 8 threads.
"""
import hashlib
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))

import connectome_gnn  # noqa: E402  (must resolve to the reference)

# this package (in this tree or installed anywhere) sets BACKEND; the reference has no such attribute
assert not hasattr(connectome_gnn, "BACKEND"), f"{connectome_gnn.__file__} is this package, not the reference"
from connectome_gnn.graph import ConnectomeDataLoader, ConnectomeGraph, collate_graphs  # noqa: E402
from connectome_gnn.models import GCNConnectome, GraphSAGEConnectome  # noqa: E402
from connectome_gnn.synthetic import REGION_NAMES, generate_connectome, generate_dataset  # noqa: E402
from connectome_gnn.train import Trainer  # noqa: E402

MODELS = {"gcn": GCNConnectome, "sage": GraphSAGEConnectome}


def h16(t) -> str:
    a = t.contiguous().numpy() if isinstance(t, torch.Tensor) else np.ascontiguousarray(t)
    return hashlib.sha256(a.tobytes()).hexdigest()[:16]


def pack(graphs) -> dict:
    """Store arrays (the layout of cgnn_store_t) of a list of reference graphs."""
    node_ptr = np.cumsum([0] + [g.num_nodes for g in graphs]).astype(np.int64)
    edge_ptr = np.cumsum([0] + [g.num_edges for g in graphs]).astype(np.int64)
    return {
        "store.x": torch.cat([g.node_features for g in graphs]).numpy(),
        "store.src": torch.cat([g.edge_index[0] for g in graphs]).numpy().astype(np.int32),
        "store.dst": torch.cat([g.edge_index[1] for g in graphs]).numpy().astype(np.int32),
        "store.w": torch.cat([g.edge_weight for g in graphs]).numpy(),
        "store.node_ptr": node_ptr,
        "store.edge_ptr": edge_ptr,
        "store.label": np.array([int(g.label) if g.label is not None else 0 for g in graphs], dtype=np.int64),
        "store.has_label": np.array([g.label is not None for g in graphs]),
    }


def structure(batch) -> dict:
    """D^, d^-1/2, w^ (models.py:94-108) and w_sum (models.py:147-148) with the reference's ops."""
    n = batch.node_features.shape[0]
    src, dst = batch.edge_index
    idx = torch.arange(n)
    src_aug, dst_aug = torch.cat([src, idx]), torch.cat([dst, idx])
    w_aug = torch.cat([batch.edge_weight, torch.ones(n)])
    deg = torch.zeros(n)
    deg.scatter_add_(0, src_aug, w_aug)
    dinv = (deg + 1e-8).pow(-0.5)
    w_norm = dinv[src_aug] * w_aug * dinv[dst_aug]
    w_sum = torch.zeros(n, 1)
    w_sum.scatter_add_(0, dst.unsqueeze(1), batch.edge_weight.unsqueeze(1))
    return {"deg": deg.numpy(), "dinv": dinv.numpy(), "w_norm": w_norm.numpy(), "wsum": w_sum[:, 0].numpy()}


def batch_fields(batch) -> dict:
    out = {
        "batch.node_features": batch.node_features.numpy(), "batch.edge_index": batch.edge_index.numpy(),
        "batch.edge_weight": batch.edge_weight.numpy(), "batch.batch": batch.batch.numpy(),
        "batch.ptr": batch.ptr.numpy(),
    }
    if batch.labels is not None:
        out["batch.labels"] = batch.labels.numpy()
    return out


def model_case(kind: str, batch, hidden: int, layers: int, tag: str, per_layer: bool = True, eval_grad: bool = True) -> dict:
    """Seeded reference model: initial weights, eval outputs, one train-mode forward/backward with
    dropout disabled (masks from the CPU generator cannot be reproduced on a GPU)."""
    torch.manual_seed(0)
    model = MODELS[kind](in_channels=batch.node_features.shape[1], hidden_dim=hidden, num_classes=2,
                         num_layers=layers, dropout=0.0)
    out = {f"{tag}.init.{k}": v.clone().numpy() for k, v in model.state_dict().items()}
    model.eval()
    with torch.no_grad():
        out[f"{tag}.eval.emb"] = model.encode(batch).numpy()
        out[f"{tag}.eval.logits"] = model(batch).numpy()
        x = batch.node_features
        for l, (conv, bn) in enumerate(zip(model.convs, model.batch_norms)):   # per-layer eval activations
            x = conv(x, batch.edge_index, batch.edge_weight)
            if per_layer:
                out[f"{tag}.eval.z{l}"] = x.numpy()
            x = bn(x)
            if kind == "gcn":
                x = torch.relu(x)
    model.train()
    logits = model(batch)
    loss = torch.nn.CrossEntropyLoss()(logits, batch.labels)
    loss.backward()
    out[f"{tag}.train.logits"] = logits.detach().numpy()
    out[f"{tag}.train.loss"] = loss.detach().numpy()
    for k, p in model.named_parameters():
        out[f"{tag}.train.grad.{k}"] = p.grad.numpy()
    for k, v in model.state_dict().items():
        if "running" in k or "num_batches" in k:
            out[f"{tag}.train.after.{k}"] = v.clone().numpy()
    if not eval_grad:
        return out
    # gradient of sum(logits) in eval mode (BatchNorm with running statistics), cf. tests/test_models.py:32-40
    model.zero_grad()
    model.eval()
    model(batch).sum().backward()
    for k, p in model.named_parameters():
        out[f"{tag}.evalgrad.{k}"] = p.grad.numpy()
    return out


def ragged_graphs():
    """Hand-made subjects exercising what tests/test_graph.py:8-26 and README.md:153-179 allow:
    different sizes, duplicate edges, explicit self loops, an isolated node, asymmetric edges, no edges."""
    g = torch.Generator().manual_seed(1234)
    graphs = []
    for k, (n, e) in enumerate([(5, 4), (12, 30), (20, 50), (7, 0), (9, 25), (3, 6)]):
        x = torch.randn(n, 3, generator=g)
        if e:
            src = torch.randint(0, n, (e,), generator=g)
            dst = torch.randint(0, n, (e,), generator=g)
            if k == 4:                     # asymmetric: one direction only, node n-1 isolated
                src, dst = src % (n - 1), dst % (n - 1)
                ei = torch.stack([src, dst])
                w = torch.rand(e, generator=g) + 0.01
            else:                          # both directions (duplicates and self loops may occur)
                ei = torch.stack([torch.cat([src, dst]), torch.cat([dst, src])])
                w0 = torch.rand(e, generator=g) + 0.01
                w = torch.cat([w0, w0])
        else:
            ei = torch.zeros(2, 0, dtype=torch.long)
            w = torch.zeros(0)
        graphs.append(ConnectomeGraph(x, ei, w, torch.tensor(k % 2, dtype=torch.long), f"ragged-{k}"))
    return graphs


def save(name: str, arrays: dict) -> None:
    path = os.path.join(HERE, name)
    np.savez_compressed(path, **arrays)
    print(f"{name}: {len(arrays)} arrays, {os.path.getsize(path) / 1024:.1f} KiB")


def main() -> None:
    torch.set_num_threads(8)
    meta = {"torch": torch.__version__, "numpy": np.__version__, "python": sys.version.split()[0],
            "threads": torch.get_num_threads()}

    # -- small: the reference's own model-test fixture (tests/test_models.py:10-14) -------------
    graphs = generate_dataset(num_subjects=8, num_regions=20, seed=0)
    batch = collate_graphs(graphs)
    arrays = {**pack(graphs), **batch_fields(batch), **structure(batch)}
    for kind in MODELS:
        arrays.update(model_case(kind, batch, hidden=16, layers=3, tag=kind))
    save("ref_small.npz", arrays)

    # -- C1 / C2: 16 x 84-node subjects, hidden 64 (BASELINE.json configs[0], configs[1]) --------
    graphs = generate_dataset(num_subjects=16, num_regions=84, k=8, beta=0.15, trait_idx=0, seed=42)
    batch = collate_graphs(graphs)
    arrays = {**pack(graphs), **structure(batch)}
    del arrays["w_norm"]                      # derivable; keeps the fixture small
    arrays["batch.ptr"] = batch.ptr.numpy()
    arrays["batch.labels"] = batch.labels.numpy()
    for kind in MODELS:
        arrays.update(model_case(kind, batch, hidden=64, layers=3, tag=kind, per_layer=False))
    save("ref_c1.npz", arrays)
    fingerprints = {
        "c1.x": h16(batch.node_features), "c1.edge_index": h16(batch.edge_index),
        "c1.edge_weight": h16(batch.edge_weight), "c1.batch": h16(batch.batch),
        "c1.labels": batch.labels.tolist(), "c1.deg": h16(torch.from_numpy(arrays["deg"])),
        "c1.wsum": h16(torch.from_numpy(arrays["wsum"])),
    }

    # -- C3: 6 x 360-node subjects, hidden 64 (the shape of BASELINE.json configs[2]) ------------------
    graphs = generate_dataset(num_subjects=6, num_regions=360, k=8, beta=0.15, trait_idx=0, seed=42)
    batch = collate_graphs(graphs)
    arrays = {**pack(graphs), **structure(batch)}
    del arrays["w_norm"]
    arrays["batch.ptr"] = batch.ptr.numpy()
    arrays["batch.labels"] = batch.labels.numpy()
    for kind in MODELS:
        arrays.update(model_case(kind, batch, hidden=64, layers=3, tag=kind, per_layer=False))
    save("ref_c3.npz", arrays)

    # -- C5: 2 x 360-node subjects, hidden 256 (the layer shape of BASELINE.json configs[4]) ------------
    graphs = graphs[:2]
    batch = collate_graphs(graphs)
    arrays = {**pack(graphs), **structure(batch)}
    del arrays["w_norm"]
    arrays["batch.ptr"] = batch.ptr.numpy()
    arrays["batch.labels"] = batch.labels.numpy()
    for kind in MODELS:
        arrays.update(model_case(kind, batch, hidden=256, layers=3, tag=kind, per_layer=False, eval_grad=False))
    save("ref_c5.npz", arrays)

    # -- ragged / degenerate inputs --------------------------------------------------------------
    graphs = ragged_graphs()
    batch = collate_graphs(graphs)
    arrays = {**pack(graphs), **batch_fields(batch), **structure(batch)}
    for kind in MODELS:
        arrays.update(model_case(kind, batch, hidden=8, layers=2, tag=kind))
    save("ref_ragged.npz", arrays)

    # -- generator fingerprints (reference synthetic.py) -------------------------------------------
    gen = {"region_names": hashlib.sha256("|".join(REGION_NAMES).encode()).hexdigest()[:16],
           "num_regions": len(REGION_NAMES)}
    for n, seed in [(83, 0), (84, 42), (20, 7), (50, 3), (360, 1), (360, 42)]:
        g = generate_connectome(num_regions=n, seed=seed)
        gen[f"n{n}.s{seed}"] = {"edge_index": h16(g.edge_index), "edge_weight": h16(g.edge_weight),
                                "node_features": h16(g.node_features), "label": int(g.label),
                                "subject_id": g.subject_id, "num_edges": g.num_edges}
    ds = generate_dataset(num_subjects=6, num_regions=84, seed=42)
    gen["dataset.84.42"] = [{"edge_index": h16(g.edge_index), "node_features": h16(g.node_features),
                             "label": int(g.label), "subject_id": g.subject_id} for g in ds]

    # -- Trainer.fit trajectory, dropout 0 (tests/test_training.py:11-33 shapes) --------------------
    graphs = generate_dataset(num_subjects=40, num_regions=20, seed=7)
    trainer_arrays = pack(graphs)
    traj = {}
    for kind in MODELS:
        torch.manual_seed(0)
        model = MODELS[kind](in_channels=5, hidden_dim=16, num_classes=2, dropout=0.0)
        for k, v in model.state_dict().items():
            trainer_arrays[f"{kind}.init.{k}"] = v.clone().numpy()
        torch.manual_seed(1)
        train_loader = ConnectomeDataLoader(graphs[:30], batch_size=10, shuffle=True)
        val_loader = ConnectomeDataLoader(graphs[30:], batch_size=10, shuffle=False)
        trainer = Trainer(model, torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=1e-4), device="cpu")
        hist = trainer.fit(train_loader, val_loader, num_epochs=3, patience=10, verbose=False)
        traj[kind] = {"history": hist, "final_eval": trainer.evaluate(val_loader)}
        for k, v in model.state_dict().items():
            trainer_arrays[f"{kind}.final.{k}"] = v.clone().numpy()
    save("ref_trainer.npz", trainer_arrays)

    with open(os.path.join(HERE, "ref_meta.json"), "w") as f:
        json.dump({"made_with": meta, "fingerprints": fingerprints, "generator": gen, "trainer": traj}, f, indent=1)
    print("ref_meta.json written")


if __name__ == "__main__":
    main()

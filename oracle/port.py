"""ORACLE - TEST INFRASTRUCTURE ONLY.  CPU restatement of the reference hot path.

Nothing under ``connectome-gnn-suite_b200/`` imports this module.  It is used by ``tests/``
(as the checker), by ``__graft_entry__.smoke()`` (as the checker) and by ``bench.py`` for the
``cpu_baseline`` leg / ``--impl reference`` arm (as the thing timed on the host cores, because the
Python reference itself is not part of this repository).

What it restates (danieleschmidt/connectome-gnn-suite, all arithmetic delegated - like the
reference - to PyTorch 2.11 CPU ATen kernels, the reference's un-pinned ``torch>=2.0`` dependency):

* ``collate``            reference ``connectome_gnn/graph.py:143-167``
* ``gcn_structure``      reference ``connectome_gnn/models.py:94-108``
* ``gcn_conv``           reference ``connectome_gnn/models.py:84-114``
* ``sage_conv``          reference ``connectome_gnn/models.py:136-152``
* ``mean_pool``          reference ``connectome_gnn/models.py:40-47,57-59``
* ``encode / forward``   reference ``connectome_gnn/models.py:203-216`` and ``256-266``
* ``train_epoch / evaluate``  reference ``connectome_gnn/train.py:41-74``

Parity is PINNED: ``tests/test_oracle.py`` checks every function here against fixtures produced
by importing the unmodified reference (``tests/golden/make_golden.py``, outputs committed under
``tests/golden/``) - bit-exact for collate / degrees and for every float tensor (same op sequence
on the same ATen build), and, when CGNN_REFERENCE names a checkout of it, against the live reference.

Parameters are plain ``dict[str, Tensor]`` with the reference's ``state_dict`` keys
(``convs.i.linear.weight``, ``convs.i.bias`` | ``convs.i.linear.bias``,
``batch_norms.i.{weight,bias,running_mean,running_var,num_batches_tracked}``,
``classifier.{0,3}.{weight,bias}``).
"""

from __future__ import annotations

import math
from typing import Optional, Sequence

import torch
import torch.nn.functional as F

BN_EPS = 1e-5
BN_MOMENTUM = 0.1


# ---------------------------------------------------------------------------
# collate (graph.py:143-167)
# ---------------------------------------------------------------------------

def collate(graphs: Sequence) -> dict:
    """Concatenate subjects; edge endpoints get the running node offset; ``batch`` is the subject
    index per node; ``ptr`` the cumulative node count; ``labels`` stacks the labels that exist."""
    xs, eis, ews, owner, ys = [], [], [], [], []
    ptr = [0]
    for k, g in enumerate(graphs):
        n = g.node_features.shape[0]
        xs.append(g.node_features)
        eis.append(g.edge_index + ptr[-1])
        ews.append(g.edge_weight)
        owner.append(torch.full((n,), k, dtype=torch.long))
        if g.label is not None:
            ys.append(g.label)
        ptr.append(ptr[-1] + n)
    return {
        "node_features": torch.cat(xs, 0),
        "edge_index": torch.cat(eis, 1),
        "edge_weight": torch.cat(ews, 0),
        "batch": torch.cat(owner, 0),
        "labels": torch.stack(ys) if ys else None,
        "ptr": torch.tensor(ptr, dtype=torch.long),
    }


# ---------------------------------------------------------------------------
# layers
# ---------------------------------------------------------------------------

def gcn_structure(edge_index: torch.Tensor, edge_weight: torch.Tensor, n: int):
    """Self-loops (weight 1) appended AFTER the real edges; D^ = row (source) sums; d^-1/2;
    w^ = d[src] * w * d[dst]   (models.py:94-108)."""
    dev = edge_weight.device   # temporaries live where the batch lives, as in the reference (models.py:95-103)
    loops = torch.arange(n, device=dev)
    src = torch.cat([edge_index[0], loops])
    dst = torch.cat([edge_index[1], loops])
    w = torch.cat([edge_weight, torch.ones(n, device=dev)])
    deg = torch.zeros(n, device=dev).scatter_add_(0, src, w)
    dinv = (deg + 1e-8).pow(-0.5)
    w_hat = dinv[src] * w * dinv[dst]
    return src, dst, w_hat, deg, dinv


def sage_wsum(edge_index: torch.Tensor, edge_weight: torch.Tensor, n: int) -> torch.Tensor:
    """w_sum[i] = sum of weights of edges arriving at i (models.py:147-148)."""
    return torch.zeros(n, 1, device=edge_weight.device).scatter_add_(0, edge_index[1].unsqueeze(1), edge_weight.unsqueeze(1))


def _segment_sum(values: torch.Tensor, index: torch.Tensor, size: int) -> torch.Tensor:
    out = torch.zeros(size, values.shape[1], dtype=values.dtype, device=values.device)
    return out.scatter_add_(0, index.unsqueeze(1).expand_as(values), values)


def gcn_conv(x, edge_index, edge_weight, weight, bias):
    """z = scatter_sum((x W^T)[src] * w^, dst) + b   (models.py:111-114)."""
    n = x.shape[0]
    src, dst, w_hat, _, _ = gcn_structure(edge_index, edge_weight, n)
    projected = F.linear(x, weight)
    return _segment_sum(projected[src] * w_hat.unsqueeze(1), dst, n) + bias


def sage_conv(x, edge_index, edge_weight, weight, bias):
    """relu(Linear([x || weighted-mean of in-neighbours]))   (models.py:146-152)."""
    n = x.shape[0]
    src, dst = edge_index
    msg = x[src] * edge_weight.unsqueeze(1)
    agg = _segment_sum(msg, dst, n) / (sage_wsum(edge_index, edge_weight, n) + 1e-8)
    return F.relu(F.linear(torch.cat([x, agg], dim=1), weight, bias))


def mean_pool(h: torch.Tensor, batch: torch.Tensor, num_graphs: int) -> torch.Tensor:
    """Per-subject mean with the reference's fp32 count and +1e-8 (models.py:40-47)."""
    total = _segment_sum(h, batch, num_graphs)
    count = torch.zeros(num_graphs, 1, device=h.device).scatter_add_(0, batch.unsqueeze(1), torch.ones(batch.shape[0], 1, device=h.device))
    return total / (count + 1e-8)


def _dropout(h, p, training, mask):
    if mask is not None:          # externally supplied keep-mask already scaled by 1/(1-p)
        return h * mask
    return F.dropout(h, p=p, training=training)


# ---------------------------------------------------------------------------
# models
# ---------------------------------------------------------------------------

def num_layers(params: dict) -> int:
    return 1 + max(int(k.split(".")[1]) for k in params if k.startswith("convs."))


def encode(kind: str, params: dict, batch: dict, training: bool = False, dropout: float = 0.0,
           masks: Optional[list] = None, collect: Optional[list] = None) -> torch.Tensor:
    """L x (conv -> BN -> [ReLU for GCN] -> dropout) -> mean pool.  BN running buffers in ``params``
    are updated in place in training mode exactly as nn.BatchNorm1d does."""
    h = batch["node_features"]
    ei, ew = batch["edge_index"], batch["edge_weight"]
    for l in range(num_layers(params)):
        if kind == "gcn":
            h = gcn_conv(h, ei, ew, params[f"convs.{l}.linear.weight"], params[f"convs.{l}.bias"])
        else:
            h = sage_conv(h, ei, ew, params[f"convs.{l}.linear.weight"], params[f"convs.{l}.linear.bias"])
        if collect is not None:
            collect.append(h)
        pre = f"batch_norms.{l}."
        if training and pre + "num_batches_tracked" in params:
            params[pre + "num_batches_tracked"] += 1
        h = F.batch_norm(h, params[pre + "running_mean"], params[pre + "running_var"], params[pre + "weight"],
                         params[pre + "bias"], training, BN_MOMENTUM, BN_EPS)
        if kind == "gcn":
            h = F.relu(h)
        h = _dropout(h, dropout, training, None if masks is None else masks[l])
    return mean_pool(h, batch["batch"], int(batch["ptr"].shape[0]) - 1)


def forward(kind: str, params: dict, batch: dict, training: bool = False, dropout: float = 0.0,
            masks: Optional[list] = None) -> torch.Tensor:
    """Class logits.  ``masks`` replaces the dropout draws: one ``[rows, H]`` multiplier per layer, then ``[B, M]`` for
    the head, each already scaled by 1 / (1 - p)."""
    emb = encode(kind, params, batch, training, dropout, masks)
    h = F.relu(F.linear(emb, params["classifier.0.weight"], params["classifier.0.bias"]))
    h = _dropout(h, dropout, training, None if masks is None else masks[-1])
    return F.linear(h, params["classifier.3.weight"], params["classifier.3.bias"])


def init_params(kind: str, in_channels: int, hidden: int = 64, classes: int = 2, layers: int = 3,
                generator: Optional[torch.Generator] = None) -> dict:
    """Fresh parameters with the reference's initialisers (xavier-uniform conv weights, zero GCN
    bias, nn.Linear / nn.BatchNorm1d defaults elsewhere; models.py:78-82,130-134,186-201).
    Draw order differs from constructing the reference modules, so use fixtures - not this - when
    the *same* weights as a seeded reference model are needed."""
    def uniform(shape, bound):
        return (torch.rand(shape, generator=generator) * 2 - 1) * bound

    p: dict = {}
    dims = [in_channels] + [hidden] * layers
    for l in range(layers):
        fan_in = dims[l] * (2 if kind == "sage" else 1)
        p[f"convs.{l}.linear.weight"] = uniform((hidden, fan_in), math.sqrt(6.0 / (fan_in + hidden)))
        if kind == "gcn":
            p[f"convs.{l}.bias"] = torch.zeros(hidden)
        else:
            p[f"convs.{l}.linear.bias"] = uniform((hidden,), 1.0 / math.sqrt(fan_in))
        p[f"batch_norms.{l}.weight"] = torch.ones(hidden)
        p[f"batch_norms.{l}.bias"] = torch.zeros(hidden)
        p[f"batch_norms.{l}.running_mean"] = torch.zeros(hidden)
        p[f"batch_norms.{l}.running_var"] = torch.ones(hidden)
        p[f"batch_norms.{l}.num_batches_tracked"] = torch.tensor(0, dtype=torch.long)
    for name, (o, i) in (("classifier.0", (hidden // 2, hidden)), ("classifier.3", (classes, hidden // 2))):
        p[name + ".weight"] = uniform((o, i), 1.0 / math.sqrt(i))
        p[name + ".bias"] = uniform((o,), 1.0 / math.sqrt(i))
    return p


def trainable(params: dict) -> list[str]:
    return [k for k in params if not k.endswith(("running_mean", "running_var", "num_batches_tracked"))]


def loss_and_grads(kind: str, params: dict, batch: dict, training: bool = True, dropout: float = 0.0,
                   masks: Optional[list] = None):
    """Mean cross-entropy (train.py:39,49) and d loss / d param for every trainable tensor.  ``masks``: as ``forward``."""
    leaves = {k: (v.detach().clone().requires_grad_(True) if k in trainable(params) else v) for k, v in params.items()}
    logits = forward(kind, leaves, batch, training, dropout, masks)
    loss = F.cross_entropy(logits, batch["labels"])
    names = trainable(params)
    grads = torch.autograd.grad(loss, [leaves[k] for k in names])
    for k in params:   # running statistics were updated in place on `leaves`' shared buffers
        if k not in names:
            params[k] = leaves[k]
    return logits.detach(), loss.detach(), dict(zip(names, grads))


# ---------------------------------------------------------------------------
# training loop (train.py:41-74) - used as the CPU baseline by bench.py
# ---------------------------------------------------------------------------

class Module(torch.nn.Module):
    """nn.Module shell around the functional port so any torch.optim optimiser can drive it."""

    def __init__(self, kind: str, params: dict, dropout: float = 0.3):
        super().__init__()
        self.kind, self.p = kind, dropout
        self._names = list(params)
        for k, v in params.items():
            key = k.replace(".", "__")
            if k in trainable(params):
                self.register_parameter(key, torch.nn.Parameter(v.clone()))
            else:
                self.register_buffer(key, v.clone())

    def tensors(self) -> dict:
        return {k: getattr(self, k.replace(".", "__")) for k in self._names}

    def forward(self, batch: dict) -> torch.Tensor:
        return forward(self.kind, self.tensors(), batch, self.training, self.p)


def batches(dataset: Sequence, batch_size: int, shuffle: bool, device=None):
    """Epoch iterator with the reference's shuffling contract (graph.py:190-197); `device` = the reference Trainer's
    `batch.to(self.device)` (train.py:47,62)."""
    order = torch.randperm(len(dataset)).tolist() if shuffle else list(range(len(dataset)))
    for s in range(0, len(order), batch_size):
        b = collate([dataset[i] for i in order[s:s + batch_size]])
        if device is not None:
            b = {k: (v.to(device) if isinstance(v, torch.Tensor) else v) for k, v in b.items()}
        yield b


def train_epoch(module: Module, optimizer, dataset, batch_size: int, shuffle: bool = True, device=None) -> float:
    module.train()
    total, seen = 0.0, 0
    for b in batches(dataset, batch_size, shuffle, device):
        optimizer.zero_grad()
        loss = F.cross_entropy(module(b), b["labels"])
        loss.backward()
        optimizer.step()
        nb = int(b["ptr"].shape[0]) - 1
        total += float(loss.detach()) * nb
        seen += nb
    return total / max(seen, 1)


@torch.no_grad()
def evaluate(module: Module, dataset, batch_size: int, device=None) -> dict:
    module.eval()
    total, correct, seen = 0.0, 0, 0
    for b in batches(dataset, batch_size, False, device):
        logits = module(b)
        nb = int(b["ptr"].shape[0]) - 1
        total += float(F.cross_entropy(logits, b["labels"])) * nb
        correct += int((logits.argmax(1) == b["labels"]).sum())
        seen += nb
    return {"accuracy": correct / max(seen, 1), "loss": total / max(seen, 1), "correct": correct, "total": seen}

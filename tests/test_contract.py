"""Every C-ABI entry point against the float64 restatement of its contract (tests/contract_ref.py), over a table of cases
that each name the kernel path they are meant to reach.

The cases the simulator can run (the warp-specialised engine, the generic SIMT kernels, pool, head, loss, BatchNorm,
fused eval) also run under -m "not gpu"; on a B200 every case runs, and each one asserts with torch.profiler that the
kernels it was written for are the ones that ran - a change to the dispatch cannot silently move coverage.
test_dispatch_table prints the table of case -> kernels.

Every undirected batch has A^ = A^T, equal in- and out-degrees and the same neighbours in the by-destination and the
by-source aggregation blobs: a kernel that aggregates in the wrong direction passes on it.  The "-directed" cases repeat
the kernel paths on one-way multigraphs (directed_graphs, |A^ - A^T| / |A^| > 0.3 asserted), with the aggregation blobs
written by the collate kernel, by k_build_agg after a device collate or a host-assembled COO batch, or by both (a
subject over the collate kernel's staging cap).  The "-salt" cases run the layer kernels' dropout with device salt words
at row offsets 2^32 - 100 and 3 * 2^32 - 50, rows crossing the 2^32 boundary inside one CTA.  test_dispatch_table also
asserts that the directed cases reach DIRECTED_REQUIRED and the salted cases SALTED_REQUIRED.

Element bar: |got - ref| <= C_ULPS * 2^-23 * mag, mag = the same computation on absolute values (contract_ref.py).
Model-level cases on ingested (real-density) connectomes compare with the oracle (oracle/port.py) by the rule
dp_parity uses: per tensor <= max(1e-5, 4 x the fp32 oracle's own distance from the fp64 evaluation), measured in
the same test; logits and loss at 1e-5.

Value mutations of the kernel sources that these cases catch on the simulator (and the first case to fail):
  drop_keep with the two 16-bit halves swapped                   mask-C64-wrap-salt (9628 of 23040 mask bits differ)
  k_gcn_fwd without the self-loop term when the CSR is read from L2   gcn-fwd-ingest360-first
  GraphSAGE w_sum + 1e-8 -> w_sum + 0 (isolated nodes)           sage-fwd-generic-n385 (tensor-core edition on a B200)
  BatchNorm backward s2 / count -> s1 / count (k_gcn_bwd)        gcn-bwd-generic-H20
  k_gcn_bwd launched on the by-destination CSR (in_rowptr / in_col / in_wn for the out_* arrays, gcn.cu)
                                                                 gcn-bwd-gemm-n385-directed (gcn-bwd-generic-H20-directed on a B200)
  k_build_agg fills each blob from the other direction's lists (rp, col and weights: dir == 0 -> dir == 1, agg.cu)
                                                                 gcn-fwd-engine-n129-directed (on a B200 too)
  k_gcn_fwd_ws hashes row grow instead of row_base + grow        gcn-fwd-engine-n384-salt
  k_gcn_fwd without act_salt(p.act)                              gcn-fwd-generic-H20-salt
  k_gcn_bwd's prev-sums mask hashes row grow instead of row_base + grow   gcn-bwd-generic-H20-salt
  (the last three together: those three cases and gcn-fwd-engine-n129-wrap3-p0.9)
Mutations of device-only kernels, one B200 run each (first case to fail):
  every k_gather<GCN_BWD> launch reads agg_in (gcn.cu, wide_tc.cu), decoded as a by-destination blob (agg.cu kPre)
                                                                 gcn-bwd-gemm-middle-directed
  k_sage_fwd_gemm's narrow-K operand path hashes row instead of row_base + row (gemm_tc.cu)
                                                                 sage-fwd-gemm-d9-hidden-salt
  k_sage_bwd_gemm without act_salt(p.act_out); act_salt(p.act_in)  sage-bwd-gemm-middle-salt

Real-density dispatch (360-region ingested subjects, q = 0.90, ~26k directed edges per subject; the table of
test_dispatch_table on a B200): GCN runs every layer, forward and backward, on k_gcn_fwd / k_gcn_bwd with the CSR read
from L2; GraphSAGE runs its first layer as k_gather + k_sage_fwd_gemm / k_sage_bwd_gemm at K = 2 and its hidden layers on
k_sage_fwd / k_sage_bwd_a / k_sage_bwd_b.
"""
import re

import numpy as np
import pytest
import torch

import contract_ref as cr
import helpers

F64 = torch.float64
ROW_BASE_WRAP = 2 ** 32 - 100          # rows 0..359 of such a tensor cross a 2^32 boundary of the global row id


# ---- inputs -----------------------------------------------------------------------------------------------------------
def rand_graphs(sizes, F, seed, isolated=True, deg=8):
    """Undirected multigraphs listed as adjacent reversed pairs; the last node of every subject of > 2 nodes has no edge
    (GraphSAGE's w_sum + 1e-8 denominator and the GCN self-loop-only row)."""
    from connectome_gnn.graph import ConnectomeGraph
    rng = np.random.default_rng(seed)
    out = []
    for n in sizes:
        hi = n - 1 if (isolated and n > 2) else n
        pairs = max(1, deg * n // 2) if n > 0 else 0
        u, v = rng.integers(0, max(hi, 1), pairs), rng.integers(0, max(hi, 1), pairs)
        w = rng.random(pairs).astype(np.float32) + 0.05
        ei = np.empty((2, 2 * pairs), dtype=np.int64)
        ei[0, 0::2], ei[1, 0::2], ei[0, 1::2], ei[1, 1::2] = u, v, v, u
        x = rng.normal(size=(n, F)).astype(np.float32)
        out.append(ConnectomeGraph(torch.from_numpy(x), torch.from_numpy(ei), torch.from_numpy(np.repeat(w, 2)),
                                   torch.tensor(int(rng.integers(0, 2)))))
    return out


def directed_graphs(sizes, F, seed, heavy=1, deg=8):
    """One-way multigraphs with independent edge weights, skewed so that the direction matters: sources are drawn from
    the lower two thirds of a subject's ids (mostly the lowest), destinations from the upper two thirds (mostly the
    highest).  The first third are out-degree hubs that no edge enters, the last third in-degree hubs that no edge
    leaves.  Every subject also gets self-loops and repeated (src, dst) pairs of other weights; the last node of a
    subject of > 2 nodes has no edge.  Subject 0 has `heavy` times the edges of the others."""
    from connectome_gnn.graph import ConnectomeGraph
    rng = np.random.default_rng(seed)
    out = []
    for s, n in enumerate(sizes):
        hi = n - 1 if n > 2 else n
        m = deg * n * (heavy if s == 0 else 1)
        span = max(1, (2 * hi) // 3)
        src = (span * rng.random(m) ** 2).astype(np.int64)
        dst = hi - 1 - (span * rng.random(m) ** 2).astype(np.int64)
        k = max(1, m // 16)
        loops, rep = rng.integers(0, hi, k), rng.integers(0, m, k)
        ei = np.stack([np.concatenate([src, loops, src[rep]]), np.concatenate([dst, loops, dst[rep]])])
        w = rng.random(ei.shape[1]).astype(np.float32) + 0.05
        x = rng.normal(size=(n, F)).astype(np.float32)
        out.append(ConnectomeGraph(torch.from_numpy(x), torch.from_numpy(ei), torch.from_numpy(w),
                                   torch.tensor(int(rng.integers(0, 2)))))
    asym = asymmetry(out)
    assert asym > 0.3, f"the directed batch is nearly symmetric: |A^ - A^T| / |A^| = {asym:.2f}"
    return out


def asymmetry(graphs):
    """|A^ - A^T|_F / |A^|_F of the batch's GCN operator A^ = D^-1/2 (A + I) D^-1/2 (A[dst, src], D^ over sources)."""
    num = den = 0.0
    for gr in graphs:
        n = gr.num_nodes
        src, dst = gr.edge_index.numpy()
        a = np.eye(n)
        np.add.at(a, (dst, src), gr.edge_weight.numpy().astype(np.float64))
        dinv = 1.0 / np.sqrt(a.sum(0))
        a = dinv[:, None] * a * dinv[None, :]
        num += float(((a - a.T) ** 2).sum())
        den += float((a ** 2).sum())
    return np.sqrt(num / den)


def host_coo(graphs):
    """(edge_index, edge_weight, ptr) of a list of subjects, concatenated on the host: what the reference is built from."""
    sizes = np.array([gr.num_nodes for gr in graphs], dtype=np.int64)
    ptr = np.concatenate([[0], np.cumsum(sizes)])
    ei = torch.cat([gr.edge_index + int(ptr[s]) for s, gr in enumerate(graphs)], 1)
    return ei, torch.cat([gr.edge_weight for gr in graphs]), torch.from_numpy(ptr)


def ingested(S, N, kind="dense", q=0.90, seed=5):
    """The README's real-data recipe on the device: packed arena of S subjects (1 feature per node)."""
    import ingest_ref
    from connectome_gnn.ingest import matrices_to_packed
    mats = ingest_ref.random_matrices(S, N, seed, kind)
    return matrices_to_packed(mats, labels=[s % 2 for s in range(S)], quantile=q, device=_DEV["device"])


def packed_graphs(p):
    """ConnectomeGraph list of a packed arena (host tensors) - what the oracle takes."""
    from connectome_gnn.graph import ConnectomeGraph
    out = []
    for s in range(len(p["node_ptr"]) - 1):
        n0, n1, e0, e1 = (int(p["node_ptr"][s]), int(p["node_ptr"][s + 1]), int(p["edge_ptr"][s]), int(p["edge_ptr"][s + 1]))
        ei = torch.stack([p["src"][e0:e1], p["dst"][e0:e1]]).long().cpu()
        out.append(ConnectomeGraph(p["x"][n0:n1].cpu(), ei, p["w"][e0:e1].cpu(), torch.tensor(int(p["label"][s]))))
    return out


def batch_of(spec, kind=None):
    """(batch, contract_ref.Graph) of a graph spec: ("rand", sizes, F, seed), ("ingest", S, N, kind, q) or
    ("directed", sizes, F, seed, blobs).  `blobs` is where the batch's aggregation blobs of model family `kind` come from:
      "lazy"      collate_graphs; k_build_agg at the first layer call
      "emit"      a lean SubjectStore.collate(prepare_for=kind): k_collate_graph writes them
      "full"      the same with lean=False (every subject small enough to be staged)
      "coo"       a ConnectomeBatch assembled from host tensors: cgnn_csr_from_coo, then k_build_agg
      "overflow"  subject 0 has 4x the edges, beyond the collate kernel's staging cap: a lean=False collate emits the
                  blobs of the others and k_build_agg those of subject 0 alone
    The reference of a directed batch is built from the host lists, not from what the collate kernel wrote."""
    from connectome_gnn.graph import ConnectomeBatch, SubjectStore, collate_graphs, pack_graphs
    if spec[0] == "rand":
        b = collate_graphs(rand_graphs(spec[1], spec[2], spec[3]))
    elif spec[0] == "directed":
        _, sizes, F, seed, blobs = spec
        gs = directed_graphs(sizes, F, seed, heavy=4 if blobs == "overflow" else 1)
        ei, w, ptr = host_coo(gs)
        dev = _DEV["device"]
        if blobs == "lazy":
            b = collate_graphs(gs)
        elif blobs == "coo":
            x = torch.cat([gr.node_features for gr in gs])
            batch = torch.repeat_interleave(torch.arange(len(gs)), ptr[1:] - ptr[:-1])
            labels = torch.stack([gr.label for gr in gs])
            b = ConnectomeBatch(x.to(dev), ei.to(dev), w.to(dev), batch.to(dev), labels.to(dev), ptr.to(dev))
            b.ensure_csr()
        else:
            assert kind is not None and blobs in ("emit", "full", "overflow"), blobs
            b = SubjectStore(pack_graphs(gs), dev).collate(np.arange(len(gs)), prepare_for=kind, lean=blobs == "emit")
        return b, cr.Graph(ei, w, ptr)
    else:
        p = ingested(*spec[1:])
        b = SubjectStore(p, _DEV["device"]).collate(np.arange(spec[1]))
    return b, cr.Graph(b.edge_index, b.edge_weight, b.ptr)


def hidden_input(rows, C, gen, relu, p_drop, site=1, row_base=0, salt=None):
    """A stored activation t and the Act that loads it: BatchNorm affine, ReLU (GCN), dropout.  t is drawn so that
    scale * t + shift stays away from 0 (an fp32 / fp64 ReLU disagreement there is round-off, not a finding)."""
    scale = torch.rand(C, generator=gen) + 0.5
    shift = (torch.rand(C, generator=gen) - 0.5) * 0.6
    y = torch.randn(rows, C, generator=gen)
    y = torch.where(y.abs() < 0.05, torch.sign(y + 1e-3) * 0.05, y)
    t = ((y - shift) / scale).float()
    return t, dict(scale=scale, shift=shift, relu=relu, p_drop=p_drop, seed=0x1234_5678_9ABC, site=site,
                   row_base=row_base, salt=salt)


def acts(spec, dev):
    """(device Act, reference Act) of an act description (None = identity)."""
    from connectome_gnn._engine import Act
    if spec is None:
        return Act(), cr.Act()
    s = dict(spec)
    salt_dev = None
    if s["salt"] is not None:
        salt_dev = torch.from_numpy(np.array(s["salt"], dtype=np.uint32).view(np.int32)).to(dev)
    d = Act(s["scale"].to(dev), s["shift"].to(dev), s["relu"], s["p_drop"], s["seed"], s["site"], s["row_base"], salt_dev)
    return d, cr.Act(s["scale"], s["shift"], s["relu"], s["p_drop"], s["seed"], s["site"], s["row_base"], s["salt"])


def worst(rs):
    return max(rs) if rs else 0.0


# ---- runners: each returns the worst error ratio of the case ----------------------------------------------------------
def run_layer_fwd(eng, kind, d_in, H, graph, hidden=True, p_drop=0.3, row_base=0, salt=None, seed=0):
    """One forward call.  hidden: the input is a stored activation loaded through BatchNorm affine, (GCN) ReLU and
    dropout, whose local row 0 is global row `row_base`, salted with the device words `salt`; else the node features."""
    dev = _DEV["device"]
    b, g = batch_of(graph, kind)
    gen = torch.Generator().manual_seed(seed)
    rows = b.num_nodes
    if hidden:
        t, a = hidden_input(rows, d_in, gen, kind == "gcn", p_drop, row_base=row_base, salt=salt)
        t = t.to(dev)
    else:                                  # a first layer reads the node features as they are
        assert b.node_features.shape[1] == d_in
        t, a = b.node_features.contiguous(), None
    act_d, act_r = acts(a, dev)
    W = (torch.randn(H, d_in * (2 if kind == "sage" else 1), generator=gen) / np.sqrt(d_in)).to(dev)
    bias = (0.1 * torch.randn(H, generator=gen)).to(dev)
    z, st, agg = eng.layer_fwd(kind, t, act_d, W, bias, b.csr, b.ptr, b.num_graphs, True)
    zr, zm, ar, am = cr.layer_fwd(kind, g, t.cpu(), act_r, W.cpu(), bias.cpu())
    rs = [cr.check(z, zr, zm, f"{kind} z")]
    if kind == "sage":
        rs.append(cr.check(agg, ar, am, "sage agg"))
    zc = z.cpu().to(F64)
    assert float(st[0]) == rows
    mean = zc.mean(0)
    rs.append(cr.check(st[1:1 + H].cpu(), mean, zc.abs().max(0).values, "statistics: mean"))
    rs.append(cr.check(st[1 + H:].cpu(), ((zc - mean) ** 2).sum(0), ((zc.abs() + mean.abs()) ** 2).sum(0) / 8,
                       "statistics: M2"))
    return worst(rs)


def run_layer_bwd(eng, kind, d_in, H, graph, first=False, hidden=None, pooled=False, bn="train", sums64=True, p_out=0.3,
                  p_in=0.3, row_base=0, salt=None, seed=0):
    """One backward call.  first: the input needs no gradient (no du_in, no prev sums); hidden (default: not first): the
    input is a stored activation with its own BatchNorm affine, ReLU and dropout, else the node features; pooled: the top
    layer (upstream = demb [B, H]); bn: "train" / "eval" / None; sums64: the double sums are handed in (and the fp32
    sums are a decoy the kernel must not read).  Both dropouts (input and output) start at global row `row_base` and are
    salted with the device words `salt`."""
    from connectome_gnn._engine import BnBwd
    dev = _DEV["device"]
    b, g = batch_of(graph, kind)
    gen = torch.Generator().manual_seed(seed)
    rows, B = b.num_nodes, b.num_graphs
    if not (not first if hidden is None else hidden):
        t, a_in = b.node_features.contiguous(), None
        assert t.shape[1] == d_in
    else:
        t, a_in = hidden_input(rows, d_in, gen, kind == "gcn", p_in, site=1, row_base=row_base, salt=salt)
        t = t.to(dev)
    act_in_d, act_in_r = acts(a_in, dev)
    W = (torch.randn(H, d_in * (2 if kind == "sage" else 1), generator=gen) / np.sqrt(d_in)).to(dev)
    agg = None
    if kind == "sage":   # the aggregate the forward stored (and with it the tensor-core path of the backward)
        _, _, agg = eng.layer_fwd(kind, t, act_in_d, W, torch.zeros(H, device=dev), b.csr, b.ptr, B, False)
    # this layer's output and its BatchNorm + (GCN) ReLU + dropout
    zt, a_out = hidden_input(rows, H, gen, kind == "gcn", p_out, site=2, row_base=row_base, salt=salt)
    if kind == "sage":
        zt = torch.clamp(torch.randn(rows, H, generator=gen), min=0.0)   # a ReLU output, exact zeros included
    z = zt.to(dev)
    act_out_d, act_out_r = acts(a_out, dev)
    mean, rstd = 0.1 * torch.randn(H, generator=gen), torch.rand(H, generator=gen) + 0.5
    s = torch.randn(2, H, generator=gen).double() * 3.0
    bn_d = bn_r = None
    if bn is not None:
        sc = a_out["scale"]
        s32 = (s * 1.5 if sums64 else s).float()
        bn_d = BnBwd(sc.to(dev), mean.to(dev), rstd.to(dev), s32.to(dev).contiguous(), float(rows), bn == "train",
                     s.to(dev).contiguous() if sums64 else None)
        used = s if sums64 else s32.double()
        bn_r = dict(scale=sc, mean=mean, rstd=rstd, s1=used[0], s2=used[1], count=float(rows), train=bn == "train")
    du = demb = None
    if pooled:
        demb = torch.randn(B, H, generator=gen).to(dev)
    else:
        du = torch.randn(rows, H, generator=gen).to(dev)
    prev = None if first else (0.1 * torch.randn(d_in, generator=gen), torch.rand(d_in, generator=gen) + 0.5)
    dW, db, du_in, ps, ps64 = eng.layer_bwd(kind, du, demb, z, act_out_d, bn_d, t, act_in_d, W, b.csr, b.ptr, B, not first,
                                            prev[0].to(dev) if prev else None, prev[1].to(dev) if prev else None, agg)
    ref = cr.layer_bwd(kind, g, zt, act_out_r, bn_r, t.cpu(), act_in_r, W.cpu(),
                       du=du.cpu() if du is not None else None, demb=demb.cpu() if demb is not None else None, prev=prev)
    rs = [cr.check(dW, *ref["dW"], f"{kind} dW"), cr.check(db, *ref["dbias"], f"{kind} dbias")]
    if not first:
        rs.append(cr.check(du_in, *ref["du_in"], f"{kind} du_in"))
        rs.append(cr.check(ps, *ref["prev_sums"], f"{kind} prev_sums"))
        rs.append(cr.check(ps64, *ref["prev_sums"], f"{kind} prev_sums64"))
    return worst(rs)


def run_mask(eng, C, p_drop, row_base, salt):
    """pool_fwd over subjects of ONE row each, input ones, dropout only: emb == keep_scale * mask, bit for bit."""
    from connectome_gnn._engine import Act
    dev = _DEV["device"]
    rows = 360
    ptr = torch.arange(rows + 1, dtype=torch.int64, device=dev)
    salt_dev = None if salt is None else torch.from_numpy(np.array(salt, dtype=np.uint32).view(np.int32)).to(dev)
    emb = eng.pool_fwd(torch.ones(rows, C, device=dev), Act(None, None, False, p_drop, 0xDEADBEEF12345, 3, row_base, salt_dev),
                       ptr, rows)
    _, ks, _, _ = cr.make_act_keys(p_drop, 0xDEADBEEF12345, 3, salt)
    mask = cr.keep_mask(p_drop, 0xDEADBEEF12345, 3, row_base, rows, C, salt)
    want = np.where(mask, np.float32(ks), np.float32(0.0)).astype(np.float32)
    got = emb.cpu().numpy()
    assert np.array_equal(got, want), f"{int((got != want).sum())} of {got.size} mask elements differ"
    assert 0.5 < mask.mean() / (1 - p_drop) < 1.5
    return 0.0


def run_pool_and_sums(eng, C, graph, p_drop=0.3, row_base=0, salt=None, seed=0):
    """cgnn_pool_fwd and cgnn_bn_bwd_sums (per-row du and pooled demb) with BatchNorm affine, ReLU and dropout."""
    dev = _DEV["device"]
    b, g = batch_of(graph)
    gen = torch.Generator().manual_seed(seed)
    rows, B = b.num_nodes, b.num_graphs
    t, a = hidden_input(rows, C, gen, True, p_drop, site=4, row_base=row_base, salt=salt)
    act_d, act_r = acts(a, dev)
    t = t.to(dev)
    emb = eng.pool_fwd(t, act_d, b.ptr, B)
    rs = [cr.check(emb, *cr.pool_fwd(g, t.cpu(), act_r), "pool")]
    mean, rstd = 0.1 * torch.randn(C, generator=gen), torch.rand(C, generator=gen) + 0.5
    du, demb = torch.randn(rows, C, generator=gen), torch.randn(B, C, generator=gen)
    for name, up_row, up_pool in (("du", du, None), ("demb", None, demb)):
        sums, sums64 = eng.bn_bwd_sums(t, act_d, mean.to(dev), rstd.to(dev), None if up_row is None else up_row.to(dev),
                                       None if up_pool is None else up_pool.to(dev), b.ptr, B)
        ref, mag = cr.bn_bwd_sums(g, t.cpu(), act_r, mean, rstd, du=up_row, demb=up_pool)
        rs += [cr.check(sums, ref, mag, f"bn_bwd_sums ({name})"), cr.check(sums64, ref, mag, f"bn_bwd_sums64 ({name})")]
    return worst(rs)


def run_head(eng, B, C, M, K, p_drop, seed=0):
    """head_fwd, ce_fwd, ce_bwd, head_bwd; labels include K - 1."""
    dev = _DEV["device"]
    gen = torch.Generator().manual_seed(seed)
    emb = torch.randn(B, C, generator=gen)
    W0, b0 = torch.randn(M, C, generator=gen) / np.sqrt(C), 0.1 * torch.randn(M, generator=gen)
    W1, b1 = torch.randn(K, M, generator=gen) / np.sqrt(M), 0.1 * torch.randn(K, generator=gen)
    salt = [0x0BADF00D, 0x600DCAFE]
    salt_dev = torch.from_numpy(np.array(salt, dtype=np.uint32).view(np.int32)).to(dev)
    d = lambda q: q.to(dev)
    hidden, logits = eng.head_fwd(d(emb), d(W0), d(b0), d(W1), d(b1), p_drop, 0xC0FFEE, 17, salt_dev if p_drop > 0 else None)
    hr, hm, lr, lm = cr.head_fwd(emb, W0, b0, W1, b1, p_drop, 0xC0FFEE, 17, salt if p_drop > 0 else None)
    rs = [cr.check(hidden, hr, hm, "head hidden"), cr.check(logits, lr, lm, "logits")]
    labels = torch.randint(0, K, (B,), generator=gen)
    labels[0] = K - 1
    labels[-1] = K - 1
    inv = 1.0 / B
    loss, nll, correct = eng.ce_fwd(logits, d(labels), inv)
    nr, nm, lsum, lmag, corr = cr.ce_fwd(logits.cpu(), labels, inv)
    rs += [cr.check(nll, nr, nm, "nll"), cr.check(loss.reshape(1), torch.tensor([lsum]), torch.tensor([lmag]), "loss")]
    assert int(correct) == corr
    gout = torch.tensor([0.7], device=dev)
    dl = eng.ce_bwd(logits, d(labels), inv, gout)
    rs.append(cr.check(dl, *cr.ce_bwd(logits.cpu(), labels, inv, 0.7), "dlogits"))
    demb, dW0, db0, dW1, db1 = eng.head_bwd(d(emb), hidden, dl, d(W0), d(W1), p_drop)
    ref = cr.head_bwd(emb, hidden.cpu(), dl.cpu(), W0, W1, p_drop)
    for name, got in (("demb", demb), ("dW0", dW0), ("db0", db0), ("dW1", dW1), ("db1", db1)):
        rs.append(cr.check(got, *ref[name], f"head {name}"))
    return worst(rs)


def run_bn_bookkeeping(eng, C=48, seed=0):
    dev = _DEV["device"]
    gen = torch.Generator().manual_seed(seed)
    recs = []
    for n in (5, 300, 1, 0, 41):
        x = torch.randn(n, C, generator=gen).double() * 2 + 0.3
        recs.append(cr.stats_of(x) if n else torch.zeros(1 + 2 * C, dtype=F64))
    parts = torch.stack(recs)
    merged = eng.bn_merge_stats(parts.to(dev), C)
    ref = cr.bn_merge_stats(parts, C)
    assert float(merged[0]) == float(ref[0]) == 347.0
    assert torch.allclose(merged.cpu(), ref, rtol=1e-12, atol=1e-12)
    gamma, beta = torch.rand(C, generator=gen) + 0.5, 0.1 * torch.randn(C, generator=gen)
    rm0, rv0 = 0.1 * torch.randn(C, generator=gen), torch.rand(C, generator=gen) + 0.5
    rm, rv, nbt = rm0.clone().to(dev), rv0.clone().to(dev), torch.zeros((), dtype=torch.int64, device=dev)
    got = eng.bn_finalize(merged, gamma.to(dev), beta.to(dev), 1e-5, 0.1, rm, rv, nbt)
    sc, sh, mean, rstd, rmr, rvr = cr.bn_finalize(ref, gamma, beta, 1e-5, 0.1, rm0, rv0)
    rs = []
    for name, gv, rv_, mg in (("scale", got[0], sc, sc.abs()), ("shift", got[1], sh, (mean * sc).abs() + beta.abs()),
                              ("mean", got[2], mean, mean.abs()), ("rstd", got[3], rstd, rstd),
                              ("running_mean", rm, rmr, rmr.abs() + rm0.abs()), ("running_var", rv, rvr, rvr)):
        rs.append(cr.check(gv, rv_, mg, f"bn_finalize {name}", c=4))
    assert int(nbt) == 1
    got = eng.bn_eval_affine(gamma.to(dev), beta.to(dev), rm0.to(dev), rv0.to(dev), 1e-5)
    sc, sh, mean, rstd = cr.bn_eval_affine(gamma, beta, rm0, rv0, 1e-5)
    for name, gv, rv_, mg in (("scale", got[0], sc, sc.abs()), ("shift", got[1], sh, (rm0 * sc).abs() + beta.abs()),
                              ("rstd", got[3], rstd, rstd)):
        rs.append(cr.check(gv, rv_, mg, f"bn_eval_affine {name}", c=4))
    return worst(rs)


def _eval_params(L, F, K, gen, M=32, H=64):
    layers = []
    for l in range(L):
        d_in = F if l == 0 else H
        layers.append((torch.randn(H, d_in, generator=gen) / np.sqrt(d_in), 0.1 * torch.randn(H, generator=gen),
                       torch.rand(H, generator=gen) + 0.5, 0.2 * torch.randn(H, generator=gen),
                       0.1 * torch.randn(H, generator=gen), torch.rand(H, generator=gen) + 0.5, 1e-5))
    head = (torch.randn(M, H, generator=gen) / 8, 0.1 * torch.randn(M, generator=gen),
            torch.randn(K, M, generator=gen) / np.sqrt(M), 0.1 * torch.randn(K, generator=gen))
    return layers, head


def run_eval_fused(eng, L, F, K, sizes=(84, 30, 130, 57, 1, 200), blobs=None, seed=0):
    """cgnn_eval_fused_fwd against the eval-mode network in float64; K > 8 must decline (None: the caller falls back).
    blobs: a directed batch whose aggregation blobs come from there (batch_of), else an undirected one."""
    dev = _DEV["device"]
    b, g = batch_of(("rand", sizes, F, 40 + L) if blobs is None else ("directed", sizes, F, 40 + L, blobs), "gcn")
    gen = torch.Generator().manual_seed(seed)
    layers, head = _eval_params(L, F, K, gen)
    to = lambda q: q.to(dev) if isinstance(q, torch.Tensor) else q
    out = eng.eval_fused("gcn", b.node_features.contiguous(), [tuple(to(q) for q in l) for l in layers],
                         tuple(to(q) for q in head), b.csr, b.ptr, b.num_graphs)
    if K > 8:
        assert out is None, "cgnn_eval_fused_fwd must decline K > 8"
        return 0.0
    assert out is not None, "cgnn_eval_fused_fwd declined a covered shape"
    emb, embm, logits, lm = cr.gcn_eval_network(g, b.node_features.cpu(), layers, head)
    return worst([cr.check(out[0], emb, embm, "fused emb"), cr.check(out[1], logits, lm, "fused logits")])


def run_fwd_pool(eng, sizes, blobs=None, seed=0):
    """cgnn_gcn_layer_fwd_pool (eval, hidden 64): emb = mean_rows relu(bn(z)); a subject of > 384 rows -> None.
    blobs: as run_eval_fused."""
    from connectome_gnn._engine import Act
    dev = _DEV["device"]
    b, g = batch_of(("rand", sizes, 3, 60) if blobs is None else ("directed", sizes, 3, 60, blobs), "gcn")
    gen = torch.Generator().manual_seed(seed)
    rows = b.num_nodes
    t, a = hidden_input(rows, 64, gen, True, 0.0)
    act_d, act_r = acts(a, dev)
    W, bias = torch.randn(64, 64, generator=gen) / 8, 0.1 * torch.randn(64, generator=gen)
    sc, sh = torch.rand(64, generator=gen) + 0.5, 0.2 * torch.randn(64, generator=gen)
    emb = eng.gcn_layer_fwd_pool(t.to(dev), act_d, W.to(dev), bias.to(dev), b.csr, b.ptr, b.num_graphs,
                                 Act(sc.to(dev), sh.to(dev), True, 0.0, 0, 1, 0))
    if max(sizes) > 384:
        assert emb is None
        return 0.0
    assert emb is not None
    z, zm, _, _ = cr.layer_fwd("gcn", g, t, act_r, W, bias)
    y = z * sc.double() + sh.double()
    u, um = torch.clamp(y, min=0.0), zm * sc.double() + sh.double().abs()
    return cr.check(emb, g.pool(u), g.pool(um), "fwd_pool emb")


# ---- the dispatch table ---------------------------------------------------------------------------------------------
# (id, runner, kwargs, runs on the simulator, kernels a B200 must show for it, kernels it must not show)
R84 = ("rand", (84, 84, 84, 84), 64, 1)
SMALL16 = ("rand", (20,) * 16, 64, 2)
CASES, EMU_CASES = [], []
DIRECTED, SALTED = set(), set()     # ids of the cases on directed batches / with salted dropout keys
BLOBS_BUILT = ("lazy", "coo", "overflow")     # batch_of modes in which k_build_agg writes (some) aggregation blobs


def case(cid, fn, kw, emu, expect=(), forbid=(), salted=False):
    """A directed case also names its collate kernel (k_collate_graph, never the pair kernel) and requires or forbids
    k_build_agg by where its blobs come from; `salted` marks a case whose dropout keys take device salt words (a `salt`
    argument marks it too)."""
    expect, forbid = set(expect), set(forbid)
    graph = kw.get("graph", ("",))
    blobs = graph[4] if graph[0] == "directed" else kw.get("blobs")
    if blobs is not None:
        DIRECTED.add(cid)
        expect.add("k_collate_graph")
        forbid.add("k_collate_pairs")
        (expect if blobs in BLOBS_BUILT else forbid).add("k_build_agg")
    if salted or kw.get("salt") is not None:
        SALTED.add(cid)
    CASES.append(pytest.param(fn, kw, expect, forbid, id=cid))
    if emu:
        EMU_CASES.append(pytest.param(fn, kw, id=cid))

# -- mask restatement first: everything else leans on it
case("mask-C64-wrap-salt", run_mask, dict(C=64, p_drop=0.3, row_base=ROW_BASE_WRAP, salt=[0x9E3779B9, 0x7F4A7C15]), True,
     ["k_pool_fwd_quad"])
case("mask-C20-wrap-salt", run_mask, dict(C=20, p_drop=0.5, row_base=ROW_BASE_WRAP, salt=[1, 2]), True, ["k_pool_fwd"])
case("mask-C64-p0.9", run_mask, dict(C=64, p_drop=0.9, row_base=7, salt=None), True, ["k_pool_fwd_quad"])
# -- gcn_layer_fwd: engine
for n in (1, 2, 8, 9, 127, 128, 129, 383, 384):
    case(f"gcn-fwd-engine-n{n}", run_layer_fwd, dict(kind="gcn", d_in=64, H=64, graph=("rand", (n, max(1, n // 3), n), 64, n)),
         n in (1, 9, 129, 384), ["k_gcn_fwd_ws<false>"])
case("gcn-fwd-engine-16-per-unit", run_layer_fwd, dict(kind="gcn", d_in=64, H=64, graph=SMALL16), True, ["k_gcn_fwd_ws<false>"])
case("gcn-fwd-engine-batch600", run_layer_fwd, dict(kind="gcn", d_in=64, H=64, graph=("rand", (84,) * 600, 64, 3)), False,
     ["k_gcn_fwd_ws<false>"])
case("gcn-fwd-engine-ingest84", run_layer_fwd, dict(kind="gcn", d_in=64, H=64, graph=("ingest", 4, 84, "dense", 0.9)), True,
     ["k_gcn_fwd_ws<false>"])
case("gcn-fwd-generic-n385", run_layer_fwd, dict(kind="gcn", d_in=64, H=64, graph=("rand", (385, 20), 64, 4)), True,
     ["k_gcn_fwd"])
# -- first layer, d_in x H
for d_in in (1, 3, 5, 8):
    for H in (32, 64, 128, 256):
        case(f"gcn-fwd-first-d{d_in}-H{H}", run_layer_fwd, dict(kind="gcn", d_in=d_in, H=H, graph=("rand", (84, 30, 1), d_in, 5),
                                                              hidden=False), False, ["k_first_fwd"])
case("gcn-fwd-d9", run_layer_fwd, dict(kind="gcn", d_in=9, H=64, graph=("rand", (84, 30), 9, 6), hidden=False), True, ["k_gcn_fwd"])
case("gcn-fwd-wide256", run_layer_fwd, dict(kind="gcn", d_in=256, H=256, graph=("rand", (84, 30, 1), 256, 7)), False,
     ["k_gather<3>", "k_wide_xw"])
for H in (20, 96):
    case(f"gcn-fwd-generic-H{H}", run_layer_fwd, dict(kind="gcn", d_in=64, H=H, graph=("rand", (84, 30, 1), 64, 8)), True,
         ["k_gcn_fwd"])
case("gcn-fwd-ingest360-first", run_layer_fwd, dict(kind="gcn", d_in=1, H=64, graph=("ingest", 2, 360, "dense", 0.9),
                                                     hidden=False), True, ["k_gcn_fwd"])
case("gcn-fwd-ingest360-hidden", run_layer_fwd, dict(kind="gcn", d_in=64, H=64, graph=("ingest", 2, 360, "dense", 0.9)), True,
     ["k_gcn_fwd"])
# -- sage_layer_fwd
case("sage-fwd-gemm-d64", run_layer_fwd, dict(kind="sage", d_in=64, H=64, graph=R84), False, ["k_gather<0>", "k_sage_fwd_gemm"])
case("sage-fwd-gemm-n384", run_layer_fwd, dict(kind="sage", d_in=64, H=64, graph=("rand", (384, 3), 64, 9)), False,
     ["k_gather<0>", "k_sage_fwd_gemm"])
case("sage-fwd-generic-n385", run_layer_fwd, dict(kind="sage", d_in=64, H=64, graph=("rand", (385, 20), 64, 4)), True,
     ["k_gather<0>", "k_sage_fwd_gemm"])
for d_in in (1, 3, 5, 8):
    for H in (32, 64, 128, 256):
        case(f"sage-fwd-first-d{d_in}-H{H}", run_layer_fwd,
             dict(kind="sage", d_in=d_in, H=H, graph=("rand", (84, 30, 1), d_in, 5), hidden=False), False, ["k_first_fwd"])
case("sage-fwd-d9", run_layer_fwd, dict(kind="sage", d_in=9, H=64, graph=("rand", (84, 30), 9, 6), hidden=False), True,
     ["k_sage_fwd_gemm"])
for d_in in (40, 48):
    case(f"sage-fwd-generic-d{d_in}", run_layer_fwd, dict(kind="sage", d_in=d_in, H=64, graph=("rand", (84, 30, 1), d_in, 10)),
         True, ["k_sage_fwd"])
case("sage-fwd-wide256", run_layer_fwd, dict(kind="sage", d_in=256, H=256, graph=("rand", (84, 30, 1), 256, 7)), False,
     ["k_wide_xw"])
for H in (20, 96):
    case(f"sage-fwd-generic-H{H}", run_layer_fwd, dict(kind="sage", d_in=64, H=H, graph=("rand", (84, 30, 1), 64, 8)), True,
         ["k_sage_fwd"])
# the contraction's operands exceed shared memory: no gather may run first only to be thrown away
case("sage-fwd-generic-d64-H128", run_layer_fwd, dict(kind="sage", d_in=64, H=128, graph=("rand", (84, 30, 1), 64, 8)), True,
     ["k_sage_fwd"], forbid=["k_gather<0>", "k_sage_fwd_gemm"])
case("sage-fwd-ingest360-first", run_layer_fwd, dict(kind="sage", d_in=1, H=64, graph=("ingest", 2, 360, "dense", 0.9),
                                                      hidden=False), True, ["k_gather<0>", "k_sage_fwd_gemm"])
case("sage-fwd-ingest360-hidden", run_layer_fwd, dict(kind="sage", d_in=64, H=64, graph=("ingest", 2, 360, "dense", 0.9)), True,
     ["k_sage_fwd"])
# -- layer backward: middle / top layer, du_in present / absent, prev sums, sums64, BatchNorm train / eval / none, dropout
for kind in ("gcn", "sage"):
    gemm = "k_gcn_bwd_gemm" if kind == "gcn" else "k_sage_bwd_gemm"
    generic = ["k_gcn_bwd"] if kind == "gcn" else ["k_sage_bwd_a", "k_sage_bwd_b"]
    gather_bwd = "k_gather<1>" if kind == "gcn" else "k_gather<2>"
    wide = ["k_gather<1>", "k_wide_xty", "k_wide_xw"] if kind == "gcn" else ["k_gather<2>", "k_wide_dz", "k_wide_xty"]
    case(f"{kind}-bwd-gemm-middle", run_layer_bwd, dict(kind=kind, d_in=64, H=64, graph=R84), False, [gemm, gather_bwd])
    case(f"{kind}-bwd-gemm-top-eval-fp32sums", run_layer_bwd, dict(kind=kind, d_in=64, H=64, graph=R84, pooled=True, bn="eval",
                                                                   sums64=False), False, [gemm])
    case(f"{kind}-bwd-gemm-top-fp32sums", run_layer_bwd, dict(kind=kind, d_in=64, H=64, graph=R84, pooled=True, sums64=False),
         False, [gemm])
    case(f"{kind}-bwd-gemm-nobn-n384", run_layer_bwd, dict(kind=kind, d_in=32, H=32, graph=("rand", (384, 5), 32, 11), bn=None),
         False, [gemm])
    case(f"{kind}-bwd-first-d1", run_layer_bwd, dict(kind=kind, d_in=1, H=64, graph=("rand", (84, 30, 1), 1, 12), first=True),
         False, ["k_first_bwd"])
    case(f"{kind}-bwd-first-d5-H256-top", run_layer_bwd, dict(kind=kind, d_in=5, H=256, graph=("rand", (84, 30, 1), 5, 12),
                                                             first=True, pooled=True), False, ["k_first_bwd"])
    case(f"{kind}-bwd-wide256", run_layer_bwd, dict(kind=kind, d_in=256, H=256, graph=("rand", (84, 30, 1), 256, 13)), False,
         wide)
    case(f"{kind}-bwd-wide256-top", run_layer_bwd, dict(kind=kind, d_in=256, H=256, graph=("rand", (84, 30, 1), 256, 13),
                                                        pooled=True, bn="eval"), False, wide)
    case(f"{kind}-bwd-generic-H20", run_layer_bwd, dict(kind=kind, d_in=64, H=20, graph=("rand", (84, 30, 1), 64, 14)), True,
         generic)
    case(f"{kind}-bwd-generic-d96", run_layer_bwd, dict(kind=kind, d_in=96, H=64, graph=("rand", (84, 30, 1), 96, 14),
                                                         pooled=True), True, generic)
    case(f"{kind}-bwd-gemm-n385", run_layer_bwd, dict(kind=kind, d_in=64, H=64, graph=("rand", (385, 20), 64, 4)), True,
         [gemm, gather_bwd])
    case(f"{kind}-bwd-gemm-first-d9", run_layer_bwd, dict(kind=kind, d_in=9, H=64, graph=("rand", (84, 30), 9, 6),
                                                           first=True, bn="eval"), True, [gemm])
    case(f"{kind}-bwd-ingest360-first", run_layer_bwd, dict(kind=kind, d_in=1, H=64, graph=("ingest", 2, 360, "dense", 0.9),
                                                             first=True), True, ["k_gcn_bwd"] if kind == "gcn" else [gemm])
    case(f"{kind}-bwd-ingest360-hidden", run_layer_bwd, dict(kind=kind, d_in=64, H=64, graph=("ingest", 2, 360, "dense", 0.9),
                                                              pooled=True), True, generic)
# du_in of 128 channels does not fit the contraction's dP operand at H = 32: no gather may run first only to be thrown away
case("gcn-bwd-generic-d128-H32", run_layer_bwd, dict(kind="gcn", d_in=128, H=32, graph=("rand", (84, 30, 1), 128, 14)), True,
     ["k_gcn_bwd"], forbid=["k_gather<1>", "k_gcn_bwd_gemm"])
# -- pool, BatchNorm backward sums
case("pool-sums-C64", run_pool_and_sums, dict(C=64, graph=R84), True, ["k_pool_fwd_quad", "k_bn_bwd_sums_quad"])
case("pool-sums-C20-wrap-salt", run_pool_and_sums, dict(C=20, graph=("rand", (360,), 20, 15), row_base=ROW_BASE_WRAP,
                                                        salt=[5, 6]), True, ["k_pool_fwd", "k_bn_bwd_sums"])
case("pool-sums-C64-wrap", run_pool_and_sums, dict(C=64, graph=("rand", (360,), 64, 15), row_base=ROW_BASE_WRAP), True,
     ["k_pool_fwd_quad", "k_bn_bwd_sums_quad"])
# -- head and loss
for K in (2, 3, 8, 9, 64):
    for M in (10, 32, 128):
        for B, p in ((1, 0.0), (4097, 0.3)):
            small = M <= 64 and K <= 8
            case(f"head-K{K}-M{M}-B{B}-p{p}", run_head, dict(B=B, C=64, M=M, K=K, p_drop=p), B == 1 or (K, M) == (9, 32),
                 ["k_head_fwd_small" if small else "k_head_fwd", "k_head_bwd", "k_ce_fwd", "k_ce_bwd"], salted=p > 0)
case("bn-bookkeeping", run_bn_bookkeeping, {}, True, [])
# -- eval-mode network in one kernel, and the pooled last layer
for L in (2, 3, 4):
    for F in (1, 5, 8):
        for K in (2, 8):
            case(f"eval-fused-L{L}-F{F}-K{K}", run_eval_fused, dict(L=L, F=F, K=K), L == 3 and K == 8, ["k_gcn_eval_fused"])
case("eval-fused-K9-declines", run_eval_fused, dict(L=3, F=5, K=9), True, [])
for sizes in ((1,), (2, 1), (9, 8, 127), (128, 129, 1), (383, 384)):
    case(f"fwd-pool-n{max(sizes)}", run_fwd_pool, dict(sizes=sizes), max(sizes) in (9, 129), ["k_gcn_fwd_ws<true>"])
case("fwd-pool-n385-declines", run_fwd_pool, dict(sizes=(385, 3)), True, [])

# -- directed twins: one-way edges, A^ != A^T, in-degree != out-degree, agg_in != agg_out.  Every mode of batch_of
#    appears on several kernel paths; the simulator runs the twins of the cases it runs above
MODES = ("emit", "lazy", "coo", "overflow")
D = lambda sizes, F, seed, blobs: ("directed", sizes, F, seed, blobs)
for n, blobs in ((9, "emit"), (129, "lazy"), (384, "coo")):
    case(f"gcn-fwd-engine-n{n}-directed", run_layer_fwd, dict(kind="gcn", d_in=64, H=64, graph=D((n, max(1, n // 3), n), 64, n, blobs)),
         True, ["k_gcn_fwd_ws<false>"])
case("gcn-fwd-engine-16-per-unit-directed", run_layer_fwd, dict(kind="gcn", d_in=64, H=64, graph=D((20,) * 16, 64, 2, "emit")),
     True, ["k_gcn_fwd_ws<false>"])
for i, (kind, d_in, H) in enumerate((k, d, h) for k in ("gcn", "sage") for d in (1, 5, 8) for h in (32, 256)):
    case(f"{kind}-fwd-first-d{d_in}-H{H}-directed", run_layer_fwd,
         dict(kind=kind, d_in=d_in, H=H, graph=D((84, 30, 1), d_in, 5, MODES[i % 4]), hidden=False), False, ["k_first_fwd"])
case("sage-fwd-gemm-d64-directed", run_layer_fwd, dict(kind="sage", d_in=64, H=64, graph=D((84,) * 4, 64, 1, "full")), False,
     ["k_gather<0>", "k_sage_fwd_gemm"])
case("sage-fwd-gemm-n384-directed", run_layer_fwd, dict(kind="sage", d_in=64, H=64, graph=D((384, 3), 64, 9, "lazy")), False,
     ["k_gather<0>", "k_sage_fwd_gemm"])
case("sage-fwd-generic-n385-directed", run_layer_fwd, dict(kind="sage", d_in=64, H=64, graph=D((385, 20), 64, 4, "coo")), True,
     ["k_gather<0>", "k_sage_fwd_gemm"])
for kind, blobs in (("gcn", "emit"), ("sage", "overflow")):
    case(f"{kind}-fwd-wide256-directed", run_layer_fwd, dict(kind=kind, d_in=256, H=256, graph=D((84, 30, 1), 256, 7, blobs)),
         False, ["k_gather<3>", "k_wide_xw"] if kind == "gcn" else ["k_wide_xw"])
for kind, blobs in (("gcn", "coo"), ("sage", "emit")):
    case(f"{kind}-fwd-generic-H20-directed", run_layer_fwd, dict(kind=kind, d_in=64, H=20, graph=D((84, 30, 1), 64, 8, blobs)),
         True, ["k_gcn_fwd" if kind == "gcn" else "k_sage_fwd"])
for kind in ("gcn", "sage"):
    gemm = "k_gcn_bwd_gemm" if kind == "gcn" else "k_sage_bwd_gemm"
    generic = ["k_gcn_bwd"] if kind == "gcn" else ["k_sage_bwd_a", "k_sage_bwd_b"]
    gather_bwd = "k_gather<1>" if kind == "gcn" else "k_gather<2>"
    wide = ["k_gather<1>", "k_wide_xty", "k_wide_xw"] if kind == "gcn" else ["k_gather<2>", "k_wide_dz", "k_wide_xty"]
    case(f"{kind}-bwd-gemm-middle-directed", run_layer_bwd, dict(kind=kind, d_in=64, H=64, graph=D((84,) * 4, 64, 1, "emit")),
         False, [gemm, gather_bwd])
    case(f"{kind}-bwd-gemm-top-directed", run_layer_bwd, dict(kind=kind, d_in=64, H=64, graph=D((84,) * 4, 64, 1, "overflow"),
                                                              pooled=True), False, [gemm])
    case(f"{kind}-bwd-gemm-n385-directed", run_layer_bwd, dict(kind=kind, d_in=64, H=64, graph=D((385, 20), 64, 4, "lazy")), True,
         [gemm, gather_bwd])
    case(f"{kind}-bwd-first-d1-directed", run_layer_bwd, dict(kind=kind, d_in=1, H=64, graph=D((84, 30, 1), 1, 12, "coo"),
                                                              first=True), False, ["k_first_bwd"])
    case(f"{kind}-bwd-first-d5-H256-top-directed", run_layer_bwd,
         dict(kind=kind, d_in=5, H=256, graph=D((84, 30, 1), 5, 12, "emit"), first=True, pooled=True), False, ["k_first_bwd"])
    case(f"{kind}-bwd-wide256-directed", run_layer_bwd, dict(kind=kind, d_in=256, H=256, graph=D((84, 30, 1), 256, 13, "lazy")),
         False, wide)
    case(f"{kind}-bwd-wide256-top-directed", run_layer_bwd, dict(kind=kind, d_in=256, H=256, graph=D((84, 30, 1), 256, 13, "coo"),
                                                                 pooled=True, bn="eval"), False, wide)
    case(f"{kind}-bwd-generic-H20-directed", run_layer_bwd, dict(kind=kind, d_in=64, H=20, graph=D((84, 30, 1), 64, 14, "emit")),
         True, generic)
    case(f"{kind}-bwd-generic-d96-directed", run_layer_bwd, dict(kind=kind, d_in=96, H=64, graph=D((84, 30, 1), 96, 14, "overflow"),
                                                                 pooled=True), True, generic)
for sizes, blobs in (((128, 129, 1), "emit"), ((9, 8, 127), "overflow"), ((383, 384), "lazy")):
    case(f"fwd-pool-n{max(sizes)}-directed", run_fwd_pool, dict(sizes=sizes, blobs=blobs), max(sizes) in (9, 129),
         ["k_gcn_fwd_ws<true>"])
for i, (L, F, K) in enumerate((l, f, k) for l in (2, 4) for f in (1, 8) for k in (2, 8)):
    case(f"eval-fused-L{L}-F{F}-K{K}-directed", run_eval_fused, dict(L=L, F=F, K=K, blobs=MODES[i % 4]), False, ["k_gcn_eval_fused"])
case("eval-fused-L3-F5-K8-directed", run_eval_fused, dict(L=3, F=5, K=8, blobs="emit"), True, ["k_gcn_eval_fused"])

# -- salted dropout keys in the layer kernels, at row offsets whose rows cross a 2^32 boundary of the global row id inside
#    one CTA's range (every batch has > 100 rows); the second offset has the high word 2, neither 0 nor 1
WRAP3 = 3 * 2 ** 32 - 50
SALT = [0x9E3779B9, 0x7F4A7C15]
SALT3 = [0xA5A5F00D, 0x0000C0DE]
S = lambda rb, salt, p=0.3: dict(row_base=rb, salt=salt, p_drop=p)
SB = lambda rb, salt: dict(row_base=rb, salt=salt)
case("gcn-fwd-engine-n384-salt", run_layer_fwd, dict(kind="gcn", d_in=64, H=64, graph=("rand", (384, 128, 384), 64, 384),
                                                     **S(ROW_BASE_WRAP, SALT)), True, ["k_gcn_fwd_ws<false>"])
case("gcn-fwd-engine-n129-wrap3-p0.9", run_layer_fwd, dict(kind="gcn", d_in=64, H=64, graph=("rand", (129, 43, 129), 64, 129),
                                                           **S(WRAP3, SALT3, 0.9)), True, ["k_gcn_fwd_ws<false>"])
for kind in ("gcn", "sage"):
    case(f"{kind}-fwd-generic-H20-salt", run_layer_fwd, dict(kind=kind, d_in=64, H=20, graph=("rand", (84, 30, 1), 64, 8),
                                                             **S(ROW_BASE_WRAP, SALT)), True, ["k_gcn_fwd" if kind == "gcn" else "k_sage_fwd"])
    case(f"{kind}-fwd-first-d5-H64-hidden-salt", run_layer_fwd, dict(kind=kind, d_in=5, H=64, graph=("rand", (84, 30, 1), 5, 5),
                                                                     **S(WRAP3, SALT3)), False, ["k_first_fwd"])
    case(f"{kind}-fwd-wide256-salt", run_layer_fwd, dict(kind=kind, d_in=256, H=256, graph=("rand", (84, 30, 1), 256, 7),
                                                         **S(ROW_BASE_WRAP, SALT)), False,
         ["k_gather<3>", "k_wide_xw"] if kind == "gcn" else ["k_wide_xw"])
    gemm = "k_gcn_bwd_gemm" if kind == "gcn" else "k_sage_bwd_gemm"
    generic = ["k_gcn_bwd"] if kind == "gcn" else ["k_sage_bwd_a", "k_sage_bwd_b"]
    gather_bwd = "k_gather<1>" if kind == "gcn" else "k_gather<2>"
    wide = ["k_gather<1>", "k_wide_xty", "k_wide_xw"] if kind == "gcn" else ["k_gather<2>", "k_wide_dz", "k_wide_xty"]
    case(f"{kind}-bwd-gemm-middle-salt", run_layer_bwd, dict(kind=kind, d_in=64, H=64, graph=R84, **SB(ROW_BASE_WRAP, SALT)), False,
         [gemm, gather_bwd])
    case(f"{kind}-bwd-gemm-n385-wrap3-salt", run_layer_bwd, dict(kind=kind, d_in=64, H=64, graph=("rand", (385, 20), 64, 4),
                                                                 **SB(WRAP3, SALT3)), False, [gemm, gather_bwd])
    case(f"{kind}-bwd-generic-H20-salt", run_layer_bwd, dict(kind=kind, d_in=64, H=20, graph=("rand", (84, 30, 1), 64, 14),
                                                             **SB(ROW_BASE_WRAP, SALT)), True, generic)
    case(f"{kind}-bwd-first-d5-H64-hidden-salt", run_layer_bwd, dict(kind=kind, d_in=5, H=64, graph=("rand", (84, 30, 1), 5, 12),
                                                                     first=True, hidden=True, **SB(WRAP3, SALT3)), False,
         ["k_first_bwd"])
    case(f"{kind}-bwd-wide256-salt", run_layer_bwd, dict(kind=kind, d_in=256, H=256, graph=("rand", (84, 30, 1), 256, 13),
                                                         **SB(ROW_BASE_WRAP, SALT)), False, wide)
case("sage-fwd-gemm-d64-salt", run_layer_fwd, dict(kind="sage", d_in=64, H=64, graph=R84, **S(WRAP3, SALT3)), False,
     ["k_gather<0>", "k_sage_fwd_gemm"])
# nine input channels: k_sage_fwd_gemm applies the input's dropout itself (the narrow-K operand path)
case("sage-fwd-gemm-d9-hidden-salt", run_layer_fwd, dict(kind="sage", d_in=9, H=64, graph=("rand", (84, 30), 9, 6),
                                                         **S(ROW_BASE_WRAP, SALT)), False, ["k_sage_fwd_gemm"])
case("pool-sums-C64-wrap3-salt", run_pool_and_sums, dict(C=64, graph=("rand", (360,), 64, 15), row_base=WRAP3, salt=SALT3), True,
     ["k_pool_fwd_quad", "k_bn_bwd_sums_quad"])

# every one of these must be reached by at least one case on a B200
REQUIRED = {"k_gcn_fwd_ws<true>", "k_gcn_fwd_ws<false>", "k_first_fwd", "k_first_bwd", "k_gather<0>", "k_gather<1>",
            "k_gather<2>", "k_gather<3>", "k_sage_fwd_gemm", "k_gcn_bwd_gemm", "k_sage_bwd_gemm", "k_wide_xw", "k_wide_xty",
            "k_wide_dz", "k_gcn_fwd", "k_gcn_bwd", "k_sage_fwd", "k_sage_bwd_a", "k_sage_bwd_b", "k_gcn_eval_fused",
            "k_pool_fwd", "k_pool_fwd_quad", "k_head_fwd", "k_head_fwd_small", "k_head_bwd", "k_ce_fwd", "k_ce_bwd",
            "k_bn_bwd_sums", "k_bn_bwd_sums_quad", "k_build_agg"}
# ... these by a directed case (every layer kernel, the blob builder and the collate kernel that emits blobs)
DIRECTED_REQUIRED = {"k_gcn_fwd_ws<true>", "k_gcn_fwd_ws<false>", "k_first_fwd", "k_first_bwd", "k_gather<0>", "k_gather<1>",
                     "k_gather<2>", "k_gather<3>", "k_sage_fwd_gemm", "k_gcn_bwd_gemm", "k_sage_bwd_gemm", "k_wide_xw",
                     "k_wide_xty", "k_wide_dz", "k_gcn_fwd", "k_gcn_bwd", "k_sage_fwd", "k_sage_bwd_a", "k_sage_bwd_b",
                     "k_gcn_eval_fused", "k_build_agg", "k_collate_graph"}
# ... and these by a salted case: every kernel that folds the device salt into its dropout keys (act_salt)
SALTED_REQUIRED = {"k_gather<0>", "k_gather<1>", "k_gather<2>", "k_gather<3>", "k_gcn_fwd_ws<false>", "k_first_fwd",
                   "k_first_bwd", "k_gcn_fwd", "k_gcn_bwd", "k_sage_fwd_gemm", "k_gcn_bwd_gemm", "k_sage_bwd_gemm", "k_pool_fwd",
                   "k_pool_fwd_quad", "k_head_fwd", "k_head_fwd_small", "k_bn_bwd_sums", "k_bn_bwd_sums_quad", "k_sage_fwd",
                   "k_sage_bwd_a", "k_sage_bwd_b", "k_wide_xty", "k_wide_dz"}

_DEV = {"device": "cpu"}


def kernel_tokens(name):
    """Kernel identifiers of one profiler event name; the warp-specialised engine and the gather kernel also by their
    first template argument (pooled / plain, gather mode)."""
    out = set()
    for m in re.finditer(r"\b(k_\w+)(?:<([^>]*)>)?", name):
        base, targs = m.group(1), m.group(2)
        out.add(base)
        if targs and base in ("k_gather", "k_gcn_fwd_ws"):
            first = targs.split(",")[0].strip().split(")")[-1]
            first = {"1": "true", "0": "false"}.get(first, first) if base == "k_gcn_fwd_ws" else first
            out.add(f"{base}<{first}>")
    return out


# ---- simulator ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fn,kw", EMU_CASES)
def test_contract_on_simulator(on_emu, fn, kw):
    _DEV["device"] = "cpu"
    r = fn(on_emu, **kw)
    print(f"worst error {r:.2f} x 2^-23 x magnitude")


def test_head_rejects_more_than_64_classes(on_emu):
    from connectome_gnn._lib import CgnnError
    z = torch.zeros
    with pytest.raises(CgnnError):
        on_emu.head_fwd(z(2, 64), z(32, 64), z(32), z(65, 32), z(65), 0.0, 0, 0)


# ---- B200 ----------------------------------------------------------------------------------------------------------------
_SEEN: dict = {}


def _run_profiled(fn, kw):
    from connectome_gnn import _engine
    from torch.profiler import ProfilerActivity, profile
    _DEV["device"] = "cuda"
    eng = _engine.engine_for(torch.empty(1, device="cuda"))
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        r = fn(eng, **kw)
        torch.cuda.synchronize()
    names = set()
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            names |= kernel_tokens(e.name)
    return r, names


@pytest.mark.gpu
@pytest.mark.parametrize("fn,kw,expect,forbid", CASES)
def test_contract_on_b200(request, fn, kw, expect, forbid):
    r, names = _run_profiled(fn, kw)
    _SEEN[request.node.callspec.id] = (names, r)
    missing = expect - names
    assert not missing, f"intended kernels {sorted(missing)} did not run; ran: {sorted(names)}"
    assert not forbid & names, f"kernels {sorted(forbid & names)} must not run; ran: {sorted(names)}"


@pytest.mark.gpu
def test_head_rejects_more_than_64_classes_b200():
    from connectome_gnn import _engine
    from connectome_gnn._lib import CgnnError
    eng = _engine.engine_for(torch.empty(1, device="cuda"))
    z = lambda *s: torch.zeros(*s, device="cuda")
    with pytest.raises(CgnnError):
        eng.head_fwd(z(2, 64), z(32, 64), z(32), z(65, 32), z(65), 0.0, 0, 0)


@pytest.mark.gpu
def test_dispatch_table():
    """Prints case -> kernels (and worst error ratio) and asserts every kernel of REQUIRED was reached, every kernel of
    DIRECTED_REQUIRED by a directed case and every kernel of SALTED_REQUIRED by a salted one.  Cases that did not run in
    this session (deselected) are run here."""
    for p in CASES:
        if p.id not in _SEEN:
            fn, kw, _, _ = p.values
            r, names = _run_profiled(fn, kw)
            _SEEN[p.id] = (names, r)
    print("\ncase | worst error (x 2^-23 x mag) | kernels")
    for cid, (names, r) in _SEEN.items():
        print(f"{cid} | {r:.2f} | {' '.join(sorted(n for n in names if n.startswith('k_')))}")
    for what, ids in (("directed", DIRECTED), ("salted", SALTED)):
        print(f"worst error of the {what} cases: {max(_SEEN[c][1] for c in ids):.2f}")
    reached = lambda ids: set().union(*(n for c, (n, _) in _SEEN.items() if c in ids))
    assert REQUIRED <= reached(_SEEN), f"never reached: {sorted(REQUIRED - reached(_SEEN))}"
    assert DIRECTED_REQUIRED <= reached(DIRECTED), f"no directed case reached: {sorted(DIRECTED_REQUIRED - reached(DIRECTED))}"
    assert SALTED_REQUIRED <= reached(SALTED), f"no salted case reached: {sorted(SALTED_REQUIRED - reached(SALTED))}"


# ---- model level: ingested (real-density) and synthetic subjects against the oracle -----------------------------------
def run_model(dev, kind, source, fused_eval="auto", K=2, lean=True, layers=3, hidden=64, seed=0):
    """A training step (logits, loss, every gradient, running statistics) and eval logits against parity.oracle_reference.
    source: ("ingest", S, N, kind, q), ("synthetic", S, N) or ("directed", sizes, F, seed) (directed_graphs).  With one all-positive feature per node the fp32 oracle
    itself sits above 1e-5 from fp64 on some tensors (BatchNorm means of nearly constant columns): bars below 1e-5 are
    scaled by the oracle's own distance, measured here.  Logits and loss at 1e-5.  (The "ties" recipe at 84 regions keeps
    no edge at all: a batch without edges, which once failed to collate.)"""
    import parity
    from connectome_gnn.graph import SubjectStore, pack_graphs
    from connectome_gnn.train import CrossEntropyLoss
    from oracle import port
    _DEV["device"] = dev
    if source[0] == "ingest":
        p = ingested(*source[1:])
        graphs = packed_graphs(p)
    elif source[0] == "directed":
        graphs = directed_graphs(*source[1:])
        for i, gr in enumerate(graphs):
            gr.label = torch.tensor(i % K)
        p = pack_graphs(graphs)
    else:
        from connectome_gnn.synthetic import generate_dataset
        graphs = generate_dataset(num_subjects=source[1], num_regions=source[2], seed=source[1] + source[2])
        for i, gr in enumerate(graphs):
            gr.label = torch.tensor(i % K)
        p = pack_graphs(graphs)
    store = SubjectStore(p, dev)
    ids = np.arange(len(graphs))
    g = torch.Generator().manual_seed(seed)
    g2 = torch.Generator().manual_seed(seed + 1)
    params = port.init_params(kind, graphs[0].num_features, hidden, K, layers, generator=g)
    for k in params:                      # non-trivial BatchNorm affine and running statistics
        if ".weight" in k and "batch_norms" in k:
            params[k] = params[k] + 0.1 * torch.randn(params[k].shape, generator=g)
        if k.endswith("running_mean"):
            params[k] = 0.05 * torch.randn(params[k].shape, generator=g2)
        if k.endswith("running_var"):
            params[k] = 1.0 + 0.2 * torch.rand(params[k].shape, generator=g2)
    refs = parity.oracle_reference(kind, params, graphs)
    a, a32 = refs["f64"], refs["f32"]
    m = parity.make_model(kind, a32, dev)
    m.fused_eval = fused_eval
    m.eval()
    with torch.no_grad():
        eb = store.collate(ids, prepare_for=kind, backward=False) if lean else store.collate(ids)
        helpers.assert_close(m(eb), a[f"{kind}.eval.logits"], "eval logits")
    m.train()
    b = store.collate(ids, prepare_for=kind) if lean else store.collate(ids)
    logits = m(b)
    loss = CrossEntropyLoss()(logits, b.labels)
    loss.backward()
    helpers.assert_close(logits, a[f"{kind}.train.logits"], "train logits")
    helpers.assert_close(loss, a[f"{kind}.train.loss"], "train loss")
    # all gradients together: max(1e-5, 10 x the fp32 oracle's distance) as parity.check_against_oracle has it; each tensor
    # within the per-tensor band of parity.py (1e-4), or 4 x the oracle's own distance where that is larger.  Measured:
    # the first-layer GCN weight gradient at 360 dense regions is 6.4e-5 (B200) / 8.6e-5 (simulator) from fp64 where the
    # fp32 oracle is at 1.6e-5 - a sum over 1080 rows of one all-positive feature cancels to 1e-3 of its magnitude, and
    # the layer-level cases above hold that very kernel (k_gcn_bwd) to 5 x 2^-23 of the magnitude.
    import parity
    names = [k for k, _ in m.named_parameters()]
    cat = lambda src: torch.cat([torch.as_tensor(src[f"{kind}.train.grad.{k}"]).reshape(-1).double() for k in names])
    got_all = torch.cat([q.grad.reshape(-1) for _, q in m.named_parameters()])
    noise_all = helpers.max_rel(cat(a32), cat(a))
    helpers.assert_close(got_all, cat(a), f"all gradients (fp32 oracle at {noise_all:.1e})", tol=max(helpers.REL_TOL, 10 * noise_all))
    scale = float(cat(a).abs().max())
    worst_bar = 0.0
    tensors = [(f"grad {k}", q.grad, f"{kind}.train.grad.{k}") for k, q in m.named_parameters()]
    tensors += [(k, v, f"{kind}.train.after.{k}") for k, v in m.state_dict().items() if "running" in k]
    for what, got, key in tensors:
        noise = helpers.max_rel(a32[key], a[key])
        bar = max(helpers.REL_TOL, 4 * noise) if what.startswith("running") else max(parity.PER_TENSOR_TOL, 4 * noise)
        worst_bar = max(worst_bar, bar)
        if kind == "gcn" and what.startswith("grad convs.") and what.endswith(".bias"):
            # analytically zero (the bias feeds BatchNorm): round-off only, held to the global gradient scale
            err = float((got.detach().cpu().double() - torch.as_tensor(a[key]).double()).abs().max())
            assert err <= max(helpers.REL_TOL, 10 * noise_all) * scale, (what, err, scale)
        else:
            helpers.assert_close(got, a[key], f"{what} (fp32 oracle at {noise:.1e})", tol=bar)
    return worst_bar


MODEL_CASES, EMU_MODEL_CASES = [], []


def model_case(cid, kw, emu):
    MODEL_CASES.append(pytest.param(kw, id=cid))
    if emu:
        EMU_MODEL_CASES.append(pytest.param(kw, id=cid))


for kind in ("gcn", "sage"):
    for N, mk in ((84, "dense"), (84, "sparse"), (84, "ties"), (360, "dense"), (360, "sparse"), (360, "ties")):
        for fe in ("auto", False):
            for K in (2, 5):
                lean = K == 2
                emu = fe == "auto" and ((N, mk, K) in ((84, "dense", 2), (84, "ties", 5), (360, "dense", 2)))
                model_case(f"{kind}-ingest{N}-{mk}-fused_{fe}-K{K}-{'lean' if lean else 'full'}",
                           dict(kind=kind, source=("ingest", 4 if N == 84 else 3, N, mk, 0.90), fused_eval=fe, K=K, lean=lean), emu)
    for q in (0.92, 0.91):     # m on either side of the first layer's and the 64-channel gather's shared-memory limits
        model_case(f"{kind}-ingest360-q{q}", dict(kind=kind, source=("ingest", 3, 360, "dense", q), lean=True), False)
    for K in (3, 9, 64):
        model_case(f"{kind}-synthetic-K{K}", dict(kind=kind, source=("synthetic", 12, 40), K=K), K == 9)
    model_case(f"{kind}-synthetic-1-layer", dict(kind=kind, source=("synthetic", 6, 84), layers=1), True)
    for fe in ("auto", False):       # one-way edges through every layer of the model, lean batches
        model_case(f"{kind}-directed-fused_{fe}", dict(kind=kind, source=("directed", (84, 60, 84, 30, 84, 9), 5, 21),
                                                       fused_eval=fe), kind == "gcn" and fe == "auto")


@pytest.mark.parametrize("kw", EMU_MODEL_CASES)
def test_model_on_simulator(on_emu, kw):
    run_model("cpu", **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("kw", MODEL_CASES)
def test_model_on_b200(kw):
    run_model("cuda", **kw)

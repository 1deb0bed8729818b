"""TEST-ONLY float64 restatement of the contracts written in include/cgnn.h.

Every function here is computed from the batch's COO (edge_index, edge_weight, ptr) - never from the kernels' CSR
arrays or aggregation blobs - in torch float64 on the CPU.  The dropout keep masks are restated bit for bit in numpy
uint32 (common.cuh: make_act, drop_row_hash, drop_keep, act_salt; head.cu: the head's stream).

Alongside each value the functions return a MAGNITUDE: the same computation on absolute values (|u|, |W|, |w^|, ...).
`check` then holds every element to its own scale,

    |got - ref| <= c * 2^-23 * mag,

which sees a wrong row however small its values are and tolerates cancellation (BatchNorm's backward subtracts the
channel means from every row).  C_ULPS below was set from the measured distribution (see test_contract.py).
"""
import numpy as np
import torch

F64 = torch.float64
EPS32 = 2.0 ** -23
# Largest error over every case of test_contract.py, in units of 2^-23 * mag: 5.2 on the simulator, 9.7 on a B200 (the
# wide GraphSAGE backward; test_dispatch_table prints the worst ratio of each case).  32 leaves a factor 3 for summation
# orders not seen yet; the value mutations listed in test_contract.py miss it by a factor 1000 or more.
C_ULPS = 32.0

M32 = np.uint64(0xFFFFFFFF)
HEAD_SITE = 0x48454144


# ---- dropout stream -------------------------------------------------------------------------------------------------
def _u32(x):
    return np.asarray(x, dtype=np.uint64) & M32


def fmix32(h):
    h = _u32(h)
    h ^= h >> np.uint64(16)
    h = (h * np.uint64(0x85EBCA6B)) & M32
    h ^= h >> np.uint64(13)
    h = (h * np.uint64(0xC2B2AE35)) & M32
    h ^= h >> np.uint64(16)
    return h


def make_act_keys(p_drop, seed, site, salt=None):
    """(thresh, keep_scale, k0, k1) as make_act derives them on the host, with the salt words folded in (act_salt)."""
    p32 = np.float32(p_drop)
    t = float(p32) * 65536.0 + 0.5
    thresh = 65535 if t >= 65535.0 else int(t)
    keep_scale = float(np.float32(1.0) / (np.float32(1.0) - p32))
    seed &= 0xFFFFFFFFFFFFFFFF
    site &= 0xFFFFFFFF
    k0 = ((seed & 0xFFFFFFFF) ^ ((site * 0x9E3779B9) & 0xFFFFFFFF)) & 0xFFFFFFFF
    k1 = ((seed >> 32) + site * 0x85EBCA6B + 0x27D4EB2F) & 0xFFFFFFFF
    if salt is not None:
        k0 ^= int(salt[0]) & 0xFFFFFFFF
        k1 = (k1 + int(salt[1])) & 0xFFFFFFFF
    return thresh, keep_scale, k0, k1


def keep_mask(p_drop, seed, site, row_base, rows, C, salt=None):
    """bool [rows, C]: dropout keeps element (r, c) of a tensor whose local row 0 is global row `row_base`."""
    thresh, _, k0, k1 = make_act_keys(p_drop, seed, site, salt)
    grow = np.arange(rows, dtype=np.int64) + np.int64(row_base)
    g = grow.astype(np.uint64)
    lo, hi = g & M32, g >> np.uint64(32)
    rh = ((lo * np.uint64(0x9E3779B1)) & M32) ^ np.uint64(k0) ^ fmix32(hi + np.uint64(k1))
    c = np.arange(C, dtype=np.uint64)
    y = fmix32(rh[:, None] + ((c >> np.uint64(2)) * np.uint64(0x632BE5AB)) + np.uint64(k1))
    w2 = (y * np.uint64(0x9E3779B1) + np.uint64(0x7F4A7C15)) & M32
    w2 ^= w2 >> np.uint64(15)
    w = np.where((c & np.uint64(2)) != 0, w2, y)
    bits = np.where((c & np.uint64(1)) != 0, w >> np.uint64(16), w & np.uint64(0xFFFF))
    return bits >= np.uint64(thresh)


class Act:
    """Host description of a cgnn_act_t for the reference: u = dropout(relu?(scale * t + shift))."""

    def __init__(self, scale=None, shift=None, relu=False, p_drop=0.0, seed=0, site=0, row_base=0, salt=None):
        self.scale, self.shift, self.relu, self.p_drop = scale, shift, relu, p_drop
        self.seed, self.site, self.row_base, self.salt = seed, site, row_base, salt

    def mask_and_scale(self, rows, C):
        """(float64 [rows, C] multiplier of the dropout: keep_scale or 0, all ones without dropout)."""
        if self.p_drop <= 0.0:
            return torch.ones(rows, C, dtype=F64)
        _, ks, _, _ = make_act_keys(self.p_drop, self.seed, self.site, self.salt)
        m = keep_mask(self.p_drop, self.seed, self.site, self.row_base, rows, C, self.salt)
        return torch.from_numpy(m.astype(np.float64)) * ks

    def pre(self, t):
        """(y, |y| scale) before ReLU and dropout."""
        t = t.to(F64)
        if self.scale is None:
            return t, t.abs()
        sc, sh = self.scale.to(F64), self.shift.to(F64)
        return t * sc + sh, (t * sc).abs() + sh.abs()


def act_fwd(act, t):
    """u = act(t) (and its magnitude); the keep mask / ReLU mask multiplier for the backward."""
    y, mag = act.pre(t)
    drop = act.mask_and_scale(*y.shape)
    gate = drop * (y > 0).to(F64) if act.relu else drop
    u = y * gate
    return u, mag * drop.abs(), gate


# ---- graph structure from the COO ----------------------------------------------------------------------------------
class Graph:
    """The batch structure the contracts are written against, from the collated COO."""

    def __init__(self, edge_index, edge_weight, ptr):
        ei = torch.as_tensor(edge_index).cpu().long()
        self.src, self.dst = ei[0], ei[1]
        self.w32 = torch.as_tensor(edge_weight).cpu().float()
        self.w = self.w32.to(F64)
        self.ptr = torch.as_tensor(ptr).cpu().long()
        self.rows = int(self.ptr[-1])
        self.B = len(self.ptr) - 1
        # D^_i = ((0 + w_e1) + w_e2 ...) + 1 over the edges with src == i in COO order, in fp32 (cgnn_csr_t: deg)
        deg = np.zeros(self.rows, dtype=np.float32)
        np.add.at(deg, self.src.numpy(), self.w32.numpy())
        self.deg = torch.from_numpy(deg + np.float32(1.0)).to(F64)
        self.dinv = (self.deg + 1e-8).rsqrt()
        self.wn = self.dinv[self.src] * self.w * self.dinv[self.dst]
        self.wsum = torch.zeros(self.rows, dtype=F64).index_add_(0, self.dst, self.w)
        self.sizes = (self.ptr[1:] - self.ptr[:-1]).to(F64)
        self.row_graph = torch.repeat_interleave(torch.arange(self.B), self.ptr[1:] - self.ptr[:-1])

    def gcn_agg(self, P, absval=False):
        """A^ P: in-edges in COO order, then the self-loop term dinv_i^2 P_i."""
        wn = self.wn.abs() if absval else self.wn
        out = torch.zeros_like(P).index_add_(0, self.dst, wn[:, None] * P[self.src])
        return out + (self.dinv * self.dinv)[:, None] * P

    def sage_agg(self, u, absval=False):
        """sum_{e: dst=i} w_e u_src / (w_sum_i + 1e-8)."""
        w = self.w.abs() if absval else self.w
        num = torch.zeros(self.rows, u.shape[1], dtype=F64).index_add_(0, self.dst, w[:, None] * u[self.src])
        return num / (self.wsum + 1e-8)[:, None]

    def pool(self, t):
        """mean over each subject's rows, / (N_g + 1e-8)."""
        s = torch.zeros(self.B, t.shape[1], dtype=F64).index_add_(0, self.row_graph, t)
        return s / (self.sizes + 1e-8)[:, None]

    def unpool(self, demb):
        """the pooled gradient broadcast to rows: demb[g] / (N_g + 1e-8)."""
        return (demb.to(F64) / (self.sizes + 1e-8)[:, None])[self.row_graph]


# ---- layer forward ---------------------------------------------------------------------------------------------------
def layer_pre(kind, graph, u, W, b, absval=False):
    """The layer's output before any ReLU: GCN A^(u W^T) + b; GraphSAGE [u || agg] W^T + b."""
    if absval:
        u, W, b = u.abs(), W.abs(), (b.abs() if b is not None else None)
    return _pre(kind, graph, u, W, b, absval)


def _pre(kind, graph, u, W, b, absgraph):
    if kind == "gcn":
        z = graph.gcn_agg(u @ W.T, absgraph)
    else:
        agg = graph.sage_agg(u, absgraph)
        z = torch.cat([u, agg], 1) @ W.T
    return z + b if b is not None else z


def layer_fwd(kind, graph, t_in, act, W, b):
    """(z, mag, agg, agg_mag): cgnn_gcn_layer_fwd / cgnn_sage_layer_fwd (SAGE: z = relu(pre))."""
    u, umag, _ = act_fwd(act, t_in)
    W, b = W.to(F64), b.to(F64)
    z = layer_pre(kind, graph, u, W, b)
    mag = layer_pre(kind, graph, umag, W, b, absval=True)
    if kind == "sage":
        z = torch.clamp(z, min=0.0)
        return z, mag, graph.sage_agg(u), graph.sage_agg(umag, absval=True)
    return z, mag, None, None


def stats_of(z):
    """{count, mean[C], M2[C]} of the rows of z (float64)."""
    z = z.to(F64)
    m = z.mean(0)
    return torch.cat([torch.tensor([float(z.shape[0])], dtype=F64), m, ((z - m) ** 2).sum(0)])


# ---- BatchNorm bookkeeping -------------------------------------------------------------------------------------------
def bn_finalize(stats, gamma, beta, eps, momentum, running_mean, running_var):
    C = gamma.shape[0]
    st = stats.to(F64)
    n, mean, m2 = float(st[0]), st[1:1 + C], st[1 + C:1 + 2 * C]
    var = m2 / n
    rstd = (var + eps).rsqrt()
    scale = gamma.to(F64) * rstd
    shift = beta.to(F64) - mean * scale
    rm = (1 - momentum) * running_mean.to(F64) + momentum * mean
    rv = (1 - momentum) * running_var.to(F64) + momentum * (m2 / (n - 1) if n > 1 else var)
    return scale, shift, mean, rstd, rm, rv


def bn_eval_affine(gamma, beta, running_mean, running_var, eps):
    rstd = (running_var.to(F64) + eps).rsqrt()
    scale = gamma.to(F64) * rstd
    return scale, beta.to(F64) - running_mean.to(F64) * scale, running_mean.to(F64), rstd


def bn_merge_stats(parts, C):
    n, mean, m2 = 0.0, torch.zeros(C, dtype=F64), torch.zeros(C, dtype=F64)
    for rec in parts.to(F64):
        nb = float(rec[0])
        if nb <= 0:
            continue
        mb, qb = rec[1:1 + C], rec[1 + C:1 + 2 * C]
        nt = n + nb
        d = mb - mean
        mean = mean + d * (nb / nt)
        m2 = m2 + qb + d * d * (n * nb / nt)
        n = nt
    return torch.cat([torch.tensor([n], dtype=F64), mean, m2])


def bn_bwd_sums(graph, z, act, mean, rstd, du=None, demb=None):
    """[2, C] = {sum dy, sum dy * xhat}, dy = d act / d y * du (du per row, or demb pooled) - and magnitudes."""
    up = du.to(F64) if du is not None else graph.unpool(demb)
    _, _, gate = act_fwd(act, z)
    dy = up * gate
    xhat = (z.to(F64) - mean.to(F64)) * rstd.to(F64)
    val = torch.stack([dy.sum(0), (dy * xhat).sum(0)])
    mag = torch.stack([dy.abs().sum(0), (dy * xhat).abs().sum(0)])
    return val, mag


# ---- layer backward --------------------------------------------------------------------------------------------------
def layer_bwd(kind, graph, z, act_out, bn, t_in, act_in, W, du=None, demb=None, prev=None):
    """Contract of cgnn_{gcn,sage}_layer_bwd.  bn = None or dict(scale, mean, rstd, s1, s2, count, train) where s1 / s2
    are the sums the kernel is handed (the literal cgnn_bn_bwd_t formula is applied to them).  prev = None or
    (prev_mean, prev_rstd): then the BatchNorm backward sums of the layer below come back too.
    Returns {name: (value, mag)} for dW, dbias, du_in, prev_sums."""
    up = du.to(F64) if du is not None else graph.unpool(demb)
    upmag = up.abs()
    _, _, gate = act_fwd(act_out, z)
    dy, dymag = up * gate, upmag * gate.abs()
    z64 = z.to(F64)
    if bn is None:
        dz, dzmag = dy, dymag
    else:
        sc = bn["scale"].to(F64)
        if bn["train"]:
            inv = 1.0 / bn["count"]
            xhat = (z64 - bn["mean"].to(F64)) * bn["rstd"].to(F64)
            s1, s2 = bn["s1"].to(F64), bn["s2"].to(F64)
            dz = sc * (dy - s1 * inv - xhat * s2 * inv)
            dzmag = sc.abs() * (dymag + (s1 * inv).abs() + (xhat * s2 * inv).abs())
        else:
            dz, dzmag = sc * dy, sc.abs() * dymag
    if kind == "sage":           # z is the post-ReLU output
        relu = (z64 > 0).to(F64)
        dz, dzmag = dz * relu, dzmag * relu
    u, umag, gate_in = act_fwd(act_in, t_in)
    W64 = W.to(F64)
    out = {}
    for tag, uu, ww, g, absval in (("val", u, W64, dz, False), ("mag", umag, W64.abs(), dzmag, True)):
        uu = uu.clone().requires_grad_(True)
        ww = ww.clone().requires_grad_(True)
        pre = _pre(kind, graph, uu, ww, None, absval)    # (the magnitude pass takes |u|, |W| as they are: no abs())
        dW, du_in = torch.autograd.grad(pre, (ww, uu), grad_outputs=g)
        out[tag] = dict(dW=dW, dbias=(g.sum(0) if tag == "val" else g.abs().sum(0)), du_in=du_in)
    res = {k: (out["val"][k], out["mag"][k]) for k in ("dW", "dbias", "du_in")}
    if prev is not None:
        pm, pr = prev
        xh = (t_in.to(F64) - pm.to(F64)) * pr.to(F64)
        dyp, dypm = out["val"]["du_in"] * gate_in, out["mag"]["du_in"] * gate_in.abs()
        res["prev_sums"] = (torch.stack([dyp.sum(0), (dyp * xh).sum(0)]),
                            torch.stack([dypm.sum(0), (dypm * xh.abs()).sum(0)]))
    return res


# ---- readout, head, loss ----------------------------------------------------------------------------------------------
def pool_fwd(graph, t, act):
    u, mag, _ = act_fwd(act, t)
    return graph.pool(u), graph.pool(mag)


def head_fwd(emb, W0, b0, W1, b1, p_drop=0.0, seed=0, graph_base=0, salt=None):
    """(hidden, logits) and their magnitudes; the dropout after the hidden ReLU draws from site HEAD_SITE, row = graph."""
    e, W0, b0, W1, b1 = (q.to(F64) for q in (emb, W0, b0, W1, b1))
    pre = e @ W0.T + b0
    premag = e.abs() @ W0.abs().T + b0.abs()
    d = Act(p_drop=p_drop, seed=seed, site=HEAD_SITE, row_base=graph_base, salt=salt).mask_and_scale(*pre.shape)
    gate = d * (pre > 0).to(F64)
    hidden, hmag = pre * gate, premag * d.abs()
    return hidden, hmag, hidden @ W1.T + b1, hmag @ W1.abs().T + b1.abs()


def ce_fwd(logits, labels, inv_count):
    l = logits.to(F64)
    lse = torch.logsumexp(l, 1)
    y = torch.as_tensor(labels).cpu().long()
    nll = lse - l[torch.arange(l.shape[0]), y]
    correct = int((torch.argmax(logits.cpu(), 1) == y).sum())     # first maximum, as the kernel's strict '>' scan
    mag = lse.abs() + l.abs().max(1).values
    return nll, mag, float((nll * inv_count).sum()), float((mag * abs(inv_count)).sum()), correct


def ce_bwd(logits, labels, inv_count, gout):
    l = logits.to(F64)
    y = torch.as_tensor(labels).cpu().long()
    sm = torch.softmax(l, 1)
    oh = torch.nn.functional.one_hot(y, l.shape[1]).to(F64)
    s = inv_count * float(gout)
    return (sm - oh) * s, (sm + oh) * abs(s)


def head_bwd(emb, hidden, dlogits, W0, W1, p_drop):
    """demb, dW0, db0, dW1, db1 with magnitudes.  The hidden units' gate is read off `hidden` (post-ReLU, post-dropout)."""
    e, h, dl, W0, W1 = (q.to(F64) for q in (emb, hidden, dlogits, W0, W1))
    ks = float(np.float32(1.0) / (np.float32(1.0) - np.float32(p_drop))) if p_drop > 0 else 1.0
    gate = (h > 0).to(F64) * ks
    dh, dhm = (dl @ W1) * gate, (dl.abs() @ W1.abs()) * gate
    return dict(demb=(dh @ W0, dhm @ W0.abs()), dW0=(dh.T @ e, dhm.T @ e.abs()), db0=(dh.sum(0), dhm.sum(0)),
                dW1=(dl.T @ h, dl.abs().T @ h.abs()), db1=(dl.sum(0), dl.abs().sum(0)))


# ---- the whole eval-mode network (cgnn_eval_fused_fwd / the pooled last layer) ---------------------------------------
def gcn_eval_network(graph, x, layers, head):
    """layers = [(W, b, gamma, beta, running_mean, running_var, eps)], head = (W0, b0, W1, b1): (emb, logits, mags)."""
    t, act = x.to(F64), Act()
    u, umag, _ = act_fwd(act, t)
    for W, b, g, be, rm, rv, eps in layers:
        z = layer_pre("gcn", graph, u, W.to(F64), b.to(F64))
        zmag = layer_pre("gcn", graph, umag, W.to(F64), b.to(F64), absval=True)
        sc, sh, _, _ = bn_eval_affine(g, be, rm, rv, eps)
        y = z * sc + sh
        u, umag = torch.clamp(y, min=0.0), zmag * sc.abs() + sh.abs()
    emb, embmag = graph.pool(u), graph.pool(umag)
    _, _, logits, lmag = head_fwd(emb, *head)
    W0, b0, W1, b1 = (q.to(F64) for q in head)
    lmag = (embmag @ W0.abs().T + b0.abs()) @ W1.abs().T + b1.abs()
    return emb, embmag, logits, lmag


# ---- the comparison ----------------------------------------------------------------------------------------------------
def ratio(got, ref, mag):
    """max over elements of |got - ref| / (2^-23 * mag) (elements with mag == 0 must match exactly)."""
    got = torch.as_tensor(got).detach().cpu().to(F64).reshape(-1)
    ref = torch.as_tensor(ref).detach().cpu().to(F64).reshape(-1)
    mag = torch.as_tensor(mag).detach().cpu().to(F64).reshape(-1)
    assert got.shape == ref.shape == mag.shape, (got.shape, ref.shape, mag.shape)
    if got.numel() == 0:
        return 0.0
    assert torch.isfinite(got).all(), "non-finite values"
    err = (got - ref).abs()
    tiny = mag == 0
    if bool(tiny.any()) and float(err[tiny].max()) > 0:
        return float("inf")
    r = err / (EPS32 * torch.where(tiny, torch.ones_like(mag), mag))
    return float(r.max())


def check(got, ref, mag, what, c=C_ULPS):
    r = ratio(got, ref, mag)
    assert r <= c, f"{what}: error {r:.1f} x 2^-23 x magnitude (bar {c:g})"
    return r

"""Typed host-side wrappers over the C ABI (``include/cgnn.h``): one method per entry point.

PyTorch is plumbing here - it owns device memory (caching allocator), the current stream and
``torch.distributed``; every bit of arithmetic on the hot path happens inside ``libcgnn.so``.
There is deliberately no CPU branch: :func:`engine_for` refuses anything that is not a CUDA
tensor, and :func:`_lib.load` raises when the CUDA library has not been built.
"""

from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional

import torch

from . import _lib
from ._lib import ActT, BnBwdT, CsrT, EvalLayerT, StoreT


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    """Device pointer of a tensor (None -> NULL).  Tensors must be contiguous."""
    if t is None:
        return None
    assert t.is_contiguous(), "cgnn kernels take dense row-major tensors"
    return t.data_ptr()


@dataclass
class Act:
    """Host mirror of ``cgnn_act_t``: how a stored tensor becomes a layer input on load."""
    scale: Optional[torch.Tensor] = None
    shift: Optional[torch.Tensor] = None
    relu: bool = False
    p_drop: float = 0.0
    seed: int = 0
    site: int = 0
    row_base: int = 0
    salt: Optional[torch.Tensor] = None    # device words folded into the mask stream (graphed steps), see cgnn_act_t

    def struct(self) -> ActT:
        return ActT(_p(self.scale), _p(self.shift), int(self.relu), float(self.p_drop),
                    int(self.seed) & 0xFFFFFFFFFFFFFFFF, int(self.site) & 0xFFFFFFFF, int(self.row_base), _p(self.salt))


@dataclass
class BnBwd:
    """Host mirror of ``cgnn_bn_bwd_t``."""
    scale: torch.Tensor
    mean: torch.Tensor
    rstd: torch.Tensor
    sums: Optional[torch.Tensor]   # [2, C]: sum dy, sum dy*xhat (global batch)
    count: float
    train: bool
    sums64: Optional[torch.Tensor] = None   # the same in float64: what the kernels read when given (see cgnn_bn_bwd_t)

    def struct(self) -> BnBwdT:
        s1 = s2 = None
        if self.sums is not None:
            c = self.scale.shape[0]
            base = self.sums.data_ptr()
            s1, s2 = base, base + 4 * c
        return BnBwdT(_p(self.scale), _p(self.mean), _p(self.rstd), s1, s2, float(self.count), int(self.train), _p(self.sums64))


_EVAL_ARRAYS: dict = {}


def _eval_layer_array(n: int):
    """ctypes array types are created per ``T * n`` expression and each one sits in a reference cycle: keep one per n."""
    t = _EVAL_ARRAYS.get(n)
    if t is None:
        t = _EVAL_ARRAYS[n] = EvalLayerT * n
    return t


class Engine:
    """Binds a loaded ABI library to one device: workspace, stream lookup, call wrappers."""

    def __init__(self, lib: C.CDLL, device: torch.device):
        self.lib = lib
        self.device = torch.device(device)
        # CUDA ordinal the C side must see as current (None: the test-only simulator engine, host pointers)
        self._index = None if self.device.type != "cuda" else (
            self.device.index if self.device.index is not None else torch.cuda.current_device())
        self.workspace_bytes = int(lib.cgnn_workspace_bytes())
        self.workspace = torch.empty(self.workspace_bytes, dtype=torch.uint8, device=self.device)
        self.launches = 0  # C-ABI calls issued (each enqueues >= 1 kernel); bench reports kernel counts separately

    # -- plumbing -------------------------------------------------------------------------
    def stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _call(self, name: str, *args) -> None:
        """One ABI call with this engine's device current: the C side launches on the *current* device and sizes its
        grids from it, so a batch on cuda:1 while cuda:0 is current must switch first (no-op when already current)."""
        self.launches += 1
        if self._index is not None and torch.cuda.current_device() != self._index:
            with torch.cuda.device(self._index):
                _lib.check(self.lib, getattr(self.lib, name)(*args), name)
        else:
            _lib.check(self.lib, getattr(self.lib, name)(*args), name)

    def empty(self, shape, dtype=torch.float32) -> torch.Tensor:
        return torch.empty(shape, dtype=dtype, device=self.device)

    # -- K0 ---------------------------------------------------------------------------------
    def new_csr(self, rows: int, edges: int, graphs: int) -> dict:
        # a batch without a single edge still gets one (unused) element per edge array: the C side reads a NULL array as
        # "not materialised" (a lean batch), and the data_ptr() of an empty tensor - even a view - is NULL
        e = lambda n, dtype=torch.float32: self.empty(max(n, 1), dtype)
        return dict(
            graph_meta=self.empty((graphs, 4), torch.int32),
            in_rowptr=e(rows + 1, torch.int32), in_col=e(edges, torch.int32), in_w=e(edges), in_wn=e(edges),
            out_rowptr=e(rows + 1, torch.int32), out_col=e(edges, torch.int32), out_w=e(edges), out_wn=e(edges),
            deg=e(rows), dinv=e(rows), wsum=e(rows))

    KINDS = {"gcn": 0, "sage": 1}

    ARRAYS = ("in_rowptr", "in_col", "in_w", "in_wn", "out_rowptr", "out_col", "out_w", "out_wn", "deg", "dinv", "wsum")

    @staticmethod
    def csr_struct(c, kind: Optional[str] = None) -> CsrT:
        """``cgnn_csr_t`` of a CSR (dict or BatchCSR); ``kind`` attaches that model family's aggregation blobs.
        A lean BatchCSR passes NULL for every array it has not materialised (``peek`` never triggers the lazy collate)."""
        g = (lambda k: c[k]) if isinstance(c, dict) else c.peek
        base = [_p(g(k)) for k in Engine.ARRAYS + ("graph_meta",)]
        blobs = None if (kind is None or isinstance(c, dict)) else (getattr(c, "agg", None) or {}).get(kind)
        if blobs is None:
            return CsrT(*base, None, None, None, -1)
        return CsrT(*base, _p(blobs[0]), _p(blobs[1]), _p(blobs[2]), Engine.KINDS[kind])

    def ensure_agg(self, csr, kind: str, num_graphs: int, rows: int, edges: int, need_out: bool = True):
        """Packed aggregation blobs of one model family for this batch (built once, cached on the CSR).  ``need_out``:
        the by-source blob (backward) is wanted too - a forward-only batch carries the by-destination blob alone."""
        if getattr(csr, "agg", None) is None:
            csr.agg = {}
        have = csr.agg.get(kind)
        if have is None or (need_out and have[1] is None):
            csr.materialize()            # the stand-alone builder reads the CSR arrays (no-op for a full batch)
            words = int(self.lib.cgnn_agg_words(rows, edges, num_graphs))
            agg_in, agg_out = self.empty(words, torch.int32), self.empty(words, torch.int32)
            row_graph = self.empty(max(rows, 1), torch.int32)
            cs = self.csr_struct(csr)
            self._call("cgnn_build_agg", C.byref(cs), Engine.KINDS[kind], num_graphs, rows, edges, csr.max_nodes,
                       _p(agg_in), _p(agg_out), _p(row_graph), self.stream())
            csr.agg[kind] = (agg_in, agg_out, row_graph)
        return csr.agg[kind]

    def _call_csr(self, name: str, csr, build_args) -> None:
        """An ABI call that takes a ``cgnn_csr_t``: a lean batch that hits a code path reading the CSR arrays
        (CGNN_ERR_NEED_CSR) materialises them once and the call is repeated."""
        try:
            self._call(name, *build_args())
        except _lib.CgnnError as e:
            if e.status != _lib.ERR_NEED_CSR or csr.is_full():
                raise
            csr.materialize()
            self._call(name, *build_args())

    def collate_csr(self, store: StoreT, ids: torch.Tensor, num_graphs: int, rows: int, edges: int, max_nodes: int,
                    max_edges: int, num_features: int, with_labels: bool, agg_kind: Optional[str] = None,
                    lean: bool = False, need_out: bool = True):
        """Returns (fields, csr arrays, blobs): ``blobs`` = (agg_in, agg_out, row_graph) of ``agg_kind`` when the
        collate kernel was asked to emit that model family's aggregation blobs in the same pass, else None.
        ``lean`` (with ``agg_kind``): only node_features, labels, ptr / eptr, graph_meta and the blobs are written -
        the COO fields, ``batch`` and every CSR array come back as None; ``need_out`` = False drops the by-source blob
        (forward-only batches).  Falls back to a full collate when the kernel cannot stage the largest subject."""
        e = self.empty
        lean = lean and agg_kind is not None and num_graphs > 0 and rows > 0
        if lean:
            out = dict(node_features=e((rows, num_features)), edge_index=None, edge_weight=None, batch=None,
                       labels=e(num_graphs, torch.int64) if with_labels else None,
                       ptr=e(num_graphs + 1, torch.int64), eptr=e(num_graphs + 1, torch.int64))
            csr = {k: None for k in Engine.ARRAYS}
            csr["graph_meta"] = e((num_graphs, 4), torch.int32)
        else:
            out = dict(
                node_features=e((rows, num_features)), edge_index=e((2, edges), torch.int64), edge_weight=e(edges),
                batch=e(rows, torch.int64), labels=e(num_graphs, torch.int64) if with_labels else None,
                ptr=e(num_graphs + 1, torch.int64), eptr=e(num_graphs + 1, torch.int64))
            csr = self.new_csr(rows, edges, num_graphs)
        cs = self.csr_struct(csr)
        blobs = None
        if agg_kind is not None and num_graphs > 0 and rows > 0:
            words = int(self.lib.cgnn_agg_words(rows, edges, num_graphs))
            blobs = (e(words, torch.int32), e(words, torch.int32) if (need_out or not lean) else None,
                     e(max(rows, 1), torch.int32))
            cs.agg_in, cs.agg_out, cs.row_graph = _p(blobs[0]), _p(blobs[1]), _p(blobs[2])
            cs.agg_kind = Engine.KINDS[agg_kind]
        try:
            self._call("cgnn_collate_csr", C.byref(store), _p(ids), num_graphs, rows, edges, max_nodes, max_edges,
                       _p(out["node_features"]), _p(out["edge_index"]), _p(out["edge_weight"]), _p(out["batch"]),
                       _p(out["labels"]), _p(out["ptr"]), _p(out["eptr"]), C.byref(cs), self.stream())
        except _lib.CgnnError as err:
            if not lean or err.status != _lib.ERR_NEED_CSR:
                raise
            return self.collate_csr(store, ids, num_graphs, rows, edges, max_nodes, max_edges, num_features, with_labels,
                                    agg_kind, lean=False)
        return out, csr, blobs

    def csr_from_coo(self, edge_index, edge_weight, ptr, num_graphs: int, rows: int, edges: int, max_nodes: int):
        csr = self.new_csr(rows, edges, num_graphs)
        eptr = self.empty(num_graphs + 1, torch.int64)
        cs = self.csr_struct(csr)
        self._call("cgnn_csr_from_coo", _p(edge_index), _p(edge_weight), _p(ptr), num_graphs, rows, edges,
                   max_nodes, _p(eptr), C.byref(cs), self.stream())
        return csr, eptr

    # -- K1 / K2 ------------------------------------------------------------------------------
    def layer_fwd(self, kind: str, t_in, act: Act, W, bias, csr, ptr, num_graphs: int, want_stats: bool):
        """Returns (z, stats, agg): ``agg`` is GraphSAGE's aggregated neighbourhood [rows, d_in] (kept for backward)."""
        rows, d_in = t_in.shape
        H = W.shape[0]
        if W.shape[1] != (2 * d_in if kind == "sage" else d_in):
            raise RuntimeError(f"{kind} layer: input has {d_in} channels but the weight is {tuple(W.shape)}")
        z = self.empty((rows, H))
        stats = self.empty(1 + 2 * H, torch.float64) if want_stats else None
        self.ensure_agg(csr, kind, num_graphs, rows, csr.num_edges, need_out=False)
        a = act.struct()
        agg = self.empty((rows, d_in)) if kind == "sage" else None

        def build():
            cs = self.csr_struct(csr, kind)
            keep.append(cs)
            args = [_p(t_in), C.byref(a), _p(W), _p(bias), C.byref(cs), _p(ptr), num_graphs, rows, d_in, H, csr.max_nodes,
                    csr.max_edges, _p(z), _p(stats)]
            if kind == "sage":
                args.append(_p(agg))
            return args + [_p(self.workspace), self.workspace_bytes, self.stream()]

        keep: list = []
        self._call_csr(f"cgnn_{kind}_layer_fwd", csr, build)
        return z, stats, agg

    def gcn_layer_fwd_pool(self, t_in, act: Act, W, bias, csr, ptr, num_graphs: int, act_out: Act):
        """Eval-mode last GCN layer with its BatchNorm affine + ReLU and the mean-pool readout folded into the kernel:
        returns emb [B, H], or None when the shape is not covered (the caller runs layer_fwd + pool_fwd)."""
        rows, d_in = t_in.shape
        H = W.shape[0]
        if W.shape[1] != d_in:
            raise RuntimeError(f"gcn layer: input has {d_in} channels but the weight is {tuple(W.shape)}")
        self.ensure_agg(csr, "gcn", num_graphs, rows, csr.num_edges, need_out=False)
        emb = self.empty((num_graphs, H))
        a, ao = act.struct(), act_out.struct()
        cs = self.csr_struct(csr, "gcn")
        try:
            self._call("cgnn_gcn_layer_fwd_pool", _p(t_in), C.byref(a), _p(W), _p(bias), C.byref(cs), _p(ptr), num_graphs, rows,
                       d_in, H, csr.max_nodes, csr.max_edges, C.byref(ao), _p(emb), self.stream())
        except _lib.CgnnError as e:
            if e.status == _lib.ERR_UNSUPPORTED:
                return None
            raise
        return emb

    # -- K9 -------------------------------------------------------------------------------------
    def eval_fused(self, kind: str, x, layers, head, csr, ptr, num_graphs: int, want_logits: bool = True):
        """The whole eval-mode network in one kernel.  ``layers`` = [(W, bias, gamma, beta, running_mean, running_var,
        eps), ...], ``head`` = (W0, b0, W1, b1).  Returns (emb, logits), or None when the shape is not covered (the
        caller then runs the per-layer entry points)."""
        rows, F = x.shape
        H = layers[0][0].shape[0]
        W0, b0, W1, b1 = head
        M, K = W0.shape[0], W1.shape[0]
        if kind != "gcn" or num_graphs == 0 or rows == 0:
            return None
        self.ensure_agg(csr, kind, num_graphs, rows, csr.num_edges, need_out=False)
        arr = _eval_layer_array(len(layers))()
        for i, (W, b, g, be, rm, rv, eps) in enumerate(layers):
            arr[i] = EvalLayerT(_p(W), _p(b), _p(g), _p(be), _p(rm), _p(rv), float(eps))
        emb = self.empty((num_graphs, H))
        logits = self.empty((num_graphs, K)) if want_logits else None
        cs = self.csr_struct(csr, kind)
        try:
            self._call("cgnn_eval_fused_fwd", Engine.KINDS[kind], _p(x), F, arr, len(layers), H, _p(W0), _p(b0), _p(W1), _p(b1),
                       M, K, C.byref(cs), _p(ptr), num_graphs, rows, csr.max_nodes, csr.max_edges, _p(emb), _p(logits),
                       _p(self.workspace), self.workspace_bytes, self.stream())
        except _lib.CgnnError as e:
            if e.status == _lib.ERR_UNSUPPORTED:
                return None
            raise
        return emb, logits

    def project_tf32x3(self, X, W):
        """P = X W^T on the tensor cores (3xTF32, fp32-grade)."""
        rows, K = X.shape
        N = W.shape[0]
        P = self.empty((rows, N))
        self._call("cgnn_project_tf32x3", _p(X), _p(W), rows, K, N, _p(P), self.stream())
        return P

    # -- K3 -------------------------------------------------------------------------------------
    def bn_merge_stats(self, parts: torch.Tensor, C_: int) -> torch.Tensor:
        out = self.empty(1 + 2 * C_, torch.float64)
        self._call("cgnn_bn_merge_stats", _p(parts), parts.shape[0], C_, _p(out), self.stream())
        return out

    def bn_finalize(self, stats, gamma, beta, eps: float, momentum: float, running_mean, running_var, nbt):
        C_ = gamma.shape[0]
        scale, shift, mean, rstd = (self.empty(C_) for _ in range(4))
        self._call("cgnn_bn_finalize", _p(stats), _p(gamma), _p(beta), C_, eps, momentum, _p(running_mean),
                   _p(running_var), _p(nbt), _p(scale), _p(shift), _p(mean), _p(rstd), self.stream())
        return scale, shift, mean, rstd

    def bn_eval_affine(self, gamma, beta, running_mean, running_var, eps: float):
        C_ = gamma.shape[0]
        scale, shift, mean, rstd = (self.empty(C_) for _ in range(4))
        self._call("cgnn_bn_eval_affine", _p(gamma), _p(beta), _p(running_mean), _p(running_var), C_, eps,
                   _p(scale), _p(shift), _p(mean), _p(rstd), self.stream())
        return scale, shift, mean, rstd

    # -- K4 -------------------------------------------------------------------------------------
    def pool_fwd(self, t_in, act: Act, ptr, num_graphs: int):
        rows, C_ = t_in.shape
        emb = self.empty((num_graphs, C_))
        a = act.struct()
        self._call("cgnn_pool_fwd", _p(t_in), C.byref(a), _p(ptr), num_graphs, rows, C_, _p(emb), self.stream())
        return emb

    def head_fwd(self, emb, W0, b0, W1, b1, p_drop: float, seed: int, graph_base: int, salt=None):
        B, C_ = emb.shape
        M, K = W0.shape[0], W1.shape[0]
        hidden, logits = self.empty((B, M)), self.empty((B, K))
        self._call("cgnn_head_fwd", _p(emb), _p(W0), _p(b0), _p(W1), _p(b1), B, C_, M, K, float(p_drop),
                   int(seed) & 0xFFFFFFFFFFFFFFFF, int(graph_base), _p(salt), _p(hidden), _p(logits), self.stream())
        return hidden, logits

    # -- the step after backward -----------------------------------------------------------------
    def step_tick(self, state: torch.Tensor) -> None:
        self._call("cgnn_step_tick", _p(state), self.stream())

    def adam_step(self, param, grad, exp_avg, exp_avg_sq, lr, beta1, beta2, eps, weight_decay, state) -> None:
        self._call("cgnn_adam_step", _p(param), _p(grad), _p(exp_avg), _p(exp_avg_sq), param.numel(), float(lr), float(beta1),
                   float(beta2), float(eps), float(weight_decay), _p(state), self.stream())

    def ce_fwd(self, logits, labels, inv_count: float):
        B, K = logits.shape
        nll, loss, correct = self.empty(B), self.empty(()), self.empty((), torch.int64)
        self._call("cgnn_ce_fwd", _p(logits), _p(labels), B, K, float(inv_count), _p(nll), _p(loss), _p(correct),
                   self.stream())
        return loss, nll, correct

    # -- K5..K7 -----------------------------------------------------------------------------------
    def ce_bwd(self, logits, labels, inv_count: float, gout):
        B, K = logits.shape
        d = self.empty((B, K))
        self._call("cgnn_ce_bwd", _p(logits), _p(labels), B, K, float(inv_count), _p(gout), _p(d), self.stream())
        return d

    def head_bwd(self, emb, hidden, dlogits, W0, W1, p_drop: float, out=None):
        B, C_ = emb.shape
        M, K = W0.shape[0], W1.shape[0]
        demb = self.empty((B, C_))
        dW0, db0, dW1, db1 = out if out is not None else (self.empty((M, C_)), self.empty(M), self.empty((K, M)), self.empty(K))
        self._call("cgnn_head_bwd", _p(emb), _p(hidden), _p(dlogits), _p(W0), _p(W1), B, C_, M, K, float(p_drop),
                   _p(demb), _p(dW0), _p(db0), _p(dW1), _p(db1), _p(self.workspace), self.workspace_bytes,
                   self.stream())
        return demb, dW0, db0, dW1, db1

    def bn_bwd_sums(self, z, act: Act, mean, rstd, du, demb, ptr, num_graphs: int, out=None):
        rows, C_ = z.shape
        sums = out if out is not None else self.empty((2, C_))
        sums64 = self.empty((2, C_), torch.float64)
        a = act.struct()
        self._call("cgnn_bn_bwd_sums", _p(z), C.byref(a), _p(mean), _p(rstd), _p(du), _p(demb), _p(ptr),
                   num_graphs, rows, C_, _p(sums), _p(sums64), _p(self.workspace), self.workspace_bytes, self.stream())
        return sums, sums64

    def layer_bwd(self, kind: str, du, demb, z, act_out: Act, bn: Optional[BnBwd], t_in, act_in: Act, W, csr, ptr,
                  num_graphs: int, need_du: bool, prev_mean, prev_rstd, agg=None, out=None, prev_out=None):
        """``out`` = (dW, db) and ``prev_out`` = the [2, d_in] BatchNorm-backward sums of the layer below, preallocated
        (views of a flat gradient buffer), or None."""
        rows, d_in = t_in.shape
        H = z.shape[1]
        dW, db = out if out is not None else (self.empty(W.shape), self.empty(H))
        du_in = self.empty((rows, d_in)) if need_du else None
        want_prev = need_du and prev_mean is not None
        prev_sums = (prev_out if prev_out is not None else self.empty((2, d_in))) if want_prev else None
        prev_sums64 = self.empty((2, d_in), torch.float64) if want_prev else None
        self.ensure_agg(csr, kind, num_graphs, rows, csr.num_edges, need_out=True)
        ao, ai = act_out.struct(), act_in.struct()
        bs = bn.struct() if bn is not None else None
        # scratch between the kernels of one call: GCN dP [rows, H]; GraphSAGE [2, rows, d_in] (d_u, d_agg), and a third
        # [rows, H] plane (dz) for the wide layers (H = d_in = 256)
        scratch = self.empty((rows, H)) if kind == "gcn" else self.empty((3 if (H == 256 and d_in == 256) else 2, rows, d_in))

        def build():
            cs = self.csr_struct(csr, kind)
            keep.append(cs)
            args = [_p(du), _p(demb), _p(z), C.byref(ao), C.byref(bs) if bs is not None else None, _p(t_in)]
            if kind == "sage":
                args.append(_p(agg))
            args += [C.byref(ai), _p(W), C.byref(cs), _p(ptr), num_graphs, rows, d_in, H, csr.max_nodes, csr.max_edges,
                     _p(dW), _p(db),
                     _p(du_in), _p(prev_mean) if want_prev else None, _p(prev_rstd) if want_prev else None,
                     _p(prev_sums), _p(prev_sums64)]
            return args + [_p(scratch), _p(self.workspace), self.workspace_bytes, self.stream()]

        keep: list = []
        self._call_csr(f"cgnn_{kind}_layer_bwd", csr, build)
        return dW, db, du_in, prev_sums, prev_sums64


_ENGINES: dict = {}


def engine_for(t: torch.Tensor) -> Engine:
    """The engine of the CUDA device `t` lives on.  No CUDA tensor, no engine: there is no CPU path."""
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(
            "connectome_gnn (B200 build) computes on CUDA only: got a "
            f"{'non-tensor' if not isinstance(t, torch.Tensor) else t.device.type} input. "
            "Move the batch with .to('cuda'); there is no CPU fallback.")
    dev = t.device
    eng = _ENGINES.get(dev)
    if eng is None:
        eng = _ENGINES[dev] = Engine(_lib.load(), dev)
    return eng


def default_device() -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("connectome_gnn (B200 build) needs a CUDA device; none is visible and there is no CPU path")
    return torch.device("cuda", torch.cuda.current_device())

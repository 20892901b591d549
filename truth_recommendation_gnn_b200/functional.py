"""``torch.autograd.Function`` wrappers around the C ABI (include/trg_b200.h).

Each function names the reference lines it replaces; all arithmetic on the hot path happens in
the sm_100a kernels -- torch supplies memory, the stream and the autograd tape.
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib, fp8
from .graph import CSR, RelationGraph, build_csr


def _long_rows_arg(csr: CSR, feat: int, dev, elem_size: int = 4):
    """ctypes ``trg_long_rows`` (+ the tensors it points to, to keep them alive) or ``(None, None)``.
    Splitting needs rows of at least 80 bytes in the table's own dtype (gather.cu ``apply_long``); narrower
    rows run unsplit -- splitting is a load-balance measure, results do not depend on it."""
    lr = csr.long_rows() if feat * elem_size >= 80 else None
    if lr is None:
        return None, None
    partial = torch.empty(lr.n_slots, feat, dtype=torch.float32, device=dev)
    s = _lib.TrgLongRows(_lib.ptr(lr.vrowptr), _lib.ptr(lr.vinfo), int(lr.vinfo.numel()), _lib.ptr(lr.long_rows),
                         _lib.ptr(lr.long_ptr), int(lr.long_rows.numel()), _lib.ptr(partial))
    return ctypes.byref(s), (s, partial)


def _check_rows(x: torch.Tensor, what: str):
    es = x.element_size()
    if x.dim() != 2 or (x.size(1) * es) % 16 != 0:
        raise _lib.TrgError(f"{what}: rows must be a multiple of 16 bytes (got shape {tuple(x.shape)}, "
                            f"{x.dtype}); pad the feature width (the reference pads to 64, inference.py:401-404)")


# ------------------------------------------------------------------------------------------
# K1 / K2: SAGEConv propagate + mean aggregation
# ------------------------------------------------------------------------------------------
def sage_agg_fwd(csr: CSR, x_src: torch.Tensor, want_inv_deg: bool = True):
    """mean over in-neighbours (train_gnn.py:177-184,194-197 -> PyG propagate/MeanAggregation)."""
    lib = _lib.load()
    _check_rows(x_src, "sage_agg_fwd")
    x_src = x_src.contiguous()
    out = torch.empty(csr.n_rows, x_src.size(1), dtype=x_src.dtype, device=x_src.device)
    inv_deg = torch.empty(csr.n_rows, dtype=torch.float32, device=x_src.device) if want_inv_deg else None
    if csr.n_rows:
        rb = x_src.size(1) * x_src.element_size()
        nbytes = csr.n_edges * (rb + 4) + 4 * (csr.n_rows + 1) + csr.n_rows * rb
        lr, keep = _long_rows_arg(csr, x_src.size(1), x_src.device, x_src.element_size())
        _lib.call("trg_sage_agg_fwd", nbytes, lib.trg_sage_agg_fwd,
                  _lib.ptr(csr.rowptr), _lib.ptr(csr.col), _lib.ptr(x_src), csr.n_rows, x_src.size(1),
                  _lib.dtype_code(x_src.dtype), _lib.ptr(out), _lib.ptr(inv_deg), lr, _lib.stream())
    return out, inv_deg


def _check_epilogue(out, relu_of, n_rows, x, who, out_dtype=None):
    for t, what, dt in ((out, "out", out_dtype or x.dtype), (relu_of, "relu_of", x.dtype)):
        if t is not None and (t.shape != (n_rows, x.size(1)) or t.dtype != dt or not t.is_contiguous()
                              or t.device != x.device):
            raise _lib.TrgError(f"{who}: {what} must be a contiguous [{n_rows}, {x.size(1)}] {dt} tensor")


def _out_dtype(x, out, out_dtype):
    """``out_dtype``: None = the table's dtype; ``torch.float32`` with a bf16 table = fp32 sum rows (partials
    a multi-GPU run reduces across ranks before the single rounding to bf16)."""
    if out_dtype is None:
        out_dtype = out.dtype if out is not None else x.dtype
    if out_dtype != x.dtype and not (x.dtype == torch.bfloat16 and out_dtype == torch.float32):
        raise _lib.TrgError(f"output dtype {out_dtype} is not supported for a {x.dtype} table")
    return out_dtype


def sage_agg_bwd(csr_t: CSR, inv_deg, g_mean: torch.Tensor, out=None, accumulate=False, relu_of=None,
                 out_dtype=None):
    """Atomic-free gradient w.r.t. the source table through the transposed CSR.  ``out`` +
    ``accumulate`` add to gradient rows already computed (a table feeding several relations);
    ``relu_of`` gates the final rows by ``relu_of > 0`` (the producing layer's ReLU backward)."""
    lib = _lib.load()
    g_mean = g_mean.contiguous()
    _check_rows(g_mean, "sage_agg_bwd")
    out_dtype = _out_dtype(g_mean, out, out_dtype)
    _check_epilogue(out, relu_of, csr_t.n_rows, g_mean, "sage_agg_bwd", out_dtype)
    if out is None:
        out = torch.empty(csr_t.n_rows, g_mean.size(1), dtype=out_dtype, device=g_mean.device)
        accumulate = False
    if csr_t.n_rows:
        rb = g_mean.size(1) * g_mean.element_size()
        ob = g_mean.size(1) * out.element_size()
        nbytes = (csr_t.n_edges * (rb + 4) + 4 * (csr_t.n_rows + 1)
                  + csr_t.n_rows * (ob * (1 + bool(accumulate)) + rb * (relu_of is not None))
                  + (4 * csr_t.n_cols if inv_deg is not None else 0))
        lr, keep = _long_rows_arg(csr_t, g_mean.size(1), g_mean.device, g_mean.element_size())
        _lib.call("trg_sage_agg_bwd", nbytes, lib.trg_sage_agg_bwd,
                  _lib.ptr(csr_t.rowptr), _lib.ptr(csr_t.col), _lib.ptr(inv_deg), _lib.ptr(g_mean),
                  csr_t.n_rows, g_mean.size(1), _lib.dtype_code(g_mean.dtype), _lib.ptr(out),
                  _lib.dtype_code(out_dtype), 1 if accumulate else 0, _lib.ptr(relu_of), lr, _lib.stream())
    return out


class SageAggFn(torch.autograd.Function):
    """mean aggregation.  ``grad_prescaled``: the incoming gradient has already been multiplied
    row-wise by 1/deg (fused into the projection backward's epilogue), so the backward is a plain
    transposed gather-sum."""

    @staticmethod
    def forward(ctx, x_src, rel: RelationGraph, grad_prescaled: bool = False):
        want_inv = rel.inv_deg is None
        mean, inv_deg = sage_agg_fwd(rel.fwd, x_src, want_inv_deg=want_inv)
        if want_inv:
            rel.inv_deg = inv_deg          # static per relation: computed by the first forward
        ctx.rel = rel
        ctx.grad_prescaled = grad_prescaled
        return mean

    @staticmethod
    def backward(ctx, g_mean):
        if not ctx.needs_input_grad[0]:
            return None, None, None
        rel = ctx.rel
        return sage_agg_bwd(rel.bwd, None if ctx.grad_prescaled else rel.inv_deg, g_mean), None, None


def sage_mean_aggregate(x_src: torch.Tensor, rel: RelationGraph, grad_prescaled: bool = False) -> torch.Tensor:
    return SageAggFn.apply(x_src, rel, grad_prescaled)


# ------------------------------------------------------------------------------------------
# generic weighted gather-sum
# ------------------------------------------------------------------------------------------
def gather_wsum(csr: CSR, coef, x: torch.Tensor, scale=None, out=None, accumulate=False, relu_of=None,
                out_dtype=None):
    lib = _lib.load()
    x = x.contiguous()
    _check_rows(x, "gather_wsum")
    out_dtype = _out_dtype(x, out, out_dtype)
    _check_epilogue(out, relu_of, csr.n_rows, x, "gather_wsum", out_dtype)
    if out is None:
        out = torch.empty(csr.n_rows, x.size(1), dtype=out_dtype, device=x.device)
        accumulate = False
    if csr.n_rows:
        rb = x.size(1) * x.element_size()
        ob = x.size(1) * out.element_size()
        nbytes = (csr.n_edges * (rb + 12) + 4 * (csr.n_rows + 1)
                  + csr.n_rows * (ob * (1 + bool(accumulate)) + rb * (relu_of is not None)))
        lr, keep = _long_rows_arg(csr, x.size(1), x.device, x.element_size())
        _lib.call("trg_gather_wsum", nbytes, lib.trg_gather_wsum,
                  _lib.ptr(csr.rowptr), _lib.ptr(csr.col), _lib.ptr(csr.eid), _lib.ptr(coef),
                  _lib.ptr(scale), _lib.ptr(x), csr.n_rows, x.size(1), _lib.dtype_code(x.dtype),
                  _lib.ptr(out), _lib.dtype_code(out_dtype), 1 if accumulate else 0, _lib.ptr(relu_of), lr,
                  _lib.stream())
    return out


def rows_finish(x, dtype, row_scale=None, add=None, relu_of=None, out=None):
    """``out = gate(row_scale[:, None] * x + add)`` rounded once to ``dtype`` (``trg_rows_finish``): the
    owned rows of a table reduced across GPUs -- 1/deg of a source-partitioned mean, the local gradient
    term, the ReLU backward -- in one pass.  ``x`` is fp32 (fp32-transported partial sums) or ``dtype``."""
    lib = _lib.load()
    x = x.contiguous()
    n, feat = x.shape
    if x.dtype != dtype and x.dtype != torch.float32:
        raise _lib.TrgError(f"rows_finish: input must be {dtype} or float32, got {x.dtype}")
    for t, what in ((add, "add"), (relu_of, "relu_of"), (out, "out")):
        if t is not None and (t.shape != x.shape or t.dtype != dtype or not t.is_contiguous()):
            raise _lib.TrgError(f"rows_finish: {what} must be a contiguous [{n}, {feat}] {dtype} tensor")
    if out is None:
        out = torch.empty(n, feat, dtype=dtype, device=x.device)
    _check_rows(out, "rows_finish")
    rs = row_scale.float().contiguous() if row_scale is not None else None
    es = out.element_size()
    nbytes = n * feat * (x.element_size() + es * (1 + (add is not None) + (relu_of is not None)))
    _lib.call("trg_rows_finish", nbytes, lib.trg_rows_finish, _lib.ptr(x), _lib.dtype_code(x.dtype), _lib.ptr(rs),
              _lib.ptr(add), _lib.ptr(relu_of), n, feat, _lib.dtype_code(dtype), _lib.ptr(out), _lib.stream())
    return out


def peer_reduce_rows(parts, row0, n_rows, dtype, row_scale=None, add=None, relu_of=None, ctas_per_sm=0):
    """``gate(row_scale * sum_g parts[g][row0:row0+n_rows] + add)`` rounded once to ``dtype``
    (``trg_peer_reduce_rows``): the reduce-scatter of a partial-sum table fused with its row finish.
    ``parts``: one ``[>= row0 + n_rows, feat]`` table per rank, in rank order -- tensors of this device or of
    peers (``peer.PeerComm`` passes raw peer-mapped pointers instead); fp32 or ``dtype``."""
    import ctypes
    lib = _lib.load()
    feat = parts[0].size(1)
    for t in parts:
        if t.dtype != parts[0].dtype or t.size(1) != feat or t.size(0) < row0 + n_rows or not t.is_contiguous():
            raise _lib.TrgError("peer_reduce_rows: partial tables must be contiguous, of one dtype and width, and "
                                "hold rows [row0, row0 + n_rows)")
    if parts[0].dtype != dtype and parts[0].dtype != torch.float32:
        raise _lib.TrgError(f"peer_reduce_rows: partial tables must be {dtype} or float32")
    for t, what in ((add, "add"), (relu_of, "relu_of")):
        if t is not None and (tuple(t.shape) != (n_rows, feat) or t.dtype != dtype or not t.is_contiguous()):
            raise _lib.TrgError(f"peer_reduce_rows: {what} must be a contiguous [{n_rows}, {feat}] {dtype} tensor")
    out = torch.empty(n_rows, feat, dtype=dtype, device=parts[0].device)
    _check_rows(out, "peer_reduce_rows")
    rs = row_scale.float().contiguous() if row_scale is not None else None
    ptrs = (ctypes.c_void_p * len(parts))(*[_lib.ptr(t) for t in parts])
    nbytes = n_rows * feat * (len(parts) * parts[0].element_size()
                              + out.element_size() * (1 + (add is not None) + (relu_of is not None)))
    _lib.call("trg_peer_reduce_rows", nbytes, lib.trg_peer_reduce_rows, ptrs, len(parts), row0,
              _lib.dtype_code(parts[0].dtype), _lib.ptr(rs), _lib.ptr(add), _lib.ptr(relu_of), n_rows, feat,
              _lib.dtype_code(dtype), _lib.ptr(out), ctas_per_sm, _lib.stream())
    return out


# ------------------------------------------------------------------------------------------
# K4: link-prediction loss (train_gnn.py:259-281) and its backward
# ------------------------------------------------------------------------------------------
class LinkStructure:
    """Static structures of the positive edge set: edges grouped by user and by post, and
    wbar = mean(interaction_type_tensor[pos_p + num_users]) (train_gnn.py:266-269,280)."""

    def __init__(self, train_edge_index, interaction_type_tensor, num_users, num_posts):
        pos_u, pos_p = train_edge_index[0], train_edge_index[1]
        self.train_edge_index = train_edge_index
        self.num_users, self.num_posts = int(num_users), int(num_posts)
        self.n_edges = int(pos_u.numel())
        self.by_user = build_csr(pos_p, pos_u, self.num_users, self.num_posts)
        self.by_post = build_csr(pos_u, pos_p, self.num_posts, self.num_users, validate=False)
        self._by_post_u = None
        self._user_of_u = None
        if self.n_edges:
            w = interaction_type_tensor[pos_p + num_users].float()
            self.wbar = w.mean().reshape(1).contiguous()
        else:
            self.wbar = torch.full((1,), float("nan"), device=pos_u.device)


    @property
    def by_post_u(self) -> CSR:
        """``by_post`` whose edge ids are BY-USER CSR POSITIONS instead of original edge positions, so
        that per-edge coefficients the user-anchored loss pass wrote sequentially (in by-user order) can
        be looked up by the post-side gather.  Static: one inverse permutation at cache-fill time."""
        if self._by_post_u is None:
            bu, bp = self.by_user, self.by_post
            inv = torch.empty(self.n_edges, dtype=torch.int32, device=bu.eid.device)
            inv[bu.eid.long()] = torch.arange(self.n_edges, dtype=torch.int32, device=bu.eid.device)
            self._by_post_u = CSR(bp.rowptr, bp.col, inv[bp.eid.long()].contiguous(), bp.n_rows, bp.n_cols, bp._long)
        return self._by_post_u

    @property
    def user_of_u(self) -> torch.Tensor:
        """int64 user id of the edge at each by-user CSR position (the expanded ``by_user.rowptr``)."""
        if self._user_of_u is None:
            rp = self.by_user.rowptr.long()
            self._user_of_u = torch.repeat_interleave(
                torch.arange(self.num_users, device=rp.device), rp[1:] - rp[:-1]).contiguous()
        return self._user_of_u


_LINK_CACHE: dict = {}


def link_structure(train_edge_index, interaction_type_tensor, num_users, num_posts) -> LinkStructure:
    key = (train_edge_index.data_ptr(), tuple(train_edge_index.shape), train_edge_index._version,
           interaction_type_tensor.data_ptr(), interaction_type_tensor._version, int(num_users),
           int(num_posts))
    s = _LINK_CACHE.get(key)
    if s is None:
        if len(_LINK_CACHE) > 8:
            _LINK_CACHE.clear()
        s = LinkStructure(train_edge_index, interaction_type_tensor, num_users, num_posts)
        s._keepalive = interaction_type_tensor
        _LINK_CACHE[key] = s
    return s


def edge_bce_fwd(ls: LinkStructure, user_emb, post_emb, neg_p, want_grad: bool):
    lib = _lib.load()
    _check_rows(user_emb, "edge_bce_fwd")
    if user_emb.dtype != post_emb.dtype or user_emb.size(1) != post_emb.size(1):
        raise _lib.TrgError("user and post embeddings must share dtype and width")
    if neg_p.dtype != torch.int64 or neg_p.numel() != ls.n_edges:
        raise _lib.TrgError("neg_p must be int64 with one entry per positive edge (train_gnn.py:272)")
    user_emb, post_emb, neg_p = user_emb.contiguous(), post_emb.contiguous(), neg_p.contiguous()
    dev = user_emb.device
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    c_pos = c_neg = g_u = None
    if want_grad:
        c_pos = torch.empty(ls.n_edges, dtype=torch.float32, device=dev)
        c_neg = torch.empty(ls.n_edges, dtype=torch.float32, device=dev)
        g_u = torch.empty_like(user_emb)
    ws_bytes = int(lib.trg_edge_bce_workspace_bytes(ls.num_users))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    e = ls.n_edges
    # 1/E scale of the means: the GLOBAL positive count when this rank holds a partition of them
    e_scale = int(getattr(ls, "n_edges_scale", e))
    rb = user_emb.size(1) * user_emb.element_size()
    nbytes = e * (2 * rb + 16 + (8 if want_grad else 0)) + ls.num_users * (rb * (2 if want_grad else 1) + 4)
    _lib.call("trg_edge_bce_fwd", nbytes, lib.trg_edge_bce_fwd,
              _lib.ptr(ls.by_user.rowptr), _lib.ptr(ls.by_user.col) if e else None,
              _lib.ptr(ls.by_user.eid) if e else None, _lib.ptr(neg_p) if e else None,
              _lib.ptr(user_emb), _lib.ptr(post_emb), ls.num_users, e_scale, user_emb.size(1),
              _lib.dtype_code(user_emb.dtype), _lib.ptr(ls.wbar), _lib.ptr(loss), _lib.ptr(c_pos),
              _lib.ptr(c_neg), _lib.ptr(g_u), _lib.ptr(ws), ws_bytes, _lib.stream())
    return loss, c_pos, c_neg, g_u


def edge_anchor_loss(csr: CSR, anchor, gathered, n_edges_scale, label, wbar, want_grad, g_anchor=None,
                     relu_gate=False, coef_in_csr_order=False):
    """One launch of the single-row anchored loss: rows of ``csr`` index ``anchor``, ``csr.col`` indexes
    ``gathered``.  Returns ``(partial loss[1], coef[E_local] | None, g_anchor | None)``.  ``relu_gate``:
    the written anchor gradient is zeroed where ``anchor <= 0`` (fused ReLU backward).
    ``coef_in_csr_order``: ``coef[e]`` belongs to the edge at CSR position ``e`` (sequential stores) instead
    of ``coef[csr.eid[e]]`` (original edge order, scattered 4-byte stores)."""
    lib = _lib.load()
    anchor, gathered = anchor.contiguous(), gathered.contiguous()
    _check_rows(anchor, "edge_anchor_loss")
    dev = anchor.device
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    coef = None
    accumulate = g_anchor is not None
    if want_grad:
        coef = torch.empty(csr.n_edges, dtype=torch.float32, device=dev)
        if g_anchor is None:
            g_anchor = torch.empty_like(anchor)
    else:
        g_anchor = None
    ws_bytes = int(lib.trg_edge_bce_workspace_bytes(csr.n_rows))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    e = csr.n_edges
    rb = anchor.size(1) * anchor.element_size()
    nbytes = e * (rb + 12) + csr.n_rows * (rb * (2 if want_grad else 1) + 4)
    _lib.call("trg_edge_anchor_loss", nbytes, lib.trg_edge_anchor_loss,
              _lib.ptr(csr.rowptr), _lib.ptr(csr.col) if e else None,
              _lib.ptr(csr.eid) if (e and not coef_in_csr_order) else None,
              _lib.ptr(anchor), _lib.ptr(gathered), csr.n_rows, int(n_edges_scale), anchor.size(1),
              _lib.dtype_code(anchor.dtype), 1 if label else 0, _lib.ptr(wbar), _lib.ptr(loss), _lib.ptr(coef),
              _lib.ptr(g_anchor), 1 if (accumulate and want_grad) else 0,
              1 if (relu_gate and want_grad) else 0, _lib.ptr(ws), ws_bytes, _lib.stream())
    return loss, coef, g_anchor


class LinkBCEFn(torch.autograd.Function):
    """loss of train_gnn.py:259-281.  Forward = two single-row passes over the positives grouped by
    user (anchor = user row, read once per user): the positive posts, then the sampled negatives
    (same grouping, column = neg_p[eid]).  Measured faster than the fused two-row kernel
    (trg_edge_bce_fwd: 12.5 ms vs 10.6 ms at config 2) because each pass keeps 8 row loads in flight
    with half the per-edge bookkeeping; dL/du is accumulated across the two passes without atomics."""

    @staticmethod
    def forward(ctx, user_emb, post_emb, neg_p, ls: LinkStructure):
        want = user_emb.requires_grad or post_emb.requires_grad
        if neg_p.dtype != torch.int64 or neg_p.numel() != ls.n_edges:
            raise _lib.TrgError("neg_p must be int64 with one entry per positive edge (train_gnn.py:272)")
        if getattr(ls, "eid_long", None) is None:
            ls.eid_long = ls.by_user.eid.long()
        e_scale = int(getattr(ls, "n_edges_scale", ls.n_edges))
        bu = ls.by_user
        # the negatives grouped by post with this step's stable sort (needed by the backward); built first
        # because its histogram pass is also the range check of caller-supplied ids (K0 aborts on an id
        # outside [0, P) before any kernel uses it as a row index)
        ctx.neg_by_post = None
        if want and ls.n_edges:
            ctx.neg_by_post = build_csr(ls.train_edge_index[0], neg_p, ls.num_posts, ls.num_users, validate=False,
                                        per_step=True)
        col_neg = neg_p.index_select(0, ls.eid_long).int()     # negatives in the by-user edge order
        neg_csr = CSR(bu.rowptr, col_neg, bu.eid, bu.n_rows, bu.n_cols)
        l_pos, c_pos, g_u = edge_anchor_loss(bu, user_emb, post_emb, e_scale, 1, ls.wbar, want, None)
        l_neg, c_neg, g_u = edge_anchor_loss(neg_csr, user_emb, post_emb, e_scale, 0, ls.wbar, want, g_u)
        ctx.ls = ls
        ctx.want = want
        if want:
            ctx.save_for_backward(user_emb, neg_p, c_pos, c_neg, g_u)
        return (l_pos + l_neg).reshape(())

    @staticmethod
    def backward(ctx, g):
        user_emb, neg_p, c_pos, c_neg, g_u = ctx.saved_tensors
        ls = ctx.ls
        g = g.reshape(1).float().contiguous()
        g_user = g_post = None
        if ctx.needs_input_grad[0]:
            g_user = g_u * g.to(g_u.dtype)
        if ctx.needs_input_grad[1]:
            # dloss/dp = sum over positive edges of the post (static structure) ...
            g_post = gather_wsum(ls.by_post, c_pos, user_emb, scale=g)
            # ... plus the sampled negatives, grouped by post (this step's stable sort, built in forward)
            if ctx.neg_by_post is not None:
                gather_wsum(ctx.neg_by_post, c_neg, user_emb, scale=g, out=g_post, accumulate=True)
        return g_user, g_post, None, None


def link_bce_loss(user_emb, post_emb, train_edge_index, neg_p, interaction_type_tensor, num_users):
    """``loss`` of train_gnn.py:259-281 given this step's negatives (``torch.randint`` at :272)."""
    ls = link_structure(train_edge_index, interaction_type_tensor, num_users, post_emb.size(0))
    return LinkBCEFn.apply(user_emb, post_emb, neg_p, ls)


# ------------------------------------------------------------------------------------------
# K3: projections + combine + ReLU
# ------------------------------------------------------------------------------------------
def _proj_bytes(n, ks, hidden, es):
    return n * (sum(ks) + hidden) * es


def sage_proj_fwd(terms, bias, relu: bool):
    """``out = act(sum_i alpha_i * A_i @ W_i^T + bias)``; terms = [(A, W, alpha), ...]."""
    lib = _lib.load()
    a0 = terms[0][0]
    n, hidden = a0.size(0), terms[0][1].size(0)
    arr = (_lib.TrgProjTerm * len(terms))()
    keep = []
    for i, (a, w, alpha) in enumerate(terms):
        a, w = a.contiguous(), w.contiguous()
        if a.dtype != a0.dtype or w.dtype != a0.dtype:
            raise _lib.TrgError("projection operands must share one dtype")
        keep += [a, w]
        arr[i].a, arr[i].w, arr[i].k, arr[i].alpha = _lib.ptr(a), _lib.ptr(w), a.size(1), float(alpha)
    out = torch.empty(n, hidden, dtype=a0.dtype, device=a0.device)
    b = bias.float().contiguous() if bias is not None else None
    ktot = sum(t[0].size(1) for t in terms)
    code = _lib.dtype_code(a0.dtype)
    ws_bytes = int(lib.trg_sage_proj_workspace_bytes(ktot, hidden, code))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=a0.device)
    _lib.call("trg_sage_proj_fwd", _proj_bytes(n, [t[0].size(1) for t in terms], hidden, a0.element_size()),
              lib.trg_sage_proj_fwd, arr, len(terms), _lib.ptr(b), n, hidden, code, 1 if relu else 0,
              _lib.ptr(out), _lib.ptr(ws), ws_bytes, _lib.stream())
    return out


def sage_proj_bwd_input(dz, terms):
    """``d_a_i = row_scale_i * (alpha_i * dZ @ W_i)``; terms = [(W[h,k], alpha, row_scale|None), ...]."""
    lib = _lib.load()
    dz = dz.contiguous()
    n, hidden = dz.shape
    arr = (_lib.TrgProjBwdTerm * len(terms))()
    outs, keep = [], []
    for i, (w, alpha, rs) in enumerate(terms):
        w = w.contiguous()
        if w.dtype != dz.dtype:
            raise _lib.TrgError("projection operands must share one dtype")
        d_a = torch.empty(n, w.size(1), dtype=dz.dtype, device=dz.device)
        rs = rs.float().contiguous() if rs is not None else None
        keep += [w, rs]
        outs.append(d_a)
        arr[i].w, arr[i].k, arr[i].alpha = _lib.ptr(w), w.size(1), float(alpha)
        arr[i].row_scale, arr[i].d_a = _lib.ptr(rs), _lib.ptr(d_a)
    ktot = sum(t[0].size(1) for t in terms)
    code = _lib.dtype_code(dz.dtype)
    ws_bytes = int(lib.trg_sage_proj_workspace_bytes(ktot, hidden, code))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dz.device)
    _lib.call("trg_sage_proj_bwd_input", n * (len(terms) * hidden + ktot) * dz.element_size(),
              lib.trg_sage_proj_bwd_input, _lib.ptr(dz), arr, len(terms), n, hidden, code,
              _lib.ptr(ws), ws_bytes, _lib.stream())
    return outs


class FusedProjFn(torch.autograd.Function):
    """``out = act(sum_t alpha_t * A_t @ W_t^T + bias)`` with its backward:
    dZ = dOut * (out > 0);  dA_t = rs_t * alpha_t * dZ @ W_t;  dW_t = alpha_t * dZ^T @ A_t;
    db = colsum(dZ).  ``row_scales[t]`` (1/deg or None) is folded into dA_t (see SageAggFn)."""

    @staticmethod
    def forward(ctx, relu, alphas, row_scales, bias, *aw):
        n_t = len(aw) // 2
        a_list, w_list = aw[:n_t], aw[n_t:]
        out = sage_proj_fwd([(a, w, al) for a, w, al in zip(a_list, w_list, alphas)], bias, relu)
        ctx.relu, ctx.alphas, ctx.row_scales, ctx.n_t = relu, alphas, row_scales, n_t
        ctx.has_bias = bias is not None
        ctx.bias_dtype = bias.dtype if bias is not None else None
        ctx.save_for_backward(out, *a_list, *w_list)
        return out

    @staticmethod
    def backward(ctx, g):
        out, *rest = ctx.saved_tensors
        n_t = ctx.n_t
        a_list, w_list = rest[:n_t], rest[n_t:]
        g = g.contiguous()
        dz = torch.ops.aten.threshold_backward(g, out, 0) if ctx.relu else g
        need_a = [ctx.needs_input_grad[4 + t] for t in range(n_t)]
        need_w = [ctx.needs_input_grad[4 + n_t + t] for t in range(n_t)]
        d_a = [None] * n_t
        idx = [t for t in range(n_t) if need_a[t]]
        if idx:
            outs = sage_proj_bwd_input(dz, [(w_list[t], ctx.alphas[t], ctx.row_scales[t]) for t in idx])
            for t, o in zip(idx, outs):
                d_a[t] = o
        d_w = [None] * n_t
        widx = [t for t in range(n_t) if need_w[t]]
        want_b = ctx.has_bias and ctx.needs_input_grad[3]
        d_b = None
        if widx or want_b:
            outs, d_b = sage_proj_bwd_weight(dz, [(a_list[t], ctx.alphas[t]) for t in widx], want_b)
            for t, o in zip(widx, outs):
                d_w[t] = o
            if d_b is not None:
                d_b = d_b.to(ctx.bias_dtype)
        return (None, None, None, d_b, *d_a, *d_w)


def sage_proj_bwd_weight(dz, terms, want_bias: bool):
    """``dW_t = alpha_t * dZ^T @ A_t`` and ``db = colsum(dZ)``; terms = [(A_t, alpha_t), ...].
    Returns ``([dW_t...], db fp32 | None)``."""
    lib = _lib.load()
    dz = dz.contiguous()
    n, hidden = dz.shape
    arr = (_lib.TrgProjDwTerm * max(len(terms), 1))()
    outs, keep = [], []
    for i, (a, alpha) in enumerate(terms):
        a = a.contiguous()
        d_w = torch.empty(hidden, a.size(1), dtype=dz.dtype, device=dz.device)
        keep.append(a)
        outs.append(d_w)
        arr[i].a, arr[i].k, arr[i].alpha, arr[i].d_w = _lib.ptr(a), a.size(1), float(alpha), _lib.ptr(d_w)
    db = torch.empty(hidden, dtype=torch.float32, device=dz.device) if want_bias else None
    ws_bytes = int(lib.trg_sage_proj_dw_workspace_bytes())
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dz.device)
    ktot = sum(t[0].size(1) for t in terms)
    _lib.call("trg_sage_proj_bwd_weight", n * (hidden + ktot) * dz.element_size(),
              lib.trg_sage_proj_bwd_weight, _lib.ptr(dz), arr, len(terms), _lib.ptr(db), n, hidden,
              _lib.dtype_code(dz.dtype), _lib.ptr(ws), ws_bytes, _lib.stream())
    return outs, db


def fused_projection(terms, bias, relu=True, row_scales=None):
    """terms = [(A, W, alpha), ...]; returns act(sum alpha A W^T + bias) with a fused backward."""
    a_list = [t[0] for t in terms]
    w_list = [t[1] for t in terms]
    alphas = tuple(float(t[2]) for t in terms)
    rs = tuple(row_scales) if row_scales is not None else (None,) * len(terms)
    return FusedProjFn.apply(relu, alphas, rs, bias, *a_list, *w_list)


# ------------------------------------------------------------------------------------------
# K5: score contraction + top-k (inference.py:427-428)
# ------------------------------------------------------------------------------------------
def score_topk(q: torch.Tensor, cat, k: int, id_offset: int = 0, exclude=None, rows=None):
    """``torch.topk(torch.mm(q, cat.T), min(k, len))`` without materialising the scores.
    Returns ``(values[B,k'] fp32 descending, ids[B,k'] int64)`` under (score desc, id asc).

    ``exclude``: an ``ExclusionIndex``; query ``b`` then never gets a post id of exclusion row
    ``rows[b]`` (``rows``: int64 ``[B]`` on the device, each in ``[0, exclude.num_rows)``; default: row
    ``b``).  A query with fewer than ``k'`` admissible posts is padded at its tail with
    ``(-inf, -1)``.  ``exclude=None`` is exactly the call without exclusions.

    ``cat`` may be an ``fp8.Fp8Catalogue``: the posts are then selected from its e4m3 copy and re-ranked
    exactly from its dense table (``fp8.score_topk``; ``q`` must have the table's dtype, ``k <= 128``)."""
    if isinstance(cat, fp8.Fp8Catalogue):
        return fp8.score_topk(q, cat, k, id_offset, exclude=exclude, rows=rows)
    if q.dim() == 1:
        q = q.unsqueeze(0)
    return _score_topk_native(q.contiguous(), cat.contiguous(), k, id_offset, exclude, rows)


def _score_topk_native(q, cat, k, id_offset, exclude, rows, code=None):
    """``trg_score_topk(_excluding)``; ``code``: the tables' dtype code (default: that of ``q.dtype``; e4m3
    tables pass ``TRG_F8E4M3``)."""
    lib = _lib.load()
    b, h = q.shape
    p = cat.size(0)
    kk = min(int(k), p)
    if exclude is None and rows is not None:
        raise ValueError("score_topk: rows selects exclusion rows and needs exclude")
    if exclude is not None:
        if rows is None:
            if b > exclude.num_rows:
                raise ValueError(f"score_topk: {b} queries but the exclusion index has {exclude.num_rows} rows; "
                                 "pass rows= to map queries to rows")
        else:
            if rows.dtype != torch.int64 or rows.dim() != 1 or rows.numel() != b:
                raise ValueError(f"score_topk: rows must be int64 [B={b}]")
            rows = rows.contiguous()
    vals = torch.empty(b, kk, dtype=torch.float32, device=q.device)
    ids = torch.empty(b, kk, dtype=torch.int64, device=q.device)
    if b == 0 or kk == 0:
        return vals, ids
    ws_bytes = int(lib.trg_score_topk_workspace_bytes(b, p, h, kk))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=q.device)
    code = _lib.dtype_code(q.dtype) if code is None else code
    if exclude is None:
        _lib.call("trg_score_topk", 2 * b * p * h, lib.trg_score_topk,  # "bytes" slot carries flops here
                  _lib.ptr(q), _lib.ptr(cat), b, p, h, code, kk, int(id_offset),
                  _lib.ptr(vals), _lib.ptr(ids), _lib.ptr(ws), ws_bytes, _lib.stream())
    else:
        _lib.call("trg_score_topk_excluding", 2 * b * p * h, lib.trg_score_topk_excluding,
                  _lib.ptr(q), _lib.ptr(cat), b, p, h, code, kk, int(id_offset),
                  # an index without any id: every row is empty and no id is read, but the pointer must be valid
                  _lib.ptr(exclude.rowptr), _lib.ptr(exclude.ids if exclude.nnz else exclude.rowptr), _lib.ptr(rows),
                  _lib.ptr(vals), _lib.ptr(ids), _lib.ptr(ws), ws_bytes, _lib.stream())
    return vals, ids


def topk_merge(vals_in: torch.Tensor, ids_in: torch.Tensor, n_lists: int, k_out: int):
    lib = _lib.load()
    b = vals_in.size(0)
    k_in = vals_in.size(1) // n_lists
    vals = torch.empty(b, k_out, dtype=torch.float32, device=vals_in.device)
    ids = torch.empty(b, k_out, dtype=torch.int64, device=vals_in.device)
    _lib.check(lib.trg_topk_merge(_lib.ptr(vals_in.contiguous()), _lib.ptr(ids_in.contiguous()), b,
                                  n_lists, k_in, k_out, _lib.ptr(vals), _lib.ptr(ids), _lib.stream()),
               "trg_topk_merge")
    return vals, ids

"""Drop-in modules for the reference's model-construction API.

``SAGEConv`` mirrors ``torch_geometric.nn.SAGEConv`` for exactly the options the reference relies
on (train_gnn.py:158-160: ``aggr='mean'``, ``root_weight=True``, ``bias=True``,
``normalize=False``, ``project=False``) with the same constructor, call signature and
``state_dict`` keys (``lin_l.weight``, ``lin_l.bias``, ``lin_r.weight``), so
``from truth_recommendation_gnn_b200.nn import SAGEConv`` replaces
``from torch_geometric.nn import SAGEConv`` (train_gnn.py:6, inference.py:117) and the scripts'
``WeightedRGCN`` class, optimizer construction, checkpointing and ``load_state_dict`` keep working
unchanged.  ``WeightedRGCN`` here is the same model with the projections, relation combine and
ReLU fused.
"""
from __future__ import annotations

import math
from typing import NamedTuple

import torch
import torch.nn.functional as F
from torch.nn.parameter import Parameter, UninitializedParameter

from . import _lib
from .functional import fused_projection, sage_mean_aggregate
from .graph import PushRelation, relation_graph

REL_DIRECT = ("post", "rev_engages", "user")
REL_SOCIAL = ("user", "social", "user")
REL_ENGAGE = ("user", "engages", "post")


class Linear(torch.nn.Module):
    """``torch_geometric.nn.dense.linear.Linear`` semantics: ``in_channels = -1`` is resolved at the
    first forward or by ``load_state_dict`` IN PLACE (the optimizer built at train_gnn.py:207
    already holds the Parameter objects).  Default init = ``torch.nn.Linear``'s."""

    def __init__(self, in_channels: int, out_channels: int, bias: bool = True):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        if in_channels > 0:
            self.weight = Parameter(torch.empty(out_channels, in_channels))
        else:
            self.weight = UninitializedParameter()
        if bias:
            self.bias = Parameter(torch.empty(out_channels))
        else:
            self.register_parameter("bias", None)
        self.reset_parameters()

    def reset_parameters(self):
        if self.in_channels <= 0:
            return
        torch.nn.init.kaiming_uniform_(self.weight, a=math.sqrt(5))
        if self.bias is not None:
            bound = 1.0 / math.sqrt(self.in_channels)
            torch.nn.init.uniform_(self.bias, -bound, bound)

    def materialize(self, in_channels: int):
        if isinstance(self.weight, UninitializedParameter):
            self.in_channels = int(in_channels)
            self.weight.materialize((self.out_channels, self.in_channels))
            self.reset_parameters()

    def _save_to_state_dict(self, destination, prefix, keep_vars):
        if isinstance(self.weight, UninitializedParameter):
            destination[prefix + "weight"] = self.weight  # like PyG: lazy weights stay placeholders
            if self.bias is not None:
                destination[prefix + "bias"] = self.bias if keep_vars else self.bias.detach()
        else:
            super()._save_to_state_dict(destination, prefix, keep_vars)

    def _load_from_state_dict(self, state_dict, prefix, local_metadata, strict, missing_keys,
                              unexpected_keys, error_msgs):
        w = state_dict.get(prefix + "weight")
        if w is not None and isinstance(self.weight, UninitializedParameter):
            self.in_channels = int(w.size(-1))
            self.weight.materialize(tuple(w.shape))
        super()._load_from_state_dict(state_dict, prefix, local_metadata, strict, missing_keys,
                                      unexpected_keys, error_msgs)

    def forward(self, x):
        self.materialize(x.size(-1))
        return F.linear(x, self.weight, self.bias)

    def extra_repr(self):
        return f"{self.in_channels}, {self.out_channels}, bias={self.bias is not None}"


class SAGEConv(torch.nn.Module):
    r"""``out = lin_l(mean_{j in N(i)} x_j) + lin_r(x_i)`` -- replaces PyG's operator at
    train_gnn.py:158-160 (ctor) and :177-184,194-197 (calls).

    ``forward((x_src, x_dst), edge_index)`` with bipartite ``edge_index[2,E]`` int64
    (``edge_index[0]`` in ``[0, N_src)``, ``edge_index[1]`` in ``[0, N_dst)``); a single tensor
    ``x`` means ``(x, x)``.  E = 0 and N_src = 0 are valid (inference.py:412-419).
    """

    def __init__(self, in_channels, out_channels: int, aggr: str = "mean", normalize: bool = False,
                 root_weight: bool = True, project: bool = False, bias: bool = True):
        super().__init__()
        if aggr != "mean" or normalize or project or not root_weight:
            raise NotImplementedError(
                "only the configuration the reference uses is accelerated: aggr='mean', "
                "normalize=False, root_weight=True, project=False (train_gnn.py:158-160)")
        if isinstance(in_channels, int):
            in_channels = (in_channels, in_channels)
        self.in_channels, self.out_channels = tuple(in_channels), out_channels
        self.lin_l = Linear(in_channels[0], out_channels, bias=bias)
        self.lin_r = Linear(in_channels[1], out_channels, bias=False)

    def reset_parameters(self):
        self.lin_l.reset_parameters()
        self.lin_r.reset_parameters()

    def forward(self, x, edge_index, size=None):
        """K0 (cached) + K1 mean aggregation, then ``lin_l(mean) + lin_r(x_dst)`` as ONE K3 launch over the
        concatenated K (bias in the epilogue, no ReLU: the caller applies its own, train_gnn.py:187-198).
        Swapping the import at train_gnn.py:6 alone therefore leaves no GEMM of the conv on cuBLAS; the
        gradient of the mean comes back pre-scaled by 1/deg (fused into the K3 input-gradient epilogue), so
        the aggregation backward is a plain transposed gather-sum (K2)."""
        if isinstance(x, torch.Tensor):
            x = (x, x)
        x_src, x_dst = x
        if not x_dst.is_cuda:
            raise _lib.TrgError("SAGEConv (B200) needs CUDA tensors; there is no CPU fallback")
        self.lin_l.materialize(x_src.size(-1))
        self.lin_r.materialize(x_dst.size(-1))
        rel = relation_graph(edge_index, x_src.size(0), x_dst.size(0))
        mean = sage_mean_aggregate(x_src, rel, True)
        return fused_projection([(mean, self.lin_l.weight, 1.0), (x_dst, self.lin_r.weight, 1.0)],
                                self.lin_l.bias, relu=False, row_scales=(rel.inv_deg, None))

    def __repr__(self):
        return f"SAGEConv({self.in_channels}, {self.out_channels}, aggr=mean)"


class FusedGemm(NamedTuple):
    """One fused K3 projection, ``relu(sum_t alphas[t] * A_t @ weights[t]^T + bias)`` with one operand A_t per
    weight, and the term lists of its forward (``terms``) and backward (``dw_terms``, ``dx_terms``) kernels."""
    weights: tuple
    alphas: tuple
    bias: torch.Tensor | None

    def terms(self, *operands):             # [(A, W, alpha)]: sage_proj_fwd, fused_projection
        return list(zip(operands, self.weights, self.alphas, strict=True))

    def dw_terms(self, *operands):          # [(A, alpha)]: sage_proj_bwd_weight
        return list(zip(operands, self.alphas, strict=True))

    def dx_terms(self, *row_scales):        # [(W, alpha, row scale)]: sage_proj_bwd_input
        return list(zip(self.weights, self.alphas, row_scales, strict=True))


def _accum(param, grad):
    """What ``loss.backward()`` does with a leaf gradient."""
    grad = grad.to(param.dtype)
    if param.grad is None:
        param.grad = grad
    else:
        param.grad.add_(grad)


class WeightedRGCN(torch.nn.Module):
    """The reference model, train_gnn.py:147-200 (dup inference.py:119-169): same attribute names,
    same fixed python-float relation weights, same ``forward(x_dict, edge_index_dict)``.

    Every path that runs the layer (autograd, tape-free, sharded, cold-start) computes it as two GEMMs
    whose operands come from ``user_gemm`` / ``post_gemm`` (wd, ws = ``w_direct``, ``w_social``)::

        user = relu([mean_d | mean_s | x_u] @ [wd W_l,d | ws W_l,s | wd W_r,d + ws W_r,s]^T + wd b_d + ws b_s)
        post = relu([mean_e | x_p] @ [W_l,e | W_r,p]^T + b_e)

    and ``accumulate_grads`` maps the GEMMs' gradients back onto the nine parameters."""

    def __init__(self, hidden_dim=64, in_channels=(-1, -1)):
        super().__init__()
        self.msg_direct = SAGEConv(in_channels, hidden_dim)   # user <- post (engagement)
        self.msg_social = SAGEConv(in_channels, hidden_dim)   # user <- user (social)
        self.post_update = SAGEConv(in_channels, hidden_dim)  # post <- user (engagement)
        self.w_direct = 1.0
        self.w_social = 0.75

    def materialize(self, user_feat: int, post_feat: int):
        """Resolve the convs' lazy in-channels from the user and post feature widths."""
        widths = ((post_feat, user_feat), (user_feat, user_feat), (user_feat, post_feat))
        for conv, (f_src, f_dst) in zip((self.msg_direct, self.msg_social, self.post_update), widths):
            conv.lin_l.materialize(f_src)
            conv.lin_r.materialize(f_dst)

    def user_gemm(self) -> FusedGemm:
        """Operands ``[mean_d | mean_s | x_u]``; the root weight and bias are combined anew by every call."""
        d, s = self.msg_direct, self.msg_social
        wd, ws = float(self.w_direct), float(self.w_social)
        w_root = wd * d.lin_r.weight + ws * s.lin_r.weight
        b_user = None
        if d.lin_l.bias is not None:
            b_user = wd * d.lin_l.bias + ws * s.lin_l.bias
        return FusedGemm((d.lin_l.weight, s.lin_l.weight, w_root), (wd, ws, 1.0), b_user)

    def post_gemm(self) -> FusedGemm:
        """Operands ``[mean_e | x_p]``."""
        p = self.post_update
        return FusedGemm((p.lin_l.weight, p.lin_r.weight), (1.0, 1.0), p.lin_l.bias)

    def accumulate_grads(self, dw_user, db_user, dw_post, db_post):
        """Add both GEMMs' gradients (one dW per operand, db) to the nine parameters as ``loss.backward()`` does."""
        d, s, p = self.msg_direct, self.msg_social, self.post_update
        wd, ws = float(self.w_direct), float(self.w_social)
        dw_d, dw_s, dw_root = dw_user
        dw_p, dw_pr = dw_post
        _accum(d.lin_l.weight, dw_d)
        _accum(s.lin_l.weight, dw_s)
        _accum(d.lin_r.weight, wd * dw_root)
        _accum(s.lin_r.weight, ws * dw_root)
        _accum(d.lin_l.bias, wd * db_user)
        _accum(s.lin_l.bias, ws * db_user)
        _accum(p.lin_l.weight, dw_p)
        _accum(p.lin_r.weight, dw_pr)
        _accum(p.lin_l.bias, db_post)

    def forward(self, x_dict, edge_index_dict):
        """Same result as train_gnn.py:166-200, computed as three K1 aggregations and two fused
        K3 projections (relation combine, biases and ReLU in the GEMM epilogue; the shared
        ``lin_r`` input of the two user convs is multiplied once by ``1.0*W_r,direct +
        0.75*W_r,social``)."""
        user_x, post_x = x_dict["user"], x_dict["post"]
        if not user_x.is_cuda:
            raise _lib.TrgError("WeightedRGCN (B200) needs CUDA tensors; there is no CPU fallback")
        n_u, n_p = user_x.size(0), post_x.size(0)
        rels = {REL_DIRECT: relation_graph(edge_index_dict[REL_DIRECT], n_p, n_u),
                REL_SOCIAL: relation_graph(edge_index_dict[REL_SOCIAL], n_u, n_u),
                REL_ENGAGE: relation_graph(edge_index_dict[REL_ENGAGE], n_u, n_p)}
        return self.forward_partitioned(x_dict, x_dict, rels, CUDA_OPS)

    def forward_partitioned(self, src_dict, dst_dict, rels, ops):
        """One hetero layer on a destination partition: ``src_dict`` holds the source tables (all
        rows: the all-gathered tables on multi-GPU), ``dst_dict`` the owned destination rows,
        ``rels`` one :class:`RelationGraph` per relation (rows = owned destinations).  Single GPU:
        ``src_dict is dst_dict``."""
        user_src, post_src = src_dict["user"], src_dict["post"]
        user_x, post_x = dst_dict["user"], dst_dict["post"]
        self.materialize(user_x.size(-1), post_x.size(-1))
        rel_d, rel_s, rel_e = rels[REL_DIRECT], rels[REL_SOCIAL], rels[REL_ENGAGE]
        mean_d = ops.aggregate(post_src, rel_d)
        mean_s = ops.aggregate(user_src, rel_s)
        mean_e = ops.aggregate(user_src, rel_e)
        ug = self.user_gemm()
        user_out = ops.project(ug.terms(mean_d, mean_s, user_x), ug.bias, True, (rel_d, rel_s, None))
        pg = self.post_gemm()
        post_out = ops.project(pg.terms(mean_e, post_x), pg.bias, True, (rel_e, None))
        return {"user": user_out, "post": post_out}


class CudaOps:
    """The sm_100a kernels behind the model (K1/K2 aggregation, K3 projections).  ``aggregate``
    returns a mean whose gradient is expected pre-scaled by 1/deg; ``project`` folds that scale
    into its input-gradient epilogue (``scale_rels`` names the relation of each mean term)."""

    @staticmethod
    def aggregate(x_src, rel):
        if isinstance(rel, PushRelation):      # multi-GPU, source-partitioned relation
            from .collectives import PushMeanAggFn
            return PushMeanAggFn.apply(x_src, rel, CudaOps.gather_sum, True)
        return sage_mean_aggregate(x_src, rel, True)

    @staticmethod
    def gather_sum(rel, which, x, out_dtype=None):
        """Plain segmented gather-sum over the forward ("fwd": rows = destinations) or transposed
        ("bwd": rows = sources) CSR of a relation -- K2 without the 1/deg scale."""
        from .functional import sage_agg_bwd
        return sage_agg_bwd(rel.fwd if which == "fwd" else rel.bwd, None, x, out_dtype=out_dtype)

    @staticmethod
    def project(terms, bias, relu, scale_rels):
        rs = tuple(r.inv_deg if r is not None else None for r in scale_rels)
        return fused_projection(terms, bias, relu=relu, row_scales=rs)


CUDA_OPS = CudaOps()


class StackedWeightedRGCN(torch.nn.Module):
    """L stacked ``WeightedRGCN`` blocks (BASELINE.json configs 1-4 ask for 2-3 layers; the
    reference has one).  Stacking rule of SURVEY.md §8: layer l has its own three convs, is fed
    the ``{'user','post'}`` output of layer l-1, and ReLU follows every layer."""

    def __init__(self, hidden_dim=64, num_layers=2, in_channels=(-1, -1)):
        super().__init__()
        self.layers = torch.nn.ModuleList(
            [WeightedRGCN(hidden_dim, in_channels if i == 0 else (hidden_dim, hidden_dim))
             for i in range(num_layers)])

    def forward(self, x_dict, edge_index_dict):
        for layer in self.layers:
            x_dict = layer(x_dict, edge_index_dict)
        return x_dict

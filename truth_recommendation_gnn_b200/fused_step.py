"""Whole-step forward + loss + backward of the reference model without the autograd tape.

``loss_and_grads`` computes exactly what ``loss = link_bce_loss(model(x)...); loss.backward()``
computes (train_gnn.py:254-283) for :class:`WeightedRGCN` / :class:`StackedWeightedRGCN`, with the
same kernels, but orders the backward by hand so that the element-wise passes autograd would launch
between them disappear into kernel epilogues:

* ReLU backward (aten ``threshold_backward``: read g, read out, write dZ) -> a ``relu_of`` gate in
  the kernel that finishes each gradient table (K2 / loss gather passes), and a free gate on the
  anchor row the loss kernel already holds in registers;
* gradient accumulation of a table that feeds several consumers (user rows: social + engages
  aggregation + root term; post rows: rev_engages aggregation + root term) -> ``accumulate`` into the
  root-term gradient written by the projection backward.

Each layer's two GEMMs take their operands from the model (``WeightedRGCN.user_gemm`` / ``post_gemm``) and
hand their gradients back through ``accumulate_grads``, as the autograd and sharded (``dist_fused``) steps do.

At config 2 this removes ~20 GB of element-wise HBM traffic per step.  The autograd path
(``functional.py`` Functions) stays the general one; ``train_step`` takes this path when the model,
inputs and parameters qualify (``eligible``) and both are checked against each other and against the
oracle in ``tests/test_gpu_model.py``.
"""
from __future__ import annotations

import torch

from . import _lib
from .functional import (edge_anchor_loss, gather_wsum, link_structure, sage_agg_bwd, sage_agg_fwd,
                         sage_proj_bwd_input, sage_proj_bwd_weight, sage_proj_fwd)
from .graph import CSR, build_csr, relation_graph
from .nn import REL_DIRECT, REL_ENGAGE, REL_SOCIAL, StackedWeightedRGCN, WeightedRGCN


def _layers(model):
    """The layers of the reference model classes (not subclasses with a changed forward), else None."""
    if type(model) is StackedWeightedRGCN:
        return list(model.layers)
    if type(model) is WeightedRGCN:
        return [model]
    return None


def model_eligible(model) -> bool:
    """The model-side conditions of the tape-free steps (this one and ``dist_fused``): a reference model class,
    every conv with its bias, every parameter requiring a gradient, grad mode enabled."""
    layers = _layers(model)
    if layers is None or not torch.is_grad_enabled():
        return False
    if any(conv.lin_l.bias is None for l in layers for conv in (l.msg_direct, l.msg_social, l.post_update)):
        return False
    return all(p.requires_grad for p in model.parameters())


def eligible(model, x_dict) -> bool:
    """True when the tape-free path computes the same thing as autograd would: ``model_eligible``, and leaf
    CUDA inputs of one dtype that need no gradient."""
    if not model_eligible(model):
        return False
    xu, xp = x_dict["user"], x_dict["post"]
    return xu.is_cuda and xp.is_cuda and not xu.requires_grad and not xp.requires_grad and xu.dtype == xp.dtype


def _agg(rel, x):
    want_inv = rel.inv_deg is None
    mean, inv_deg = sage_agg_fwd(rel.fwd, x, want_inv_deg=want_inv)
    if want_inv:
        rel.inv_deg = inv_deg
    return mean


@torch.no_grad()
def loss_and_grads(model, x_dict, edge_index_dict, train_edge_index, interaction_type_tensor, num_users,
                   neg_p, neg_ready=None):
    """Returns the 0-d loss tensor; parameter gradients are accumulated into ``.grad``.  ``neg_ready``: an
    event after which ``neg_p`` is valid (its host -> device copy runs on a side stream during the forward)."""
    layers = _layers(model)
    if layers is None:
        raise _lib.TrgError("loss_and_grads: model must be WeightedRGCN or StackedWeightedRGCN")
    hu, hp = x_dict["user"].contiguous(), x_dict["post"].contiguous()
    n_u, n_p = hu.size(0), hp.size(0)
    rel_d = relation_graph(edge_index_dict[REL_DIRECT], n_p, n_u)
    rel_s = relation_graph(edge_index_dict[REL_SOCIAL], n_u, n_u)
    rel_e = relation_graph(edge_index_dict[REL_ENGAGE], n_u, n_p)

    # ---- forward (train_gnn.py:166-200 per layer) ----
    saved = []
    for layer in layers:
        layer.materialize(hu.size(-1), hp.size(-1))
        mean_d, mean_s, mean_e = _agg(rel_d, hp), _agg(rel_s, hu), _agg(rel_e, hu)
        ug, pg = layer.user_gemm(), layer.post_gemm()
        hu_n = sage_proj_fwd(ug.terms(mean_d, mean_s, hu), ug.bias, True)
        hp_n = sage_proj_fwd(pg.terms(mean_e, hp), pg.bias, True)
        saved.append((hu, hp, mean_d, mean_s, mean_e, ug, pg))
        hu, hp = hu_n, hp_n

    # ---- loss (train_gnn.py:259-281) + its backward onto the last layer's pre-activations ----
    ls = link_structure(train_edge_index, interaction_type_tensor, num_users, n_p)
    if neg_ready is not None:
        torch.cuda.current_stream().wait_event(neg_ready)
    if neg_p.dtype != torch.int64 or neg_p.numel() != ls.n_edges:
        raise _lib.TrgError("neg_p must be int64 with one entry per positive edge (train_gnn.py:272)")
    if getattr(ls, "eid_long", None) is None:
        ls.eid_long = ls.by_user.eid.long()
    bu = ls.by_user
    # negatives in by-user edge order; every per-edge array of the loss lives in that order from here on:
    # the user-anchored passes write their coefficients sequentially, and the post-side gathers look them
    # up through edge ids that ARE by-user positions (static remap for the positives; for the negatives
    # the per-step sort is run on the by-user-ordered arrays, so its edge ids come out that way)
    col_neg64 = neg_p.index_select(0, ls.eid_long)
    # this step's by-post grouping first: its histogram pass is also the range check of the caller's
    # negatives (an id outside [0, P) aborts there, before any kernel uses it as a row index)
    neg_by_post = build_csr(ls.user_of_u, col_neg64, n_p, n_u, validate=False, per_step=True)
    neg_by_user = CSR(bu.rowptr, col_neg64.int(), bu.eid, bu.n_rows, bu.n_cols)
    l_pos, c_pos, dz_u = edge_anchor_loss(bu, hu, hp, ls.n_edges, 1, ls.wbar, True, None, coef_in_csr_order=True)
    l_neg, c_neg, dz_u = edge_anchor_loss(neg_by_user, hu, hp, ls.n_edges, 0, ls.wbar, True, dz_u,
                                          relu_gate=True, coef_in_csr_order=True)
    dz_p = gather_wsum(ls.by_post_u, c_pos, hu)
    gather_wsum(neg_by_post, c_neg, hu, out=dz_p, accumulate=True, relu_of=hp)
    del col_neg64
    loss = (l_pos + l_neg).reshape(())
    del neg_by_user, neg_by_post, c_pos, c_neg, hu, hp

    # ---- backward through the layers (train_gnn.py:283) ----
    for li in range(len(layers) - 1, -1, -1):
        hu_in, hp_in, mean_d, mean_s, mean_e, ug, pg = saved.pop()
        dw_u, db_u = sage_proj_bwd_weight(dz_u, ug.dw_terms(mean_d, mean_s, hu_in), True)
        dw_p, db_p = sage_proj_bwd_weight(dz_p, pg.dw_terms(mean_e, hp_in), True)
        del mean_d, mean_s, mean_e
        layers[li].accumulate_grads(dw_u, db_u, dw_p, db_p)
        if li == 0:
            break
        # gradients w.r.t. this layer's inputs = the previous layer's outputs; the mean terms come out
        # pre-scaled by 1/deg, so the transposed aggregations below are plain gather-sums
        g_md, g_ms, g_hu = sage_proj_bwd_input(dz_u, ug.dx_terms(rel_d.inv_deg, rel_s.inv_deg, None))
        g_me, g_hp = sage_proj_bwd_input(dz_p, pg.dx_terms(rel_e.inv_deg, None))
        del dz_u, dz_p
        sage_agg_bwd(rel_s.bwd, None, g_ms, out=g_hu, accumulate=True)
        sage_agg_bwd(rel_e.bwd, None, g_me, out=g_hu, accumulate=True, relu_of=hu_in)
        sage_agg_bwd(rel_d.bwd, None, g_md, out=g_hp, accumulate=True, relu_of=hp_in)
        dz_u, dz_p = g_hu, g_hp
    return loss

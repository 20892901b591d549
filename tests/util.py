"""Shared helpers for the parity tests (tolerances are BASELINE.json's north_star)."""
import os

import torch

from oracle import sage as osage
from truth_recommendation_gnn_b200 import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

TOL_F32 = 1e-5   # relative, fp32 embeddings / losses / scores
TOL_BF16 = 1e-2  # relative, bf16 storage with fp32 accumulation


def load_golden(name):
    return torch.load(os.path.join(GOLDEN, name + ".pt"), weights_only=False)


def golden_graph(fix, device="cpu"):
    ei = {eval(k): v.to(device) for k, v in fix["edge_index"].items()}
    m = fix["meta"]
    return synth.SynthGraph({"user": fix["x_user"].to(device), "post": fix["x_post"].to(device)}, ei,
                            ei[synth.REL_ENGAGE], fix["w"].to(device), m["u"], m["p"])


def oracle_model(h, layers, sd, fin=None):
    fin = fin or h
    m = (osage.WeightedRGCNOracle(h, (fin, fin)) if layers == 1
         else osage.StackedWeightedRGCNOracle(h, layers, (fin, fin)))
    m.load_state_dict(sd)
    return m


def assert_close(a, b, tol, what=""):
    """NORM form, ``max|a-b| / max|b|``: for tensors whose entries are sums of many SIGNED terms (GEMMs and
    gather-sums of zero-mean data, every gradient).  Such sums cancel, so an entry can be arbitrarily small
    next to the terms that produced it and its element-wise relative error says nothing about the
    arithmetic (measured: the fp32 CPU oracle itself is 5e-3 .. 1e-1 away from the fp64 oracle
    element-wise on 2-3 layer embeddings with the 1e-6 floor, and 2e-7 in this form)."""
    err = osage.rel_err_norm(a, b)
    assert err <= tol, f"{what}: rel err {err:.3e} > {tol:.1e}"
    return err


def rel_err_elementwise(a, b, floor_frac=1e-6):
    """SURVEY.md §8(c): ``max_i |a_i - b_i| / max(|b_i|, floor)`` with ``floor = floor_frac * max|b|`` (the
    absolute floor is needed because post-ReLU outputs contain exact zeros)."""
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    if b.numel() == 0:
        return 0.0
    floor = max(floor_frac * float(b.abs().max()), 1e-30)
    return float(((a - b).abs() / b.abs().clamp(min=floor)).max())


def assert_close_elementwise(a, b, tol, what="", floor_frac=1e-6):
    """ELEMENT-WISE relative error with an absolute floor, for tensors WITHOUT cancellation: scores and
    means of non-negative (post-ReLU) rows, top-k values, losses."""
    err = rel_err_elementwise(a, b, floor_frac)
    assert err <= tol, f"{what}: element-wise rel err {err:.3e} > {tol:.1e}"
    return err


def assert_as_accurate_as_fp32(a, b32, b64, tol, what="", floor_frac=1e-3, slack=8.0):
    """Parity for tensors WITH cancellation (embeddings = ReLU of signed sums, gradients), judged against an
    fp64 run of the oracle: ``a`` (the CUDA result) must be (1) within ``tol`` of the fp64 oracle relative
    to the tensor's scale, and (2) element-wise (floor ``floor_frac * max|b|``) no further from the fp64
    oracle than ``slack`` x the distance of the reference's OWN fp32 arithmetic (``b32``, the fp32 CPU
    oracle) -- i.e. wherever the reference's fp32 result is itself well determined, ours matches it to
    ``tol``; where rounding (or a ReLU gate within rounding of 0) makes the reference's own result
    uncertain, ours is no more uncertain.  ``slack``: the statistic is a MAXIMUM over all elements of a noisy
    ratio, dominated by the few entries near the floor (1e-3 of the scale, where tol x floor = 1e-8 of the
    scale is below what any fp32 summation order resolves); two correct fp32 evaluations differ by a factor of
    a few there (measured: 3.2x on the skewed fixture, 3xTF32 products + another summation order).  No seed
    search."""
    e_norm = osage.rel_err_norm(a, b64)
    assert e_norm <= tol, f"{what}: rel err vs fp64 oracle {e_norm:.3e} > {tol:.1e}"
    e_a = rel_err_elementwise(a, b64, floor_frac)
    e_ref = rel_err_elementwise(b32, b64, floor_frac)
    assert e_a <= max(tol, slack * e_ref), (f"{what}: element-wise err vs fp64 oracle {e_a:.3e} > max({tol:.1e}, "
                                            f"{slack} x fp32-oracle err {e_ref:.3e})")
    return e_a, e_ref


def product_gates(model, x_dict, edge_index_dict):
    """ReLU gates the product applied, layer by layer (``out > 0`` of every block), as CPU bool masks."""
    layers = list(model.layers) if hasattr(model, "layers") else [model]
    gates, x = [], x_dict
    with torch.no_grad():
        for layer in layers:
            x = layer(x, edge_index_dict)
            gates.append({k: (v > 0).cpu() for k, v in x.items()})
    return gates


def oracle_grads_with_gates(h, layers, sd, g, neg, gates, dtype=torch.float32, kink=1e-5, fin=None):
    """Gradients of the reference loss (train_gnn.py:259-283) from the oracle with the ReLU gates forced to
    ``gates`` (see ``oracle.sage.forward_gated``), after checking against an fp64 run that those gates differ
    from the exact ones ONLY where the pre-activation is within ``kink`` (relative to the layer's scale) of 0.
    Returns ``(loss, {param name: grad}, n_ambiguous_gates)``."""
    m64 = oracle_model(h, layers, sd, fin).double()
    x64 = {k: v.double() for k, v in g.x_dict.items()}
    with torch.no_grad():
        _, zs = osage.forward_gated(m64, x64, g.edge_index_dict, gates)
    n_amb = 0
    for l, (z_u, z_p) in enumerate(zs):
        for z, gate, what in ((z_u, gates[l]["user"], "user"), (z_p, gates[l]["post"], "post")):
            if not z.numel():
                continue
            wrong = gate != (z > 0)
            if bool(wrong.any()):
                worst = float(z[wrong].abs().max() / z.abs().max())
                assert worst <= kink, f"layer {l} {what}: a gate differs where |z| = {worst:.2e} of the scale"
                n_amb += int(wrong.sum())
    m = oracle_model(h, layers, sd, fin).to(dtype)
    out, _ = osage.forward_gated(m, {k: v.to(dtype) for k, v in g.x_dict.items()}, g.edge_index_dict, gates)
    loss = osage.link_loss(out["user"], out["post"], g.train_edge_index[0], g.train_edge_index[1], neg,
                           g.interaction_type_tensor.to(dtype), g.num_users)
    loss.backward()
    return float(loss), {n: p.grad for n, p in m.named_parameters()}, n_amb


def oracle_grads_bf16(h, layers, sd, g, neg, fin=None):
    """Gradients of the reference loss from the oracle run in bf16: parameters, inputs and every intermediate
    table rounded to bf16 as each op produces it (PyTorch's bf16 CPU ops), the loss taken in fp32 on the bf16
    embeddings.  Their distance from the fp32 oracle is what bf16 storage alone costs on that input."""
    m = oracle_model(h, layers, sd, fin).to(torch.bfloat16)
    out = m({k: v.to(torch.bfloat16) for k, v in g.x_dict.items()}, g.edge_index_dict)
    loss = osage.link_loss(out["user"].float(), out["post"].float(), g.train_edge_index[0], g.train_edge_index[1],
                           neg, g.interaction_type_tensor.float(), g.num_users)
    loss.backward()
    return {n: p.grad.float() for n, p in m.named_parameters()}

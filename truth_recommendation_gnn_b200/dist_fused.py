"""Tape-free, communication-overlapped train step on a destination partition (SURVEY.md §8e).

Same partitioning and the same result as ``dist.train_step_sharded`` (autograd Functions +
blocking collectives); here the forward, the loss and the backward are ordered by hand so that
every collective of the step is in flight while an independent kernel runs:

  forward, layer l    all-gather(user rows)            ||  push partial sums over the local posts
                      reduce-scatter(push partials)    ||  social + engages aggregation, post projection
  loss                all-gather(final user rows)      ||  this step's negative-edge CSRs (by post, by user)
                      reduce-scatter(dL/du partials)   ||  post-side projection backward + engages^T gather
  backward, layer l   all-gather(d mean_direct)        ||  social^T gather
                      reduce-scatter(d user partials)  ||  rev_engages^T gather over the local posts and
                                                           the next (lower) layer's post-side backward

Collectives are ``torch.distributed`` async ops (NCCL runs them on its own stream over NVLink /
NVSwitch); ``wait()`` only orders the consuming kernel after them.  ReLU backward and gradient
accumulation ride in kernel epilogues and the layer's GEMMs come from the model, as in ``fused_step``;
the graphed step is a ``train.GraphedStep``.  ``prims`` supplies the compute
primitives: the CUDA kernels in the product (``CUDA_STEP_PRIMS``), oracle ops in the CPU (gloo)
tests of this host logic (``tests/oracle_ops.OracleStepPrims``).
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from . import _lib
from .dist import PaddedPairs, ShardedGraph, allreduce_grads
from .fused_step import _agg, _layers, model_eligible
from .graph import PushRelation
from .nn import REL_DIRECT, REL_ENGAGE, REL_SOCIAL
from .train import GraphedStep


# ------------------------------------------------------------------------------------------
# async collectives
# ------------------------------------------------------------------------------------------
class _Pending:
    """Result of an async collective: ``wait()`` orders the current stream after it."""

    def __init__(self, work, out, keep=None, post=None):
        self.work, self.out, self.keep, self.post = work, out, keep, post

    def wait(self):
        if self.work is not None:
            self.work.wait()
            self.work = None
        out = self.post(self.out) if self.post is not None else self.out
        self.keep = self.post = None
        return out


def all_gather_rows_async(x_local: torch.Tensor) -> _Pending:
    world = dist.get_world_size()
    x_local = x_local.contiguous()
    out = torch.empty(world * x_local.size(0), *x_local.shape[1:], dtype=x_local.dtype, device=x_local.device)
    return _Pending(dist.all_gather_into_tensor(out, x_local, async_op=True), out, keep=x_local)


def reduce_scatter_rows_async(g_full: torch.Tensor) -> _Pending:
    world, rank = dist.get_world_size(), dist.get_rank()
    chunk = g_full.size(0) // world
    g_full = g_full.contiguous()
    if dist.get_backend() == "gloo":      # gloo has no reduce_scatter: all_reduce + slice
        buf = g_full.clone()
        return _Pending(dist.all_reduce(buf, async_op=True), buf,
                        post=lambda b: b[rank * chunk:(rank + 1) * chunk].clone())
    out = torch.empty(chunk, *g_full.shape[1:], dtype=g_full.dtype, device=g_full.device)
    return _Pending(dist.reduce_scatter_tensor(out, g_full, op=dist.ReduceOp.SUM, async_op=True), out, keep=g_full)


class _Finished:
    """A reduce-scatter in flight whose owned rows are finished (1/deg, local term, ReLU backward) by a
    separate pass on the consumer's stream when they are first needed."""

    def __init__(self, pending, finish):
        self.pending, self.finish = pending, finish

    def wait(self):
        return self.finish(self.pending.wait())


class LibraryComm:
    """The bandwidth collectives as ``torch.distributed`` calls (NCCL kernels on the GPU box -- the A/B of the
    peer-memory path --, gloo in the CPU tests of this host logic)."""

    def begin_step(self):
        pass

    def all_gather_rows_async(self, x_local):
        return all_gather_rows_async(x_local)

    def partial(self, rows, feat, dtype):
        return None                                    # the producing kernel allocates its own table

    def reduce_finish_async(self, part, dtype, prims, row_scale=None, add=None, relu_of=None):
        return _Finished(reduce_scatter_rows_async(part),
                         lambda t: prims.rows_finish(t, dtype, row_scale=row_scale, add=add, relu_of=relu_of))


class PeerMemoryComm:
    """The bandwidth collectives over peer memory (``peer.PeerComm``): copy-engine all-gather, and the
    reduce-scatter fused with the row finish in ``trg_peer_reduce_rows``."""

    def __init__(self, pc):
        self.pc = pc

    def begin_step(self):
        self.pc.begin_step()

    def all_gather_rows_async(self, x_local):
        return self.pc.all_gather_rows_async(x_local)

    def partial(self, rows, feat, dtype):
        return self.pc.acquire_partial(rows, feat, dtype)

    def reduce_finish_async(self, part, dtype, prims, row_scale=None, add=None, relu_of=None):
        return self.pc.reduce_rows_async(part, dtype, row_scale=row_scale, add=add, relu_of=relu_of)


LIBRARY_COMM = LibraryComm()


def comm_for(model, shard: ShardedGraph):
    """Peer-memory collectives for CUDA shards whose ranks can map each other's memory (one NVLink / NVSwitch
    node); ``TRG_DIST_COMM=nccl`` keeps the library collectives (A/B).  The choice is made once per shard."""
    c = getattr(shard, "_comm", None)
    if c is not None:
        return c
    x = shard.x_local["user"]
    c = LIBRARY_COMM
    import os
    # peer (= peer-staged) | peer-direct | nccl; a shard may pin its own mode (``shard.comm_mode``)
    mode = getattr(shard, "comm_mode", None) or os.environ.get("TRG_DIST_COMM", "peer")
    if x.is_cuda and dist.get_backend() == "nccl" and mode != "nccl":
        from .peer import peer_comm_for
        feat = max([x.size(1), shard.x_local["post"].size(1)] + [int(p.size(0)) for p in model.parameters() if p.dim() == 2])
        c = PeerMemoryComm(peer_comm_for(shard, feat, x.dtype, transport_dtype(x.dtype),
                                         reduce_mode="direct" if mode == "peer-direct" else "staged"))
    shard._comm = c
    return c


# ------------------------------------------------------------------------------------------
# compute primitives (CUDA)
# ------------------------------------------------------------------------------------------
class CudaStepPrims:
    """The sm_100a kernels, by the names the step below uses."""

    agg_mean = staticmethod(_agg)                       # (rel, x_src)

    @staticmethod
    def gather_sum(rel, which, x, out=None, accumulate=False, relu_of=None, out_dtype=None):
        from .functional import sage_agg_bwd
        return sage_agg_bwd(rel.fwd if which == "fwd" else rel.bwd, None, x, out=out, accumulate=accumulate,
                            relu_of=relu_of, out_dtype=out_dtype)

    @staticmethod
    def rows_finish(x, dtype, row_scale=None, add=None, relu_of=None):
        from .functional import rows_finish
        return rows_finish(x, dtype, row_scale=row_scale, add=add, relu_of=relu_of)

    @staticmethod
    def proj_fwd(terms, bias, relu):
        from .functional import sage_proj_fwd
        return sage_proj_fwd(terms, bias, relu)

    @staticmethod
    def proj_bwd_weight(dz, terms, want_bias):
        from .functional import sage_proj_bwd_weight
        return sage_proj_bwd_weight(dz, terms, want_bias)

    @staticmethod
    def proj_bwd_input(dz, terms):
        from .functional import sage_proj_bwd_input
        return sage_proj_bwd_input(dz, terms)

    @staticmethod
    def csr(other, key, n_key, n_other, per_step=False, sentinel=False):
        """``sentinel``: the pairs are padded with key = n_key (PaddedPairs); the structure is built with one
        extra row that collects the padding and is never visited (consumers walk rows [0, n_key))."""
        from .graph import build_csr
        c = build_csr(other, key, n_key + (1 if sentinel else 0), n_other, validate=False, per_step=per_step)
        c.n_rows = n_key
        return c

    @staticmethod
    def select_negatives(shard, neg_p_global, capacity=None):
        return shard.select_negatives(neg_p_global, capacity)

    @staticmethod
    def anchor_loss(csr, anchor, gathered, n_edges, label, wbar, g_anchor, relu_gate, coef_in_csr_order=False):
        from .functional import edge_anchor_loss
        return edge_anchor_loss(csr, anchor, gathered, n_edges, label, wbar, True, g_anchor, relu_gate=relu_gate,
                                coef_in_csr_order=coef_in_csr_order)

    @staticmethod
    def wsum(csr, coef, x, out=None, accumulate=False, out_dtype=None):
        from .functional import gather_wsum
        return gather_wsum(csr, coef, x, out=out, accumulate=accumulate, out_dtype=out_dtype)


CUDA_STEP_PRIMS = CudaStepPrims()


def transport_dtype(dtype):
    """dtype in which partial sums cross NVLink: bf16 tables send fp32 partials (each rank's fp32
    accumulation is NOT rounded before the cross-rank add; the owner rounds once, in ``rows_finish``), so
    the sharded bf16 result has the single-GPU kernel's rounding behaviour.  fp32 tables: fp32."""
    return torch.float32 if dtype == torch.bfloat16 else None


def eligible(model, shard: ShardedGraph) -> bool:
    """``fused_step.model_eligible`` on a shard of two or more ranks with the post -> user relation pushed."""
    return shard.world >= 2 and isinstance(shard.rels[REL_DIRECT], PushRelation) and model_eligible(model)


def _host_slice_gather(shard: ShardedGraph, host: torch.Tensor):
    """The shard's ``HostSliceGather`` for host arrays the size of ``host``, cached as ``shard._neg_gather``."""
    hg = getattr(shard, "_neg_gather", None)
    if hg is None or hg.n != host.numel():
        from .peer import HostSliceGather
        hg = shard._neg_gather = HostSliceGather(host.numel(), host.dtype, shard.x_local["user"].device)
    return hg


@torch.no_grad()
def loss_and_grads_sharded(model, shard: ShardedGraph, neg_p_local, prims=CUDA_STEP_PRIMS, neg_ready=None,
                           neg_p_global=None, neg_capacity=None, comm=None):
    """Forward + link loss + backward on this rank's partition.  Returns the LOCAL partial loss
    (0-d); local parameter-gradient partials are accumulated into ``.grad`` (the caller all-reduces
    both).  Negatives: ``neg_p_local`` = ``shard.local_negatives(neg_p)`` (or a ``PaddedPairs``), or
    ``neg_p_global`` = the step's full ``neg_p`` -- this rank's share is then selected here, on the device
    and without a host sync, while the final user rows are being all-gathered."""
    layers = _layers(model)
    if layers is None:
        raise _lib.TrgError("loss_and_grads_sharded: model must be WeightedRGCN or StackedWeightedRGCN")
    prel_d, rel_s, rel_e = shard.rels[REL_DIRECT], shard.rels[REL_SOCIAL], shard.rels[REL_ENGAGE]
    rel_d = prel_d.rel                                  # rows ("fwd") = all users, sources = local posts
    hu, hp = shard.x_local["user"], shard.x_local["post"]
    n_u_pad = shard.cu * shard.world
    dtype = hu.dtype
    xfer = transport_dtype(dtype)
    pdt = xfer or dtype                                 # element type of the partial-sum tables
    comm = comm or LIBRARY_COMM
    comm.begin_step()

    # ---- forward ----
    saved = []
    for i, layer in enumerate(layers):
        layer.materialize(hu.size(-1), hp.size(-1))
        ag = None if i == 0 else comm.all_gather_rows_async(hu)
        part = prims.gather_sum(rel_d, "fwd", hp, out=comm.partial(n_u_pad, hp.size(1), pdt),
                                out_dtype=xfer)                          # [U_pad, F] partial sums  || all-gather
        rs = comm.reduce_finish_async(part, dtype, prims, row_scale=prel_d.inv_deg)   # sum / global in-degree
        del part
        user_full = shard.layer0_sources()["user"] if i == 0 else ag.wait()
        mean_s = prims.agg_mean(rel_s, user_full)                        # || reduce-scatter
        mean_e = prims.agg_mean(rel_e, user_full)
        del user_full
        pg = layer.post_gemm()
        hp_n = prims.proj_fwd(pg.terms(mean_e, hp), pg.bias, True)
        mean_d = rs.wait()
        ug = layer.user_gemm()
        hu_n = prims.proj_fwd(ug.terms(mean_d, mean_s, hu), ug.bias, True)
        saved.append((hu, hp, mean_d, mean_s, mean_e, ug, pg))
        hu, hp = hu_n, hp_n

    # ---- loss: every <u, p> term is evaluated by the owner of the post (dist.ShardedGraph) ----
    ag = comm.all_gather_rows_async(hu)
    st = shard.loss_structures(prims)
    if neg_ready is not None:          # host negatives: their copy ran on a side stream during the forward
        torch.cuda.current_stream().wait_event(neg_ready)
    if neg_p_local is None:
        neg_p_local = prims.select_negatives(shard, neg_p_global, neg_capacity)                    # || all-gather
    padded = isinstance(neg_p_local, PaddedPairs)
    neg_u, neg_pl = (neg_p_local.user, neg_p_local.post) if padded else (neg_p_local[0], neg_p_local[1])
    kw = {"sentinel": True} if padded else {}
    neg_by_post = prims.csr(neg_u, neg_pl, shard.cp, n_u_pad, per_step=True, **kw)                  # || all-gather
    neg_by_user = prims.csr(neg_pl, neg_u, n_u_pad, shard.cp, per_step=True, **kw)
    user_full = ag.wait()
    e_glob = shard.n_pos_global
    seq = "pos_by_user_p" in st     # positives: coefficients written in by-post order (static remap)
    l_pos, c_pos, g_p = prims.anchor_loss(st["pos_by_post"], hp, user_full, e_glob, 1, shard.wbar, None, False,
                                          **({"coef_in_csr_order": True} if seq else {}))
    l_neg, c_neg, dz_p = prims.anchor_loss(neg_by_post, hp, user_full, e_glob, 0, shard.wbar, g_p, True)
    del user_full
    g_uf = prims.wsum(st["pos_by_user_p" if seq else "pos_by_user"], c_pos, hp,
                      out=comm.partial(n_u_pad, hp.size(1), pdt), out_dtype=xfer)              # dL/du partials, all users
    g_uf = prims.wsum(neg_by_user, c_neg, hp, out=g_uf, accumulate=True)
    # partials in flight; the owner adds its local term and applies the ReLU backward (gate = hu)
    pend_u = comm.reduce_finish_async(g_uf, dtype, prims, relu_of=hu)
    loss_local = (l_pos + l_neg).reshape(())
    del g_uf, c_pos, c_neg, neg_by_post, neg_by_user, hu, hp

    # ---- backward ----
    for li in range(len(layers) - 1, -1, -1):
        hu_in, hp_in, mean_d, mean_s, mean_e, ug, pg = saved.pop()
        # post side first: it does not depend on the user-gradient reduce-scatter still in flight
        dw_p, db_p = prims.proj_bwd_weight(dz_p, pg.dw_terms(mean_e, hp_in), True)
        g_uf = g_hp = None
        if li > 0:
            g_me, g_hp = prims.proj_bwd_input(dz_p, pg.dx_terms(rel_e.inv_deg, None))
            g_uf = prims.gather_sum(rel_e, "bwd", g_me, out=comm.partial(n_u_pad, g_me.size(1), pdt),
                                    out_dtype=xfer)                      # d user_full partials (engages^T)
            del g_me
        del dz_p, mean_e
        dz_u = pend_u.wait()                                  # reduced (+ local term), ReLU backward applied
        del pend_u
        dw_u, db_u = prims.proj_bwd_weight(dz_u, ug.dw_terms(mean_d, mean_s, hu_in), True)
        del mean_d, mean_s
        layers[li].accumulate_grads(dw_u, db_u, dw_p, db_p)
        if li == 0:
            break
        g_md, g_ms, g_hu = prims.proj_bwd_input(dz_u, ug.dx_terms(prel_d.inv_deg, rel_s.inv_deg, None))
        del dz_u
        ag = comm.all_gather_rows_async(g_md)                         # every post owner needs d mean_direct
        g_uf = prims.gather_sum(rel_s, "bwd", g_ms, out=g_uf, accumulate=True)      # || all-gather
        pend_u = comm.reduce_finish_async(g_uf, dtype, prims, add=g_hu, relu_of=hu_in)
        del g_uf, g_ms, g_hu
        g_md_full = ag.wait()
        dz_p = prims.gather_sum(rel_d, "bwd", g_md_full, out=g_hp, accumulate=True, relu_of=hp_in)  # || reduce-scatter
        del g_md_full, g_md
    return loss_local


class GraphedShardedStep(GraphedStep):
    """The sharded step -- forward, loss, backward, every collective, the gradient all-reduce -- captured ONCE
    into a CUDA graph and replayed per step (``train_step_sharded_fused(..., cuda_graph=True)``; the capture and
    replay are :class:`train.GraphedStep`'s).

    At 8 GPUs one step is ~9 ms of GPU work behind ~85 kernel launches, ~60 copy-engine transfers and ~120
    stream/event operations: enqueueing them from Python takes as long as executing them (9 - 11 ms measured),
    so the eager step is host-bound.  The replay is one launch.  Host negatives are uploaded with the shard's
    ``HostSliceGather`` when the ranks share peer memory."""

    def __init__(self, model, optimizer, shard: ShardedGraph, neg_capacity=None):
        if not eligible(model, shard) or not shard.x_local["user"].is_cuda:
            raise ValueError("GraphedShardedStep needs a CUDA shard and a model the tape-free sharded step accepts")
        super().__init__(model, optimizer, shard.n_pos_global, shard.x_local["user"].device)
        self.shard, self.neg_capacity = shard, neg_capacity
        self.comm = comm_for(model, shard)

    def _body(self):
        loss = loss_and_grads_sharded(self.model, self.shard, None, CUDA_STEP_PRIMS, neg_ready=self.neg_ready,
                                      neg_p_global=self.neg, neg_capacity=self.neg_capacity, comm=self.comm).clone()
        lw = dist.all_reduce(loss, async_op=True)
        allreduce_grads(list(self.model.parameters()))
        lw.wait()
        return loss

    def _draw_negatives(self):
        return self.shard.draw_negatives()

    def _upload(self, neg_p_global):
        if not neg_p_global.is_cuda and isinstance(self.comm, PeerMemoryComm):
            hg = _host_slice_gather(self.shard, neg_p_global)
            hg.gather_async(neg_p_global, out=self.neg, event=self.neg_ready)     # side stream: overlaps the forward
        else:
            self.neg.copy_(neg_p_global, non_blocking=True)
            self.neg_ready.record()

    def _before_capture(self):
        dist.barrier()
        if isinstance(self.comm, PeerMemoryComm):
            self.comm.pc._last_barrier = None        # an event recorded outside the capture cannot be waited inside


def train_step_sharded_fused(model, optimizer, shard: ShardedGraph, neg_p_global=None, neg_p_local=None,
                             prims=CUDA_STEP_PRIMS, return_tensor=False, neg_capacity=None, cuda_graph=False):
    """``dist.train_step_sharded`` without the tape and with the collectives overlapped.

    ``neg_p_global``: the step's ``torch.randint(0, P, (E,))`` (train_gnn.py:272) -- the SAME array on every
    rank, device or (pinned) host; ``None`` draws it from the shard's rank-synchronised generator.  Each rank
    keeps the pairs whose negative post it owns; that selection runs on the device inside the step with no
    host synchronisation (``ShardedGraph.select_negatives``; ``neg_capacity`` overrides its room).
    ``neg_p_local``: a share already selected by the caller (``shard.local_negatives``).
    ``cuda_graph``: replay the step from a CUDA graph captured on the first call (``GraphedShardedStep``)."""
    if cuda_graph:
        if neg_p_local is not None or prims is not CUDA_STEP_PRIMS:
            raise ValueError("cuda_graph=True takes the step's global negatives and the CUDA primitives")
        gs = getattr(shard, "_graphed", None)
        if gs is None or gs.model is not model or gs.optimizer is not optimizer:
            gs = shard._graphed = GraphedShardedStep(model, optimizer, shard, neg_capacity)
        return gs(neg_p_global, return_tensor=return_tensor)
    model.train()
    optimizer.zero_grad()
    is_cuda = shard.x_local["user"].is_cuda
    neg_ready = None
    if neg_p_local is None:
        if neg_p_global is None:
            neg_p_global = shard.draw_negatives()          # rank-synchronised generator: same array everywhere
        if not neg_p_global.is_cuda and is_cuda:
            if prims is CUDA_STEP_PRIMS and isinstance(comm_for(model, shard), PeerMemoryComm):
                # every rank holds the same host array: upload 1/G of it, pull the rest over NVLink
                neg_p_global, neg_ready = _host_slice_gather(shard, neg_p_global).gather_async(neg_p_global)
            else:
                from .train import stage_negatives
                neg_p_global, neg_ready = stage_negatives(neg_p_global, shard.x_local["user"].device)
    elif torch.is_tensor(neg_p_local) and not neg_p_local.is_cuda and is_cuda:
        from .train import stage_negatives
        neg_p_local, neg_ready = stage_negatives(neg_p_local, shard.x_local["user"].device)
    loss = loss_and_grads_sharded(model, shard, neg_p_local, prims, neg_ready=neg_ready, neg_p_global=neg_p_global,
                                  neg_capacity=neg_capacity,
                                  comm=comm_for(model, shard) if prims is CUDA_STEP_PRIMS else LIBRARY_COMM).clone()
    lw = dist.all_reduce(loss, async_op=True)
    allreduce_grads(list(model.parameters()))
    optimizer.step()
    lw.wait()
    return loss if return_tensor else loss.item()

"""Multi-GPU execution of the hot path: destination-node partitioning (SURVEY.md §8e).

One process per GPU (``torch.distributed``; NCCL over NVLink on the B200 box, gloo in the CPU
tests of this host logic).  Rank g owns a contiguous range of users and of posts, the CSR rows of
all three relations whose destination falls in its ranges, and the matching activation rows.
Per layer the user table and the post table are all-gathered ONCE each (users feed two relations);
the backward of that gather is a reduce-scatter of the source-gradient partials; weight gradients
are all-reduced as one flat buffer.  The loss partitions the positive edges by owner of ``pos_u``.
Inference shards the catalogue by post-id range and merges per-shard top-k lists.

The reference has no distributed code at all (single process, single device: train_gnn.py:205);
this is the scaling axis BASELINE.json asks for.
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from .graph import PushRelation, RelationGraph
from .nn import CUDA_OPS, REL_DIRECT, REL_ENGAGE, REL_SOCIAL, StackedWeightedRGCN, WeightedRGCN


def chunk_of(n: int, world: int) -> int:
    return (n + world - 1) // world


from .collectives import all_gather_rows, all_gather_rows_raw as _all_gather_rows  # noqa: E402


# ------------------------------------------------------------------------------------------
# partitioned graph
# ------------------------------------------------------------------------------------------
class ShardedGraph:
    """This rank's share of the graph, built from the full COO ``edge_index_dict`` (reference
    format).  Source ids stay global (row r of an all-gathered table is global id r because the
    ranges are contiguous chunks); destination ids become local."""

    def __init__(self, x_dict, edge_index_dict, train_edge_index, interaction_type_tensor,
                 num_users, num_posts, rank=None, world=None):
        self.rank = dist.get_rank() if rank is None else rank
        self.world = dist.get_world_size() if world is None else world
        self.num_users, self.num_posts = int(num_users), int(num_posts)
        self.cu, self.cp = chunk_of(num_users, self.world), chunk_of(num_posts, self.world)
        self.u0, self.p0 = self.rank * self.cu, self.rank * self.cp
        self.u1, self.p1 = min(self.u0 + self.cu, num_users), min(self.p0 + self.cp, num_posts)
        n_of = {"user": (self.u0, self.u1, self.cu), "post": (self.p0, self.p1, self.cp)}
        # owned feature rows, zero-padded to the chunk size so every rank gathers equal shapes
        self.x_local = {}
        for t, (a, b, c) in n_of.items():
            x = x_dict[t]
            xl = torch.zeros(c, x.size(1), dtype=x.dtype, device=x.device)
            xl[:max(b - a, 0)] = x[a:b]
            self.x_local[t] = xl
        # per relation: edges whose destination is owned; dst -> local id
        self.rels = {}
        self.n_local_edges = {}
        for rel in (REL_DIRECT, REL_SOCIAL, REL_ENGAGE):
            ei = edge_index_dict[rel]
            if rel == REL_DIRECT and self.world > 1:
                # post -> user is partitioned by SOURCE: partial sums for all users are pushed to
                # their owners (U x H moves instead of an all-gather of the 5x larger post table)
                a, b, c = n_of["post"]
                m = (ei[0] >= a) & (ei[0] < b)
                loc = torch.stack([ei[0][m] - a, ei[1][m]]).contiguous()
                deg = torch.bincount(ei[1], minlength=num_users)[self.u0:self.u1].float()
                inv = torch.ones(self.cu, device=ei.device)
                inv[:deg.numel()] = 1.0 / deg.clamp(min=1.0)
                self.rels[rel] = PushRelation(RelationGraph(loc, c, self.cu * self.world), inv)
                self.n_local_edges[rel] = int(loc.size(1))
                continue
            a, b, c = n_of[rel[2]]
            m = (ei[1] >= a) & (ei[1] < b)
            loc = torch.stack([ei[0][m], ei[1][m] - a]).contiguous()
            n_src_pad = n_of[rel[0]][2] * self.world
            self.rels[rel] = RelationGraph(loc, n_src_pad, c)
            self.n_local_edges[rel] = int(loc.size(1))
        # loss (train_gnn.py:259-281): every term <u, p> is evaluated by the OWNER OF THE POST against
        # the all-gathered user table (U x H moves instead of the 5x larger post table): positives
        # with pos_p owned here (static), negatives with neg_p owned here (selected every step)
        pos_u, pos_p = train_edge_index[0], train_edge_index[1]
        self.pos_u_global = pos_u.contiguous()
        self.pos_mask = (pos_p >= self.p0) & (pos_p < self.p1)
        self.pos_local = torch.stack([pos_u[self.pos_mask], pos_p[self.pos_mask] - self.p0]).contiguous()
        self.n_pos_global = int(train_edge_index.size(1))
        w = interaction_type_tensor[pos_p[self.pos_mask] + num_users].float()
        wsum = torch.stack([w.sum(), torch.tensor(float(w.numel()), device=w.device)])
        if self.world > 1:
            dist.all_reduce(wsum)
        self.wbar = (wsum[0] / wsum[1]).reshape(1).float().contiguous()
        self._layer0_src = None
        self._neg_gen = None

    def draw_negatives(self):
        """``neg_p = torch.randint(0, num_posts, (E,))`` of train_gnn.py:272 for a step whose caller supplies
        none.  Every rank must see the SAME array (each keeps the entries whose post it owns, and their union
        has to be one negative per positive edge): it is drawn from a dedicated device generator seeded with
        a value broadcast from rank 0 when first used and advanced identically on every rank afterwards --
        never from the ranks' own default generators, whose states are unrelated."""
        dev = self.pos_u_global.device
        if self._neg_gen is None:
            seed = torch.randint(0, 2**62, (1,), dtype=torch.int64)
            if self.world > 1:
                seed = seed.to(dev) if dist.get_backend() == "nccl" else seed
                dist.broadcast(seed, src=0)
            self._neg_gen = torch.Generator(device=dev).manual_seed(int(seed.item()))
        return torch.randint(0, self.num_posts, (self.n_pos_global,), generator=self._neg_gen, device=dev)

    def local_negatives(self, neg_p_global):
        """This rank's share of ``neg_p = torch.randint(0, P, (E,))`` (train_gnn.py:272): the pairs
        (pos_u[e], neg_p[e]) whose negative post is owned here, as (global user, local post)."""
        m = (neg_p_global >= self.p0) & (neg_p_global < self.p1)
        return torch.stack([self.pos_u_global[m], neg_p_global[m] - self.p0]).contiguous()

    @classmethod
    def from_generator(cls, cg, device, dtype=torch.float32, rank=None, world=None, chunk=32_000_000):
        """This rank's share of a counter-based graph (``synth.CounterGraph``), produced ON THIS DEVICE without
        the full graph ever existing anywhere: the edge streams are generated ``chunk`` edges at a time and
        filtered by ownership, feature rows are generated for the owned ranges only.  Same attributes, same
        edge order and therefore bit-identical structures as ``ShardedGraph(cg.materialize(...))`` (tested);
        this is how BASELINE config 4 (1B edges, H = 256) is set up on 8 x 180 GB."""
        self = cls.__new__(cls)
        self.rank = dist.get_rank() if rank is None else rank
        self.world = dist.get_world_size() if world is None else world
        U, P = cg.num_users, cg.num_posts
        self.num_users, self.num_posts = U, P
        self.cu, self.cp = chunk_of(U, self.world), chunk_of(P, self.world)
        self.u0, self.p0 = self.rank * self.cu, self.rank * self.cp
        self.u1, self.p1 = min(self.u0 + self.cu, U), min(self.p0 + self.cp, P)
        self.x_local = {}
        for t, (a, b, c) in (("user", (self.u0, self.u1, self.cu)), ("post", (self.p0, self.p1, self.cp))):
            xl = torch.zeros(c, cg.feat, dtype=dtype, device=device)
            if b > a:
                xl[:b - a] = cg.features(t, a, b, device, dtype)
            self.x_local[t] = xl

        def stream(rel, keep):
            """Concatenate ``keep(edge chunk)`` over the whole edge stream of ``rel``."""
            parts = []
            for a in range(0, cg.n_edges(rel), chunk):
                parts.append(keep(cg.edges(rel, a, min(a + chunk, cg.n_edges(rel)), device)))
            if not parts:
                return torch.empty(2, 0, dtype=torch.int64, device=device)
            return torch.cat(parts, dim=1).contiguous()

        def by_dst(a, b):
            return lambda ei: torch.stack([ei[0], ei[1] - a])[:, (ei[1] >= a) & (ei[1] < b)]

        self.rels, self.n_local_edges = {}, {}
        n_u_pad, n_p_pad = self.cu * self.world, self.cp * self.world
        if self.world > 1:
            # post -> user partitioned by SOURCE post (see __init__); global in-degree of the owned users
            deg = torch.zeros(self.cu, dtype=torch.int64, device=device)
            parts = []
            for a in range(0, cg.e_eng, chunk):
                ei = cg.edges(REL_DIRECT, a, min(a + chunk, cg.e_eng), device)
                m = (ei[0] >= self.p0) & (ei[0] < self.p1)
                parts.append(torch.stack([ei[0] - self.p0, ei[1]])[:, m])
                own = ei[1][(ei[1] >= self.u0) & (ei[1] < self.u1)] - self.u0
                deg += torch.bincount(own, minlength=self.cu)
            loc = torch.cat(parts, dim=1).contiguous() if parts else torch.empty(2, 0, dtype=torch.int64, device=device)
            inv = 1.0 / deg.clamp(min=1).float()
            self.rels[REL_DIRECT] = PushRelation(RelationGraph(loc, self.cp, n_u_pad), inv)
        else:
            loc = stream(REL_DIRECT, by_dst(self.u0, self.u1))
            self.rels[REL_DIRECT] = RelationGraph(loc, n_p_pad, self.cu)
        self.n_local_edges[REL_DIRECT] = int(loc.size(1))
        loc = stream(REL_SOCIAL, by_dst(self.u0, self.u1))
        self.rels[REL_SOCIAL] = RelationGraph(loc, n_u_pad, self.cu)
        self.n_local_edges[REL_SOCIAL] = int(loc.size(1))
        loc = stream(REL_ENGAGE, by_dst(self.p0, self.p1))
        self.rels[REL_ENGAGE] = RelationGraph(loc, n_u_pad, self.cp)
        self.n_local_edges[REL_ENGAGE] = int(loc.size(1))
        # loss: positives = the engagement edges, evaluated by the owner of the post -> exactly the local
        # engages edges (same filter, same order): (global user, local post)
        self.pos_local = loc
        self.pos_mask = None                       # a full-length mask is never built here
        self.n_pos_global = cg.e_eng
        self.pos_u_global = torch.cat([cg.edges(REL_ENGAGE, a, min(a + chunk, cg.e_eng), device)[0]
                                       for a in range(0, cg.e_eng, chunk)]).contiguous() if cg.e_eng else \
            torch.empty(0, dtype=torch.int64, device=device)
        w = cg.post_weight(loc[1] + self.p0)
        wsum = torch.stack([w.sum(), torch.tensor(float(w.numel()), device=device)])
        if self.world > 1:
            dist.all_reduce(wsum)
        self.wbar = (wsum[0] / wsum[1]).reshape(1).float().contiguous()
        self._layer0_src = None
        self._neg_gen = None
        return self

    def neg_capacity(self):
        """Room for this rank's share of E uniformly drawn negatives: mean E/G plus 8 standard deviations of
        the binomial count (overflow probability ~1e-15) plus slack."""
        import math
        # torch.randint (train_gnn.py:272) maps a 32-bit draw with `% P` when P < 2^32: the low
        # (2^32 mod P) values come up floor(2^32 / P) + 1 times in 2^32, the rest floor(2^32 / P) times.
        # At P = 50M that is a +1.2 % share for the low ids -- more than 8 sigma of a 100M-entry share --
        # so the bound uses the largest per-value probability, not 1 / P.
        p_max = 1.0 / self.num_posts
        if self.num_posts < 2**32:
            p_max = (2**32 // self.num_posts + 1) / 2.0**32
        mean = self.n_pos_global * min(1.0, self.cp * p_max)
        return int(min(self.n_pos_global, mean + 8.0 * math.sqrt(max(mean, 1.0)) + 1024))

    def select_negatives(self, neg_p_global, capacity=None):
        """``local_negatives`` without a host synchronisation (``trg_select_range``): the pairs
        (pos_u[e], neg_p[e] - p0) with neg_p[e] owned here, in edge order, padded to ``capacity`` entries with the
        sentinel pair (n_users_padded, posts_per_rank) that CSR builds with one extra row absorb.  The count
        never travels to the host, so the CPU keeps enqueueing ahead of the GPU; more than ``capacity`` local
        negatives (a caller whose negatives are far from ``torch.randint``'s uniform draw, train_gnn.py:272)
        abort the kernel with a message -- pass ``capacity=E`` or use ``local_negatives`` for such inputs."""
        from . import _lib
        lib = _lib.load()
        e = self.n_pos_global
        if neg_p_global.dtype != torch.int64 or neg_p_global.numel() != e:
            raise _lib.TrgError("neg_p must be int64 with one entry per positive edge (train_gnn.py:272)")
        cap = int(self.neg_capacity() if capacity is None else capacity)
        dev = self.pos_u_global.device
        user = torch.empty(cap, dtype=torch.int64, device=dev)
        post = torch.empty(cap, dtype=torch.int64, device=dev)
        count = torch.empty(1, dtype=torch.int32, device=dev)
        ws_bytes = int(lib.trg_select_range_workspace_bytes(e))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        _lib.call("trg_select_range", e * 16 + cap * 32, lib.trg_select_range, _lib.ptr(neg_p_global.contiguous()),
                  _lib.ptr(self.pos_u_global), e, self.p0, self.p1, cap, self.cp, self.cu * self.world,
                  _lib.ptr(post), _lib.ptr(user), _lib.ptr(count), _lib.ptr(ws), ws_bytes, _lib.stream())
        return PaddedPairs(user, post, count)

    def layer0_sources(self):
        """Input features are static: gather them once (train_gnn.py:211 moves the graph once)."""
        if self._layer0_src is None:
            self._layer0_src = {"user": _all_gather_rows(self.x_local["user"]), "post": self.x_local["post"]}
        return self._layer0_src


class PaddedPairs:
    """(global user, local post) pairs of this rank's negatives padded to a fixed capacity with sentinel ids
    (``ShardedGraph.select_negatives``); ``count`` is a device int32 -- nothing here is known on the host."""

    def __init__(self, user, post, count):
        self.user, self.post, self.count = user, post, count


def forward_sharded(model, shard: ShardedGraph, ops=CUDA_OPS):
    """Forward of ``WeightedRGCN`` / ``StackedWeightedRGCN`` on this rank's destination rows."""
    layers = list(model.layers) if isinstance(model, StackedWeightedRGCN) else [model]
    dst = shard.x_local
    for i, layer in enumerate(layers):
        # only the user table is gathered: posts are consumed where they live (PushRelation)
        src = shard.layer0_sources() if i == 0 else {"user": all_gather_rows(dst["user"]), "post": dst["post"]}
        dst = layer.forward_partitioned(src, dst, shard.rels, ops)
    return dst


class AnchoredLinkLossFn(torch.autograd.Function):
    """Partial link loss of this rank (post-owner partition) and its backward.  ``prims`` supplies the
    compute primitives (CUDA kernels in the product, oracle ops in the CPU host-logic tests):
      prims.anchor_loss(csr, post_local, user_full, E, label, wbar, want_grad, g_post) -> (loss, coef, g_post)
      prims.wsum(csr, coef, post_local, scale, out) -> out
      prims.csr(other, key, n_key, n_other) -> CSR"""

    @staticmethod
    def forward(ctx, user_full, post_local, neg_pairs, shard, prims):
        want = user_full.requires_grad or post_local.requires_grad
        st = shard.loss_structures(prims)
        n_u_pad = shard.cu * shard.world
        neg_by_post = prims.csr(neg_pairs[0], neg_pairs[1], shard.cp, n_u_pad, per_step=True)
        lp, c_pos, g_p = prims.anchor_loss(st["pos_by_post"], post_local, user_full, shard.n_pos_global, 1,
                                           shard.wbar, want, None)
        ln, c_neg, g_p = prims.anchor_loss(neg_by_post, post_local, user_full, shard.n_pos_global, 0,
                                           shard.wbar, want, g_p)
        ctx.shard, ctx.prims, ctx.st, ctx.want = shard, prims, st, want
        if want:
            ctx.save_for_backward(post_local, neg_pairs, c_pos, c_neg, g_p)
        return (lp + ln).reshape(())

    @staticmethod
    def backward(ctx, g):
        post_local, neg_pairs, c_pos, c_neg, g_p = ctx.saved_tensors
        shard, prims, st = ctx.shard, ctx.prims, ctx.st
        g = g.reshape(1).float().contiguous()
        g_user = g_post = None
        if ctx.needs_input_grad[1]:
            g_post = g_p * g.to(g_p.dtype)
        if ctx.needs_input_grad[0]:
            n_u_pad = shard.cu * shard.world
            # dloss/du for ALL users touched by local edges; AllGatherRows.backward reduce-scatters it
            g_user = prims.wsum(st["pos_by_user"], c_pos, post_local, g, None)
            neg_by_user = prims.csr(neg_pairs[1], neg_pairs[0], n_u_pad, shard.cp, per_step=True)
            g_user = prims.wsum(neg_by_user, c_neg, post_local, g, g_user)
        return g_user, g_post, None, None, None


class CudaLossPrims:
    @staticmethod
    def csr(other, key, n_key, n_other, per_step=False):
        from .graph import build_csr
        return build_csr(other, key, n_key, n_other, validate=False, per_step=per_step)

    @staticmethod
    def anchor_loss(csr, post_local, user_full, n_edges, label, wbar, want, g_post):
        from .functional import edge_anchor_loss
        return edge_anchor_loss(csr, post_local, user_full, n_edges, label, wbar, want, g_post)

    @staticmethod
    def wsum(csr, coef, post_local, scale, out):
        from .functional import gather_wsum
        return gather_wsum(csr, coef, post_local, scale=scale, out=out, accumulate=out is not None)


CUDA_LOSS_OPS = CudaLossPrims()


def _loss_structures(self, prims):
    st = getattr(self, "_loss_st", None)
    if st is None:
        pu, pp = self.pos_local[0], self.pos_local[1]
        n_u_pad = self.cu * self.world
        st = {"pos_by_post": prims.csr(pu, pp, self.cp, n_u_pad),
              "pos_by_user": prims.csr(pp, pu, n_u_pad, self.cp)}
        # pos_by_user with edge ids that are BY-POST CSR POSITIONS: the post-anchored loss pass can then
        # write its per-edge coefficients sequentially (dist_fused); static, built once
        bp, bu = st["pos_by_post"], st["pos_by_user"]
        if hasattr(bp, "eid") and hasattr(bu, "eid") and torch.is_tensor(getattr(bp, "eid", None)):
            from .graph import CSR
            inv = torch.empty(bp.eid.numel(), dtype=torch.int32, device=bp.eid.device)
            inv[bp.eid.long()] = torch.arange(bp.eid.numel(), dtype=torch.int32, device=bp.eid.device)
            st["pos_by_user_p"] = CSR(bu.rowptr, bu.col, inv[bu.eid.long()].contiguous(), bu.n_rows, bu.n_cols, bu._long)
        self._loss_st = st
    return st


ShardedGraph.loss_structures = _loss_structures


def allreduce_grads(params):
    """One flat all-reduce (sum) of every weight gradient (9*L small tensors: latency-bound)."""
    grads = [p.grad for p in params if p.grad is not None]
    if not grads or dist.get_world_size() == 1:
        return
    flat = torch.cat([g.reshape(-1).float() for g in grads])
    dist.all_reduce(flat)
    off = 0
    for p in params:
        g = p.grad
        if g is None:
            continue
        n = g.numel()
        if g.dtype == torch.float32:
            p.grad = flat[off:off + n].view_as(g)      # a view of the reduced buffer: no copy-back kernel
        else:
            g.copy_(flat[off:off + n].view_as(g))
        off += n


def train_step_sharded(model, optimizer, shard: ShardedGraph, neg_p_global=None, neg_p_local=None,
                       ops=CUDA_OPS, loss_ops=CUDA_LOSS_OPS, return_tensor=False):
    """The body of ``train()`` (train_gnn.py:242-285) on a destination partition.  Every rank holds
    the same weights; the returned loss is the global loss (identical on all ranks).
    ``neg_p_global``: the step's ``torch.randint(0, P, (E,))`` -- it MUST be the same array on every rank;
    ``None`` draws it from the shard's rank-synchronised generator (``ShardedGraph.draw_negatives``) --
    or ``neg_p_local``: this rank's share already selected with ``shard.local_negatives``."""
    model.train()
    optimizer.zero_grad()
    out = forward_sharded(model, shard, ops)
    user_full = all_gather_rows(out["user"])
    if neg_p_local is None:
        if neg_p_global is None:
            neg_p_global = shard.draw_negatives()
        neg_p_local = shard.local_negatives(neg_p_global)
    loss_local = AnchoredLinkLossFn.apply(user_full, out["post"], neg_p_local, shard, loss_ops)
    loss_local.backward()
    allreduce_grads(list(model.parameters()))
    optimizer.step()
    loss = loss_local.detach().clone()
    if shard.world > 1:
        dist.all_reduce(loss)
    return loss if return_tensor else loss.item()


@torch.no_grad()
def recommend_sharded(q, cat_local, k, id_offset, score_topk_fn=None, merge_fn=None, exclude=None, rows=None):
    """Catalogue sharded by post-id range: local score + top-k, all-gather of the per-shard
    ``(values, global ids)``, merge under (score desc, id asc) == the unsharded result.
    ``exclude`` / ``rows`` (see ``score_topk``): every rank passes the same index, since its ids are
    global; rows short of admissible posts end in ``(-inf, -1)`` pads, as unsharded."""
    from . import functional as Fn
    score_topk_fn = score_topk_fn or Fn.score_topk
    merge_fn = merge_fn or Fn.topk_merge
    world = dist.get_world_size()
    if exclude is None and rows is None:
        vals, ids = score_topk_fn(q, cat_local, k, id_offset)
    else:
        vals, ids = score_topk_fn(q, cat_local, k, id_offset, exclude=exclude, rows=rows)
    kk = vals.size(1)
    if world == 1:
        return vals, ids
    pad_id = torch.iinfo(torch.int64).max
    if exclude is not None:
        # the merge treats only id INT64_MAX as padding
        ids = torch.where(ids < 0, torch.full_like(ids, pad_id), ids)
    # shards may hold fewer than k posts: pad lists so every rank contributes k columns
    if kk < k:
        pad = k - kk
        vals = torch.cat([vals, torch.full((vals.size(0), pad), float("-inf"), device=vals.device)], 1)
        ids = torch.cat([ids, torch.full((ids.size(0), pad), pad_id, device=ids.device)], 1)
    b = vals.size(0)
    av = torch.empty(world * b, k, dtype=vals.dtype, device=vals.device)
    ai = torch.empty(world * b, k, dtype=ids.dtype, device=ids.device)
    dist.all_gather_into_tensor(av, vals.contiguous())
    dist.all_gather_into_tensor(ai, ids.contiguous())
    av = av.view(world, b, k).permute(1, 0, 2).reshape(b, -1).contiguous()
    ai = ai.view(world, b, k).permute(1, 0, 2).reshape(b, -1).contiguous()
    return merge_fn(av, ai, world, k)

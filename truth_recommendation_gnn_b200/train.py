"""The reference's training step and recommendation call, on the B200 kernels.

``train_step`` is the body of ``train()`` (train_gnn.py:242-285) with the same order of
operations: zero_grad -> forward -> positive/negative scoring -> loss -> backward -> Adam step.
``recommend`` is inference.py:427-428.
"""
from __future__ import annotations

import torch

from . import _lib, fused_step
from .functional import link_bce_loss, score_topk


_COPY_STREAMS: dict = {}


def stage_negatives(neg_p, device):
    """This step's host input (the sampled negatives, train_gnn.py:272, when they are drawn on the host):
    start the host -> device copy on a side stream so that it overlaps the forward pass, which does not
    need them.  Returns ``(device tensor, event)``; the consumer waits on the event right before the loss.
    Device tensors pass through (``event`` is None)."""
    if neg_p is None or neg_p.is_cuda or torch.device(device).type != "cuda":
        return neg_p, None       # (host features: the model itself raises TrgError -- there is no CPU path)
    device = torch.device(device)
    side = _COPY_STREAMS.get(device)
    if side is None:
        side = _COPY_STREAMS[device] = torch.cuda.Stream(device=device)
    with torch.cuda.stream(side):
        dev_t = neg_p.to(device, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(side)
    dev_t.record_stream(torch.cuda.current_stream(device))
    return dev_t, ev


class GraphedStep:
    """A tape-free train step (subclasses supply ``_body``, ``_draw_negatives``, ``_upload``) captured into a
    CUDA graph on the first call, after two warm-up passes with that call's negatives (structures and lazy
    weights materialise there; the optimiser is NOT stepped), and replayed as one launch per step.  Outside the
    graph: ``_upload`` of the step's negatives into the static input ``neg``, ending with ``neg_ready``, an
    ``external`` event whose wait node sits right before the loss, so a host array still uploads during the
    replayed forward; the caller's ``optimizer.step()``; the loss read-back.  The ``.grad`` tensors live in the
    graph's pool and are rewritten by every replay: ``optimizer.zero_grad()`` must not set them to None."""

    def __init__(self, model, optimizer, n_neg, device):
        self.model, self.optimizer = model, optimizer
        self.neg = torch.empty(n_neg, dtype=torch.int64, device=device)
        self.neg_ready = torch.cuda.Event(external=True)
        self.graph = self.loss = None
        self.params, self.grads, self.launches_per_replay = [], [], 0

    def _before_capture(self):
        pass

    def _capture(self):
        if _lib.PROF.enabled:
            raise _lib.TrgError(f"{type(self).__name__}: per-call event timing (PROF) cannot run in a graph capture")
        cur = torch.cuda.current_stream()
        warm = torch.cuda.Stream(self.neg.device)
        warm.wait_stream(cur)
        with torch.cuda.stream(warm):
            for _ in range(2):            # structures (CSRs), lazy weights, allocator; the optimiser is not stepped
                self.optimizer.zero_grad(set_to_none=True)
                self._body()
        cur.wait_stream(warm)
        torch.cuda.synchronize()
        self._before_capture()
        self.optimizer.zero_grad(set_to_none=True)
        g = torch.cuda.CUDAGraph()
        n0 = _lib.launch_count()
        with torch.cuda.graph(g, capture_error_mode="thread_local"):
            self.loss = self._body()
        self.launches_per_replay = _lib.launch_count() - n0      # kernels of this library inside one replay
        self.params = [p for p in self.model.parameters() if p.grad is not None]
        self.grads = [p.grad for p in self.params]               # static: rewritten by every replay
        self.graph = g

    def close(self):
        """Drop the captured graph (and with it any collective work it holds): a process group must not be
        destroyed while a graph that captured its collectives is alive."""
        self.graph = None
        self.loss = None
        self.params, self.grads = [], []

    def __call__(self, neg_p=None, return_tensor=False):
        self.model.train()
        if neg_p is None:
            neg_p = self._draw_negatives()
        self._upload(neg_p)
        if self.graph is None:
            self._capture()
        self.graph.replay()
        for p, g in zip(self.params, self.grads):                # (an eager step in between may have re-pointed them)
            p.grad = g
        self.optimizer.step()
        return self.loss if return_tensor else self.loss.item()


class GraphedTrainStep(GraphedStep):
    """``train_step`` replayed from a CUDA graph (:class:`GraphedStep`).  At the reference's own scale (BASELINE
    config 1: 10k users / 50k posts / 500k edges) a step is ~32 launches of a few microseconds each and the eager
    step is bound by Python's launch path (~1 ms); the replay is one launch.  At config 2 the step is GPU-bound
    and the graph changes nothing.  The static inputs (features, edge lists) are the tensors of the first call:
    a different graph object needs a new ``GraphedTrainStep``."""

    def __init__(self, model, optimizer, x_dict, edge_index_dict, train_edge_index, interaction_type_tensor,
                 num_users, num_posts):
        if not fused_step.eligible(model, x_dict):
            raise ValueError("GraphedTrainStep needs CUDA inputs and a model the tape-free step accepts")
        dev = x_dict["user"].device
        super().__init__(model, optimizer, train_edge_index.size(1), dev)
        self.args = (x_dict, edge_index_dict, train_edge_index, interaction_type_tensor, num_users)
        self.num_posts = int(num_posts)
        self.side = torch.cuda.Stream(dev)

    def matches(self, model, optimizer, x_dict, edge_index_dict, train_edge_index):
        a = self.args
        return (model is self.model and optimizer is self.optimizer and x_dict["user"] is a[0]["user"]
                and x_dict["post"] is a[0]["post"] and train_edge_index is a[2]
                and all(edge_index_dict[k] is a[1][k] for k in a[1]))

    def _body(self):
        x_dict, edge_index_dict, train_edge_index, itt, num_users = self.args
        return fused_step.loss_and_grads(self.model, x_dict, edge_index_dict, train_edge_index, itt, num_users,
                                         self.neg, neg_ready=self.neg_ready).clone()

    def _draw_negatives(self):
        return torch.randint(0, self.num_posts, (self.neg.numel(),), device=self.neg.device)

    def _upload(self, neg_p):
        if neg_p.is_cuda:
            self.neg.copy_(neg_p)
            self.neg_ready.record()
        else:                              # host array: upload on a side stream, during the replayed forward
            self.side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(self.side):
                self.neg.copy_(neg_p, non_blocking=True)
                self.neg_ready.record(self.side)


def train_step(model, optimizer, x_dict, edge_index_dict, train_edge_index, interaction_type_tensor,
               num_users, num_posts, neg_p=None, return_tensor=False, fused=None, cuda_graph=False):
    """One full-batch step.  ``neg_p`` defaults to ``torch.randint(0, num_posts, (E,), device)`` as
    at train_gnn.py:272.  Returns ``loss.item()`` (train_gnn.py:285) or the 0-d device tensor when
    ``return_tensor`` (no host sync).

    ``fused``: ``None`` = take the tape-free forward+loss+backward (``fused_step.loss_and_grads``)
    whenever the model qualifies, ``False`` = always build the autograd tape and call
    ``loss.backward()`` (same kernels plus torch's element-wise ReLU-backward / accumulation passes),
    ``True`` = require the fused path.  ``cuda_graph``: replay the (tape-free) step from a CUDA graph captured
    on the first call with these inputs (:class:`GraphedTrainStep`, cached on the model)."""
    if cuda_graph:
        gs = getattr(model, "_trg_graphed_step", None)
        if gs is None or not gs.matches(model, optimizer, x_dict, edge_index_dict, train_edge_index):
            gs = GraphedTrainStep(model, optimizer, x_dict, edge_index_dict, train_edge_index,
                                  interaction_type_tensor, num_users, num_posts)
            object.__setattr__(model, "_trg_graphed_step", gs)
        return gs(neg_p, return_tensor=return_tensor)
    model.train()
    optimizer.zero_grad()
    use_fused = fused_step.eligible(model, x_dict) if fused is None else bool(fused)
    neg_p, neg_ready = stage_negatives(neg_p, x_dict["user"].device)     # host negatives: copy overlaps the forward
    if use_fused:
        if neg_p is None:
            neg_p = torch.randint(0, num_posts, (train_edge_index.size(1),), device=x_dict["user"].device)
        loss = fused_step.loss_and_grads(model, x_dict, edge_index_dict, train_edge_index,
                                         interaction_type_tensor, num_users, neg_p, neg_ready=neg_ready)
    else:
        out = model(x_dict, edge_index_dict)
        user_emb, post_emb = out["user"], out["post"]
        if neg_ready is not None:
            torch.cuda.current_stream().wait_event(neg_ready)
        if neg_p is None:
            neg_p = torch.randint(0, num_posts, (train_edge_index.size(1),), device=user_emb.device)
        loss = link_bce_loss(user_emb, post_emb, train_edge_index, neg_p, interaction_type_tensor, num_users)
        loss.backward()
    optimizer.step()
    return loss.detach() if return_tensor else loss.item()


@torch.no_grad()
def recommend(user_emb, known_post_emb, k=10, id_offset=0, exclude=None, rows=None):
    """``scores = torch.mm(user_emb, known_post_emb.T); torch.topk(scores, min(K, len(scores)))``
    (inference.py:427-428) for one user row or a batch.  Returns ``(top scores, top post ids)``.
    ``exclude`` / ``rows``: drop each user's history (an ``ExclusionIndex``), see ``score_topk``."""
    return score_topk(user_emb, known_post_emb, k, id_offset, exclude=exclude, rows=rows)

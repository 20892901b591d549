"""Batched, device-side ``evaluate()`` and cold-start recommendation (SURVEY.md §8f N1 / N2).

``evaluate`` replaces the per-user python loop of train_gnn.py:290-367 (``.item()`` per test edge,
one ``torch.mm`` + ``torch.topk`` + sklearn call per user) with ONE K5 launch over all test users
against the candidate pool, plus a few device tensor ops for Recall@K / NDCG@K.
``recommend_cold_users`` batches inference.py:378-441: the 1-node / 0-edge forward collapses to
``relu(1.0*(b_d + x W_r,d^T) + 0.75*(b_s + x W_r,s^T))`` (one K3 launch), followed by K5.
"""
from __future__ import annotations

import torch

from .functional import sage_proj_fwd, score_topk


@torch.no_grad()
def evaluate(test_edges, user_emb, post_emb, K=10, num_users=None):
    """Recall@K and NDCG@K over the test split, semantics of train_gnn.py:290-367:

    * ``test_edges[0]`` user ids, ``test_edges[1]`` GLOBAL post ids (``local + num_users``, :316);
    * candidate pool = sorted unique test posts (:321); every test user is scored against it;
    * recall = |top-K ∩ true posts| / len(true posts) with duplicates counted in the denominator (:346);
    * NDCG@K with binary relevance, ``sklearn.metrics.ndcg_score`` definition (:359-363).  sklearn
      averages gains inside groups of TIED scores; here ties are ranked canonically (id ascending), so
      the two agree whenever a user's top-(K+1) scores are distinct.
    Returns ``(mean_recall, mean_ndcg)`` as python floats (one host read at the end)."""
    num_users = user_emb.size(0) if num_users is None else int(num_users)
    dev = user_emb.device
    u = test_edges[0].to(dev).long()
    p = test_edges[1].to(dev).long() - num_users
    keep = u < num_users                                     # :327 skip invalid user indices
    u, p = u[keep], p[keep]
    if u.numel() == 0:
        return float("nan"), float("nan")
    cands = torch.unique(p)                                  # sorted unique candidate posts
    users, inv = torch.unique(u, return_inverse=True)
    n_true = torch.bincount(inv, minlength=users.numel()).double()          # len(true_posts), dups counted
    n_post = int(post_emb.size(0))
    pair_keys = torch.unique(u * n_post + p)                 # distinct (user, post) test pairs, sorted
    n_rel = torch.bincount(torch.searchsorted(users, pair_keys // n_post), minlength=users.numel())
    kk = min(int(K), int(cands.numel()))
    _, idx = score_topk(user_emb[users].contiguous(), post_emb[cands].contiguous(), kk)
    top_posts = cands[idx]                                   # [n_users, kk] local post ids, rank order
    keys = users[:, None] * n_post + top_posts
    pos = torch.searchsorted(pair_keys, keys.reshape(-1)).clamp(max=pair_keys.numel() - 1)
    hit = (pair_keys[pos] == keys.reshape(-1)).reshape(keys.shape)
    recall = hit.sum(1).double() / n_true
    disc = 1.0 / torch.log2(torch.arange(2, kk + 2, device=dev, dtype=torch.float64))
    dcg = (hit.double() * disc).sum(1)
    cum = torch.cat([torch.zeros(1, device=dev, dtype=torch.float64), disc.cumsum(0)])
    idcg = cum[n_rel.clamp(max=kk)]
    ndcg = dcg / idcg
    return float(recall.mean()), float(ndcg.mean())


@torch.no_grad()
def embed_cold_users(model, x_user):
    """Embeddings of users with no edges (inference.py:397-424): every SAGEConv sees E = 0, so
    ``user_emb = relu(w_direct*(b_d + x W_r,d^T) + w_social*(b_s + x W_r,s^T))`` -- one fused K3
    launch for the whole batch instead of a 1-node ``HeteroData`` + forward per user."""
    model.msg_direct.lin_r.materialize(x_user.size(-1))
    model.msg_social.lin_r.materialize(x_user.size(-1))
    ug = model.user_gemm()
    # both means are zero: only the root term, the user GEMM's last operand, remains
    return sage_proj_fwd([(x_user.contiguous(), ug.weights[-1], ug.alphas[-1])], ug.bias, True)


@torch.no_grad()
def recommend_cold_users(model, x_user, known_post_emb, k=10):
    """Batched ``recommend_for_user_inductive`` (inference.py:378-441): cold-start embedding, then
    ``mm`` + ``topk`` against the stored post table (inference.py:427-428).  Returns
    ``(top scores [B,k], top post ids [B,k])``."""
    return score_topk(embed_cold_users(model, x_user), known_post_emb, k)

"""CPU oracle of top-k with per-query exclusions.  TEST INFRASTRUCTURE.

Dense scores, the excluded (row, global id) pairs removed, the canonical (score desc, id asc) top-k of
what is left (``oracle.topk.topk_canonical``'s order), and ``(-inf, -1)`` pads for rows with fewer than
min(k, P) admissible posts -- the contract of ``trg_score_topk_excluding`` (``include/trg_b200.h``).
"""
import torch


def score_topk_excluding(q: torch.Tensor, cat: torch.Tensor, k: int, excl_pairs: torch.Tensor,
                         id_offset: int = 0, rows=None):
    """Query ``b`` (exclusion row ``rows[b]``, default ``b``) never gets a global id ``g`` for which
    ``(row, g)`` is in ``excl_pairs`` (int64 ``[2, E]``: exclusion row, global post id = local +
    ``id_offset``).  The top min(k, P) of what is left under (score desc, id asc); rows with fewer
    admissible posts end in ``(-inf, -1)``."""
    scores = torch.mm(q, cat.T)
    b, p = scores.shape
    kk = min(k, p)
    r = torch.arange(b) if rows is None else torch.as_tensor(rows, dtype=torch.int64).cpu()
    er, g = excl_pairs[0].cpu(), excl_pairs[1].cpu() - id_offset
    inside = (g >= 0) & (g < p)
    n_rows = int(max(int(er.max()) + 1 if er.numel() else 0, int(r.max()) + 1 if b else 0))
    dense = torch.zeros(n_rows, p, dtype=torch.bool)
    dense[er[inside], g[inside]] = True
    excluded = dense[r]
    # (admissible first, score desc, id asc): a stable sort on the flag after the canonical sort
    vals, idx = torch.sort(scores, dim=-1, descending=True, stable=True)
    flag = excluded.gather(-1, idx)
    o = torch.argsort(flag.to(torch.int8), dim=-1, stable=True)
    vals, idx, flag = vals.gather(-1, o)[..., :kk], idx.gather(-1, o)[..., :kk], flag.gather(-1, o)[..., :kk]
    vals = vals.masked_fill(flag, float("-inf"))
    ids = (idx + id_offset).masked_fill(flag, -1)
    return vals.contiguous(), ids.contiguous()

"""Per-user exclusion lists for top-k recommendation (``score_topk(..., exclude=...)``).

A recommender does not show a user the posts they have already engaged with, yet those are the posts
that score highest against an embedding trained on them.  ``ExclusionIndex`` holds, for every
"exclusion row" (usually a user), the sorted list of post ids that row must never be recommended.
K5 reads it on the device inside the selection itself, so the top-k stays exact whatever the size of a
history (see ``include/trg_b200.h``, ``trg_score_topk_excluding``).
"""
from __future__ import annotations

import torch

from .graph import build_csr

_INT32_MAX = (1 << 31) - 1


class ExclusionIndex:
    """CSR over exclusion rows: ``rowptr int32[num_rows + 1]``; ``ids int32[nnz]`` are post ids in
    the FULL catalogue's numbering (the id space of ``score_topk``'s output, i.e. local +
    ``id_offset``), ascending within each row.  Duplicates are harmless; so are ids outside a given
    catalogue or shard, which simply never match.  Because ids are global, one index serves every
    shard of a sharded catalogue."""

    def __init__(self, rowptr: torch.Tensor, ids: torch.Tensor, num_rows: int):
        if rowptr.dtype != torch.int32 or ids.dtype != torch.int32:
            raise TypeError("ExclusionIndex: rowptr and ids must be int32")
        if rowptr.dim() != 1 or rowptr.numel() != int(num_rows) + 1:
            raise ValueError(f"ExclusionIndex: rowptr must have num_rows + 1 = {int(num_rows) + 1} entries")
        self.rowptr = rowptr.contiguous()
        self.ids = ids.contiguous()
        self.num_rows = int(num_rows)

    @classmethod
    def from_edges(cls, edge_index: torch.Tensor, num_rows: int, num_ids: int, validate: bool = True):
        """Index from a ``[2, E]`` int64 COO of (row, post id), e.g. the training ``engages`` edges
        (user, post).  Two stable K0 sorts -- by post, then by row -- are an LSD sort on (row, post):
        every row's ids come out ascending.  ``validate`` checks the id ranges with one host sync, as
        ``build_csr`` does."""
        if edge_index.dim() != 2 or edge_index.size(0) != 2:
            raise ValueError("edge_index must have shape [2, E]")
        if int(num_ids) > _INT32_MAX + 1:
            raise ValueError(f"num_ids={int(num_ids)}: post ids must fit in int32")
        row, post = edge_index[0], edge_index[1]
        by_post = build_csr(row, post, int(num_ids), int(num_rows), validate=validate, per_step=True)
        post_sorted = post.contiguous().index_select(0, by_post.eid.long())
        by_row = build_csr(post_sorted, by_post.col.long(), int(num_rows), int(num_ids), validate=False,
                           per_step=True)
        return cls(by_row.rowptr, by_row.col, num_rows)

    @property
    def nnz(self) -> int:
        return int(self.ids.numel())

    def to(self, device):
        return ExclusionIndex(self.rowptr.to(device), self.ids.to(device), self.num_rows)

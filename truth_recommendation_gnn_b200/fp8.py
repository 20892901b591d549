"""Top-k recommendation from an e4m3 copy of the post catalogue, re-ranked exactly in the table's precision.

Stage 1 scores every post on the tensor cores from 8-bit operands (``trg_score_topk`` with
``TRG_F8E4M3``: half the catalogue bytes and half the tensor time of bf16) and keeps ``N_CAND`` candidates
per query.  Stage 2 (``trg_rescore_topk``) re-scores those candidates from the dense fp32 / bf16 table and
returns the top k of them.  The result is the exact top-k whenever the exact top-k is among the candidates.

Scales are powers of two, so dividing by them is exact: one per catalogue (every shard shares it when the
caller passes the all-reduced ``amax``) and one per query row (a positive per-row factor does not change
that row's ranking).  All of it runs on the device without a host synchronisation.
"""
from __future__ import annotations

import torch

from . import _lib

N_CAND = 128           # stage-1 candidates per query (the tensor-core kernel's lists hold at most 128)
CHUNK_ROWS = 1 << 20   # rows quantised at a time: no full-size fp32 temporary of a 50M-row table
HIDDEN = (128, 256)


def pow2_scale(amax: torch.Tensor) -> torch.Tensor:
    """Elementwise smallest power of two ``s`` with ``amax / s <= 448`` (fp32, on ``amax``'s device); 1 where
    ``amax == 0``.  Exact: with ``amax = m * 2^e``, ``m`` in [0.5, 1) and ``448 = 0.875 * 2^9``, the exponent is
    ``e - 9``, plus one when ``m > 0.875``."""
    amax = amax.float()
    m, e = torch.frexp(amax)
    n = e - 9 + (m > 0.875).to(e.dtype)
    s = ((n + 127).clamp(1, 254) << 23).view(torch.float32)   # 2^n from its exponent bits
    return torch.where(amax == 0, torch.ones_like(s), s)


def table_amax(table: torch.Tensor) -> torch.Tensor:
    """``max |table|`` as a 0-dim fp32 device tensor, read in row chunks (sharded callers all-reduce it with MAX
    and pass it to ``Fp8Catalogue.from_dense``)."""
    amax = torch.zeros((), dtype=torch.float32, device=table.device)
    for i in range(0, table.size(0), CHUNK_ROWS):
        amax = torch.maximum(amax, table[i:i + CHUNK_ROWS].abs().amax().float())
    return amax


def _check_dense(t: torch.Tensor, what: str):
    if t.dtype not in (torch.float32, torch.bfloat16):
        raise _lib.TrgError(f"{what}: table must be float32 or bfloat16, got {t.dtype}")
    if t.dim() != 2 or t.size(1) not in HIDDEN:
        raise _lib.TrgError(f"{what}: table must be [P, H] with H in {HIDDEN}, got shape {tuple(t.shape)}")
    if not t.is_cuda:
        raise _lib.TrgError(f"{what}: the e4m3 path runs on CUDA tensors only; got a {t.device} tensor")


class Fp8Catalogue:
    """A post table with its e4m3 copy: ``data`` (``float8_e4m3fn [P, H]``) = ``dense / scale`` rounded to
    nearest even, ``scale`` a 0-dim fp32 power of two, and ``dense`` the table itself (not a copy), which
    stage 2 re-scores from.  Build it once per embedding refresh."""

    def __init__(self, data: torch.Tensor, scale: torch.Tensor, dense: torch.Tensor):
        self.data, self.scale, self.dense = data, scale, dense

    @classmethod
    @torch.no_grad()
    def from_dense(cls, table: torch.Tensor, amax=None) -> "Fp8Catalogue":
        """``amax``: ``max |table|`` over the whole catalogue (a number or a device scalar); default: this
        table's.  Shards of one catalogue pass the all-reduced value so that they share one scale."""
        _check_dense(table, "Fp8Catalogue.from_dense")
        table = table.contiguous()
        if amax is None:
            amax = table_amax(table)
        amax = torch.as_tensor(amax, dtype=torch.float32, device=table.device).reshape(())
        scale = pow2_scale(amax)
        inv = 1.0 / scale                      # a power of two: multiplying by it is dividing by scale
        data = torch.empty(table.shape, dtype=torch.float8_e4m3fn, device=table.device)
        for i in range(0, table.size(0), CHUNK_ROWS):
            data[i:i + CHUNK_ROWS] = (table[i:i + CHUNK_ROWS].float() * inv).to(torch.float8_e4m3fn)
        return cls(data, scale, table)

    def __len__(self):
        return self.data.size(0)


def quantize_rows(q: torch.Tensor):
    """Per-row e4m3 copy of ``q [B, H]``: ``(q8, s)`` with ``q8[b] = q[b] / s[b]`` rounded to nearest even and
    ``s [B]`` fp32 powers of two (``pow2_scale`` of each row's ``max |q|``)."""
    s = pow2_scale(q.abs().amax(dim=1))
    return (q.float() * (1.0 / s)[:, None]).to(torch.float8_e4m3fn), s


def _check_query(q, cat: Fp8Catalogue, k):
    if q.dim() != 2 or q.size(1) != cat.data.size(1):
        raise _lib.TrgError(f"score_topk(e4m3): queries must be [B, {cat.data.size(1)}], got {tuple(q.shape)}")
    if q.dtype != cat.dense.dtype:
        raise _lib.TrgError(f"score_topk(e4m3): queries are {q.dtype} but the catalogue's table is "
                            f"{cat.dense.dtype}; they must match")
    if not 1 <= int(k) <= N_CAND:
        raise _lib.TrgError(f"score_topk(e4m3): k={k} must be in [1, {N_CAND}]")
    if not q.is_cuda:
        raise _lib.TrgError("score_topk(e4m3): queries must be CUDA tensors")


@torch.no_grad()
def _fp8_candidates(q, cat: Fp8Catalogue, k=N_CAND, id_offset=0, exclude=None, rows=None):
    """Stage 1 alone: the top ``min(k, P)`` of the e4m3 scores, ``(values, ids)``, values dequantised
    (``q8 . c8 * s_q[b] * scale``, exact power-of-two factors).  Exclusions apply here."""
    from .functional import _score_topk_native
    q = q.unsqueeze(0) if q.dim() == 1 else q
    _check_query(q, cat, k)
    q8, s = quantize_rows(q.contiguous())
    vals, ids = _score_topk_native(q8, cat.data, k, id_offset, exclude, rows, code=_lib.TRG_F8E4M3)
    return vals * (s[:, None] * cat.scale), ids


def rescore_topk(q, table, cand_ids, k, id_offset=0):
    """Stage 2 alone: exact scores of the candidate ids ``cand_ids [B, C]`` (global ids; -1 or out-of-range ids
    are skipped) from the dense table, and the top ``min(k, C)`` of them under (score desc, id asc); rows with
    fewer valid candidates end in ``(-inf, -1)``."""
    lib = _lib.load()
    q, table, cand_ids = q.contiguous(), table.contiguous(), cand_ids.contiguous()
    if q.dtype != table.dtype or cand_ids.dtype != torch.int64 or cand_ids.dim() != 2 \
            or cand_ids.size(0) != q.size(0):
        raise _lib.TrgError("rescore_topk: q and table must share a dtype, cand_ids must be int64 [B, C]")
    b, h = q.shape
    c = cand_ids.size(1)
    kk = min(int(k), c)
    vals = torch.empty(b, kk, dtype=torch.float32, device=q.device)
    ids = torch.empty(b, kk, dtype=torch.int64, device=q.device)
    if b == 0 or kk == 0:
        return vals, ids
    ws_bytes = int(lib.trg_rescore_topk_workspace_bytes(b, c))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=q.device)
    _lib.call("trg_rescore_topk", b * c * h * table.element_size(), lib.trg_rescore_topk,
              _lib.ptr(q), _lib.ptr(table), b, table.size(0), h, _lib.dtype_code(q.dtype), _lib.ptr(cand_ids), c,
              int(id_offset), kk, _lib.ptr(vals), _lib.ptr(ids), _lib.ptr(ws), ws_bytes, _lib.stream())
    return vals, ids


@torch.no_grad()
def score_topk(q, cat: Fp8Catalogue, k, id_offset=0, exclude=None, rows=None):
    """``functional.score_topk`` on an ``Fp8Catalogue``: e4m3 stage 1 (``N_CAND`` candidates per query,
    exclusions applied), then exact re-ranking from ``cat.dense``.  Returns ``(values [B, min(k, P)] fp32,
    ids int64)``; values are the dense table's scores (the fp32 FMA chain of ``trg_rescore_topk``)."""
    q = q.unsqueeze(0) if q.dim() == 1 else q
    _check_query(q, cat, k)
    _, cand = _fp8_candidates(q, cat, N_CAND, id_offset, exclude, rows)
    return rescore_topk(q, cat.dense, cand, min(int(k), len(cat)), id_offset)

"""CPU oracle of the e4m3 top-k (``truth_recommendation_gnn_b200.fp8``).  TEST INFRASTRUCTURE.

Written independently of torch's float8 cast: e4m3 (4 exponent bits, bias 7, 3 mantissa bits, largest
finite 448, subnormal step 2^-9) round-to-nearest-even in numpy, the power-of-two scale rule, the stage-1
ranking of the dequantised values in fp64, and the stage-2 re-scoring chain in fp32.
"""
import numpy as np
import torch

from tests import oracle_exclude as oexcl

E4M3_MAX = 448.0


def e4m3_round(x) -> np.ndarray:
    """``x`` (|x| <= 448) rounded to the nearest e4m3 value, ties to even, as float64."""
    x = np.asarray(x, dtype=np.float64)
    ax = np.abs(x)
    _, e = np.frexp(ax)                          # ax in [2^(e-1), 2^e)
    q = np.maximum(e - 4, -9)                    # 3 mantissa bits below the leading one; subnormal step 2^-9
    step = np.ldexp(1.0, q)
    return np.copysign(np.rint(ax / step) * step, x)


def pow2_scale(amax: float) -> float:
    """Smallest power of two ``s`` with ``amax / s <= 448``; 1 for ``amax == 0``."""
    amax = float(amax)
    if amax == 0.0:
        return 1.0
    n = int(np.floor(np.log2(amax))) - 9
    while amax > E4M3_MAX * 2.0 ** n:
        n += 1
    while amax <= E4M3_MAX * 2.0 ** (n - 1):
        n -= 1
    return 2.0 ** n


def quantize_table(t: torch.Tensor, amax=None):
    """``(codes as float64 values, scale)`` of a whole table with one scale."""
    x = t.detach().cpu().double().numpy()
    s = pow2_scale(np.abs(x).max() if amax is None else amax)
    return e4m3_round(x / s), s


def quantize_rows(q: torch.Tensor):
    """``(values float64 [B, H], scales [B])``: one scale per row."""
    x = q.detach().cpu().double().numpy()
    s = np.array([pow2_scale(a) for a in np.abs(x).max(axis=1)], dtype=np.float64)
    return e4m3_round(x / s[:, None]), s


def dequantized(q: torch.Tensor, cat: torch.Tensor, amax=None):
    """The fp64 values the e4m3 stage multiplies: ``q8 * s_q`` and ``c8 * s_c``."""
    q8, sq = quantize_rows(q)
    c8, sc = quantize_table(cat, amax)
    return torch.from_numpy(q8 * sq[:, None]), torch.from_numpy(c8 * sc)


def stage1_topk(q, cat, k, excl_pairs=None, id_offset=0, rows=None, amax=None):
    """Top min(k, P) of the fp64 dot products of the dequantised inputs under (score desc, id asc), with the
    exclusions of ``oracle_exclude`` (``excl_pairs`` int64 [2, E] of (row, global id)); values fp64."""
    qd, cd = dequantized(q, cat, amax)
    if excl_pairs is None:
        excl_pairs = torch.zeros(2, 0, dtype=torch.int64)
    return oexcl.score_topk_excluding(qd, cd, k, excl_pairs, id_offset, rows)


def rescore_chain(q: torch.Tensor, table: torch.Tensor, cand: torch.Tensor, id_offset=0):
    """fp32 scores of candidates ``cand [B, C]`` (global ids; invalid -> -inf), the sequential chain
    ``s = s + q[h] * t[h]`` in fp32, one rounding per operation.  For bf16 inputs every product is exact in
    fp32, so this equals the kernel's fmaf chain."""
    qn = q.detach().cpu().float().numpy()
    tn = table.detach().cpu().float().numpy()
    c = cand.cpu().numpy() - id_offset
    ok = (cand.cpu().numpy() >= 0) & (c >= 0) & (c < tn.shape[0])
    rows = tn[np.where(ok, c, 0)]                          # [B, C, H]
    s = np.zeros(c.shape, dtype=np.float32)
    for h in range(qn.shape[1]):
        s = (s + (qn[:, None, h] * rows[:, :, h]).astype(np.float32)).astype(np.float32)
    return torch.from_numpy(np.where(ok, s, np.float32(-np.inf)))

"""CPU checks of the e4m3 top-k: the numpy oracle against torch's cast, the scale rule at its boundaries,
the package's quantisers against the oracle, and the inputs the e4m3 path refuses."""
import numpy as np
import pytest
import torch

from tests import oracle_fp8 as o8
from truth_recommendation_gnn_b200 import _lib, fp8
from truth_recommendation_gnn_b200.fp8 import Fp8Catalogue


def test_oracle_rounding_matches_torch_on_every_bf16_value():
    bits = torch.arange(1 << 16, dtype=torch.int32).to(torch.int16).view(torch.bfloat16)
    x = bits.float()
    x = x[torch.isfinite(x) & (x.abs() <= 448)]
    ref = torch.from_numpy(o8.e4m3_round(x.double().numpy()))
    got = x.to(torch.float8_e4m3fn).double()
    assert torch.equal(got, ref)


def test_oracle_rounding_ties_go_to_even():
    # midpoints between neighbours: 1 + 1/16 (between 1 and 1.125) -> 1; 1 + 3/16 -> 1.25; subnormal 2^-10 -> 0
    assert o8.e4m3_round([1 + 1 / 16, 1 + 3 / 16, 2.0 ** -10, 3 * 2.0 ** -10, -(1 + 1 / 16)]).tolist() == \
        [1.0, 1.25, 0.0, 2.0 ** -8, -1.0]


@pytest.mark.parametrize("n", range(-30, 31, 3))
def test_scale_boundaries(n):
    at = 448.0 * 2.0 ** n
    above = float(np.nextafter(np.float32(at), np.float32(np.inf)))
    below = float(np.nextafter(np.float32(at), np.float32(0)))
    amax = torch.tensor([at, above, below, 0.0])
    want = [2.0 ** n, 2.0 ** (n + 1), 2.0 ** n, 1.0]
    assert [o8.pow2_scale(a) for a in amax.tolist()] == want
    assert fp8.pow2_scale(amax).tolist() == want
    assert fp8.pow2_scale(amax.bfloat16().float()[:1]).tolist() == [o8.pow2_scale(float(amax.bfloat16()[0]))]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_row_quantiser_matches_oracle(dtype):
    g = torch.Generator().manual_seed(3)
    q = (torch.randn(300, 128, generator=g) * torch.logspace(-8, 8, 300)[:, None]).to(dtype)
    q[7] = 0
    q8, s = fp8.quantize_rows(q)
    r8, rs = o8.quantize_rows(q)
    assert torch.equal(s.double(), torch.from_numpy(rs))
    assert torch.equal(q8.double(), torch.from_numpy(r8))


def _cat(dtype=torch.float32, h=128):
    t = torch.randn(50, h).to(dtype)
    return Fp8Catalogue(t.to(torch.float8_e4m3fn), torch.ones(()), t)


def test_host_tables_are_refused():
    with pytest.raises(_lib.TrgError, match="CUDA"):
        Fp8Catalogue.from_dense(torch.randn(100, 128))
    with pytest.raises(_lib.TrgError, match="CUDA"):
        fp8.score_topk(torch.randn(4, 128), _cat(), 10)


def test_widths_k_and_dtypes_are_refused():
    with pytest.raises(_lib.TrgError, match="H in"):
        fp8._check_dense(torch.randn(10, 64), "from_dense")
    with pytest.raises(_lib.TrgError, match="float32 or bfloat16"):
        fp8._check_dense(torch.randn(10, 128).half(), "from_dense")
    with pytest.raises(_lib.TrgError, match="k=129"):
        fp8.score_topk(torch.randn(4, 128), _cat(), 129)
    with pytest.raises(_lib.TrgError, match="must match"):
        fp8.score_topk(torch.randn(4, 128).bfloat16(), _cat(torch.float32), 10)
    with pytest.raises(_lib.TrgError, match="queries must be"):
        fp8.score_topk(torch.randn(4, 256), _cat(), 10)

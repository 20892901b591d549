"""K3, the projection GEMMs, at every kernel path the library dispatches to.

``trg_sage_proj_fwd``, ``trg_sage_proj_bwd_input`` and ``trg_sage_proj_bwd_weight`` each pick a kernel from
(dtype, hidden, k).  Every case here names the path it is meant to reach and checks, through the library's
launch counter, that the call took that path; a later change of the dispatch rules cannot silently move a
case off the kernel it covers.  The checks:

* an element-wise bound against an fp64 reference on the same (dtype-rounded) inputs, relative to the
  absolute-value product, with rows drawn at scales 2^-30 .. 2^30 so that an error confined to small rows
  cannot hide behind large ones;
* exact integer signatures at n >= 3 * 148 * 128 rows, where every CTA of the persistent kernels takes at
  least three tiles and every ring and both accumulator buffers are reused;
* bounds: inputs are prefix views of NaN-padded buffers, the workspace starts as NaN, and outputs are views
  into NaN-guarded buffers whose guards must come back bit for bit;
* determinism, row independence and zero-row calls.
"""
import ctypes
import math

import pytest
import torch

from truth_recommendation_gnn_b200 import _lib

pytestmark = pytest.mark.gpu

F32, BF16 = torch.float32, torch.bfloat16
NSM = 148
RAGGED = 2 * NSM * 128 + 77          # every CTA of a persistent kernel takes two tiles, plus a partial tile
SIG_ROWS = 3 * NSM * 128 + 77        # every CTA takes at least three tiles
GUARD_ROWS = 130                     # more than one tile of rows past the end of every output


# ------------------------------------------------------------------------------------------------
# Python mirror of the dispatch rules (api.cu, proj_tc.cu: proj_tc_eligible / launch_gemm,
# proj_dw_tc.cu: proj_dw_eligible / proj_tc_bwd_weight).  Each returns (path, launches).
# ------------------------------------------------------------------------------------------------
def _kblock(dtype):
    """Elements in one 128-byte k-block."""
    return 32 if dtype == F32 else 64


def _tc_kernel(dtype, bn):
    if dtype == F32:
        return f"proj_tc_f32a_kernel<{bn}>" if bn <= 128 else "proj_tc_kernel<true,256>"
    return f"proj_tc_kernel<false,{bn}>"


def fwd_path(dtype, hidden, ks, n):
    if hidden in (64, 128, 256) and all(k % _kblock(dtype) == 0 for k in ks):
        path, launches = _tc_kernel(dtype, hidden), 2            # prep_weights + GEMM
    else:
        path, launches = "proj_simt", 1
    return path, (launches if n else 0)


def bwd_input_path(dtype, hidden, ks, n):
    if len(set(ks)) == 1 and ks[0] in (64, 128, 256) and hidden % _kblock(dtype) == 0:
        path, launches = _tc_kernel(dtype, ks[0]), 2              # one n-block of width k per term
    else:
        path, launches = "proj_simt", 1 + len(ks)                 # prep_weights + one GEMM per term
    return path, (launches if n else 0)


def dw_packs(dtype, ks, bias):
    """Greedy packing of the terms (and the bias column sums) into launches, per 128-wide block of hidden:
    a list of (term indices, carries the bias)."""
    epc = _kblock(dtype)
    cap = 512 - 128 if dtype == F32 else 512      # fp32 keeps 128 TMEM columns for its dZ^T ring
    packs, t0, bias_done = [], 0, not bias
    while t0 < len(ks) or not bias_done:
        cols, nt = 0, 0
        while t0 + nt < len(ks) and nt < 4 and cols + ks[t0 + nt] <= cap:
            cols += ks[t0 + nt]
            nt += 1
        b = not bias_done and cols + epc <= 512
        bias_done = bias_done or b
        packs.append((tuple(range(t0, t0 + nt)), b))
        t0 += nt
    return packs


def bwd_weight_path(dtype, hidden, ks, bias, n):
    epc = _kblock(dtype)
    if n == 0:
        return ("zero rows", 0)
    if hidden % epc == 0 and all(k % epc == 0 and k <= 256 for k in ks):
        return (f"proj_dw_kernel<{'F32' if dtype == F32 else 'BF16'}>",
                2 * len(dw_packs(dtype, ks, bias)) * math.ceil(hidden / 128))
    return "dw_simt", 2 * len(ks) + (2 if bias else 0)


def test_dispatch_mirror_examples():
    """The two packings the weight-gradient cases rely on."""
    assert dw_packs(BF16, (256, 256, 256), True) == [((0, 1), False), ((2,), True)]
    assert bwd_weight_path(BF16, 256, (256, 256, 256), True, 1) == ("proj_dw_kernel<BF16>", 8)
    assert dw_packs(F32, (128, 128, 128, 128), True) == [((0, 1, 2), True), ((3,), False)]
    assert bwd_weight_path(F32, 128, (128, 128, 128, 128), True, 1) == ("proj_dw_kernel<F32>", 4)
    assert dw_packs(BF16, (256, 256), True) == [((0, 1), False), ((), True)]          # bias-only launch
    assert dw_packs(F32, (), True) == [((), True)]


# ------------------------------------------------------------------------------------------------
# direct C-ABI calls (as functional.py makes them) on caller-owned, guarded buffers
# ------------------------------------------------------------------------------------------------
def _bits(t):
    return t.view(torch.int32 if t.element_size() == 4 else torch.int16)


class Guarded:
    """A [shape] output viewed inside a NaN-filled buffer with guard regions before and after it."""

    def __init__(self, shape, dtype, dev, tail=None):
        numel = math.prod(shape)
        self.lead = 64                                 # 16-byte aligned for both dtypes
        tail = tail if tail is not None else GUARD_ROWS * (shape[-1] if len(shape) > 1 else 1) + 64
        self.buf = torch.full((self.lead + numel + tail,), float("nan"), dtype=dtype, device=dev)
        self.view = self.buf[self.lead:self.lead + numel].view(shape)
        self.numel = numel
        self.snap = self.buf.clone()

    def check_guards(self, what):
        b, s, e = _bits(self.buf), _bits(self.snap), self.lead + self.numel
        assert torch.equal(b[:self.lead], s[:self.lead]), f"{what}: wrote before the output"
        assert torch.equal(b[e:], s[e:]), f"{what}: wrote past the output"


def nan_padded(x, dev, extra=GUARD_ROWS + 1):
    """``x`` on the device as the prefix view of a buffer whose remaining rows are NaN."""
    big = torch.full((x.shape[0] + extra, *x.shape[1:]), float("nan"), dtype=x.dtype, device=dev)
    big[:x.shape[0]] = x.to(dev)
    return big[:x.shape[0]]


def _nan_workspace(nbytes, dev):
    return torch.full((max(int(nbytes), 16),), 0xFF, dtype=torch.uint8, device=dev)   # NaN in fp32 and bf16


def abi_fwd(terms, bias, relu, out):
    """terms = [(A, W, alpha)] device tensors; out [n, hidden].  Returns the launch-count delta."""
    lib = _lib.load()
    n, hidden = out.shape
    arr = (_lib.TrgProjTerm * len(terms))()
    for i, (a, w, alpha) in enumerate(terms):
        arr[i].a, arr[i].w, arr[i].k, arr[i].alpha = _lib.ptr(a), _lib.ptr(w), a.size(1), float(alpha)
    code = _lib.dtype_code(out.dtype)
    ws_bytes = int(lib.trg_sage_proj_workspace_bytes(sum(a.size(1) for a, _, _ in terms), hidden, code))
    ws = _nan_workspace(ws_bytes, out.device)
    n0 = _lib.launch_count()
    _lib.check(lib.trg_sage_proj_fwd(arr, len(terms), _lib.ptr(bias), n, hidden, code, int(relu), _lib.ptr(out),
                                     _lib.ptr(ws), ws_bytes, _lib.stream()), "trg_sage_proj_fwd")
    return _lib.launch_count() - n0


def abi_bwd_input(dz, terms):
    """terms = [(W, alpha, row_scale | None, d_a)].  Returns the launch-count delta."""
    lib = _lib.load()
    n, hidden = dz.shape
    arr = (_lib.TrgProjBwdTerm * len(terms))()
    for i, (w, alpha, rs, d_a) in enumerate(terms):
        arr[i].w, arr[i].k, arr[i].alpha = _lib.ptr(w), w.size(1), float(alpha)
        arr[i].row_scale, arr[i].d_a = _lib.ptr(rs), _lib.ptr(d_a)
    code = _lib.dtype_code(dz.dtype)
    ws_bytes = int(lib.trg_sage_proj_workspace_bytes(sum(t[0].size(1) for t in terms), hidden, code))
    ws = _nan_workspace(ws_bytes, dz.device)
    n0 = _lib.launch_count()
    _lib.check(lib.trg_sage_proj_bwd_input(_lib.ptr(dz), arr, len(terms), n, hidden, code, _lib.ptr(ws), ws_bytes,
                                           _lib.stream()), "trg_sage_proj_bwd_input")
    return _lib.launch_count() - n0


def abi_bwd_weight(dz, terms, db):
    """terms = [(A, alpha, d_w)]; db [hidden] fp32 or None.  Returns the launch-count delta."""
    lib = _lib.load()
    n, hidden = dz.shape
    arr = (_lib.TrgProjDwTerm * max(len(terms), 1))()
    for i, (a, alpha, d_w) in enumerate(terms):
        arr[i].a, arr[i].k, arr[i].alpha, arr[i].d_w = _lib.ptr(a), a.size(1), float(alpha), _lib.ptr(d_w)
    ws_bytes = int(lib.trg_sage_proj_dw_workspace_bytes())
    ws = _nan_workspace(ws_bytes, dz.device)
    n0 = _lib.launch_count()
    _lib.check(lib.trg_sage_proj_bwd_weight(_lib.ptr(dz), arr if terms else None, len(terms), _lib.ptr(db), n,
                                            hidden, _lib.dtype_code(dz.dtype), _lib.ptr(ws), ws_bytes,
                                            _lib.stream()), "trg_sage_proj_bwd_weight")
    return _lib.launch_count() - n0


# ------------------------------------------------------------------------------------------------
# inputs and the fp64 reference
# ------------------------------------------------------------------------------------------------
def scaled_rows(n, k, lo, hi, g, dtype):
    """randn rows, each scaled by 2^e with e uniform in [lo, hi], rounded to the storage dtype."""
    x = torch.randn(n, k, generator=g, dtype=torch.float64)
    e = torch.randint(lo, hi + 1, (n, 1), generator=g).double()
    return (x * torch.pow(2.0, e)).to(dtype)


def row_scale(mode, n, g):
    if mode is None:
        return None
    rs = torch.rand(n, generator=g) * 2 + 0.25
    if mode == "zeros":
        rs[torch.rand(n, generator=g) < 0.3] = 0
        rs[:1] = 0
    return rs


def scaled_weight(w, alpha, dtype, rounded):
    """alpha * W as the kernel's weight operand: the bf16 weight preparation stores alpha * W in bf16
    (one rounding when alpha is not a power of two); everywhere else it stays exact or fp32-accurate."""
    v = w.double() * alpha
    return v.to(BF16).double() if rounded else v


def check_bound(out, ref, absdot, dtype, what):
    """fp32: |out - ref| <= 1e-5 * absdot.  bf16 (exact products, fp32 accumulate, one rounding):
    |out - ref| <= 2^-8 |ref| + 1e-5 * absdot.  ``absdot`` is the same expression evaluated on absolute
    values (it includes |bias| and |row_scale|), so the bound holds element by element, at every scale."""
    out = out.detach().double().cpu()
    assert bool(torch.isfinite(out).all()), f"{what}: non-finite output"
    bound = 1e-5 * absdot
    if dtype == BF16:
        bound = bound + 2.0 ** -8 * ref.abs()
    err = (out - ref).abs()
    bad = err > bound
    if bool(bad.any()):
        ratio = float((err / bound.clamp(min=1e-300)).max())
        idx = tuple(int(i) for i in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {out.numel()} entries out of bound (worst "
                             f"err/bound {ratio:.3g}; first at {idx}: got {float(out[idx])!r}, "
                             f"want {float(ref[idx])!r} +- {float(bound[idx]):.3g})")


ALPHAS = (1.0, 0.75, 0.0, -1.5)


# ------------------------------------------------------------------------------------------------
# b. fp64 matrix over every path
# ------------------------------------------------------------------------------------------------
FWD_CASES = [
    # dtype, hidden, ks, n, alphas, bias, relu
    (F32, 64, (32,), 1, (1.0,), True, False),                                     # one k-block, one row
    (F32, 64, (32, 96, 64, 128), 129, ALPHAS, True, True),                        # 4 terms, odd chunk count
    (F32, 128, (96, 32), 127, (-1.5, 1.0), False, True),
    (F32, 128, (128, 128, 128), RAGGED, (1.0, 0.75, -1.5), True, True),           # persistent loop wraps
    (F32, 256, (256, 32, 96), 128, (0.75, 1.0, 0.0), True, False),
    (F32, 256, (256, 256), RAGGED, (1.0, 0.75), True, True),                      # 256-wide fp32 wraps
    (F32, 96, (16, 48), 300, (1.0, 0.75), True, True),                            # hidden not 64/128/256
    (F32, 128, (40, 128), 129, (-1.5, 1.0), False, False),                        # k not a whole k-block
    (BF16, 64, (64,), 1, (0.75,), True, True),
    (BF16, 64, (64, 192, 128, 64), 129, ALPHAS, True, True),
    (BF16, 128, (192, 64), 127, (1.0, -1.5), False, False),
    (BF16, 128, (128, 128, 128), RAGGED, (1.0, 0.75, -1.5), True, True),
    (BF16, 256, (256, 256, 256), RAGGED, (1.0, 0.75, 1.0), True, True),           # config 4's layer shape
    (BF16, 256, (64,), 128, (0.0,), True, False),                                 # alpha 0: out = bias
    (BF16, 96, (64, 32), 300, (1.0, 0.75), True, True),                           # bf16 generic kernel
    (BF16, 128, (8, 40), 129, (-1.5, 1.0), False, True),
]


def _fwd_inputs(dtype, hidden, ks, n, bias, seed):
    g = torch.Generator().manual_seed(seed)
    A = [scaled_rows(n, k, -30, 30, g, dtype) for k in ks]
    W = [scaled_rows(hidden, k, -10, 10, g, dtype) for k in ks]
    b = torch.randn(hidden, generator=g) if bias else None
    return A, W, b


def fwd_reference(A, W, alphas, b, relu, dtype, tc):
    ref = torch.zeros(A[0].shape[0], W[0].shape[0], dtype=torch.float64)
    absdot = torch.zeros_like(ref)
    for a, w, al in zip(A, W, alphas):
        wa = scaled_weight(w, al, dtype, dtype == BF16 and tc)
        ref += a.double() @ wa.t()
        absdot += a.double().abs() @ wa.abs().t()
    if b is not None:
        ref += b.double()
        absdot += b.double().abs()
    return (torch.relu(ref) if relu else ref), absdot


@pytest.mark.parametrize("dtype,hidden,ks,n,alphas,bias,relu", FWD_CASES)
def test_fwd_matches_fp64(dev, dtype, hidden, ks, n, alphas, bias, relu):
    path, launches = fwd_path(dtype, hidden, ks, n)
    A, W, b = _fwd_inputs(dtype, hidden, ks, n, bias, seed=n + hidden + len(ks))
    out = Guarded((n, hidden), dtype, dev)
    got = abi_fwd([(nan_padded(a, dev), nan_padded(w, dev), al) for a, w, al in zip(A, W, alphas)],
                  nan_padded(b, dev) if b is not None else None, relu, out.view)
    assert got == launches, f"expected {path} ({launches} launches), saw {got}"
    out.check_guards(path)
    ref, absdot = fwd_reference(A, W, alphas, b, relu, dtype, path != "proj_simt")
    check_bound(out.view, ref, absdot, dtype, path)


BWD_INPUT_CASES = [
    # dtype, hidden, ks, n, alphas, row-scale modes
    (F32, 128, (64, 64, 64), 129, (1.0, 0.75, -1.5), (None, "pos", "zeros")),      # k < hidden
    (F32, 32, (128, 128, 128, 128), RAGGED, ALPHAS, ("zeros", None, "pos", None)),  # K = one k-block
    (F32, 128, (256, 256), 127, (0.75, 1.0), ("pos", None)),                      # k > hidden
    (F32, 256, (256,), 1, (-1.5,), ("zeros",)),
    (F32, 128, (64, 128), 300, (1.0, 0.75), ("pos", "zeros")),                    # mixed k: generic kernel
    (F32, 96, (96,), 128, (0.75,), (None,)),
    (BF16, 128, (64, 64), 128, (1.0, 0.75), ("zeros", None)),
    (BF16, 64, (128, 128, 128), RAGGED, (1.0, -1.5, 0.0), (None, "pos", "zeros")),
    (BF16, 128, (256,), 129, (0.75,), ("pos",)),
    (BF16, 256, (256, 256, 256), RAGGED, (1.0, 0.75, 1.0), ("pos", "zeros", None)),  # config 4
    (BF16, 128, (64, 192), 300, (1.0, -1.5), (None, "zeros")),                    # generic kernel
    (BF16, 192, (192,), 127, (0.75,), ("pos",)),
]


def _bwd_input_inputs(dtype, hidden, ks, n, modes, seed):
    g = torch.Generator().manual_seed(seed)
    dz = scaled_rows(n, hidden, -30, 30, g, dtype)
    W = [scaled_rows(hidden, k, -10, 10, g, dtype) for k in ks]
    rs = [row_scale(m, n, g) for m in modes]
    return dz, W, rs


@pytest.mark.parametrize("dtype,hidden,ks,n,alphas,modes", BWD_INPUT_CASES)
def test_bwd_input_matches_fp64(dev, dtype, hidden, ks, n, alphas, modes):
    path, launches = bwd_input_path(dtype, hidden, ks, n)
    dz, W, rs = _bwd_input_inputs(dtype, hidden, ks, n, modes, seed=3 * n + hidden + len(ks))
    outs = [Guarded((n, k), dtype, dev) for k in ks]
    got = abi_bwd_input(nan_padded(dz, dev), [(nan_padded(w, dev), al, nan_padded(r, dev) if r is not None else None,
                                               o.view) for w, al, r, o in zip(W, alphas, rs, outs)])
    assert got == launches, f"expected {path} ({launches} launches), saw {got}"
    for t, (o, w, al, r) in enumerate(zip(outs, W, alphas, rs)):
        o.check_guards(f"{path} term {t}")
        wa = scaled_weight(w, al, dtype, dtype == BF16)
        ref, absdot = dz.double() @ wa, dz.double().abs() @ wa.abs()
        if r is not None:
            ref, absdot = ref * r.double()[:, None], absdot * r.double()[:, None]
        check_bound(o.view, ref, absdot, dtype, f"{path} term {t}")


BWD_WEIGHT_CASES = [
    # dtype, hidden, ks, n, alphas, bias
    (F32, 64, (32, 96), 1, (1.0, 0.75), True),                                    # hidden < 128
    (F32, 96, (128,), 127, (-1.5,), True),                                        # hidden not a multiple of 128
    (F32, 128, (128, 128, 128, 128), RAGGED, ALPHAS, True),                       # two packs: [t0..t2 + b], [t3]
    (F32, 256, (256, 32), 129, (0.75, 1.0), False),
    (F32, 512, (64,), 128, (1.0,), True),
    (F32, 192, (64, 160), 3000, (1.0, -1.5), True),
    (F32, 96, (), 2000, (), True),                                                # bias only
    (BF16, 64, (64, 128), 129, (1.0, 0.75), True),
    (BF16, 192, (192, 64), 127, (-1.5, 1.0), True),
    (BF16, 256, (256, 256, 256), 20_000, (1.0, 0.75, -1.5), True),                # [t0, t1], [t2 + b] per block
    (BF16, 512, (128,), 128, (1.0,), False),
    (BF16, 128, (256, 256), 1, (1.0, 0.0), True),                                 # [t0, t1], [b]
    (BF16, 256, (), 3000, (), True),                                              # bias only
    (F32, 128, (16, 48), 300, (1.0, 0.75), True),                                 # generic kernels
    (BF16, 96, (64, 32), 300, (0.75, 1.0), True),
    (F32, 64, (384,), 129, (-1.5,), True),                                        # k > 256
]


def _bwd_weight_inputs(dtype, hidden, ks, n, seed):
    g = torch.Generator().manual_seed(seed)
    dz = scaled_rows(n, hidden, -30, 30, g, dtype)
    A = [scaled_rows(n, k, -30, 30, g, dtype) for k in ks]
    return dz, A


def run_bwd_weight_case(dev, dtype, hidden, ks, n, alphas, bias, seed):
    path, launches = bwd_weight_path(dtype, hidden, ks, bias, n)
    dz, A = _bwd_weight_inputs(dtype, hidden, ks, n, seed)
    dws = [Guarded((hidden, k), dtype, dev) for k in ks]
    db = Guarded((hidden,), F32, dev) if bias else None
    got = abi_bwd_weight(nan_padded(dz, dev), [(nan_padded(a, dev), al, o.view) for a, al, o in zip(A, alphas, dws)],
                         db.view if db is not None else None)
    assert got == launches, f"expected {path} ({launches} launches), saw {got}"
    for t, (o, a, al) in enumerate(zip(dws, A, alphas)):
        o.check_guards(f"{path} dW{t}")
        ref = al * (dz.double().t() @ a.double())
        absdot = abs(al) * (dz.double().abs().t() @ a.double().abs())
        check_bound(o.view, ref, absdot, dtype, f"{path} dW{t}")
    if db is not None:
        db.check_guards(f"{path} db")
        check_bound(db.view, dz.double().sum(0), dz.double().abs().sum(0), F32, f"{path} db")
    return path


@pytest.mark.parametrize("dtype,hidden,ks,n,alphas,bias", BWD_WEIGHT_CASES)
def test_bwd_weight_matches_fp64(dev, dtype, hidden, ks, n, alphas, bias):
    run_bwd_weight_case(dev, dtype, hidden, ks, n, alphas, bias, seed=7 * n + hidden + len(ks))


@pytest.mark.parametrize("dtype", [F32, BF16])
@pytest.mark.parametrize("hidden,k", [(256, 384), (512, 512)])
def test_bwd_weight_wide_k_fits_workspace(dev, dtype, hidden, k):
    """k > 256 takes the generic weight-gradient kernels, whose per-CTA [hidden, k] partials must fit the
    fixed workspace: at hidden 256 / k 384 (384-d input features) 148 partials would need 58 MB."""
    assert run_bwd_weight_case(dev, dtype, hidden, (k,), 10_000, (0.75,), True, seed=hidden + k) == "dw_simt"


# ------------------------------------------------------------------------------------------------
# c. exact signatures at n >= 3 * 148 * 128 rows, every tensor-core instantiation
# ------------------------------------------------------------------------------------------------
SIG_ALPHAS = (1.0, 0.5, 2.0, -1.0)


def _codes(shape, g):
    return torch.randint(1, 8, shape, generator=g).double()


@pytest.mark.parametrize("dtype,hidden,ks", [
    (F32, 64, (32, 96, 128)), (F32, 128, (128, 64)), (F32, 256, (96, 256)),
    (BF16, 64, (64, 192)), (BF16, 128, (128, 128, 64)), (BF16, 256, (256, 256, 256)),
])
def test_fwd_signature_bit_exact(dev, dtype, hidden, ks):
    """A_t[r, c_t(r)] = 1 with c_t(r) pseudo-random (so every column of every k-block is hit, and rows of
    consecutive tiles of one CTA differ), W_t codes in 1..7, power-of-two alphas, integer bias: the output
    Σ_t α_t W_t[h, c_t(r)] + b[h] is exact in both dtypes.  A dropped, doubled, stale or misplaced k-block,
    row, tile or pipeline stage changes it."""
    n = SIG_ROWS
    path, launches = fwd_path(dtype, hidden, ks, n)
    assert path != "proj_simt"
    g = torch.Generator().manual_seed(hidden + len(ks))
    rows = torch.arange(n)
    cols = [torch.randint(0, k, (n,), generator=g) for k in ks]
    W = [_codes((hidden, k), g) for k in ks]
    b = torch.randint(-8, 9, (hidden,), generator=g).float()
    A = []
    for k, c in zip(ks, cols):
        a = torch.zeros(n, k, dtype=dtype, device=dev)
        a[rows.to(dev), c.to(dev)] = 1
        A.append(a)
    exp = b.double().expand(n, hidden).clone()
    for w, c, al in zip(W, cols, SIG_ALPHAS):
        exp += al * w.t()[c]
    out = Guarded((n, hidden), dtype, dev)
    got = abi_fwd([(a, w.to(dtype).to(dev), al) for a, w, al in zip(A, W, SIG_ALPHAS)], b.to(dev), False, out.view)
    assert got == launches
    out.check_guards(path)
    bad = out.view.double().cpu() != exp
    assert not bool(bad.any()), f"{path}: {int(bad.sum())} entries differ, rows {bad.any(1).nonzero()[:8, 0].tolist()}"


@pytest.mark.parametrize("dtype,hidden,k,n_terms", [
    (F32, 128, 64, 3), (F32, 96, 128, 2), (F32, 128, 256, 2),
    (BF16, 192, 64, 3), (BF16, 128, 128, 2), (BF16, 256, 256, 3),
])
def test_bwd_input_signature_bit_exact(dev, dtype, hidden, k, n_terms):
    """dZ one-hot at h(r) with value ±1 or 2, row_scale powers of two and zeros:
    d_a_t[r, c] = rs_t[r] α_t v(r) W_t[h(r), c], exact; each entry depends on its row, term and the
    k-block of hidden that holds h(r)."""
    n = SIG_ROWS
    ks = (k,) * n_terms
    path, launches = bwd_input_path(dtype, hidden, ks, n)
    assert path != "proj_simt"
    g = torch.Generator().manual_seed(hidden * 3 + k + n_terms)
    h_of = torch.randint(0, hidden, (n,), generator=g)
    v = torch.tensor([1.0, -1.0, 2.0])[torch.randint(0, 3, (n,), generator=g)]
    dz = torch.zeros(n, hidden, dtype=dtype, device=dev)
    dz[torch.arange(n, device=dev), h_of.to(dev)] = v.to(dtype).to(dev)
    W = [_codes((hidden, k), g) for _ in ks]
    rs = [torch.tensor([0.0, 0.5, 1.0, 2.0, 4.0])[torch.randint(0, 5, (n,), generator=g)] for _ in ks]
    rs[0] = None
    outs = [Guarded((n, k), dtype, dev) for _ in ks]
    got = abi_bwd_input(dz, [(w.to(dtype).to(dev), al, r.to(dev) if r is not None else None, o.view)
                             for w, al, r, o in zip(W, SIG_ALPHAS, rs, outs)])
    assert got == launches
    for t, (o, w, al, r) in enumerate(zip(outs, W, SIG_ALPHAS, rs)):
        o.check_guards(f"{path} term {t}")
        exp = (al * v.double())[:, None] * w[h_of]
        if r is not None:
            exp = exp * r.double()[:, None]
        bad = o.view.double().cpu() != exp
        assert not bool(bad.any()), f"{path} term {t}: {int(bad.sum())} entries differ"


@pytest.mark.parametrize("dtype,hidden,ks,bias", [
    (F32, 128, (128, 128, 128, 128), True),    # two packs, 4 terms
    (F32, 256, (32, 96, 256), True),           # two blocks of hidden
    (F32, 96, (), True),                       # bias only
    (BF16, 256, (256, 256, 256), True),        # [t0, t1], [t2 + b] in each of two blocks
    (BF16, 128, (256, 256), True),             # [t0, t1], [b]
    (BF16, 192, (64, 128), False),
])
def test_bwd_weight_signature_bit_exact(dev, dtype, hidden, ks, bias):
    """One-hot dZ (±1, 2 at h(r)) and one-hot A_t (1 at c_t(r)): dW_t[h, c] = α_t Σ_{r: h(r)=h, c_t(r)=c} v(r)
    is an integer scatter count, rounded once; db[h] = Σ_{r: h(r)=h} v(r).  Every CTA accumulates many row
    stages, so a dropped, doubled or stale stage, or a misplaced row, n-block or pack, changes a count."""
    n = SIG_ROWS
    path, launches = bwd_weight_path(dtype, hidden, ks, bias, n)
    assert path.startswith("proj_dw_kernel")
    g = torch.Generator().manual_seed(hidden * 5 + sum(ks))
    h_of = torch.randint(0, hidden, (n,), generator=g)
    v = torch.tensor([1.0, -1.0, 2.0])[torch.randint(0, 3, (n,), generator=g)]
    rows = torch.arange(n, device=dev)
    dz = torch.zeros(n, hidden, dtype=dtype, device=dev)
    dz[rows, h_of.to(dev)] = v.to(dtype).to(dev)
    cols = [torch.randint(0, k, (n,), generator=g) for k in ks]
    A = []
    for k, c in zip(ks, cols):
        a = torch.zeros(n, k, dtype=dtype, device=dev)
        a[rows, c.to(dev)] = 1
        A.append(a)
    dws = [Guarded((hidden, k), dtype, dev) for k in ks]
    db = Guarded((hidden,), F32, dev) if bias else None
    got = abi_bwd_weight(dz, [(a, al, o.view) for a, al, o in zip(A, SIG_ALPHAS, dws)], db.view if bias else None)
    assert got == launches
    for t, (o, k, c, al) in enumerate(zip(dws, ks, cols, SIG_ALPHAS)):
        o.check_guards(f"{path} dW{t}")
        cnt = torch.zeros(hidden * k, dtype=torch.float64).index_add_(0, h_of * k + c, v.double()).view(hidden, k)
        exp = (al * cnt).to(dtype).double()
        bad = o.view.double().cpu() != exp
        assert not bool(bad.any()), f"{path} dW{t}: {int(bad.sum())} entries differ"
    if bias:
        db.check_guards(f"{path} db")
        exp = torch.zeros(hidden, dtype=torch.float64).index_add_(0, h_of, v.double())
        assert torch.equal(db.view.double().cpu(), exp), f"{path} db"


# ------------------------------------------------------------------------------------------------
# d/e. padding, determinism and row independence
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,hidden,ks", [
    (F32, 128, (128, 96)), (F32, 256, (256, 64)), (F32, 96, (16, 48)),
    (BF16, 256, (256, 256, 256)), (BF16, 64, (64, 128)), (BF16, 128, (8, 40)),
])
def test_fwd_deterministic_padding_free_and_row_independent(dev, dtype, hidden, ks):
    """Bitwise: a repeated call, a call on exact-size (unpadded) inputs, and rows [r0, r0 + m) of a
    multi-tile call recomputed on their own, all give the same output."""
    n = RAGGED
    path, launches = fwd_path(dtype, hidden, ks, n)
    A, W, b = _fwd_inputs(dtype, hidden, ks, n, True, seed=hidden + 11)
    alphas = ALPHAS[:len(ks)]
    Ad, Wd, bd = [a.to(dev) for a in A], [w.to(dev) for w in W], b.to(dev)
    outs = []
    for padded in (True, True, False):
        o = Guarded((n, hidden), dtype, dev)
        terms = [(nan_padded(a, dev) if padded else a, w, al) for a, w, al in zip(Ad, Wd, alphas)]
        assert abi_fwd(terms, bd, True, o.view) == launches
        outs.append(o.view)
    assert torch.equal(_bits(outs[0]), _bits(outs[1])), f"{path}: repeated call differs"
    assert torch.equal(_bits(outs[0]), _bits(outs[2])), f"{path}: NaN padding past n_rows changed the output"
    for r0, m in ((0, 1), (128 * 150 + 3, 129), (n - 77, 77), (5000, 1000)):
        part = Guarded((m, hidden), dtype, dev)
        assert abi_fwd([(a[r0:r0 + m], w, al) for a, w, al in zip(Ad, Wd, alphas)], bd, True, part.view) == \
            fwd_path(dtype, hidden, ks, m)[1]
        assert torch.equal(_bits(part.view), _bits(outs[0][r0:r0 + m])), f"{path}: rows {r0}+{m} differ alone"


@pytest.mark.parametrize("dtype,hidden,ks", [
    (F32, 128, (64, 64)), (F32, 128, (256,)), (F32, 128, (64, 128)),
    (BF16, 256, (256, 256, 256)), (BF16, 192, (64, 64)), (BF16, 128, (64, 192)),
])
def test_bwd_input_deterministic_padding_free_and_row_independent(dev, dtype, hidden, ks):
    n = RAGGED
    path, launches = bwd_input_path(dtype, hidden, ks, n)
    dz, W, rs = _bwd_input_inputs(dtype, hidden, ks, n, ("zeros", "pos", None)[:len(ks)], seed=hidden + 13)
    alphas = ALPHAS[:len(ks)]
    dzd, Wd = dz.to(dev), [w.to(dev) for w in W]
    rsd = [r.to(dev) if r is not None else None for r in rs]

    def run(dz_in, rows):
        outs = [Guarded((rows.stop - rows.start, k), dtype, dev) for k in ks]
        got = abi_bwd_input(dz_in, [(w, al, r[rows] if r is not None else None, o.view)
                                    for w, al, r, o in zip(Wd, alphas, rsd, outs)])
        assert got == bwd_input_path(dtype, hidden, ks, rows.stop - rows.start)[1]
        return [o.view for o in outs]

    full = slice(0, n)
    o1, o2, o3 = run(nan_padded(dz, dev), full), run(nan_padded(dz, dev), full), run(dzd, full)
    for t in range(len(ks)):
        assert torch.equal(_bits(o1[t]), _bits(o2[t])), f"{path}: repeated call differs"
        assert torch.equal(_bits(o1[t]), _bits(o3[t])), f"{path}: NaN padding past n_rows changed the output"
    for r0, m in ((0, 1), (128 * 150 + 3, 129), (n - 77, 77), (5000, 1000)):
        part = run(dzd[r0:r0 + m], slice(r0, r0 + m))
        for t in range(len(ks)):
            assert torch.equal(_bits(part[t]), _bits(o1[t][r0:r0 + m])), f"{path}: rows {r0}+{m} differ alone"


@pytest.mark.parametrize("dtype,hidden,ks", [
    (F32, 128, (128, 128, 128, 128)), (F32, 64, (384,)), (BF16, 256, (256, 256, 256)), (BF16, 96, (64, 32)),
])
def test_bwd_weight_deterministic_and_padding_free(dev, dtype, hidden, ks):
    n = 20_000
    path, launches = bwd_weight_path(dtype, hidden, ks, True, n)
    dz, A = _bwd_weight_inputs(dtype, hidden, ks, n, seed=hidden + 17)
    res = []
    for padded in (True, True, False):
        dws = [Guarded((hidden, k), dtype, dev) for k in ks]
        db = Guarded((hidden,), F32, dev)
        put = (lambda x: nan_padded(x, dev)) if padded else (lambda x: x.to(dev))
        assert abi_bwd_weight(put(dz), [(put(a), al, o.view) for a, al, o in zip(A, ALPHAS, dws)], db.view) == launches
        res.append([o.view for o in dws] + [db.view])
    for x, y, z in zip(*res):
        assert torch.equal(_bits(x), _bits(y)), f"{path}: repeated call differs"
        assert torch.equal(_bits(x), _bits(z)), f"{path}: NaN padding past n_rows changed the output"


# ------------------------------------------------------------------------------------------------
# f. zero rows
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [F32, BF16])
@pytest.mark.parametrize("hidden,k", [(128, 128), (96, 48)])     # tensor-core and generic shapes
def test_zero_rows(dev, dtype, hidden, k):
    """n_rows = 0: nothing launches; forward and input gradient write nothing, the weight gradient is
    dW = 0 and db = 0 (an empty sum), on both the tensor-core and the generic path."""
    g = torch.Generator().manual_seed(hidden + k)
    w = torch.randn(hidden, k, generator=g).to(dtype).to(dev)
    empty_a = torch.empty(GUARD_ROWS, k, dtype=dtype, device=dev)[:0]
    empty_z = torch.empty(GUARD_ROWS, hidden, dtype=dtype, device=dev)[:0]
    out = Guarded((0, hidden), dtype, dev)
    assert abi_fwd([(empty_a, w, 1.0), (empty_a, w, 0.75)], torch.ones(hidden, device=dev), True, out.view) == 0
    out.check_guards("fwd")
    d_a = [Guarded((0, k), dtype, dev) for _ in range(2)]
    assert abi_bwd_input(empty_z, [(w, 1.0, None, d_a[0].view), (w, 0.75, None, d_a[1].view)]) == 0
    for o in d_a:
        o.check_guards("bwd_input")
    for n_terms in (2, 0):
        dws = [Guarded((hidden, k), dtype, dev) for _ in range(n_terms)]
        db = Guarded((hidden,), F32, dev)
        assert abi_bwd_weight(empty_z, [(empty_a, 0.75, o.view) for o in dws], db.view) == 0
        for o in dws + [db]:
            o.check_guards("bwd_weight")
            assert not bool(o.view.any()) and bool(torch.isfinite(o.view).all()), "bwd_weight with 0 rows must be 0"

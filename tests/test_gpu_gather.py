"""K1 / K2 / wsum, the gather-reduce kernels, at every kernel form the library dispatches to, and the row-finish
kernels of the sharded step at the sizes they run at.

``launch_gather`` (gather.cu) picks one of nine kernel forms from the row width in 16-byte vectors; each form
comes in three modes (mean, neighbour scale, edge coefficient), the non-mean modes with the ``accumulate`` and
``relu_of`` epilogues and, for bf16 tables, fp32 output rows; forms of rows >= 80 bytes also have a long-row
instantiation plus ``gather_combine_long``.  Every case names the form it is meant to reach (``gather_form``
restates the dispatch chain) and checks, through the library's launch counter, the launches that form makes.
The checks:

* graphs built to hit the walk's boundaries (``boundary_degrees``): degrees 0, 1, LPR - 1, LPR, LPR + 1, the
  unroll count +- 1 and 2 LPR + 1; rows ending on the last lane of a chunk; runs of empty rows longer than a
  group and than a CTA; an empty last row and a partial last CTA; duplicate edges and source ids 0 and
  N_src - 1; for long rows, rows of T, T + 1, 2T and 2T + 1 edges next to short ones in one group; plus one
  random skewed graph per dtype;
* mean: bit-exact against the sequential CSR-order fp32 sum divided in IEEE fp32, ``inv_deg`` bit-exact;
* K2 / wsum, every epilogue combination: exact signatures (integer tables, dyadic weights and scales, so every
  sum is exact in fp32 in any order) must equal the fp64 reference bit for bit after the output rounding; on
  random rows drawn at scales 2^-30 .. 2^30 the error is bounded element by element by
  (deg + slices + 4) 2^-24 (sum |terms| + |base|), plus 2^-8 |ref| when the output is bf16;
* bounds: inputs are prefix views of NaN-padded buffers and outputs are views into NaN-guarded buffers whose
  guards must come back bit for bit; long-row results must be bitwise repeatable;
* host-side rejections (rows wider than 2048 bytes, long rows on rows under 80 bytes) launch nothing.

The row-finish kernels run at row counts that take every thread of the grid-stride loops through three or more
iterations.  ``trg_rows_finish`` and ``trg_peer_reduce_rows`` compute ``row_scale * x + add`` as an FMUL and an
FADD (no FFMA in the sm_100a SASS of either kernel); the tests accept the fused or the unfused fp32 result per
element, since both are a correct compilation of the source.
"""
import ctypes
import math

import pytest
import torch

import truth_recommendation_gnn_b200 as trg
from oracle import sage as osage
from truth_recommendation_gnn_b200 import _lib
from truth_recommendation_gnn_b200 import functional as Fn
from truth_recommendation_gnn_b200 import graph as G
from truth_recommendation_gnn_b200.graph import CSR

pytestmark = pytest.mark.gpu

F32, BF16 = torch.float32, torch.bfloat16
TRG_E_UNSUPPORTED = 4
MAX_SMS = 148                     # grid_sms(): the device's SM count, capped at the B200's
LONG_T = 40                       # long-row threshold of the long-row cases
N_SRC = 131                       # source table of the boundary graphs: every id is used many times
U = 2.0 ** -24                    # fp32 unit roundoff


# ------------------------------------------------------------------------------------------------
# Python mirror of launch_gather's dispatch (gather.cu)
# ------------------------------------------------------------------------------------------------
#: form -> (LPR lanes per row group, R rows per group, VPL 16-byte vectors per lane)
FORMS = {
    "gather_reduce<LPR 1>": (1, 1, 1),
    "gather_reduce<LPR 2>": (2, 1, 1),
    "gather_reduce<LPR 4>": (4, 1, 1),
    "seg<LPR 8, R 4>": (8, 4, 1),
    "seg<LPR 16, R 8>": (16, 8, 1),
    "SEG8": (32, 8, 1),
    "seg<LPR 32, VPL 1>": (32, 8, 1),
    "seg<LPR 32, VPL 2>": (32, 8, 2),
    "seg<LPR 32, VPL 4>": (32, 8, 4),
}
UNROLL = {1: 8, 2: 4, 4: 2}       # row loads in flight per lane, by VPL


def row_vecs(dtype, feat):
    return feat * (4 if dtype == F32 else 2) // 16


def gather_form(dtype, feat):
    rv = row_vecs(dtype, feat)
    if rv <= 1:
        return "gather_reduce<LPR 1>"
    if rv <= 2:
        return "gather_reduce<LPR 2>"
    if rv <= 4:
        return "gather_reduce<LPR 4>"
    if rv <= 8:
        return "seg<LPR 8, R 4>"
    if rv == 16:
        return "SEG8"
    if rv <= 16:
        return "seg<LPR 16, R 8>"
    if rv <= 32:
        return "seg<LPR 32, VPL 1>"
    if rv <= 64:
        return "seg<LPR 32, VPL 2>"
    if rv <= 128:
        return "seg<LPR 32, VPL 4>"
    return "unsupported"


def cta_rows(form):
    lpr, r, _ = FORMS[form]
    return 256 // lpr * r


WIDTHS = {F32: (4, 8, 12, 16, 20, 32, 48, 64, 96, 128, 132, 192, 256, 260, 384, 512),
          BF16: (8, 16, 24, 32, 40, 64, 96, 128, 192, 256, 264, 512, 520, 1024)}
SKEWED_WIDTHS = {F32: (8, 64, 384), BF16: (24, 128, 1024)}
_DT = {F32: "f32", BF16: "bf16"}

CASES = ([(dt, f, "edges") for dt in (F32, BF16) for f in WIDTHS[dt]]
         + [(dt, f, "long") for dt in (F32, BF16) for f in WIDTHS[dt] if row_vecs(dt, f) >= 5]
         + [(dt, f, "skewed") for dt in (F32, BF16) for f in SKEWED_WIDTHS[dt]])
CASE_IDS = [f"{_DT[dt]}-F{f}-{g}" for dt, f, g in CASES]
MEAN_CASES = CASES
WEIGHTED_CASES = [(m, *c) for m in ("k2", "wsum") for c in CASES]
WEIGHTED_IDS = [f"{m}-{i}" for m in ("k2", "wsum") for i in CASE_IDS]


def test_dispatch_mirror_covers_every_form():
    """Runs without a GPU: every form is reached by the cases of every mode and dtype, and the long-row cases
    reach every form with rows of >= 5 vectors."""
    assert [gather_form(F32, 4 * rv) for rv in (1, 2, 3, 4, 5, 8, 9, 15, 16, 17, 32, 33, 64, 65, 128, 129)] == [
        "gather_reduce<LPR 1>", "gather_reduce<LPR 2>", "gather_reduce<LPR 4>", "gather_reduce<LPR 4>",
        "seg<LPR 8, R 4>", "seg<LPR 8, R 4>", "seg<LPR 16, R 8>", "seg<LPR 16, R 8>", "SEG8",
        "seg<LPR 32, VPL 1>", "seg<LPR 32, VPL 1>", "seg<LPR 32, VPL 2>", "seg<LPR 32, VPL 2>",
        "seg<LPR 32, VPL 4>", "seg<LPR 32, VPL 4>", "unsupported"]
    assert gather_form(BF16, 8 * 16) == "SEG8" and gather_form(BF16, 1032) == "unsupported"
    long_forms = {f for f in FORMS if FORMS[f][0] >= 8}
    assert long_forms == {gather_form(F32, 4 * rv) for rv in range(5, 129)}
    for mode, cases in (("mean", [(None, *c) for c in MEAN_CASES]), ("k2/wsum", WEIGHTED_CASES)):
        modes = {c[0] for c in cases}
        for m in modes:
            for dt in (F32, BF16):
                mine = [(f, g) for mm, d, f, g in cases if mm == m and d == dt]
                assert {gather_form(dt, f) for f, _ in mine} == set(FORMS), (mode, m, dt)
                assert {gather_form(dt, f) for f, g in mine if g == "long"} == long_forms, (mode, m, dt)
                assert {g for _, g in mine} == {"edges", "long", "skewed"}


# ------------------------------------------------------------------------------------------------
# graphs
# ------------------------------------------------------------------------------------------------
class Graph:
    """A CSR built on the host from per-row degrees: rows in order, edges of a row back to back."""

    def __init__(self, deg, n_src, gen, col=None, eid=None, long_t=None):
        self.deg = torch.as_tensor(deg, dtype=torch.long)
        self.n_rows, self.n_src = self.deg.numel(), n_src
        self.rowptr = torch.zeros(self.n_rows + 1, dtype=torch.long)
        self.rowptr[1:] = torch.cumsum(self.deg, 0)
        e = int(self.rowptr[-1])
        self.dst = torch.repeat_interleave(torch.arange(self.n_rows), self.deg)
        if col is None:
            col = torch.randint(0, n_src, (e,), generator=gen)
            col[::17] = 0                                            # the first and the last source row
            col[5::23] = n_src - 1
            first = self.rowptr[:-1][self.deg >= 2]                  # duplicate edges: a row's last edge
            col[first + self.deg[self.deg >= 2] - 1] = col[first]    # repeats its first source
        self.col = col
        self.eid = torch.randperm(e, generator=gen) if eid is None else eid
        self.long_t = long_t
        self.slices = (torch.where(self.deg > long_t, (self.deg + long_t - 1) // long_t, 1) if long_t
                       else torch.ones_like(self.deg))

    @property
    def n_edges(self):
        return self.col.numel()

    def csr(self, dev):
        return CSR(self.rowptr.int().to(dev), self.col.int().to(dev), self.eid.int().to(dev), self.n_rows,
                   self.n_src)


def boundary_degrees(form):
    """Row degrees that walk ``form`` across its boundaries (see the module docstring)."""
    lpr, r, vpl = FORMS[form]
    un, cta = UNROLL[vpl], cta_rows(form)
    special = sorted({0, 1, lpr - 1, lpr, lpr + 1, un - 1, un, un + 1, 2 * lpr + 1})
    degs = []

    def align(m, fill):
        while len(degs) % m:
            degs.append(fill)

    for s in range(r + 1):               # every special degree at several offsets inside a group
        k = s % len(special)
        degs += [2] * s + special[k:] + special[:k]
    align(r, 1)
    # rows whose last edge is the last lane of a chunk (chunks start at the group's first edge)
    degs += [lpr - 3, 3, lpr, 2 * lpr - 1, 1] if r > 1 else [lpr, 2 * lpr, 3 * lpr]
    align(r, 1)
    degs += [0] * (r + 1) + [5, 1]       # a group whose rows are all empty, and a run longer than R
    align(cta, 1)
    degs += [0] * (cta + r + 1)          # a whole CTA of empty rows
    degs += special + [2 * lpr + 1, 0, lpr]
    degs.append(2)
    while (len(degs) + 1) % cta == 0 or (r > 1 and (len(degs) + 1) % r == 0):
        degs.append(1)
    degs.append(0)                       # an empty last row; the last group and CTA are partial
    return degs


def long_degrees(form, t=LONG_T):
    """``boundary_degrees`` with rows of T, T + 1, 2T, 2T + 1 and more edges between the short ones: at a
    group's start, next to short and empty rows, back to back, and just before the empty last row."""
    longs = [t, t + 1, 2 * t, 2 * t + 1, 5 * t + 3, t + 1, 2 * t + 1]
    degs = [2 * t + 1]
    for i, d in enumerate(boundary_degrees(form)[:-1]):
        degs.append(d)
        if i % 11 == 5:
            degs.append(longs[(i // 11) % len(longs)])
    return degs + [2 * t, t + 1, 0]


@pytest.mark.parametrize("form", list(FORMS))
def test_boundary_graphs_reach_every_boundary(form):
    """Runs without a GPU: the generated graphs contain what their docstrings promise."""
    lpr, r, vpl = FORMS[form]
    cta, un = cta_rows(form), UNROLL[vpl]
    graph = make_graph("edges", form, seed=0)
    deg = graph.deg.tolist()
    assert {0, 1, lpr - 1, lpr, lpr + 1, un - 1, un, un + 1, 2 * lpr + 1} <= set(deg)
    assert deg[-1] == 0 and graph.n_rows % cta != 0 and (r == 1 or graph.n_rows % r != 0)
    group_empty = [all(d == 0 for d in deg[i:i + r]) for i in range(0, graph.n_rows - r + 1, r)]
    cta_empty = [all(d == 0 for d in deg[i:i + cta]) for i in range(0, graph.n_rows - cta + 1, cta)]
    assert any(group_empty) and any(cta_empty)
    if r > 1:      # a row that ends on the last lane of a chunk, the chunk not being the row's first
        ends = [(int(graph.rowptr[i + 1]) - int(graph.rowptr[i - i % r])) for i in range(graph.n_rows)]
        assert any(e % lpr == 0 and e > lpr and d > 0 and i % r for i, (e, d) in enumerate(zip(ends, deg)))
    col = graph.col.tolist()
    assert 0 in col and N_SRC - 1 in col
    assert any(col[a] == col[b - 1] for a, b in zip(graph.rowptr[:-1].tolist(), graph.rowptr[1:].tolist())
               if b - a >= 2)
    if lpr >= 8:
        ld = long_degrees(form)
        assert {LONG_T, LONG_T + 1, 2 * LONG_T, 2 * LONG_T + 1} <= set(ld)
        assert ld[-1] == 0 and ld[0] > LONG_T
        assert any(a > LONG_T and 0 < b <= LONG_T for a, b in zip(ld, ld[1:]))      # long next to short
        assert any(a > LONG_T and b > LONG_T for a, b in zip(ld, ld[1:]))           # two long rows in a row


def make_graph(kind, form, seed):
    gen = torch.Generator().manual_seed(seed)
    if kind == "edges":
        return Graph(boundary_degrees(form), N_SRC, gen)
    if kind == "long":
        return Graph(long_degrees(form), N_SRC, gen, long_t=LONG_T)
    # random skewed: destinations ~ rand^3 (a few hubs of hundreds of edges, many empty rows), sorted stably
    n_rows, n_src, e = 1200, 500, 8000
    dst = (n_rows * torch.rand(e, generator=gen, dtype=torch.float64).pow(3)).long().clamp_(0, n_rows - 1)
    src = torch.randint(0, n_src, (e,), generator=gen)
    order = torch.sort(dst, stable=True)[1]
    return Graph(torch.bincount(dst, minlength=n_rows), n_src, gen, col=src[order], eid=order)


# ------------------------------------------------------------------------------------------------
# buffers and direct C-ABI calls
# ------------------------------------------------------------------------------------------------
def _bits(t):
    return t.view(torch.int32 if t.element_size() == 4 else torch.int16)


class Guarded:
    """A [shape] output viewed inside a NaN-filled buffer with guard regions before and after it."""

    def __init__(self, shape, dtype, dev, fill=None):
        numel = math.prod(shape)
        self.lead = 64                                 # 16-byte aligned for both dtypes
        tail = 64 * (shape[-1] if len(shape) > 1 else 1) + 64
        self.buf = torch.full((self.lead + numel + tail,), float("nan"), dtype=dtype, device=dev)
        self.view = self.buf[self.lead:self.lead + numel].view(shape)
        if fill is not None:
            self.view.copy_(fill)
        self.numel = numel
        self.snap = self.buf.clone()

    def check_guards(self, what):
        b, s, e = _bits(self.buf), _bits(self.snap), self.lead + self.numel
        assert torch.equal(b[:self.lead], s[:self.lead]), f"{what}: wrote before the output"
        assert torch.equal(b[e:], s[e:]), f"{what}: wrote past the output"


def nan_padded(x, dev, extra=67):
    """``x`` on the device as the prefix view of a buffer whose remaining rows are NaN."""
    big = torch.full((x.shape[0] + extra, *x.shape[1:]), float("nan"), dtype=x.dtype, device=dev)
    big[:x.shape[0]] = x.to(dev)
    return big[:x.shape[0]]


def long_rows_arg(csr, feat, threshold):
    """ctypes ``trg_long_rows`` for ``csr`` split at ``threshold`` (its partial-sum slots start as NaN), the
    objects to keep alive, and the number of long rows."""
    lr = csr.long_rows(threshold)
    if lr is None:
        return None, None, 0
    partial = torch.full((lr.n_slots, feat), float("nan"), dtype=F32, device=csr.rowptr.device)
    s = _lib.TrgLongRows(_lib.ptr(lr.vrowptr), _lib.ptr(lr.vinfo), int(lr.vinfo.numel()), _lib.ptr(lr.long_rows),
                         _lib.ptr(lr.long_ptr), int(lr.long_rows.numel()), _lib.ptr(partial))
    return ctypes.byref(s), (s, partial), int(lr.long_rows.numel())


def abi_gather(mode, csr, x, out, *, lr=None, inv_deg=None, nbr_scale=None, coef=None, scale=None,
               accumulate=False, relu_of=None, n_rows=None):
    """One call of trg_sage_agg_fwd ("mean"), trg_sage_agg_bwd ("k2") or trg_gather_wsum ("wsum").
    Returns (return code, launch-count delta)."""
    lib = _lib.load()
    p = _lib.ptr
    n = csr.n_rows if n_rows is None else n_rows
    feat, code, st = x.size(1), _lib.dtype_code(x.dtype), _lib.stream()
    n0 = _lib.launch_count()
    if mode == "mean":
        rc = lib.trg_sage_agg_fwd(p(csr.rowptr), p(csr.col), p(x), n, feat, code, p(out), p(inv_deg), lr, st)
    elif mode == "k2":
        rc = lib.trg_sage_agg_bwd(p(csr.rowptr), p(csr.col), p(nbr_scale), p(x), n, feat, code, p(out),
                                  _lib.dtype_code(out.dtype), int(accumulate), p(relu_of), lr, st)
    else:
        rc = lib.trg_gather_wsum(p(csr.rowptr), p(csr.col), p(csr.eid), p(coef), p(scale), p(x), n, feat, code,
                                 p(out), _lib.dtype_code(out.dtype), int(accumulate), p(relu_of), lr, st)
    return rc, _lib.launch_count() - n0


# ------------------------------------------------------------------------------------------------
# inputs and references
# ------------------------------------------------------------------------------------------------
def scaled_rows(n, k, g, dtype, lo=-30, hi=30):
    """randn rows, each scaled by 2^e with e uniform in [lo, hi], rounded to the storage dtype."""
    x = torch.randn(n, k, generator=g, dtype=torch.float64)
    e = torch.randint(lo, hi + 1, (n, 1), generator=g).double()
    return (x * torch.pow(2.0, e)).to(dtype)


def small_ints(shape, g, dtype, lo=-3, hi=3):
    return torch.randint(lo, hi + 1, shape, generator=g).to(dtype)


def dyadic(n, g):
    """+-2^j, j in [-2, 1]: products with small integers stay exact in fp32."""
    sign = torch.randint(0, 2, (n,), generator=g).float() * 2 - 1
    return sign * torch.pow(2.0, torch.randint(-2, 2, (n,), generator=g).float())


def gather_sums(graph, w_edge, x):
    """fp64 ``sum_j w[j] x[col[j]]`` per row and the same sum of absolute values (w_edge None = 1)."""
    terms = x.double()[graph.col]
    if w_edge is not None:
        terms = terms * w_edge.double()[:, None]
    zeros = torch.zeros(graph.n_rows, x.size(1), dtype=torch.float64)
    return zeros.index_add(0, graph.dst, terms), zeros.index_add(0, graph.dst, terms.abs())


def assert_bits(got, want, what):
    got = got.detach().cpu()
    assert got.dtype == want.dtype and got.shape == want.shape, (what, got.dtype, got.shape, want.shape)
    bad = ~((got == want) | (torch.isnan(got) & torch.isnan(want)))
    if bool(bad.any()):
        idx = tuple(int(i) for i in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {got.numel()} entries differ (first at {idx}: got "
                             f"{float(got[idx])!r}, want {float(want[idx])!r})")


def check_bound(out, ref, absr, steps, out_dtype, what):
    """|out - ref| <= steps 2^-24 absr (+ 2^-8 |ref| after a bf16 rounding), element by element; ``steps``
    is per row."""
    out = out.detach().double().cpu()
    assert bool(torch.isfinite(out).all()), f"{what}: non-finite output"
    bound = steps.double()[:, None] * U * absr
    if out_dtype == BF16:
        bound = bound * (1 + 2.0 ** -8) + 2.0 ** -8 * ref.abs()       # bf16 unit roundoff: 8-bit significand
    err = (out - ref).abs()
    bad = err > bound
    if bool(bad.any()):
        ratio = float((err / bound.clamp(min=1e-300)).max())
        idx = tuple(int(i) for i in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {out.numel()} entries out of bound (worst err/bound "
                             f"{ratio:.3g}; first at {idx}: got {float(out[idx])!r}, want {float(ref[idx])!r} "
                             f"+- {float(bound[idx]):.3g})")


def expected_launches(graph, n_long):
    return 0 if graph.n_rows == 0 else 1 + (n_long > 0)


# ------------------------------------------------------------------------------------------------
# K1: mean
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,feat,kind", MEAN_CASES, ids=CASE_IDS)
def test_mean_every_form(dev, dtype, feat, kind):
    form = gather_form(dtype, feat)
    graph = make_graph(kind, form, seed=feat + 7 * len(kind))
    csr = graph.csr(dev)
    lr, keep, n_long = long_rows_arg(csr, feat, graph.long_t) if graph.long_t else (None, None, 0)
    assert (n_long > 0) == (kind == "long")
    gen = torch.Generator().manual_seed(feat)
    cnt = graph.deg.clamp(min=1).float()
    for data in ("exact", "random"):
        x = small_ints((graph.n_src, feat), gen, dtype) if data == "exact" else scaled_rows(graph.n_src, feat, gen,
                                                                                             dtype)
        xd = nan_padded(x, dev)
        what = f"{form} mean {data}"
        if data == "exact" or graph.long_t is None:
            if data == "exact":             # integer sums: exact in fp32 in any order, one IEEE division
                want = gather_sums(graph, None, x)[0].float() / cnt[:, None]
            else:                           # the sequential CSR-order fp32 sum, divided in IEEE fp32
                nt = torch.get_num_threads()
                torch.set_num_threads(1)
                try:
                    want = osage.scatter_mean(x.float()[graph.col], graph.dst, graph.n_rows)[0]
                finally:
                    torch.set_num_threads(nt)
            want = want.to(dtype)           # bf16: the fp32 mean rounded once
        else:
            s, a = gather_sums(graph, None, x)
            want = None
        outs = []
        for want_inv in (True, False):
            out = Guarded((graph.n_rows, feat), dtype, dev)
            inv = Guarded((graph.n_rows,), F32, dev) if want_inv else None
            rc, launches = abi_gather("mean", csr, xd, out.view, lr=lr, inv_deg=inv.view if inv else None)
            assert rc == 0, _lib.load().trg_last_error().decode()
            assert launches == expected_launches(graph, n_long), f"{what}: {launches} launches"
            out.check_guards(what)
            if inv is not None:
                inv.check_guards(what + " inv_deg")
                assert_bits(inv.view, 1.0 / cnt, what + " inv_deg")
            if want is not None:
                assert_bits(out.view, want, what)
            else:
                check_bound(out.view, s / cnt.double()[:, None], a / cnt.double()[:, None],
                            graph.deg + graph.slices + 4, dtype, what)
            outs.append(out.view)
        assert_bits(outs[1], outs[0].cpu(), what + ": repeated call")


# ------------------------------------------------------------------------------------------------
# K2 and wsum, every epilogue
# ------------------------------------------------------------------------------------------------
def weighted_inputs(mode, data, graph, dtype, feat, gen):
    exact = data == "exact"
    x = small_ints((graph.n_src, feat), gen, dtype) if exact else scaled_rows(graph.n_src, feat, gen, dtype)
    if mode == "k2":        # neighbour scale (1 / deg of the forward's destinations), indexed by col
        w = dyadic(graph.n_src, gen) if exact else torch.rand(graph.n_src, generator=gen) * 0.99 + 0.01
        scale = None
    else:                   # edge coefficient, indexed by eid; a device scalar scale
        w = dyadic(graph.n_edges, gen) if exact else torch.randn(graph.n_edges, generator=gen)
        scale = torch.tensor([-0.5 if exact else 0.7310586])
    base = (small_ints((graph.n_rows, feat), gen, torch.float64, -8, 8) * 0.25 if exact
            else scaled_rows(graph.n_rows, feat, gen, torch.float64))
    relu_of = small_ints((graph.n_rows, feat), gen, dtype, -2, 2)            # a third of the gate entries are 0
    return x, w, scale, base, relu_of


def epilogue_variants(dtype):
    outs = (dtype, F32) if dtype == BF16 else (dtype,)
    return [(acc, relu, given, od) for acc in (False, True) for relu in (False, True) for given in (False, True)
            for od in outs]


@pytest.mark.parametrize("mode,dtype,feat,kind", WEIGHTED_CASES, ids=WEIGHTED_IDS)
def test_weighted_gather_every_form_and_epilogue(dev, mode, dtype, feat, kind):
    form = gather_form(dtype, feat)
    graph = make_graph(kind, form, seed=feat + 7 * len(kind) + len(mode))
    csr = graph.csr(dev)
    lr, keep, n_long = long_rows_arg(csr, feat, graph.long_t) if graph.long_t else (None, None, 0)
    gen = torch.Generator().manual_seed(3 * feat + len(mode))
    steps = graph.deg + graph.slices + 4
    for data in ("exact", "random"):
        x, w, scale, base, relu_of = weighted_inputs(mode, data, graph, dtype, feat, gen)
        xd, wd, relud = nan_padded(x, dev), nan_padded(w, dev), nan_padded(relu_of, dev)
        scaled = {False: gather_sums(graph, None if mode == "k2" else w[graph.eid], x)}
        scaled[True] = gather_sums(graph, w[graph.col] if mode == "k2" else w[graph.eid], x)
        for acc, relu, given, od in epilogue_variants(dtype):
            what = (f"{form} {mode} {data}: accumulate={acc} relu_of={relu} "
                    f"{'inv_deg' if mode == 'k2' else 'scale'}={given} out={_DT[od]}")
            s, a = scaled[given] if mode == "k2" else scaled[False]
            post = float(scale) if (mode == "wsum" and given) else 1.0
            b = base.to(od)
            kw = dict(lr=lr, accumulate=acc, relu_of=relud if relu else None)
            if mode == "k2":
                kw["nbr_scale"] = wd if given else None
            else:
                kw.update(coef=wd, scale=scale.to(dev) if given else None)
            runs = 2 if kind == "long" and data == "random" and acc and relu else 1
            outs = []
            for _ in range(runs):
                out = Guarded((graph.n_rows, feat), od, dev, fill=b.to(dev) if acc else None)
                rc, launches = abi_gather(mode, csr, xd, out.view, **kw)
                assert rc == 0, _lib.load().trg_last_error().decode()
                assert launches == expected_launches(graph, n_long), f"{what}: {launches} launches"
                out.check_guards(what)
                outs.append(out.view.cpu())
            if runs == 2:
                assert_bits(outs[1], outs[0], what + ": repeated call")
            ref, absr = s * post, a * abs(post)
            if acc:
                ref, absr = ref + b.double(), absr + b.double().abs()
            if relu:
                keep_ = relu_of.double() > 0
                ref, absr = torch.where(keep_, ref, 0.0), torch.where(keep_, absr, 0.0)
            if data == "exact":
                assert_bits(outs[0], ref.to(od), what)
            else:
                check_bound(outs[0], ref, absr, steps, od, what)


# ------------------------------------------------------------------------------------------------
# zero rows and host-side rejections
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["mean", "k2", "wsum"])
def test_gather_zero_rows_launch_nothing(dev, mode):
    graph = Graph([], N_SRC, torch.Generator().manual_seed(0))
    csr = graph.csr(dev)
    x = torch.ones(N_SRC, 64, device=dev)
    out = Guarded((0, 64), F32, dev)
    rc, launches = abi_gather(mode, csr, x, out.view, coef=torch.ones(1, device=dev))
    assert rc == 0 and launches == 0
    out.check_guards(f"{mode}, zero rows")


@pytest.mark.parametrize("mode", ["mean", "k2", "wsum"])
@pytest.mark.parametrize("dtype,feat", [(F32, 516), (BF16, 1032), (F32, 1024)])
def test_gather_rejects_rows_wider_than_2048_bytes(dev, mode, dtype, feat):
    graph = make_graph("edges", "seg<LPR 32, VPL 4>", seed=1)
    csr = graph.csr(dev)
    x = torch.ones(N_SRC, feat, dtype=dtype, device=dev)
    out = Guarded((graph.n_rows, feat), dtype, dev)
    rc, launches = abi_gather(mode, csr, x, out.view, coef=torch.ones(graph.n_edges, device=dev))
    assert rc == TRG_E_UNSUPPORTED and launches == 0
    out.check_guards(f"{mode} rejected")
    n0 = _lib.launch_count()
    with pytest.raises(_lib.TrgError):
        if mode == "mean":
            Fn.sage_agg_fwd(csr, x)
        elif mode == "k2":
            Fn.sage_agg_bwd(csr, None, x)
        else:
            Fn.gather_wsum(csr, torch.ones(graph.n_edges, device=dev), x)
    assert _lib.launch_count() == n0


@pytest.mark.parametrize("mode", ["mean", "k2", "wsum"])
@pytest.mark.parametrize("dtype,feat", [(F32, 16), (F32, 4), (BF16, 32)])
def test_long_rows_need_rows_of_80_bytes(dev, mode, dtype, feat):
    """Long-row splitting is only instantiated for rows of >= 5 vectors; the library refuses it below."""
    graph = make_graph("long", "seg<LPR 8, R 4>", seed=2)
    csr = graph.csr(dev)
    lr, keep, n_long = long_rows_arg(csr, feat, LONG_T)
    assert n_long > 0
    x = torch.ones(N_SRC, feat, dtype=dtype, device=dev)
    out = Guarded((graph.n_rows, feat), dtype, dev)
    rc, launches = abi_gather(mode, csr, x, out.view, lr=lr, coef=torch.ones(graph.n_edges, device=dev))
    assert rc == TRG_E_UNSUPPORTED and launches == 0
    out.check_guards(f"{mode} rejected")


# ------------------------------------------------------------------------------------------------
# the functional wrappers on a library-built CSR
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,feat,long_rows", [(F32, 64, False), (F32, 128, True), (F32, 8, False),
                                                  (BF16, 128, False), (BF16, 256, True), (BF16, 16, False)])
def test_functional_wrappers_exact(dev, dtype, feat, long_rows, monkeypatch):
    """``sage_agg_fwd`` / ``sage_agg_bwd`` / ``gather_wsum`` as the model calls them (a CSR from
    ``RelationGraph``, hub rows split at the library's threshold, fp32 sum rows of a bf16 table accumulated
    across two relations, the ReLU gate), on integer data: every result is exact."""
    monkeypatch.setattr(G, "LONG_ROW_THRESHOLD", 64 if long_rows else 1 << 30)
    gen = torch.Generator().manual_seed(feat + long_rows)
    n_src, n_dst, e = 300, 200, 6000
    src = torch.randint(0, n_src, (e,), generator=gen)
    dst = (n_dst * torch.rand(e, generator=gen, dtype=torch.float64).pow(3)).long().clamp_(0, n_dst - 1)
    x = small_ints((n_src, feat), gen, dtype)
    coef = dyadic(e, gen)
    act = small_ints((n_dst, feat), gen, dtype, -2, 2)
    base = small_ints((n_dst, feat), gen, dtype)
    csr = trg.RelationGraph(torch.stack([src, dst]).to(dev), n_src, n_dst).fwd
    assert (csr.long_rows() is not None) == long_rows
    zeros = torch.zeros(n_dst, feat, dtype=torch.float64)
    s_plain = zeros.index_add(0, dst, x.double()[src])
    s_coef = zeros.index_add(0, dst, coef.double()[:, None] * x.double()[src])
    xd, cd, actd = x.to(dev), coef.to(dev), act.to(dev)

    out = Fn.sage_agg_bwd(csr, None, xd, out_dtype=F32)               # fp32 sum rows, also of a bf16 table
    assert out.dtype == F32
    assert_bits(out, s_plain.float(), "agg_bwd, fp32 rows")
    Fn.gather_wsum(csr, cd, xd, scale=torch.tensor([0.5], device=dev), out=out, accumulate=True)
    assert_bits(out, (s_plain + 0.5 * s_coef).float(), "wsum accumulating into fp32 rows")
    r = Fn.gather_wsum(csr, cd, xd, relu_of=actd)
    assert_bits(r, torch.where(act > 0, s_coef, 0.0).to(dtype), "wsum, gate only")
    r = Fn.sage_agg_bwd(csr, None, xd, out=base.to(dev), accumulate=True, relu_of=actd)
    assert_bits(r, torch.where(act > 0, base.double() + s_plain, 0.0).to(dtype), "agg_bwd, accumulate + gate")
    mean, inv = Fn.sage_agg_fwd(csr, xd)
    cnt = torch.bincount(dst, minlength=n_dst).clamp(min=1).float()
    assert_bits(mean, (s_plain.float() / cnt[:, None]).to(dtype), "mean")
    assert_bits(inv, 1.0 / cnt, "inv_deg")
    with pytest.raises(_lib.TrgError):
        Fn.sage_agg_bwd(csr, None, x.float().to(dev), out_dtype=BF16)   # only bf16 -> fp32 rows exist


# ------------------------------------------------------------------------------------------------
# row finish at production sizes
# ------------------------------------------------------------------------------------------------
def grid_sms(dev):
    return min(torch.cuda.get_device_properties(dev).multi_processor_count, MAX_SMS)


def signed_mags(shape, g, dtype):
    """Values of magnitude [0.25, 4) with random signs, multiples of 2^-25 (and so are their fp32 sums).  With
    ``row_scale = k / 64``, k <= 256, the exact ``row_scale * x + add`` spans fewer than 53 bits: it is exact
    in fp64, and its fp32 rounding is the fused (FMA) result."""
    m = torch.rand(shape, generator=g, device=g.device) * 3.75 + 0.25
    s = torch.randint(0, 2, shape, generator=g, device=g.device).float() * 2 - 1
    return (m * s).to(dtype)


def finish_inputs(n, feat, dt, g, dev):
    rs = torch.randint(0, 257, (n,), generator=g, device=dev).float() / 64          # includes 0
    add = signed_mags((n, feat), g, dt)
    act = torch.randint(-2, 3, (n, feat), generator=g, device=dev).to(dt)           # a fifth of the gates are 0
    return rs, add, act


def assert_either(out, unfused, fused, what):
    """Per element, the unfused ``row_scale * x + add`` (two fp32 roundings) or the fused one (one)."""
    ok = (out == unfused) | (out == fused)
    if not bool(ok.all()):
        idx = tuple(int(i) for i in (~ok).nonzero()[0])
        raise AssertionError(f"{what}: {int((~ok).sum())} of {out.numel()} entries are neither result (first at "
                             f"{idx}: got {float(out[idx])!r}, unfused {float(unfused[idx])!r}, fused "
                             f"{float(fused[idx])!r})")


def finish_refs(xf, rs, add, act, dt):
    """torch fp32 references (each op rounded once, as the kernels' FMUL / FADD) and the fused candidate."""
    af = add.float()
    gate = act.float() > 0
    unfused = torch.where(gate, xf * rs[:, None] + af, 0.0).to(dt)
    fused = torch.where(gate, (xf.double() * rs.double()[:, None] + af.double()).float(), 0.0).to(dt)
    return {"row_scale": (xf * rs[:, None]).to(dt), "add": (xf + af).to(dt),
            "relu_of": torch.where(gate, xf, 0.0).to(dt), "add+relu_of": torch.where(gate, xf + af, 0.0).to(dt),
            "all": (unfused, fused)}


FINISH_VARIANTS = [("f32", F32, F32), ("bf16", BF16, BF16), ("f32->bf16", F32, BF16)]
FINISH_CASES = [(name, ti, dt, f) for name, ti, dt in FINISH_VARIANTS
                for f in ((4,) if dt == F32 else (8,)) + (64, 128, 256, 1024)]


@pytest.mark.parametrize("name,in_dtype,dtype,feat", FINISH_CASES,
                         ids=[f"{c[0]}-F{c[3]}" for c in FINISH_CASES])
def test_rows_finish_grid_stride(dev, name, in_dtype, dtype, feat):
    """Row counts that send every thread of the (SMs x 8)-CTA grid through >= 3 iterations, plus a ragged tail;
    every epilogue alone bit-exact against torch's fp32 ops, all of them together with ``out`` aliasing ``add``."""
    vpr = feat * (4 if dtype == F32 else 2) // 16
    per_iter = grid_sms(dev) * 8 * 256
    n = 3 * per_iter // vpr + 7
    assert n * vpr > 3 * per_iter
    g = torch.Generator(device=dev).manual_seed(feat + len(name))
    x = nan_padded(signed_mags((n, feat), g, in_dtype), dev, extra=5)
    rs, add, act = finish_inputs(n, feat, dtype, g, dev)
    refs = finish_refs(x.float(), rs, add, act, dtype)
    for what, kw in (("row_scale", dict(row_scale=rs)), ("add", dict(add=add)), ("relu_of", dict(relu_of=act)),
                     ("add+relu_of", dict(add=add, relu_of=act)), ("all", dict(row_scale=rs, add=add, relu_of=act))):
        out = Guarded((n, feat), dtype, dev)
        n0 = _lib.launch_count()
        Fn.rows_finish(x, dtype, out=out.view, **kw)
        assert _lib.launch_count() - n0 == 1
        out.check_guards(f"rows_finish {name} {what}")
        if what == "all":
            assert_either(out.view, *refs[what], f"rows_finish {name} {what}")
        else:
            assert torch.equal(out.view, refs[what]), f"rows_finish {name} {what}"
    inplace = add.clone()                                                # out aliases add (allowed)
    Fn.rows_finish(x, dtype, row_scale=rs, add=inplace, relu_of=act, out=inplace)
    assert_either(inplace, *refs["all"], f"rows_finish {name}, out aliasing add")
    n0 = _lib.launch_count()
    assert Fn.rows_finish(x[:0], dtype).shape == (0, feat) and _lib.launch_count() == n0


PEER_FEAT = {1: 24, 2: 40, 3: 8, 4: 128, 5: 72, 8: 40, 16: 24}


@pytest.mark.parametrize("name,in_dtype,dtype", FINISH_VARIANTS, ids=[v[0] for v in FINISH_VARIANTS])
@pytest.mark.parametrize("n_peers", [1, 2, 3, 4, 5, 8, 16])
def test_peer_reduce_rows_grid_stride(dev, name, in_dtype, dtype, n_peers):
    """``n_units`` past three full iterations of the default grid at the widest unroll (UN = 4 units per thread,
    G = 2), so the j >= 1 units and the stride loop run for every compile-time rank count; ``ctas_per_sm`` 0, 1
    and 8; ``row0 > 0`` in partial tables taller than ``row0 + n_rows`` whose other rows are NaN.  The G tables
    live on this device; over NVLink they are the peers' mapped buffers."""
    feat = PEER_FEAT[n_peers]
    upr = feat * (4 if dtype == F32 else 2) // 16
    n = 3 * 4 * grid_sms(dev) * 2 * 256 // upr + 1001
    row0, tail = 1237, 333
    g = torch.Generator(device=dev).manual_seed(n_peers * 10 + len(name))
    parts = []
    for _ in range(n_peers):
        t = torch.full((row0 + n + tail, feat), float("nan"), dtype=in_dtype, device=dev)
        t[row0:row0 + n] = signed_mags((n, feat), g, in_dtype)
        parts.append(t)
    seq = parts[0][row0:row0 + n].float()
    for p in parts[1:]:
        seq = seq + p[row0:row0 + n].float()                             # fp32, rank order
    rs, add, act = finish_inputs(n, feat, dtype, g, dev)
    refs = finish_refs(seq, rs, add, act, dtype)
    calls = [("row_scale", 0, dict(row_scale=rs)), ("add", 0, dict(add=add)), ("relu_of", 0, dict(relu_of=act)),
             ("add+relu_of", 0, dict(add=add, relu_of=act))]
    calls += [("all", c, dict(row_scale=rs, add=add, relu_of=act)) for c in (0, 1, 8)]
    for what, ctas, kw in calls:
        n0 = _lib.launch_count()
        out = Fn.peer_reduce_rows(parts, row0, n, dtype, ctas_per_sm=ctas, **kw)
        assert _lib.launch_count() - n0 == 1
        tag = f"peer_reduce_rows {name} G={n_peers} ctas_per_sm={ctas} {what}"
        assert out.dtype == dtype and out.shape == (n, feat)
        if what == "all":
            assert_either(out, *refs[what], tag)
        else:
            assert torch.equal(out, refs[what]), tag
    n0 = _lib.launch_count()
    assert Fn.peer_reduce_rows(parts, 0, 0, dtype).shape == (0, feat) and _lib.launch_count() == n0

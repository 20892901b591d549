"""K4, the link-prediction loss kernels (edge_bce.cu), at every kernel form the library dispatches to, every
epilogue and the call sequences the train steps make, against an fp64 reference.

``launch_bce`` picks one of six ``edge_bce<T, LPR, VPL, R, TWO>`` forms from the row width in 16-byte vectors,
for the two-row entry point ``trg_edge_bce_fwd`` (TWO) and the single-row ``trg_edge_anchor_loss``; 512-byte rows
of the single-row entry point take ``edge_anchor_ring`` instead.  ``bce_form`` restates that dispatch and a test
that needs no GPU checks that the widths below reach every form of both entry points.  The checks:

* graphs built to hit each form's walk (``boundary_degrees``): degrees 0, 1, the unroll count +- 1, LPR - 1, LPR,
  LPR + 1, 2 LPR + 1 and 3 LPR + 1 (and the ring's group and slot wraps); rows that start inside a chunk and end
  on its last lane; runs of empty rows longer than a group and than a CTA; empty first and last rows, a partial
  last group and CTA; duplicate edges and gathered ids 0 and N - 1; one random skewed graph per dtype; a hub row
  of 2^21 edges per entry point;
* exact-signature inputs: small integers times per-row powers of two, so every logit ``x_e`` is exact in fp32 in
  any summation order and the only rounding left is the loss arithmetic's.  The bounds follow from it (u = 2^-24,
  gamma(n) = n u / (1 - n u)):
  - per-edge coefficient: ``expf`` (2 ulp <= 4u relative) plus five correctly rounded operations (``1 + e``, the
    division, ``* wbar``, ``* inv_e`` and ``inv_e`` itself) give gamma(9) |c| -- the error of ``e`` reaches
    ``e / (1 + e)`` and ``1 / (1 + e)`` with a factor <= 1 -- plus 2^-146 max(1, wbar) absolute for underflow;
    where fp32 sigmoid is exactly 1 (z >= 17, e < 2^-24 even with its 2 ulp) the coefficient is bit-exact;
  - anchor gradient, per element: gamma(chain + 9) sum_e |c_e g_e| (chain = deg FMAs, 2 deg in the two-row
    form), plus u |ref| when ``accumulate`` adds a base row, plus 2^-8 |ref| for bf16 rows; gated elements are
    exactly +0, rows without edges exactly 0 or their (gated) base row;
  - loss: each fp32 term ``softplus(z)`` is within 7u (``expf`` 4u, ``log1pf`` 2u, one addition); a lane sums
    at most m of them in fp32 before it folds that sum into its fp64 running sum (once per chunk; m and the
    number of chunks k from ``lane_chain``); the fixed-order fp64 reduction of the CTA partials adds a few more
    fp64 additions; then three fp32 roundings (the mean, ``* wbar``, the sum of the two means):
    gamma(m + 9) S + (k + tree) 2^-53 S, S = the fp64 loss.  Every case also keeps the 1e-5 relative promise;
* every case runs twice and must be bitwise identical; the loss does not depend on ``want_grad``, ``eid``,
  ``accumulate`` or ``relu_gate``; coefficients do not depend on where ``eid`` puts them;
* bounds: tables are prefix views of NaN-padded buffers, index arrays prefix views of buffers whose padding points
  at a NaN row (or at a guard slot), so a read past the end shows up as a NaN; outputs, the loss and the
  workspace are views into NaN-guarded buffers whose guards must come back bit for bit, and coefficient slots
  that no edge owns must stay untouched;
* launches: 2 per call (1 for zero rows); rows wider than 1024 bytes and a short workspace are refused on the
  host, whatever the row count, with no launch.
"""
import math

import pytest
import torch

import truth_recommendation_gnn_b200 as trg
from tests.util import U, Guarded, _bits, check_bound, nan_padded
from truth_recommendation_gnn_b200 import _lib
from truth_recommendation_gnn_b200 import functional as Fn
from truth_recommendation_gnn_b200.graph import CSR

pytestmark = pytest.mark.gpu

F32, BF16 = torch.float32, torch.bfloat16
TRG_E_WORKSPACE, TRG_E_UNSUPPORTED = 2, 4
N_SRC = 131                       # gathered table of the boundary graphs: every id is used many times
HUB = 1 << 21                     # edges of the hub row
WBAR = 1.2999999523162842         # fp32(1.3): wbar * x rounds
D64 = torch.float64


def gamma(n):
    return n * U / (1 - n * U)


# ------------------------------------------------------------------------------------------------
# Python mirror of the dispatch (edge_bce.cu: launch_bce, trg_edge_anchor_loss)
# ------------------------------------------------------------------------------------------------
RING = "edge_anchor_ring"
#: form -> (LPR lanes per row group, VPL 16-byte vectors per lane, R rows per group)
FORMS = {
    "edge_bce<LPR 2, VPL 1, R 1>": (2, 1, 1),
    "edge_bce<LPR 4, VPL 1, R 2>": (4, 1, 2),
    "edge_bce<LPR 8, VPL 1, R 4>": (8, 1, 4),
    "edge_bce<LPR 16, VPL 1, R 4>": (16, 1, 4),
    "edge_bce<LPR 32, VPL 1, R 4>": (32, 1, 4),
    "edge_bce<LPR 32, VPL 2, R 4>": (32, 2, 4),
}
RING_G, RING_R = 8, 4             # edges per cp.async group, rows per warp
RING_DEGREES = {7, 8, 9, 15, 16, 17, 24, 25, 33}


def row_vecs(dtype, h):
    return h * (4 if dtype == F32 else 2) // 16


def bce_form(dtype, h, two):
    rv = row_vecs(dtype, h)
    if not two and rv == 32:
        return RING
    for limit, form in zip((2, 4, 8, 16, 32, 64), FORMS):
        if rv <= limit:
            return form
    return "unsupported"


def unroll(form, two):
    """kUnroll: edges of one batch (all in flight at once)."""
    if form == RING:
        return RING_G
    lpr, vpl, _ = FORMS[form]
    return (1 if lpr < 4 else 2 if lpr < 8 else 4 if vpl == 1 else 2) * (1 if two else 2)


def chunk_edges(form):
    """Edges of one step of a row group's walk (one per lane; the ring: one cp.async group)."""
    return RING_G if form == RING else FORMS[form][0]


def group_rows(form):
    return RING_R if form == RING else FORMS[form][2]


def cta_rows(form):
    return 256 // 32 * RING_R if form == RING else 256 // FORMS[form][0] * FORMS[form][2]


WIDTHS = {F32: (4, 8, 12, 16, 20, 32, 36, 64, 68, 124, 128, 132, 256),
          BF16: (8, 16, 24, 32, 40, 64, 72, 128, 136, 248, 256, 264, 512)}
TOO_WIDE = {F32: 260, BF16: 520}
_DT = {F32: "f32", BF16: "bf16"}
CASES = ([(dt, h, "edges") for dt in (F32, BF16) for h in WIDTHS[dt]]
         + [(F32, 64, "skewed"), (BF16, 256, "skewed"), (F32, 16, "saturated"), (BF16, 256, "saturated")])
CASE_IDS = [f"{_DT[dt]}-H{h}-{k}" for dt, h, k in CASES]


def test_dispatch_mirror_covers_every_form():
    """Runs without a GPU: the widths reach every form of both entry points, with inactive lanes (rv 3, 5, 33)."""
    assert [bce_form(F32, 4 * rv, True) for rv in (1, 2, 3, 4, 5, 8, 9, 16, 17, 32, 33, 64, 65)] == [
        *[list(FORMS)[0]] * 2, *[list(FORMS)[1]] * 2, *[list(FORMS)[2]] * 2, *[list(FORMS)[3]] * 2,
        *[list(FORMS)[4]] * 2, *[list(FORMS)[5]] * 2, "unsupported"]
    assert bce_form(F32, 128, False) == RING and bce_form(BF16, 256, False) == RING
    assert bce_form(F32, 124, False) == bce_form(F32, 128, True) == list(FORMS)[4]
    assert [unroll(f, True) for f in FORMS] == [1, 2, 4, 4, 4, 2]
    assert [unroll(f, False) for f in FORMS] == [2, 4, 8, 8, 8, 4] and unroll(RING, False) == 8
    assert [cta_rows(f) for f in FORMS] == [128, 128, 128, 64, 32, 32] and cta_rows(RING) == 32
    for dt in (F32, BF16):
        assert bce_form(dt, TOO_WIDE[dt], True) == bce_form(dt, TOO_WIDE[dt], False) == "unsupported"
        assert {bce_form(dt, h, True) for h in WIDTHS[dt]} == set(FORMS)
        assert {bce_form(dt, h, False) for h in WIDTHS[dt]} == set(FORMS) | {RING}
        assert {row_vecs(dt, h) for h in WIDTHS[dt]} >= {3, 5, 33}      # inactive lanes; a partial 2nd vector
    for dt, h, _ in CASES:
        assert bce_form(dt, h, False) != "unsupported"
    assert {bce_form(dt, h, two) for dt, h, _ in HUB_CASES for two in (True, False)} >= {RING, list(FORMS)[3]}


# ------------------------------------------------------------------------------------------------
# graphs
# ------------------------------------------------------------------------------------------------
class LossGraph:
    """A CSR of the loss kernels built on the host from per-row degrees: rows in order, a row's edges back to
    back.  ``slot[e]`` is edge e's coefficient slot (its ``eid``), an injective map into ``n_slots`` > E slots
    so that some slots own no edge; ``neg[s]`` is the two-row form's negative of slot s."""

    def __init__(self, deg, n_src, gen, col=None):
        self.deg = torch.as_tensor(deg, dtype=torch.long)
        self.n_rows, self.n_src = self.deg.numel(), n_src
        self.rowptr = torch.zeros(self.n_rows + 1, dtype=torch.long)
        self.rowptr[1:] = torch.cumsum(self.deg, 0)
        e = int(self.rowptr[-1])
        self.dst = torch.repeat_interleave(torch.arange(self.n_rows), self.deg)
        if col is None:
            col = torch.randint(0, n_src, (e,), generator=gen)
            col[::17] = 0                                            # the first and the last gathered row
            col[5::23] = n_src - 1
            first = self.rowptr[:-1][self.deg >= 2]                  # duplicate edges: a row's last edge
            col[first + self.deg[self.deg >= 2] - 1] = col[first]    # repeats its first
        self.col = col
        self.n_slots = e + e // 7 + 3
        self.slot = torch.randperm(self.n_slots, generator=gen)[:e]
        self.neg = torch.randint(0, n_src, (self.n_slots,), generator=gen)
        self.neg[::13] = n_src - 1
        self.neg[3::19] = 0

    @property
    def n_edges(self):
        return self.col.numel()

    def eid_perm(self):
        """The edges' ``slot`` order as a permutation of [0, E): the ``eid`` of a CSR the library built, which
        the wrappers' E-entry coefficient arrays are indexed with."""
        return torch.argsort(torch.argsort(self.slot))

    def neg_col(self):
        """The negative of every edge, in CSR order."""
        return self.neg[self.slot]

    def device(self, dev):
        """rowptr / col / eid / neg_p (eid-indexed) / neg_p (CSR-indexed) as prefix views of padded device
        buffers; padding points at the gathered table's first NaN row, the first coefficient slot past the
        output (a guard), or edges that lie in that padding."""
        e = self.n_edges
        return dict(rowptr=idx_padded(self.rowptr, e + 5, dev), col=idx_padded(self.col, self.n_src, dev),
                    eid=idx_padded(self.slot, self.n_slots, dev),
                    neg=idx_padded(self.neg, self.n_src, dev, torch.int64),
                    neg_csr=idx_padded(self.neg_col(), self.n_src, dev, torch.int64))


def idx_padded(x, fill, dev, dtype=torch.int32, extra=67):
    big = torch.full((x.numel() + extra,), fill, dtype=dtype, device=dev)
    big[:x.numel()] = x.to(dev, dtype)
    return big[:x.numel()]


def boundary_degrees(form, two):
    """Row degrees that walk ``form`` across its boundaries (see the module docstring)."""
    lpr, r, cta, un = chunk_edges(form), group_rows(form), cta_rows(form), unroll(form, two)
    special = {0, 1, un - 1, un, un + 1, lpr - 1, lpr, lpr + 1, 2 * lpr + 1, 3 * lpr + 1}
    special = sorted(special | (RING_DEGREES if form == RING else set()))
    degs = []

    def align(m, fill):
        while len(degs) % m:
            degs.append(fill)

    for s in range(r + 1):               # every special degree at several offsets inside a group
        k = s % len(special)
        degs += [2] * s + special[k:] + special[:k]
    align(r, 1)
    # rows that start inside a chunk and end on the last lane of a later one (chunks start at the group's first
    # edge), and a row that fills its chunk
    degs += [lpr - 3, lpr + 3, lpr, 2 * lpr - 1, 1] if r > 1 else [lpr, 2 * lpr, 3 * lpr]
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


def make_graph(kind, form, two, seed):
    gen = torch.Generator().manual_seed(seed)
    if kind != "skewed":
        return LossGraph(boundary_degrees(form, two), N_SRC, gen)
    # random skewed: rows ~ rand^3 (a few rows of hundreds of edges, many empty rows)
    n_rows, n_src, e = 1200, 500, 8000
    dst = (n_rows * torch.rand(e, generator=gen, dtype=D64).pow(3)).long().clamp_(0, n_rows - 1)
    src = torch.randint(0, n_src, (e,), generator=gen)
    return LossGraph(torch.bincount(dst, minlength=n_rows), n_src, gen, col=src[torch.sort(dst, stable=True)[1]])


def hub_graph(seed):
    """One row of 2^21 edges among short and empty rows, starting inside a group."""
    gen = torch.Generator().manual_seed(seed)
    return LossGraph([0, 3, 1, HUB, 2, 0, 9, 1, 0, 33, 5], N_SRC, gen)


def lane_chain(form, two, rowptr):
    """(m, k): the most fp32 loss terms one lane sums before folding them into its fp64 running sum, and the
    most chunks one row group walks (one fold each).  A row group walks its edges in chunks of ``chunk_edges``
    and each chunk in batches of at most ``unroll`` edges that do not cross a row boundary; each batch adds one
    term to the fp32 sum of the lane finishing its first score, and every chunk ends with the fold."""
    deg = rowptr[1:] - rowptr[:-1]
    if int(rowptr[-1]) == 0:
        return 0, 0
    lpr, r, un = chunk_edges(form), group_rows(form), unroll(form, two)
    row = torch.repeat_interleave(torch.arange(deg.numel()), deg)
    grp = row // r
    chunk = (torch.arange(row.numel()) - rowptr[grp * r]) // lpr
    new_gc = torch.ones(row.numel(), dtype=torch.bool)
    new_gc[1:] = (grp[1:] != grp[:-1]) | (chunk[1:] != chunk[:-1])     # a (group, chunk) starts
    new = new_gc.clone()
    new[1:] |= row[1:] != row[:-1]                                      # a (row, chunk) segment starts
    seg_len = torch.bincount(torch.cumsum(new.long(), 0) - 1)
    gc_of_seg = (torch.cumsum(new_gc.long(), 0) - 1)[new]
    batches = torch.zeros(int(new_gc.sum()), dtype=torch.long).index_add_(0, gc_of_seg, (seg_len + un - 1) // un)
    return int(batches.max()), int(chunk.max()) + 1


@pytest.mark.parametrize("form,two", [(f, t) for f in FORMS for t in (True, False)] + [(RING, False)],
                         ids=[f"{f}-{'two' if t else 'single'}" for f in FORMS for t in (True, False)] + [RING])
def test_boundary_graphs_reach_every_boundary(form, two):
    """Runs without a GPU: the generated graphs contain what their docstrings promise."""
    lpr, r, cta, un = chunk_edges(form), group_rows(form), cta_rows(form), unroll(form, two)
    graph = make_graph("edges", form, two, seed=0)
    deg = graph.deg.tolist()
    want = {0, 1, un - 1, un, un + 1, lpr - 1, lpr, lpr + 1, 2 * lpr + 1, 3 * lpr + 1}
    assert want | (RING_DEGREES if form == RING else set()) <= set(deg)
    assert deg[0] == 0 and deg[-1] == 0 and graph.n_rows % cta != 0 and (r == 1 or graph.n_rows % r != 0)
    runs, run = [], 0
    for d in deg:
        run = run + 1 if d == 0 else 0
        runs.append(run)
    assert max(runs) > cta and any(all(d == 0 for d in deg[i:i + r]) for i in range(0, graph.n_rows - r + 1, r))
    rp = graph.rowptr.tolist()
    ends = [rp[i + 1] - rp[i - i % r] for i in range(graph.n_rows)]       # row end, from its group's first edge
    starts = [rp[i] - rp[i - i % r] for i in range(graph.n_rows)]
    assert any(e % lpr == 0 and s % lpr and d > 0 for e, s, d in zip(ends, starts, deg)) or r == 1
    assert any(e % lpr == 0 and e > lpr and d > 0 for e, d in zip(ends, deg))
    col = graph.col.tolist()
    assert 0 in col and N_SRC - 1 in col and 0 in graph.neg_col().tolist()
    assert any(col[a] == col[b - 1] for a, b in zip(rp[:-1], rp[1:]) if b - a >= 2)
    m, k = lane_chain(form, two, graph.rowptr)
    assert 1 <= m <= lpr and k >= 4          # a lane finishes <= 1 term per batch; a row of 3 LPR + 1 edges


def test_hub_graph():
    """Runs without a GPU: one row of 2^21 edges next to short and empty rows; one lane of the ring adds 2^18
    of its loss terms."""
    hub = hub_graph(0)
    assert int(hub.deg.max()) == HUB and int((hub.deg > 0).sum()) >= 6 and hub.deg[0] == 0
    m, k = lane_chain(RING, False, hub.rowptr)
    assert m <= RING_G and k >= HUB // RING_G


# ------------------------------------------------------------------------------------------------
# inputs and references
# ------------------------------------------------------------------------------------------------
def exact_rows(n, h, gen, dtype, lo, hi, neg_zeros=False):
    """Integers in [-3, 3] times 2^k per row, k uniform in [lo, hi]; ``neg_zeros``: half the zeros are -0.0."""
    x = torch.randint(-3, 4, (n, h), generator=gen).double()
    x = x * torch.pow(2.0, torch.randint(lo, hi + 1, (n, 1), generator=gen).double())
    if neg_zeros:
        flip = (x == 0) & (torch.rand(n, h, generator=gen) < 0.5)
        x = torch.where(flip, torch.tensor(-0.0, dtype=D64), x)
    return x.to(dtype)


def loss_inputs(graph, dtype, h, kind, gen):
    """Anchor rows (with +-0 entries for the ReLU gate), gathered rows and accumulate base rows."""
    sh = round(math.log2(h) / 4)                 # logits mostly within tens at every width
    lo, hi, glo, ghi = (2, 2, 4, 6) if kind == "saturated" else (-3 - sh, 1 - sh, -3 - sh, 1 - sh)
    anchor = exact_rows(graph.n_rows, h, gen, dtype, lo, hi, neg_zeros=True)
    gathered = exact_rows(graph.n_src, h, gen, dtype, glo, ghi)
    base = exact_rows(graph.n_rows, h, gen, dtype, -14, -10, neg_zeros=True)
    return anchor, gathered, base


class Ref:
    """fp64 reference of one launch over ``edges`` = [(col, label)] sets of the same rows (one set for the
    single-row form, positives and negatives for the two-row form)."""

    def __init__(self, graph, anchor, gathered, sets, e_scale, wbar=WBAR):
        a64, g64 = anchor.double(), gathered.double()
        s = a64 @ g64.T                                     # every logit, exact
        self.e_scale, self.wbar = e_scale, wbar
        inv_e = 1.0 / e_scale if e_scale else float("nan")
        w = torch.zeros(graph.n_rows, graph.n_src, dtype=D64)
        wabs = torch.zeros_like(w)
        self.coef, self.z, self.loss = [], [], 0.0
        for col, label in sets:
            x = s[graph.dst, col]
            z = -x if label else x
            c = (-wbar if label else 1.0) * torch.sigmoid(z) * inv_e
            sp = float(torch.logaddexp(torch.zeros_like(z), z).sum())
            self.loss += (wbar if label else 1.0) * sp * inv_e
            self.coef.append(c)
            self.z.append(z)
            w.index_put_((graph.dst, col), c, accumulate=True)
            wabs.index_put_((graph.dst, col), c.abs(), accumulate=True)
        self.labels = [lab for _, lab in sets]
        self.grad = w @ g64                                  # sum_e c_e g[col_e]
        self.absr = wabs @ g64.abs() + 2.0 ** -100           # sum_e |c_e g[col_e]|; floor: underflow
        self.chain = graph.deg * len(sets)                   # fp32 FMAs per anchor element


WORST = {}                        # quantity -> (worst error / bound, case): reported at the end of the module


def note(what, ratio, case):
    if ratio > WORST.get(what, (-1.0, None))[0]:
        WORST[what] = (ratio, case)


@pytest.fixture(scope="module", autouse=True)
def report_worst():
    yield
    for what, (ratio, case) in sorted(WORST.items()):
        print(f"\nK4 worst error/bound, {what}: {ratio:.3g} ({case})")


def check_coef(got, ref, z, label, e_scale, what):
    """Per-edge coefficients (CSR order) against fp64: gamma(9) |c| + underflow; bit-exact where fp32
    sigmoid is 1."""
    got = got.detach().cpu()
    assert bool(torch.isfinite(got).all()), f"{what}: non-finite coefficient"
    bound = gamma(9) * ref.abs() + 2.0 ** -146 * max(1.0, WBAR)
    err = (got.double() - ref).abs()
    if bool((err > bound).any()):
        i = int((err / bound).argmax())
        raise AssertionError(f"{what}: {int((err > bound).sum())} coefficients out of bound (worst err/bound "
                             f"{float(err[i] / bound[i]):.3g} at edge {i}: got {float(got[i])!r}, want "
                             f"{float(ref[i])!r}, z = {float(z[i])})")
    note("coefficient", float((err / bound).max()) if err.numel() else 0.0, what)
    sat = z >= 17
    inv_e = torch.tensor(1.0 / e_scale, dtype=F32)
    lim = (torch.tensor(-WBAR, dtype=F32) if label else torch.tensor(1.0, dtype=F32)) * inv_e
    assert bool((got[sat] == lim).all()), f"{what}: coefficient of a saturated sigmoid is not {float(lim)!r}"


def check_grad(got, ref, anchor, base, accumulate, relu, dtype, what, extra_abs=None):
    """Anchor gradient rows against fp64 (see the module docstring); exact on gated elements and empty rows."""
    got = got.detach().cpu()
    want = ref.grad + (base.double() if accumulate else 0.0)
    steps = ref.chain.double()[:, None] + 9 + (1 if accumulate else 0)
    absr = gamma(steps) / U * ref.absr + (want.abs() if accumulate else 0.0)
    if extra_abs is not None:
        absr = absr + extra_abs
    if relu:
        keep = anchor.float() > 0
        want, absr = torch.where(keep, want, 0.0), torch.where(keep, absr, 0.0)
        gated = _bits(got)[~keep]
        assert bool((gated == 0).all()), f"{what}: a gated element is not +0"
    check_bound(got, want, absr, torch.ones(got.size(0), dtype=D64), dtype, what)
    bound = U * absr
    if dtype == BF16:
        bound = bound * (1 + 2.0 ** -8) + 2.0 ** -8 * want.abs()
    note(f"gradient ({_DT[dtype]} rows)", float(((got.double() - want).abs() / bound.clamp(min=1e-300)).max()), what)
    empty = ref.chain == 0
    exp = base.float() + 0.0 if accumulate else torch.zeros(base.shape, dtype=F32)    # 0 + -0.0 = +0
    if relu:
        exp = torch.where(anchor.float() > 0, exp, 0.0)
    assert torch.equal(_bits(got[empty]), _bits(exp.to(dtype)[empty])), f"{what}: a row without edges"


def check_loss(got, ref, m, n_parts, what):
    """The launch's loss against fp64: gamma(m + 9) S + (k + tree) 2^-53 S with (m, k) = ``m``, and the 1e-5
    promise."""
    s = ref.loss
    if ref.e_scale == 0:
        assert math.isnan(got), f"{what}: E = 0 must give NaN, like torch's mean"
        return
    m, k = m
    tree = 5 + 8 + (n_parts + 1023) // 1024 + 5 + 32     # warp, CTA, strided finish, warp, finish
    bound = gamma(m + 9) * s + (k + tree) * 2.0 ** -53 * s + 2.0 ** -140
    err = abs(got - s)
    assert math.isfinite(got) and err <= bound, f"{what}: loss {got!r}, fp64 {s!r}: err/bound {err / bound:.3g}"
    assert err <= 1e-5 * s, f"{what}: loss {got!r} is {err / s:.3g} from fp64 {s!r}"
    note("loss", err / bound, what)
    note("loss, relative to fp64" + (" (hub rows)" if "hub" in what else ""), err / s if s else 0.0, what)


# ------------------------------------------------------------------------------------------------
# direct C-ABI calls
# ------------------------------------------------------------------------------------------------
def workspace(n_rows, dev):
    nbytes = int(_lib.load().trg_edge_bce_workspace_bytes(n_rows))
    return Guarded((nbytes // 4,), F32, dev), nbytes


def gptr(b):
    """Device pointer of a Guarded output (None -> NULL); a zero-size output still gets its address."""
    return None if b is None else b.buf.data_ptr() + b.lead * b.buf.element_size()


def wbar_dev(dev):
    return nan_padded(torch.tensor([WBAR], dtype=F32), dev, extra=3)


def abi_two_row(gd, n_rows, u, p, e_scale, want_grad, with_eid, n_out, dtype, h, dev, ws_bytes=None):
    """One trg_edge_bce_fwd call.  Returns (rc, launches, loss, c_pos, c_neg, g_u) as Guarded buffers."""
    lib, ptr = _lib.load(), _lib.ptr
    loss = Guarded((1,), F32, dev)
    cp = Guarded((n_out,), F32, dev) if want_grad else None
    cn = Guarded((n_out,), F32, dev) if want_grad else None
    gu = Guarded((n_rows, h), dtype, dev) if want_grad else None
    ws, nbytes = workspace(n_rows, dev)
    n0 = _lib.launch_count()
    rc = lib.trg_edge_bce_fwd(ptr(gd["rowptr"]), ptr(gd["col"]), ptr(gd["eid"]) if with_eid else None,
                              ptr(gd["neg"] if with_eid else gd["neg_csr"]), ptr(u), ptr(p), n_rows, e_scale, h,
                              _lib.dtype_code(dtype), ptr(gd["wbar"]), gptr(loss), gptr(cp), gptr(cn), gptr(gu),
                              gptr(ws),
                              nbytes if ws_bytes is None else ws_bytes, _lib.stream())
    launches = _lib.launch_count() - n0
    for b, w in ((loss, "loss"), (cp, "c_pos"), (cn, "c_neg"), (gu, "g_u"), (ws, "workspace")):
        if b is not None:
            b.check_guards(f"trg_edge_bce_fwd {w}")
    return rc, launches, loss, cp, cn, gu


def abi_anchor(gd, n_rows, anchor, gathered, e_scale, label, want_grad, with_eid, n_out, dtype, h, dev,
               base=None, accumulate=False, relu_gate=False, ws_bytes=None):
    """One trg_edge_anchor_loss call.  Returns (rc, launches, loss, coef, g_anchor) as Guarded buffers."""
    lib, ptr = _lib.load(), _lib.ptr
    loss = Guarded((1,), F32, dev)
    coef = Guarded((n_out,), F32, dev) if want_grad else None
    ga = Guarded((n_rows, h), dtype, dev, fill=base.to(dev) if accumulate else None) if want_grad else None
    ws, nbytes = workspace(n_rows, dev)
    n0 = _lib.launch_count()
    rc = lib.trg_edge_anchor_loss(ptr(gd["rowptr"]), ptr(gd["col"]), ptr(gd["eid"]) if with_eid else None,
                                  ptr(anchor), ptr(gathered), n_rows, e_scale, h, _lib.dtype_code(dtype), label,
                                  ptr(gd["wbar"]), gptr(loss), gptr(coef), gptr(ga), int(accumulate),
                                  int(relu_gate), gptr(ws),
                                  nbytes if ws_bytes is None else ws_bytes, _lib.stream())
    launches = _lib.launch_count() - n0
    for b, w in ((loss, "loss"), (coef, "coef"), (ga, "g_anchor"), (ws, "workspace")):
        if b is not None:
            b.check_guards(f"trg_edge_anchor_loss {w}")
    return rc, launches, loss, coef, ga


def coef_csr(buf, graph, with_eid, what):
    """Coefficients in CSR order; with ``eid`` the slots no edge owns must be untouched."""
    v = buf.view.cpu()
    if not with_eid:
        return v
    free = torch.ones(graph.n_slots, dtype=torch.bool)
    free[graph.slot] = False
    snap = buf.snap[buf.lead:buf.lead + buf.numel].cpu()
    assert torch.equal(_bits(v)[free], _bits(snap)[free]), f"{what}: wrote a slot that owns no edge"
    return v[graph.slot]


def same_bits(a, b, what):
    assert torch.equal(_bits(a.cpu()), _bits(b.cpu())), what


def device_case(graph, dev):
    gd = graph.device(dev)
    gd["wbar"] = wbar_dev(dev)
    return gd


# ------------------------------------------------------------------------------------------------
# trg_edge_bce_fwd: the two-row form
# ------------------------------------------------------------------------------------------------
def run_two_row(dev, graph, dtype, h, kind, seed, runs=2):
    form = bce_form(dtype, h, True)
    gen = torch.Generator().manual_seed(seed)
    u, p, _ = loss_inputs(graph, dtype, h, kind, gen)
    ud, pd = nan_padded(u, dev), nan_padded(p, dev)
    gd = device_case(graph, dev)
    e = graph.n_edges
    ref = Ref(graph, u, p, [(graph.col, 1), (graph.neg_col(), 0)], e)
    m = lane_chain(form, True, graph.rowptr)
    n_parts = -(-graph.n_rows // cta_rows(form))
    results = {}
    for with_eid in (True, False):
        for want_grad in (True, False):
            what = f"{form} two-row {_DT[dtype]} H={h} {kind}: eid={with_eid} want_grad={want_grad}"
            outs = []
            for _ in range(runs):
                rc, launches, loss, cp, cn, gu = abi_two_row(gd, graph.n_rows, ud, pd, e, want_grad, with_eid,
                                                             graph.n_slots if with_eid else e, dtype, h, dev)
                assert rc == 0, _lib.load().trg_last_error().decode()
                assert launches == (2 if graph.n_rows else 1), f"{what}: {launches} launches"
                outs.append([loss.view.cpu()] + ([coef_csr(cp, graph, with_eid, what),
                                                  coef_csr(cn, graph, with_eid, what), gu.view.cpu()]
                                                 if want_grad else []))
            for a, b in zip(outs[0], outs[-1]):
                same_bits(a, b, f"{what}: repeated call")
            results[(with_eid, want_grad)] = outs[0]
            check_loss(float(outs[0][0]), ref, m, n_parts, what)
            if want_grad:
                check_coef(outs[0][1], ref.coef[0], ref.z[0], 1, e, what + " c_pos")
                check_coef(outs[0][2], ref.coef[1], ref.z[1], 0, e, what + " c_neg")
                check_grad(outs[0][3], ref, u, u, False, False, dtype, what + " g_u")
    base = results[(True, True)]
    for key, r in results.items():
        for a, b in zip(base, r):
            same_bits(a, b, f"{form} two-row {_DT[dtype]} H={h}: {key} differs from eid=True want_grad=True")
    return ref


@pytest.mark.parametrize("dtype,h,kind", CASES, ids=CASE_IDS)
def test_two_row_every_form(dev, dtype, h, kind):
    graph = make_graph(kind, bce_form(dtype, h, True), True, seed=h + 3 * len(kind))
    run_two_row(dev, graph, dtype, h, kind, seed=h)


# ------------------------------------------------------------------------------------------------
# trg_edge_anchor_loss: the single-row form and the ring, every epilogue
# ------------------------------------------------------------------------------------------------
VARIANTS = [(acc, relu, eid) for acc in (False, True) for relu in (False, True) for eid in (True, False)]


def run_anchor(dev, graph, dtype, h, kind, seed, labels=(1, 0), variants=VARIANTS, runs=2, e_scale=None):
    form = bce_form(dtype, h, False)
    gen = torch.Generator().manual_seed(seed)
    anchor, gathered, base = loss_inputs(graph, dtype, h, kind, gen)
    ad, gdv = nan_padded(anchor, dev), nan_padded(gathered, dev)
    gd = device_case(graph, dev)
    e = graph.n_edges
    e_scale = e if e_scale is None else e_scale
    m = lane_chain(form, False, graph.rowptr)
    n_parts = -(-graph.n_rows // cta_rows(form))
    for label in labels:
        ref = Ref(graph, anchor, gathered, [(graph.col, label)], e_scale)
        losses, coefs, grads = [], [], {}
        for acc, relu, with_eid in variants + [(False, False, True), (False, False, False)]:
            want_grad = len(losses) < len(variants)
            what = (f"{form} {_DT[dtype]} H={h} {kind} label={label}: accumulate={acc} relu_gate={relu} "
                    f"eid={with_eid} want_grad={want_grad}")
            outs = []
            for _ in range(runs if want_grad else 1):
                rc, launches, loss, coef, ga = abi_anchor(gd, graph.n_rows, ad, gdv, e_scale, label, want_grad,
                                                          with_eid, graph.n_slots if with_eid else e, dtype, h,
                                                          dev, base=base, accumulate=acc, relu_gate=relu)
                assert rc == 0, _lib.load().trg_last_error().decode()
                assert launches == (2 if graph.n_rows else 1), f"{what}: {launches} launches"
                outs.append([loss.view.cpu()] + ([coef_csr(coef, graph, with_eid, what), ga.view.cpu()]
                                                 if want_grad else []))
            for a, b in zip(outs[0], outs[-1]):
                same_bits(a, b, f"{what}: repeated call")
            losses.append(outs[0][0])
            if not want_grad:
                continue
            check_loss(float(outs[0][0]), ref, m, n_parts, what)
            check_coef(outs[0][1], ref.coef[0], ref.z[0], label, e_scale, what)
            check_grad(outs[0][2], ref, anchor, base, acc, relu, dtype, what)
            coefs.append(outs[0][1])
            grads.setdefault((acc, relu), []).append(outs[0][2])
        for i, l in enumerate(losses):
            same_bits(l, losses[0], f"{form} {_DT[dtype]} H={h} label={label}: the loss of call {i} differs")
        for i, c in enumerate(coefs):
            same_bits(c, coefs[0], f"{form} {_DT[dtype]} H={h} label={label}: the coefficients of call {i} differ")
        for key, gs in grads.items():
            for g in gs:
                same_bits(g, gs[0], f"{form} {_DT[dtype]} H={h} label={label} {key}: eid changes the gradient")


@pytest.mark.parametrize("dtype,h,kind", CASES, ids=CASE_IDS)
def test_anchor_loss_every_form_and_epilogue(dev, dtype, h, kind):
    graph = make_graph(kind, bce_form(dtype, h, False), False, seed=h + 5 * len(kind))
    run_anchor(dev, graph, dtype, h, kind, seed=2 * h + 1)


# ------------------------------------------------------------------------------------------------
# hub rows
# ------------------------------------------------------------------------------------------------
HUB_CASES = [(F32, 128, "ring"), (BF16, 256, "ring"), (F32, 64, "register")]


@pytest.mark.parametrize("dtype,h,what", HUB_CASES, ids=[f"{_DT[d]}-H{h}-{w}" for d, h, w in HUB_CASES])
@pytest.mark.parametrize("entry", ["two_row", "anchor"])
def test_hub_row(dev, entry, dtype, h, what):
    """A row of 2^21 edges is walked by one row group: its loss terms are summed by a handful of lanes (2^18
    each in the ring form).  The loss must stay within 1e-5 of fp64."""
    graph = hub_graph(h)
    if entry == "two_row":
        run_two_row(dev, graph, dtype, h, "hub", seed=h, runs=1)
    else:
        run_anchor(dev, graph, dtype, h, "hub", seed=h, variants=[(True, True, True), (False, False, False)])


# ------------------------------------------------------------------------------------------------
# zero edges, zero rows, rejections
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("entry", ["two_row", "anchor"])
def test_empty_edge_sets(dev, entry):
    """E = 0: the loss is NaN (like torch's mean), gradient rows are 0 (or the base).  Zero rows with E > 0: the
    loss is exactly 0 from the finish launch alone."""
    gen = torch.Generator().manual_seed(0)
    h = 64
    for deg, e_scale in (([0] * 300, 0), ([], 0), ([], 5)):
        graph = LossGraph(deg, N_SRC, gen)
        a, g, base = loss_inputs(graph, F32, h, "edges", gen)
        ad, gdv = nan_padded(a, dev), nan_padded(g, dev)
        gd = device_case(graph, dev)
        what = f"{entry}: {graph.n_rows} rows, n_edges_scale={e_scale}"
        if entry == "two_row":
            rc, launches, loss, _, _, gu = abi_two_row(gd, graph.n_rows, ad, gdv, e_scale, True, True,
                                                       graph.n_slots, F32, h, dev)
            out, exp = gu.view.cpu(), torch.zeros(graph.n_rows, h)
        else:
            rc, launches, loss, _, ga = abi_anchor(gd, graph.n_rows, ad, gdv, e_scale, 0, True, True,
                                                   graph.n_slots, F32, h, dev, base=base, accumulate=True,
                                                   relu_gate=True)
            out, exp = ga.view.cpu(), torch.where(a > 0, base + 0.0, 0.0)
        assert rc == 0 and launches == (2 if graph.n_rows else 1), what
        assert torch.equal(_bits(out), _bits(exp)), what
        lv = float(loss.view)
        assert (math.isnan(lv) if e_scale == 0 else _bits(loss.view.cpu()).item() == 0), f"{what}: loss {lv}"


@pytest.mark.parametrize("n_rows", [0, 40])
@pytest.mark.parametrize("dtype", [F32, BF16])
@pytest.mark.parametrize("entry", ["two_row", "anchor"])
def test_rejects_rows_wider_than_1024_bytes(dev, entry, dtype, n_rows):
    """Refused on the host whatever the row count, with no launch and nothing written."""
    h = TOO_WIDE[dtype]
    graph = LossGraph([3] * n_rows, N_SRC, torch.Generator().manual_seed(1))
    x = nan_padded(torch.ones(max(n_rows, N_SRC), h, dtype=dtype), dev)
    gd = device_case(graph, dev)
    if entry == "two_row":
        rc, launches, loss, cp, cn, gu = abi_two_row(gd, n_rows, x, x, graph.n_edges, True, True, graph.n_slots,
                                                     dtype, h, dev)
        outs = (loss, cp, cn, gu)
    else:
        rc, launches, loss, coef, ga = abi_anchor(gd, n_rows, x, x, graph.n_edges, 1, True, True, graph.n_slots,
                                                  dtype, h, dev)
        outs = (loss, coef, ga)
    assert rc == TRG_E_UNSUPPORTED and launches == 0, (rc, launches)
    for b in outs:
        assert torch.equal(_bits(b.buf), _bits(b.snap)), "a refused call wrote an output"


@pytest.mark.parametrize("entry", ["two_row", "anchor"])
def test_rejects_short_workspace(dev, entry):
    graph = make_graph("edges", bce_form(F32, 64, entry == "two_row"), entry == "two_row", seed=3)
    x = nan_padded(torch.ones(max(graph.n_rows, N_SRC), 64), dev)
    gd = device_case(graph, dev)
    need = int(_lib.load().trg_edge_bce_workspace_bytes(graph.n_rows))
    for short in (need - 1, 0):
        if entry == "two_row":
            rc, launches, *_ = abi_two_row(gd, graph.n_rows, x, x, graph.n_edges, True, True, graph.n_slots, F32,
                                           64, dev, ws_bytes=short)
        else:
            rc, launches, *_ = abi_anchor(gd, graph.n_rows, x, x, graph.n_edges, 1, True, True, graph.n_slots,
                                          F32, 64, dev, ws_bytes=short)
        assert rc == TRG_E_WORKSPACE and launches == 0, (short, rc, launches)


# ------------------------------------------------------------------------------------------------
# the call sequences of the train steps
# ------------------------------------------------------------------------------------------------
SEQ_CASES = [(dt, h) for dt in (F32, BF16) for h in WIDTHS[dt]]
SEQ_IDS = [f"{_DT[dt]}-H{h}" for dt, h in SEQ_CASES]


def two_launch_grad_check(got, refs, anchor, relu, dtype, what):
    """Gradient rows of launch 1 (written) then launch 2 (accumulating, optionally gated): the first result is
    rounded to the row dtype before the second adds to it."""
    r1, r2 = refs
    merged = Ref.__new__(Ref)
    merged.grad, merged.absr, merged.chain = r1.grad + r2.grad, r1.absr + r2.absr, r1.chain + r2.chain
    extra = (2.0 ** -8 / U) * (1 + 2.0 ** -8) * r1.grad.abs() if dtype == BF16 else None   # launch 1's rounding
    # launch 2 adds its sum to launch 1's row: the accumulate epilogue on a zero base
    check_grad(got, merged, anchor, torch.zeros_like(anchor), True, relu, dtype, what, extra_abs=extra)


def sequence_case(dtype, h, seed):
    form = bce_form(dtype, h, False)
    graph = make_graph("edges", form, False, seed=seed)
    gen = torch.Generator().manual_seed(seed)
    anchor, gathered, _ = loss_inputs(graph, dtype, h, "edges", gen)
    return form, graph, anchor, gathered


@pytest.mark.parametrize("dtype,h", SEQ_CASES, ids=SEQ_IDS)
def test_one_gpu_step_sequence(dev, dtype, h):
    """fused_step.loss_and_grads: user-anchored positives then negatives, coefficients in CSR order, the second
    launch accumulating into the first's rows with the ReLU gate; n_edges_scale = E."""
    form, graph, hu, hp = sequence_case(dtype, h, seed=h + 11)
    e = graph.n_edges
    bu = CSR(graph.rowptr.int().to(dev), graph.col.int().to(dev), graph.eid_perm().int().to(dev), graph.n_rows,
             N_SRC)
    neg_by_user = CSR(bu.rowptr, graph.neg_col().int().to(dev), bu.eid, bu.n_rows, bu.n_cols)
    wbar = torch.tensor([WBAR], device=dev)
    hud, hpd = hu.to(dev), hp.to(dev)
    n0 = _lib.launch_count()
    l_pos, c_pos, dz_u = Fn.edge_anchor_loss(bu, hud, hpd, e, 1, wbar, True, None, coef_in_csr_order=True)
    l_neg, c_neg, dz_u = Fn.edge_anchor_loss(neg_by_user, hud, hpd, e, 0, wbar, True, dz_u, relu_gate=True,
                                             coef_in_csr_order=True)
    assert _lib.launch_count() - n0 == 4
    refs = (Ref(graph, hu, hp, [(graph.col, 1)], e), Ref(graph, hu, hp, [(graph.neg_col(), 0)], e))
    both = Ref(graph, hu, hp, [(graph.col, 1), (graph.neg_col(), 0)], e)
    what = f"one-GPU step {form} {_DT[dtype]} H={h}"
    m = lane_chain(form, False, graph.rowptr)
    n_parts = -(-graph.n_rows // cta_rows(form))
    total = float(l_pos.cpu() + l_neg.cpu())       # the step adds the two partial losses in fp32
    check_loss(float(l_pos), refs[0], m, n_parts, what + " positives")
    check_loss(float(l_neg), refs[1], m, n_parts, what + " negatives")
    assert abs(total - both.loss) <= 1e-5 * both.loss, (total, both.loss)
    check_coef(c_pos.cpu(), refs[0].coef[0], refs[0].z[0], 1, e, what + " c_pos")
    check_coef(c_neg.cpu(), refs[1].coef[0], refs[1].z[0], 0, e, what + " c_neg")
    two_launch_grad_check(dz_u.cpu(), refs, hu, True, dtype, what + " dz_u")


@pytest.mark.parametrize("dtype,h", SEQ_CASES, ids=SEQ_IDS)
def test_sharded_step_sequence(dev, dtype, h):
    """dist_fused.loss_and_grads_sharded: post-anchored (anchor = this rank's posts, gathered = the all-gathered
    user rows), coefficients at ``eid``, the GLOBAL positive count as n_edges_scale, the negatives' launch
    accumulating with the ReLU gate."""
    form, graph, hp, user_full = sequence_case(dtype, h, seed=h + 13)
    e_glob = 3 * graph.n_edges + 11
    neg_anchor_graph = LossGraph(graph.deg.flip(0), N_SRC, torch.Generator().manual_seed(h))  # the negatives
    pos_csr = CSR(graph.rowptr.int().to(dev), graph.col.int().to(dev), graph.eid_perm().int().to(dev),
                  graph.n_rows, N_SRC)
    neg_csr = CSR(neg_anchor_graph.rowptr.int().to(dev), neg_anchor_graph.col.int().to(dev),
                  neg_anchor_graph.eid_perm().int().to(dev), graph.n_rows, N_SRC)
    wbar = torch.tensor([WBAR], device=dev)
    hpd, ufd = hp.to(dev), user_full.to(dev)
    l_pos, c_pos, g_p = Fn.edge_anchor_loss(pos_csr, hpd, ufd, e_glob, 1, wbar, True, None, relu_gate=False)
    l_neg, c_neg, dz_p = Fn.edge_anchor_loss(neg_csr, hpd, ufd, e_glob, 0, wbar, True, g_p, relu_gate=True)
    r_pos = Ref(graph, hp, user_full, [(graph.col, 1)], e_glob)
    r_neg = Ref(neg_anchor_graph, hp, user_full, [(neg_anchor_graph.col, 0)], e_glob)
    what = f"sharded step {form} {_DT[dtype]} H={h}"
    n_parts = -(-graph.n_rows // cta_rows(form))
    check_loss(float(l_pos), r_pos, lane_chain(form, False, graph.rowptr), n_parts, what + " positives")
    check_loss(float(l_neg), r_neg, lane_chain(form, False, neg_anchor_graph.rowptr), n_parts, what + " negatives")
    # coefficients in original edge order: c[eid[e]]
    check_coef(c_pos.cpu()[graph.eid_perm()], r_pos.coef[0], r_pos.z[0], 1, e_glob, what + " c_pos")
    check_coef(c_neg.cpu()[neg_anchor_graph.eid_perm()], r_neg.coef[0], r_neg.z[0], 0, e_glob, what + " c_neg")
    two_launch_grad_check(dz_p.cpu(), (r_pos, r_neg), hp, True, dtype, what + " dz_p")


LINK_CASES = [(dt, min(h for h in WIDTHS[dt] if bce_form(dt, h, False) == f)) for dt in (F32, BF16)
              for f in list(FORMS) + [RING]]


@pytest.mark.parametrize("dtype,h", LINK_CASES, ids=[f"{_DT[dt]}-H{h}" for dt, h in LINK_CASES])
def test_link_bce_loss_every_form(dev, dtype, h):
    """``link_bce_loss`` forward and backward: dL/du from the two anchored launches, dL/dp through
    ``gather_wsum`` over the positives grouped by post and this step's negatives grouped by post."""
    n_u, n_p, e = 300, 500, 4000
    gen = torch.Generator().manual_seed(h)
    sh = round(math.log2(h) / 4)
    u = exact_rows(n_u, h, gen, dtype, -3 - sh, 1 - sh, neg_zeros=True)
    p = exact_rows(n_p, h, gen, dtype, -3 - sh, 1 - sh)
    tei = torch.stack([torch.randint(0, n_u, (e,), generator=gen), torch.randint(0, n_p, (e,), generator=gen)])
    tei = torch.cat([tei, tei[:, :50]], dim=1)                      # duplicate positives
    tei[1, :40] = n_p - 1
    tei[0, 40:80] = 0
    e = tei.size(1)
    neg = torch.randint(0, n_p, (e,), generator=gen)
    neg[::31] = 0
    w = torch.zeros(n_u + n_p)
    w[n_u:] = torch.where(torch.rand(n_p, generator=gen) < 0.25, 3.0, 1.0)
    ud, pd = u.to(dev).requires_grad_(True), p.to(dev).requires_grad_(True)
    teid, wd = tei.to(dev), w.to(dev)
    loss = trg.link_bce_loss(ud, pd, teid, neg.to(dev), wd, n_u)
    (2.0 * loss).backward()
    wbar = float(Fn.link_structure(teid, wd, n_u, n_p).wbar)       # the kernels' wbar (the cached structure)
    # fp64 reference
    u64, p64 = u.double(), p.double()
    xp, xn = (u64[tei[0]] * p64[tei[1]]).sum(1), (u64[tei[0]] * p64[neg]).sum(1)
    cp, cn = -wbar * torch.sigmoid(-xp) / e, torch.sigmoid(xn) / e
    s_loss = (wbar * torch.logaddexp(torch.zeros_like(xp), -xp).sum() / e
              + torch.logaddexp(torch.zeros_like(xn), xn).sum() / e)
    what = f"link_bce_loss {bce_form(dtype, h, False)} {_DT[dtype]} H={h}"
    assert abs(float(loss) - float(s_loss)) <= 1e-5 * float(s_loss), (what, float(loss), float(s_loss))
    zu = torch.zeros(n_u, h, dtype=D64)
    gu_pos = zu.index_add(0, tei[0], cp[:, None] * p64[tei[1]])
    gu = gu_pos + zu.index_add(0, tei[0], cn[:, None] * p64[neg])
    au = zu.index_add(0, tei[0], cp.abs()[:, None] * p64[tei[1]].abs() + cn.abs()[:, None] * p64[neg].abs())
    deg_u = 2 * torch.bincount(tei[0], minlength=n_u).double()[:, None]
    absr_u = gamma(deg_u + 10) / U * au + gu.abs()
    if dtype == BF16:
        absr_u = absr_u + (2.0 ** -8 / U) * (1 + 2.0 ** -8) * gu_pos.abs()
    check_bound(ud.grad.cpu(), 2 * gu, 2 * absr_u, torch.ones(n_u, dtype=D64), dtype, what + " dL/du")
    zp = torch.zeros(n_p, h, dtype=D64)
    gp_pos = zp.index_add(0, tei[1], cp[:, None] * u64[tei[0]])
    gp = gp_pos + zp.index_add(0, neg, cn[:, None] * u64[tei[0]])
    ap = zp.index_add(0, tei[1], cp.abs()[:, None] * u64[tei[0]].abs()).index_add(
        0, neg, cn.abs()[:, None] * u64[tei[0]].abs())
    deg_p = (torch.bincount(tei[1], minlength=n_p) + torch.bincount(neg, minlength=n_p)).double()[:, None]
    # gather_wsum: (deg + slices + 4) u per pass (test_gpu_gather), the coefficients' own 9u, the second pass's add
    absr_p = gamma(deg_p + 15) / U * ap + gp.abs()
    if dtype == BF16:
        absr_p = absr_p + (2.0 ** -8 / U) * (1 + 2.0 ** -8) * gp_pos.abs()
    check_bound(pd.grad.cpu(), 2 * gp, 2 * absr_p, torch.ones(n_p, dtype=D64), dtype, what + " dL/dp")

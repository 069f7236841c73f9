"""The row-wise, SpecialSpmm, ConvKB-head, ELU-epilogue and SGD kernels against fp64 at every branch they dispatch to.

Each of these kernels picks a kernel, a vector width or an epilogue from the shape, stride and alignment of its operands.
Section 0 restates every such predicate in Python and pins a table of cases that reaches each branch (CPU). The -m gpu
tests take their cases from that table and compare each kernel with an fp64 reference computed on the CPU from the same
fp32 inputs, under bounds derived from the operation:

- sums and dots of n fp32 terms (spmm, mlp_head_fwd, rank_scores): |err| <= (n + 8) 2^-24 sum |term_i| per entry;
- rownorm / residual_norm forward: one relative error of the row scale for the whole row, so <= 2e-6 per element;
  zero rows come out exactly 0, rows below the 1e-12 clamp as x / 1e-12;
- residual_norm backward: |err| <= 1e-6 ||g_row|| inv_row per row (the unclamped formula (g - o (o.g)) inv cancels, so a
  per-element relative bound does not apply there); dx2 is exactly 0 where mask = 0;
- tanh: forward within 2^-22 |tanh x| (libdevice tanhf is 2 ulp); backward |err| <= 2^-22 |dout| on the kernel's own y;
- ELU on x <= 0: |err| <= 2.5e-7 (a CPU emulation of the fp32 formula reaches 7.6e-8 on the exp2f branch; the device
  exp2f adds at most 2 ulp), and within 2.5e-7 relative on the polynomial branch; exact for x > 0;
- copies and gathers (gather_concat, the spmm backward, the LeakyReLU outputs of mlp_head_bwd): bit-equal;
- SGD: within 1 ulp of the fp64 update p - fp32(lr) g (the kernel is one fmaf; only double rounding can differ).

The kernels are reached through the public Python wrappers; branches those cannot reach (strided or misaligned outputs,
LeakyReLU slopes other than 0.01, D = 513 in rank_scores, a zero-length tensor inside one SGD launch) go through the C ABI.
"""
import pytest
import torch
import torch.nn.functional as F

from helpers import B200_SMS, gemm_nn_branch

U = 2.0 ** -24                    # fp32 unit roundoff
EPS = 1e-12                       # F.normalize's eps (models.py:160-161, 175-179)
RK_REG = 16                       # spk_convkb.cu: rank_scores keeps a row in RK_REG 32-float register chunks
LRELU_SLOPE = 0.01                # convkb.LRELU_SLOPE, nn.LeakyReLU()'s default
SENTINEL = -1234.5                # fills every padding column and every row past n; no kernel here writes it


# ---- 0. branch table (CPU) ------------------------------------------------------------------------------------------
def rownorm_kernel(width, ldx, ldy, x_off, y_off):
    """spk_rowops.cu rownorm(): offsets are in floats from a 16-byte aligned allocation."""
    vec2 = width % 2 == 0 and width <= 256 and ldx % 2 == 0 and ldy % 2 == 0 and x_off % 2 == 0 and y_off % 2 == 0
    if vec2 and width <= 64:
        return "vec2<1,4>"                      # 4 rows per warp, 32 rows per CTA
    return "vec2<4,1>" if vec2 else "scalar"


def spmm_branch(width):
    """spk_api.cu spmm_rowsum_kernel: lanes walk the edges of a row (then one warp sum) for width 1, columns otherwise."""
    return "lanes-over-edges" if width == 1 else "per-column"


def rank_scores_rc(d):
    """spk_convkb.cu launch_rank_scores: a pair row lives in RK_REG register chunks of 32 floats; wider rows are code 2."""
    return 0 if d <= 32 * RK_REG else 2


ROWNORM_WIDTHS = [1, 2, 7, 50, 63, 64, 66, 200, 255, 256, 258, 400, 512]
ROWNORM_ROWS = [1, 3, 31, 33, 1000]
ROWNORM_BIG = 100_000             # rows of the extra contiguous case at every width


def rownorm_layout(width, layout):
    """(row stride, base offset) in floats of the view a rownorm case reads and writes."""
    return {"contig": (width, 0),
            "padded": (width + 6, 0),                                  # same parity as width: padding columns only
            "odd_ld": (width + 1 if width % 2 == 0 else width + 2, 0),  # odd row stride
            "offset": (width + 2 + width % 2, 1)}[layout]              # even stride, base one float past 8-byte alignment


ROWNORM_CASES = [(w, lay) for w in ROWNORM_WIDTHS for lay in ("contig", "padded", "odd_ld", "offset")]
RESNORM_WIDTHS = [1, 31, 32, 33, 200, 512, 700]
SPMM_WIDTHS = [1, 2, 7, 32, 33, 200]
HEAD_D = [1, 12, 31, 32, 33, 200, 512, 1000]
HEAD_B = [1, 7, 9, 100_000]
RANK_D = [1, 31, 32, 33, 200, 511, 512]
# (T, R): every T and R of the issue at every D, with the T x R x D work of the fp64 reference kept small
RANK_TR = [(1, 1), (7, 2), (9, 1000), (1000, 1), (1000, 2)]
RANK_BIG_TR_D = [1, 33]           # D that also run T = R = 1000
GEMM_SHAPES = [(1000, 200, 200), (5000, 40, 37), (37_760, 64, 96), (37_888, 64, 96), (40_000, 200, 200)]
GEMM_PATHS = ["tc", "simt", "tc-pair", "tc-cluster"]


def gemm_layouts(k, n):
    """(name, lda, ldc, accumulate) of one GEMM case: aligned and unaligned C, with and without accumulate, and an A whose
    row stride is not a multiple of 4 (tcgen05 cannot load it by TMA: gemm_nn takes the SIMT GEMM)."""
    al, un = (n + 3) // 4 * 4, (n + 1 if (n + 1) % 4 else n + 2)
    return [("aligned C", k, al, False), ("aligned C", k, al, True), ("unaligned C", k, un, False),
            ("unaligned C", k, un, True), ("A lda % 4 != 0", k + 1 if (k + 1) % 4 else k + 2, al, False)]


GEMM_CASES = [(m, k, n, path) for m, k, n in GEMM_SHAPES for path in GEMM_PATHS]


def test_branch_table_covers_every_dispatch():
    # rownorm: the three kernels, the width bounds of both vec2 instantiations, and the alignment predicate
    got = {}
    for w, lay in ROWNORM_CASES:
        ld, off = rownorm_layout(w, lay)
        assert ld >= w
        got.setdefault(rownorm_kernel(w, ld, ld, off, off), set()).add((w, lay))
    assert set(got) == {"vec2<1,4>", "vec2<4,1>", "scalar"}
    assert (64, "contig") in got["vec2<1,4>"] and (66, "contig") in got["vec2<4,1>"] and (256, "contig") in got["vec2<4,1>"]
    assert (258, "contig") in got["scalar"] and (63, "contig") in got["scalar"] and (512, "padded") in got["scalar"]
    for lay in ("odd_ld", "offset"):                        # even widths <= 256 the stride or the base alone sends to scalar
        assert {(2, lay), (64, lay), (256, lay)} <= got["scalar"]
    assert rownorm_kernel(64, 64, 66, 0, 0) == "vec2<1,4>" and rownorm_kernel(64, 64, 65, 0, 0) == "scalar"
    assert rownorm_kernel(64, 64, 64, 0, 1) == "scalar"
    # spmm: width 1 against the per-column kernel, widths past one warp
    assert {spmm_branch(w) for w in SPMM_WIDTHS} == {"lanes-over-edges", "per-column"}
    assert any(w > 32 for w in SPMM_WIDTHS)
    # rank_scores: the largest D fills every register chunk, one more float is rejected
    assert max(RANK_D) == 32 * RK_REG and rank_scores_rc(max(RANK_D)) == 0 and rank_scores_rc(max(RANK_D) + 1) == 2
    assert {(d + 31) // 32 for d in RANK_D} >= {1, 2, RK_REG} and any(d % 32 for d in RANK_D)
    # GEMM with the ELU epilogue: every (kernel, epilogue) pair, and the pair / cluster threshold at 2 x 148 x 128 rows
    seen = set()
    for m, k, n, path in GEMM_CASES:
        for _, lda, ldc, acc in gemm_layouts(k, n):
            seen.add(gemm_nn_branch(m, n, lda, ldc, acc, 1, path))
    assert seen == {("simt", "elu_inplace"), ("tc", "tma"), ("tc", "row-vec4"), ("tc", "row-scalar"), ("pair", "tma"),
                    ("cluster", "tma"), ("cluster", "row-scalar")}, seen
    assert 2 * B200_SMS * 128 == 37_888
    assert gemm_nn_branch(37_888, 96, 64, 96, False, 1, "tc-pair") == ("pair", "tma")
    assert gemm_nn_branch(37_760, 96, 64, 96, False, 1, "tc-pair") == ("tc", "tma")
    assert gemm_nn_branch(37_888, 96, 64, 96, True, 1, "tc-pair") == ("tc", "row-vec4")      # act && accumulate
    assert gemm_nn_branch(37_888, 96, 64, 96, True, 0, "tc-pair") == ("pair", "tma")
    assert gemm_nn_branch(37_888, 96, 64, 96, True, 1, "tc-cluster") == ("tc", "row-vec4")
    assert gemm_nn_branch(37_760, 96, 64, 96, False, 1, "tc-cluster") == ("tc", "tma")
    assert gemm_nn_branch(5000, 37, 40, 40, False, 0, "tc") == ("tc", "row-vec4")           # N % 4 != 0


# ---- shared harness -------------------------------------------------------------------------------------------------
_WORST = {}


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    """Prints (with -s) the largest error and the largest error / bound each kernel family reached."""
    yield
    if _WORST:
        print("\nlargest |err| and |err| / bound per kernel family:")
        for fam, (e, r) in sorted(_WORST.items()):
            print(f"  {fam:24s} {e:10.3e} {r:8.4f}")


def _within(family, err, bound):
    err, bound = err.double().flatten(), bound.double().flatten()
    bad = ~(err <= bound)                               # a NaN error is out of bound too
    if bool(bad.any()):
        i = int(bad.nonzero()[0])
        pytest.fail(f"{family}: {int(bad.sum())} of {err.numel()} entries out of bound; first at flat index {i}: "
                    f"|err| {float(err[i]):.3e} > {float(bound[i]):.3e}")
    if err.numel():
        ratio = torch.where(bound > 0, err / bound, torch.zeros_like(err))
        w = _WORST.setdefault(family, [0.0, 0.0])
        w[0], w[1] = max(w[0], float(err.max())), max(w[1], float(ratio.max()))


def _dev():
    return torch.device("cuda:0")


def _lib():
    from recon_b200 import _lib as L
    return L


def _call(fn_name, *args):
    L = _lib()
    L.check(getattr(L.load(), fn_name)(*args, L.stream_ptr()), fn_name)


def _bits(x):
    return x.detach().contiguous().view(torch.int32).cpu()


def _strided(vals, ld, off=0):
    """vals [n, w] as a device view with row stride ld whose first element is float `off` of a SENTINEL-filled buffer.
    Returns (buffer, view, mask of the buffer elements outside the view)."""
    n, w = vals.shape
    total = off + (n + 1) * ld
    buf = torch.full((total,), SENTINEL)
    view = buf.as_strided((n, w), (ld, 1), off)
    view.copy_(vals)
    outside = torch.ones(total, dtype=torch.bool)
    outside.as_strided((n, w), (ld, 1), off).fill_(False)
    buf = buf.to(_dev())
    return buf, buf.as_strided((n, w), (ld, 1), off), outside


def _outside_unchanged(buf, outside):
    b = buf.cpu()
    assert bool((b[outside] == SENTINEL).all()), "a kernel wrote outside its view"


def _sum_bound(n_terms, abs_sum):
    return (n_terms + 8) * U * abs_sum


# ---- 1. rownorm -----------------------------------------------------------------------------------------------------
def _rownorm_input(n, w, seed):
    """Random rows plus, from 3 rows on, zero rows (row 0 among them), rows of norm 1e-14 and 5e-13 (below the clamp) and
    rows of norm 1e18 (the last row among them)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, w, generator=g, dtype=torch.float64) * torch.exp(torch.randn(n, 1, generator=g, dtype=torch.float64))
    if n >= 3:
        k = torch.arange(n) % 7
        last = torch.zeros(n, dtype=torch.bool)
        last[-1] = True
        for norm, sel in ((1e-14, k == 2), (5e-13, k == 4), (1e18, (k == 5) | last)):
            x[sel] = x[sel] / x[sel].norm(dim=1, keepdim=True) * norm
        x[(k == 0) & ~last] = 0
    return x.float()


def _check_rownorm(y, x, family):
    ref = F.normalize(x.double(), dim=1, eps=EPS)
    y = y.detach().cpu().double()
    _within(family, (y - ref).abs(), 2e-6 * ref.abs())        # zero rows: bound 0, so exactly 0


@pytest.mark.gpu
@pytest.mark.parametrize("width,layout", ROWNORM_CASES)
def test_rownorm(width, layout):
    from recon_b200 import functional as SF
    L = _lib()
    ld, off = rownorm_layout(width, layout)
    rows = ROWNORM_ROWS + ([ROWNORM_BIG] if layout == "contig" else [])
    for n in rows:
        x = _rownorm_input(n, width, seed=n * 1000 + width)
        fam = "rownorm " + rownorm_kernel(width, ld, ld, off, off)
        # out of place: the public wrapper for contiguous rows, the C ABI for strided / offset views
        xb, xv, xout = _strided(x, ld, off)
        yb, yv, yout = _strided(torch.zeros(n, width), ld, off)
        if layout == "contig":
            y = SF.rownorm(xv)
        else:
            _call("spk_rownorm", L.ptr(xv), ld, L.ptr(yv), ld, n, width)
            y = yv
            _outside_unchanged(yb, yout)
        _check_rownorm(y, x, fam)
        assert torch.equal(xb.cpu().as_strided((n, width), (ld, 1), off), x)       # the input is read only
        if n == ROWNORM_BIG:
            continue
        # in place through rownorm_ (any row stride, any base)
        SF.rownorm_(xv)
        _check_rownorm(xv, x, fam)
        _outside_unchanged(xb, xout)


# ---- 2. residual_norm -----------------------------------------------------------------------------------------------
def _resnorm_input(n, w, seed):
    """EW, x2, mask with rows of 8 kinds: ordinary (random 0/1 mask, twice), v exactly 0 (EW = -x2, mask 1), ||v|| = 1e-14
    with mask 1 / mask 0, ||v|| = 5e-13, and ||v|| = 1.001e-12 (just above the clamp) with mask 1 / mask 0."""
    g = torch.Generator().manual_seed(seed)
    ew = torch.randn(n, w, generator=g, dtype=torch.float64)
    x2 = torch.randn(n, w, generator=g, dtype=torch.float64)
    mask = (torch.rand(n, generator=g) < 0.5).double()
    k = torch.arange(n) % 8
    for kind, norm, m in ((2, 1e-14, 1.0), (3, 1e-14, 0.0), (4, 5e-13, 1.0), (5, 1.001e-12, 1.0), (6, 1.001e-12, 0.0)):
        sel = k == kind
        ew[sel] = ew[sel] / ew[sel].norm(dim=1, keepdim=True) * norm
        mask[sel] = m
        if m:
            x2[sel] = 0                                                 # v = EW exactly
    x2, mask = x2.float(), mask.float()
    ew = ew.float()
    ew[k == 1] = -x2[k == 1]
    mask[k == 1] = 1
    return ew, x2, mask


@pytest.mark.gpu
@pytest.mark.parametrize("width", RESNORM_WIDTHS)
def test_residual_norm_fwd_bwd(width):
    from recon_b200.functional import ResidualNormFn
    n = 2000
    ew, x2, mask = _resnorm_input(n, width, seed=width)
    g = torch.randn(n, width, generator=torch.Generator().manual_seed(width + 1))
    e_d = ew.to(_dev()).requires_grad_()
    x_d = x2.to(_dev()).requires_grad_()
    out = ResidualNormFn.apply(e_d, x_d, mask.to(_dev()))
    out.backward(g.to(_dev()))

    e64, x64 = ew.double().requires_grad_(), x2.double().requires_grad_()
    v64 = e64 + mask.double()[:, None] * x64
    ref = F.normalize(v64, dim=1, eps=EPS)
    ref.backward(g.double())
    k = torch.arange(n) % 8
    assert bool((v64.detach()[k == 1] == 0).all())
    nv = v64.detach().norm(dim=1)
    assert bool((nv[(k >= 2) & (k <= 4)] < EPS).all()) and bool((nv[(k == 5) | (k == 6)] > EPS).all())

    o = out.detach().cpu().double()
    _within("residual_norm fwd", (o - ref.detach()).abs(), 2e-6 * ref.detach().abs())
    inv = 1.0 / nv.clamp_min(EPS)
    row_bound = (1e-6 * g.double().norm(dim=1) * inv)[:, None].expand(n, width)
    dew, dx2 = e_d.grad.cpu(), x_d.grad.cpu()
    _within("residual_norm bwd", (dew.double() - e64.grad).abs(), row_bound)
    _within("residual_norm bwd", (dx2.double() - x64.grad).abs(), row_bound)
    assert bool((dx2[mask == 0] == 0).all())
    assert torch.equal(dx2[mask == 1], dew[mask == 1])


# ---- 3. SpecialSpmm (spmm_rowsum) and GatherRowsFn ---------------------------------------------------------------------
def _spmm_edges(n, seed):
    """[2, E] edges over n rows: a 5000-edge hub row (row 5), 500 duplicated edges, and empty rows (row 0, row n - 1 and
    every row = 3 mod 10)."""
    g = torch.Generator().manual_seed(seed)
    live = torch.arange(1, n - 1)
    live = live[live % 10 != 3]
    rows = torch.cat((live[torch.randint(0, live.numel(), (20_000,), generator=g)], torch.full((5000,), 5)))
    rows = torch.cat((rows, rows[:500]))
    rows = rows[torch.randperm(rows.numel(), generator=g)]
    return torch.stack((rows, torch.randint(0, n, (rows.numel(),), generator=g)))


@pytest.mark.gpu
@pytest.mark.parametrize("width", SPMM_WIDTHS)
def test_spmm_rowsum(width):
    from recon_b200.layers import SpecialSpmmFunctionFinal
    n = 3000
    edge = _spmm_edges(n, seed=width)
    e = edge.shape[1]
    g = torch.Generator().manual_seed(width + 7)
    w = torch.randn(e, width, generator=g) * torch.exp(torch.randn(e, 1, generator=g))
    w_d = w.to(_dev()).requires_grad_()
    out = SpecialSpmmFunctionFinal.apply(edge.to(_dev()), w_d, n, e, width)
    ref = torch.zeros(n, width, dtype=torch.float64).index_add_(0, edge[0], w.double())
    absum = torch.zeros(n, width, dtype=torch.float64).index_add_(0, edge[0], w.double().abs())
    deg = torch.bincount(edge[0], minlength=n).double()[:, None]
    assert deg[5] >= 5000 and deg[0] == 0 and deg[n - 1] == 0
    _within(f"spmm fwd ({spmm_branch(width)})", (out.detach().cpu().double() - ref).abs(), _sum_bound(deg, absum))
    gout = torch.randn(n, width, generator=g)
    out.backward(gout.to(_dev()))
    assert torch.equal(_bits(w_d.grad), _bits(gout[edge[0]]))


@pytest.mark.gpu
@pytest.mark.parametrize("width", [1, 7])
def test_spmm_rowsum_no_edges(width):
    from recon_b200.layers import SpecialSpmmFunctionFinal
    w = torch.zeros(0, width, device=_dev(), requires_grad=True)
    out = SpecialSpmmFunctionFinal.apply(torch.zeros(2, 0, dtype=torch.int64, device=_dev()), w, 9, 0, width)
    assert out.shape == (9, width) and bool((out == 0).all())
    out.backward(torch.ones(9, width, device=_dev()))
    assert w.grad.shape == (0, width)


@pytest.mark.gpu
def test_gather_rows_hub_entity():
    """GatherRowsFn (the embedding lookups of GAT/models.py:295-296): forward bit-equal to table[idx], backward (row sums
    on the spmm kernel at the embedding width) against fp64 index_add, with a 2000-triple hub entity."""
    from recon_b200.convkb import GatherRowsFn
    n_ent, d = 5000, 200
    g = torch.Generator().manual_seed(3)
    idx = torch.cat((torch.full((2000,), 7), torch.randint(0, n_ent - 100, (3000,), generator=g)))
    idx = idx[torch.randperm(idx.numel(), generator=g)]
    table = torch.randn(n_ent, d, generator=g)
    t_d = table.to(_dev()).requires_grad_()
    rows = GatherRowsFn.apply(t_d, idx.to(_dev()))
    assert torch.equal(_bits(rows), _bits(table[idx]))
    gout = torch.randn(idx.numel(), d, generator=g)
    rows.backward(gout.to(_dev()))
    ref = torch.zeros(n_ent, d, dtype=torch.float64).index_add_(0, idx, gout.double())
    absum = torch.zeros(n_ent, d, dtype=torch.float64).index_add_(0, idx, gout.double().abs())
    deg = torch.bincount(idx, minlength=n_ent).double()[:, None]
    assert deg[7] >= 2000
    _within("GatherRowsFn bwd", (t_d.grad.cpu().double() - ref).abs(), _sum_bound(deg, absum))


# ---- 4. ConvKB head: mlp_head, gather_concat, tanh, rank_scores --------------------------------------------------------
def _head_input(b, d, seed):
    """H1 [b, d] with exact-zero pre-activations (H1 = -b1) at every column = 0 mod 3 of every row = 0 mod 5."""
    g = torch.Generator().manual_seed(seed)
    h1 = torch.randn(b, d, generator=g) * 2
    b1 = torch.randn(d, generator=g) * 0.5
    w2 = torch.randn(1, d, generator=g)
    b2 = torch.randn(1, generator=g)
    zr, zc = torch.arange(0, b, 5), torch.arange(0, d, 3)
    h1[zr[:, None], zc[None, :]] = -b1[zc]
    return h1, b1, w2, b2


def _lrelu_sum64(pre, w2, b2, slope):
    """b2 + sum_d w2[d] lrelu(pre[., d]) in fp64, and sum |term| (b2 included), row by row in chunks."""
    outs, sums = [], []
    for c in range(0, pre.shape[0], 8192):
        p = pre[c:c + 8192]
        t = w2.double() * torch.where(p > 0, p, slope * p)
        outs.append(t.sum(1) + float(b2))
        sums.append(t.abs().sum(1) + abs(float(b2)))
    return torch.cat(outs), torch.cat(sums)


@pytest.mark.gpu
@pytest.mark.parametrize("slope", [LRELU_SLOPE, 0.0, 1.0])
@pytest.mark.parametrize("d", HEAD_D)
def test_mlp_head(d, slope):
    L = _lib()
    s32 = float(torch.tensor(slope, dtype=torch.float32))
    for b in (HEAD_B if slope == LRELU_SLOPE else [1, 7, 9, 1000]):
        h1, b1, w2, b2 = _head_input(b, d, seed=b + d)
        hb, hv, _ = _strided(h1, d + 3)                                   # row stride > D
        b1_d, w2_d, b2_d = b1.to(_dev()), w2.to(_dev()), b2.to(_dev())
        dout = torch.randn(b, generator=torch.Generator().manual_seed(d))
        dout_d = dout.to(_dev())
        if slope == LRELU_SLOPE:                                          # the public path: ConvKB's fused head
            from recon_b200.convkb import MLPHeadFn
            out = MLPHeadFn.apply(hv, b1_d, w2_d, b2_d).reshape(b)
        else:
            out = torch.empty(b, device=_dev())
            _call("spk_mlp_head_fwd", L.ptr(hv), d + 3, L.ptr(b1_d), L.ptr(w2_d), L.ptr(b2_d), s32, b, d, L.ptr(out))
        pre64 = h1.double() + b1.double()
        ref, absum = _lrelu_sum64(pre64, w2, b2, s32)
        _within("mlp_head fwd", (out.cpu().double() - ref).abs(), _sum_bound(d + 1, absum))

        dbuf, dv, dout_mask = _strided(torch.zeros(b, d), d + 5)
        abuf, av, aout_mask = _strided(torch.zeros(b, d), d + 2)
        _call("spk_mlp_head_bwd", L.ptr(hv), d + 3, L.ptr(b1_d), L.ptr(w2_d), s32, L.ptr(dout_d), b, d,
              L.ptr(dv), d + 5, L.ptr(av), d + 2)
        _outside_unchanged(dbuf, dout_mask)
        _outside_unchanged(abuf, aout_mask)
        pre32 = h1 + b1                                                    # fp32, as the kernel forms it
        g32 = dout[:, None] * w2
        s = torch.tensor(s32, dtype=torch.float32)
        assert torch.equal(_bits(dv), _bits(torch.where(pre32 > 0, g32, s * g32)))
        assert torch.equal(_bits(av), _bits(torch.where(pre32 > 0, pre32, s * pre32)))
        if b <= 1000:                                                      # torch's LeakyReLU: slope * g at pre = 0
            p = pre64.clone().requires_grad_()
            (F.leaky_relu(p, s32) * (dout.double()[:, None] * w2.double())).sum().backward()
            _within("mlp_head bwd", (dv.cpu().double() - p.grad).abs(), 3 * U * p.grad.abs())
            zero = pre32 == 0
            assert bool(zero.any())
            assert torch.equal(p.grad[zero], ((dout.double()[:, None] * w2.double()) * s32)[zero])


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 33, 513])
@pytest.mark.parametrize("indexed", [False, True])
@pytest.mark.parametrize("n_pieces", [1, 2, 3])
def test_gather_concat(n_pieces, indexed, d):
    from recon_b200.convkb import _gather_concat
    g = torch.Generator().manual_seed(n_pieces * 1000 + d + indexed)
    b = 1000
    sizes = [700, 40, 700] if indexed else [b, b + 5, b + 300]
    tables = [torch.randn(r, d, generator=g) for r in sizes]
    tri = torch.stack([torch.randint(0, r, (b,), generator=g) for r in sizes], dim=1).to(_dev())     # [B, 3]
    pieces = []
    for p in range(n_pieces):
        _, tv, _ = _strided(tables[p], d + 3)                              # tables with a row stride > D
        pieces.append((tv, tri[:, p] if indexed else None, 3))
    out = _gather_concat(pieces, b, d)
    rows = [tables[p][tri[:, p].cpu()] if indexed else tables[p][:b] for p in range(n_pieces)]
    assert torch.equal(_bits(out), _bits(torch.cat(rows, dim=1)))
    if indexed:
        for p in range(n_pieces):
            for bad in (-1, sizes[p]):
                t2 = tri.clone()
                t2[17, p] = bad
                with pytest.raises(IndexError):
                    _gather_concat([(tv, t2[:, q], 3) for q, (tv, _, _) in enumerate(pieces)], b, d)
    else:
        with pytest.raises(IndexError):                                    # idx = None: row b of every table, b < rows
            _gather_concat([(pieces[0][0][:b - 1], None, 3)], b, d)


_TANH_SPECIALS = [0.0, -0.0, 1e-30, -1e-30, 0.5, -0.55, 4.0, 9.01, -9.01, 20.0, -20.0, 1e30, -1e30,
                  float("inf"), float("-inf"), float("nan")]


@pytest.mark.gpu
@pytest.mark.parametrize("width", [1, 33])
def test_tanh_fwd_bwd(width):
    L = _lib()
    n = 600
    g = torch.Generator().manual_seed(width)
    x = (torch.randn(n, width, generator=g) * 3).flatten()
    x[:len(_TANH_SPECIALS)] = torch.tensor(_TANH_SPECIALS)
    x = x.reshape(n, width)
    xb, xv, xout = _strided(x, width + 3)
    _call("spk_tanh_fwd", L.ptr(xv), width + 3, n, width)
    _outside_unchanged(xb, xout)
    y = xv.cpu()
    ref = torch.tanh(x.double())
    fin = ~torch.isnan(x)
    _within("tanh fwd", (y.double() - ref)[fin].abs(), 2.0 ** -22 * ref[fin].abs())
    assert bool(torch.isnan(y[~fin]).all())
    zero = x == 0
    assert torch.equal(torch.signbit(y[zero]), torch.signbit(x[zero]))
    assert bool((y[x.abs() >= 20] == torch.sign(x[x.abs() >= 20])).all())       # +-20, +-1e30, +-inf: exactly +-1

    dout = torch.randn(n, width, generator=g)
    _, dov, _ = _strided(dout, width + 2)
    pb, pv, pout = _strided(torch.zeros(n, width), width + 5)
    _call("spk_tanh_bwd", L.ptr(xv), width + 3, L.ptr(dov), width + 2, n, width, L.ptr(pv), width + 5)
    _outside_unchanged(pb, pout)
    dpre = pv.cpu()
    ref_b = dout.double() * (1 - y.double() ** 2)                          # on the kernel's own y
    _within("tanh bwd", (dpre.double() - ref_b)[fin].abs(), 2.0 ** -22 * dout.double()[fin].abs())
    assert bool(torch.isnan(dpre[~fin]).all())

    from recon_b200.convkb import TanhFn                                   # the public autograd wrapper, contiguous rows
    xd = x.to(_dev()).requires_grad_()
    yt = TanhFn.apply(xd)
    yt.backward(dout.to(_dev()))
    assert torch.equal(_bits(yt), _bits(y)) and torch.equal(_bits(xd.grad), _bits(dpre))


RANK_CASES = [(d, t, r) for d in RANK_D for t, r in RANK_TR + ([(1000, 1000)] if d in RANK_BIG_TR_D else [])]


@pytest.mark.gpu
@pytest.mark.parametrize("d,t,r", RANK_CASES)
def test_rank_scores(d, t, r):
    L = _lib()
    g = torch.Generator().manual_seed(d * 7 + t + r)
    u = torch.randn(t, d, generator=g)
    bt = torch.randn(r, d, generator=g)
    w2 = torch.randn(1, d, generator=g)
    b2 = torch.randn(1, generator=g)
    u[0, :d // 2] = -bt[0, :d // 2]                                        # exact-zero pre-activations
    _, uv, _ = _strided(u, d + 5)
    _, bv, _ = _strided(bt, d + 1)
    ob, ov, oout = _strided(torch.zeros(t, r), r + 3)                      # output row stride > R
    s32 = float(torch.tensor(LRELU_SLOPE, dtype=torch.float32))
    w2_d, b2_d = w2.to(_dev()), b2.to(_dev())
    _call("spk_rank_scores", L.ptr(uv), d + 5, L.ptr(bv), d + 1, L.ptr(w2_d), L.ptr(b2_d), s32, t, r, d, L.ptr(ov), r + 3)
    _outside_unchanged(ob, oout)
    got = ov.cpu().double()
    u64, b64 = u.double(), bt.double()
    for c in range(0, t, 64):
        pre = u64[c:c + 64, None, :] + b64[None, :, :]                       # [tc, R, D]
        ref, absum = _lrelu_sum64(pre.reshape(-1, d), w2, b2, s32)
        _within("rank_scores", (got[c:c + 64].reshape(-1) - ref).abs(), _sum_bound(d + 1, absum))


@pytest.mark.gpu
def test_rank_scores_rejects_rows_past_the_register_tile():
    import types
    from recon_b200 import convkb
    L = _lib()
    d = 32 * RK_REG + 1
    u = torch.zeros(4, d, device=_dev())
    bt = torch.zeros(3, d, device=_dev())
    w2, b2 = torch.zeros(1, d, device=_dev()), torch.zeros(1, device=_dev())
    out = torch.full((4, 3), SENTINEL, device=_dev())
    rc = L.load().spk_rank_scores(L.ptr(u), d, L.ptr(bt), d, L.ptr(w2), L.ptr(b2), LRELU_SLOPE, 4, 3, d, L.ptr(out), 3,
                                  L.stream_ptr())
    assert rc == 2
    assert bool((out == SENTINEL).all())
    model = types.SimpleNamespace(final_entity_embeddings=torch.randn(20, d, device=_dev()),
                                  final_relation_embeddings=torch.randn(5, d, device=_dev()),
                                  convKB=types.SimpleNamespace(fc1=torch.nn.Linear(3 * d, d).to(_dev()),
                                                               fc2=torch.nn.Linear(d, 1).to(_dev())))
    with pytest.raises(RuntimeError):
        convkb.relation_scores(model, torch.tensor([[0, 1, 2], [3, 4, 5]]))


# ---- 5. ELU: the GEMM epilogue (act = 1) and spk_elu_inplace ---------------------------------------------------------
@pytest.fixture
def gemm_env(monkeypatch):
    """Sets functional.USE_TC and the opt-in GEMM variants (pair-CTA kernel, 2-CTA clusters) for one path."""
    from recon_b200 import functional as SF
    old = SF.USE_TC

    def set_path(path):
        SF.USE_TC = path != "simt"
        if path == "tc-pair":
            monkeypatch.setenv("SPK_TC_PAIR", "1")
        if path == "tc-cluster":
            monkeypatch.setenv("SPK_TC_CLUSTER", "2")
    yield set_path
    SF.USE_TC = old


def _elu_inplace(x):
    L = _lib()
    _call("spk_elu_inplace", L.ptr(x), x.stride(0), x.shape[0], x.shape[1])


@pytest.mark.gpu
@pytest.mark.parametrize("m,k,n,path", GEMM_CASES)
def test_gemm_nn_elu_epilogue_bit_equal(m, k, n, path, gemm_env):
    """gemm_nn(act=1), the ELU of the aggregate path's projection (functional.py AggGroupFn), is bit-equal to gemm_nn
    followed by spk_elu_inplace on every (kernel, epilogue) of the branch table. Inputs include overflowing products,
    +-inf, NaN and tiny rows; the products are ~N(0, 1), so both ELU branches and the switch at -0.125 are hit. No
    path writes the padding columns of C's rows."""
    from recon_b200.functional import gemm_nn
    gemm_env(path)
    g = torch.Generator().manual_seed(m + k + n)
    a0 = torch.randn(m, k, generator=g) / k ** 0.5
    a0[0, :] = 3e38
    a0[1, 0], a0[2, 1], a0[3, 2] = float("inf"), float("-inf"), float("nan")
    a0[4, :] = 1e-30
    b = torch.randn(k, n, generator=g).to(_dev())
    for name, lda, ldc, acc in gemm_layouts(k, n):
        _, a, _ = _strided(a0, lda)
        c0 = torch.randn(m, ldc, generator=g).to(_dev())
        ref, got = c0.clone(), c0.clone()
        pre = gemm_nn(a, b, out=ref[:, :n], accumulate=acc)
        assert bool(((pre > -0.2) & (pre <= -0.125)).any())
        _elu_inplace(ref[:, :n])
        gemm_nn(a, b, out=got[:, :n], accumulate=acc, act=1)
        assert torch.equal(_bits(got), _bits(ref)), (name, acc, gemm_nn_branch(m, n, lda, ldc, acc, 1, path))
        assert torch.equal(_bits(ref[:, n:]), _bits(c0[:, n:])), (name, acc, gemm_nn_branch(m, n, lda, ldc, acc, 0, path))
    assert bool(torch.isnan(got).any())


@pytest.mark.gpu
def test_elu_inplace_against_expm1():
    """spk_elu_inplace over 2M points of [-20, 0], +-16 ulp around the switch at -0.125, +-0, +-inf, NaN, denormals and
    positive values, in a strided view, against fp64 expm1."""
    sw = torch.tensor([-0.125])
    near = [sw]
    for direction in (-1.0, 1.0):
        v = sw
        for _ in range(16):
            v = torch.nextafter(v, torch.tensor([direction]))
            near.append(v)
    x = torch.cat([torch.linspace(-20, 0, 2_000_000), torch.cat(near), torch.linspace(-0.3, 0, 100_000),
                   torch.linspace(0, 20, 10_000),
                   torch.tensor([0.0, -0.0, float("inf"), float("-inf"), float("nan"), 1e-45, -1e-45, 1e-38, -1e-38,
                                 -1e-8, -88.0, -104.0, -3e38, 3e38])])
    w = 1000
    pad = (-x.numel()) % w
    x = torch.cat((x, torch.zeros(pad))).reshape(-1, w)
    xb, xv, xout = _strided(x, w + 3)
    _elu_inplace(xv)
    _outside_unchanged(xb, xout)
    y = xv.cpu()
    pos = x > 0
    assert torch.equal(_bits(y[pos]), _bits(x[pos]))
    assert bool(torch.isnan(y[torch.isnan(x)]).all())
    assert bool((y[x == float("-inf")] == -1).all()) and bool((y[x == 0] == 0).all())
    neg = (x <= 0) & torch.isfinite(x)
    ref = torch.expm1(x[neg].double())
    err = (y[neg].double() - ref).abs()
    _within("elu x <= 0 (abs)", err, torch.full_like(err, 2.5e-7))
    poly = x[neg] > -0.125
    _within("elu poly branch (rel)", err[poly], 2.5e-7 * ref[poly].abs())


# ---- 6. sgd_step ----------------------------------------------------------------------------------------------------
def _sgd_params(count, seed):
    """`count` parameters; with count >= 33 one has 0 elements and one has no .grad; with count 1 or 33 one has 700k
    elements (more than 148 x 16 x 256: the kernel's grid-stride loop)."""
    g = torch.Generator().manual_seed(seed)
    sizes = [(i * 37) % 500 + 1 for i in range(count)]
    if count in (1, 33):
        sizes[0] = 700_000
    ps = []
    for i, s in enumerate(sizes):
        if count >= 33 and i == 3:
            s = 0
        p = torch.nn.Parameter(torch.randn(s, generator=g).to(_dev()))
        if not (count >= 33 and i == 5):
            p.grad = torch.randn(s, generator=g).to(_dev())
        ps.append(p)
    return ps


def _sgd_ulps(got, p0, grad, lr32):
    ref = (p0.double() - lr32 * grad.double()).float()
    return (got.view(torch.int32).long() - ref.view(torch.int32).long()).abs()


@pytest.mark.gpu
@pytest.mark.parametrize("count", [1, 16, 17, 33])
def test_sgd_step(count):
    from recon_b200.loss import sgd_step
    assert 700_000 > B200_SMS * 16 * 256
    lr = 0.3
    lr32 = float(torch.tensor(lr, dtype=torch.float32))
    ps = _sgd_params(count, seed=count)
    before = [p.detach().cpu().clone() for p in ps]
    sgd_step(ps, lr)
    for p, p0 in zip(ps, before):
        got = p.detach().cpu()
        if p.grad is None or p.numel() == 0:
            assert torch.equal(_bits(got), _bits(p0))
            continue
        d = _sgd_ulps(got, p0, p.grad.cpu(), lr32)
        _within("sgd_step (ulp)", d.double(), torch.ones_like(d, dtype=torch.float64))


@pytest.mark.gpu
def test_sgd_step_skips_empty_tensor_inside_one_launch():
    """A zero-length entry between two tensors of one spk_sgd_step call (the C ABI compacts the list)."""
    L = _lib()
    g = torch.Generator().manual_seed(5)
    p = [torch.randn(n, generator=g).to(_dev()) for n in (300, 0, 1000)]
    gr = [torch.randn(n, generator=g).to(_dev()) for n in (300, 0, 1000)]
    before = [t.cpu() for t in p]
    a = L.SgdArgs()
    for j in range(3):
        a.param[j] = p[j].data_ptr() if p[j].numel() else None
        a.grad[j] = gr[j].data_ptr() if gr[j].numel() else None
        a.numel[j] = p[j].numel()
    a.count, a.lr = 3, 0.3
    L.check(L.load().spk_sgd_step(a, L.stream_ptr()), "sgd_step")
    lr32 = float(torch.tensor(0.3, dtype=torch.float32))
    for j in (0, 2):
        d = _sgd_ulps(p[j].cpu(), before[j], gr[j].cpu(), lr32)
        _within("sgd_step (ulp)", d.double(), torch.ones_like(d, dtype=torch.float64))

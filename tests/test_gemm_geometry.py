"""The dense GEMMs element-wise against fp64 at every tile geometry, pipeline depth and epilogue they dispatch to.

Section 0 (CPU) restates the plans of spk_gemm_tc.cu (gemm_nn_tc, tn_plan) and spk_gemm_simt.cu (row bands, TN splits)
in tests/helpers.py and checks that the case table below reaches every class of them. The -m gpu tests run each case
through functional.gemm_nn / gemm_tn (spk_gemm_nn_tc_act directly for N > 512, which gemm_nn sends to SIMT) on operands
that are views inside larger buffers: A and B with NaN in their padding columns and in the rows past the view, C inside
a buffer of sentinel bits with padding columns and rows above and below. Every case checks

1. |C - C64| <= gamma (|A| @ |B|) element-wise (+ 2^-23 |C64| for C +=), C64 the fp64 product of the same fp32 inputs.
   3xTF32 (A = A_hi + A_lo, hi = the top 10 explicit mantissa bits, so |lo| <= 2^-10 |x|): the dropped lo * lo product
   is <= 2^-20 |a b|, and the MMA reads each lo as TF32 (10 mantissa bits), which costs <= 2^-20 |a b| in each of the
   two correction products, so 3 * 2^-20; the fp32 accumulator in TMEM takes three MMAs per K step of 8, each allowed
   2^-23 of the running |sum|, and the epilogue / split reduction a few more roundings:
       tc:   gamma = 3 * 2^-20 + (3 * ceil(L / 8) + splits + 2) * 2^-23      (L = K for NN, M for TN; splits = 0 for NN)
       SIMT: gamma = (L + splits + 1) * 2^-24                                 (one fmaf chain per split, then the splits)
   This worst-case bound grows with L and only catches gross errors;
2. per 128-row x 32-column block of C (the kernels' M tile by one store box), rel-L2 against C64 <= BLOCK_TOL of the
   kernel family: a lost correction product in one k-block, a wrong K tail or a stale tile shows up here even when the
   whole-matrix rel-L2 stays small;
3. every sentinel outside C's view keeps its bits, and C is finite (the NaN padding is never read);
4. a second identical call is bit-identical;
5. with NaN planted in A (rows at the first and last M tile and at a 32-row boundary) and in B (the first and last column
   of every N tile), exactly those rows and columns of C are NaN; for TN, NaN in A's columns and B's columns give NaN
   rows and columns of C. This pins the tile origins, swizzles and descriptors at every geometry.

Tall outputs compare a sample of rows with fp64: every row of the first two and the last two M tiles and 2048 others.
"""
import math

import pytest
import torch

from helpers import (B200_SMS, SIMT_BAND, TC_BM, gemm_nn_branch, simt_nn_bands, simt_tn_splits, tc_nn_plan,
                     tc_tn_plan)

SENTINEL_BITS = 0x7FA5A5A5       # a signalling-NaN pattern: no kernel produces it, and reading it into a sum shows
SAMPLE_ABOVE = 40_000            # outputs with more rows compare a sample of rows with fp64
# Per-block rel-L2 limit per kernel family, under 4x the largest value this table reached on one NVIDIA B200 (1000 W
# power limit). The tcgen05 families grow about linearly with the reduction length (~8e-9 L for NN: the tensor cores'
# fp32 accumulation truncates), so their largest values come from K = 1000 (NN) and the 32-split TN case; the pair and
# cluster cases run K <= 72. A correction product lost for one k-block costs ~4e-4 sqrt(k-block columns / L) in rel-L2.
BLOCK_TOL = {"nn-tc": 2e-5,        # measured 7.6e-6
             "nn-pair": 2.5e-6,    # measured 8.7e-7
             "nn-cluster": 2.5e-6,  # measured 8.7e-7
             "nn-simt": 1e-6,      # measured 2.7e-7
             "tn-tc": 2.5e-5,      # measured 8.9e-6
             "tn-simt": 2e-6}      # measured 7.1e-7

# ---- the case table -----------------------------------------------------------------------------------------------
# NN: (path, M, K, N). "tc-pair" / "tc-cluster" set SPK_TC_PAIR=1 / SPK_TC_CLUSTER=2; "direct" calls spk_gemm_nn_tc_act
NN_CASES = [
    ("tc", 300, 3, 52),            # K < 8; 3 M tiles; 4 stages
    ("tc", 1000, 17, 35),          # K in 9..31; float4 row epilogue with N % 4 == 3; 4 stages
    ("tc", 700, 384, 64),          # K % 32 == 0, 12 k-blocks = 3 x 4 stages
    ("tc", 5000, 225, 100),        # K % 8 != 0 past 32; 3 stages
    ("tc", 19000, 33, 151),        # 149 M tiles: 2 per CTA; K = 33 (one column in the last k-block)
    ("tc", 38000, 64, 200),        # 297 M tiles: 3 per CTA; 2 stages
    ("tc", 2000, 1000, 256),       # BN = 256; 32 k-blocks over 2 stages; K % 32 == 8
    ("tc", 3000, 200, 203),        # 2 stages, float4 row epilogue
    ("tc", 20000, 40, 272),        # 2 N tiles of 160 (not a multiple of 32 at ceil(N / 2) = 136); 314 items: 3 per CTA
    ("tc", 1500, 300, 303),        # 2 N tiles, float4 row epilogue, 3 stages over 10 k-blocks
    ("tc", 900, 129, 416),         # 2 N tiles of 224
    ("tc", 4097, 256, 511),        # 2 N tiles of 256, one-row last M tile
    ("tc", 513, 96, 512),          # 2 N tiles of 256, TMA epilogue
    ("direct", 2000, 200, 600),    # 3 N tiles
    ("direct", 1000, 300, 603),    # 3 N tiles, float4 row epilogue
    ("tc", 1000, 64, 701),         # N > 512 through gemm_nn: the SIMT GEMM
    ("tc-pair", 37_938, 72, 96),   # 297 M tiles (odd) >= 2 x 148: pair kernel at one N tile
    ("tc-pair", 19_021, 50, 300),  # 149 M tiles (odd) x 2 N tiles >= 2 x 148
    ("tc-cluster", 37_938, 72, 96),
    ("tc-cluster", 19_021, 50, 300),
    ("simt", SIMT_BAND + 1, 5, 7),  # two row bands
    ("simt", 3001, 37, 131),
    ("simt", 2000, 200, 203),
]
# TN: (path, M, Ka, Nb): C[Ka, Nb] = A[M, Ka]^T B[M, Nb]
TN_CASES = [
    ("tc", 500, 40, 52),           # one split, 4 stages
    ("tc", 31_761, 129, 256),      # second Ka tile of one column; BN = 256, 2 stages; 32 splits, the last of 17 rows
    ("tc", 3000, 200, 600),        # 3 Nb tiles, 3 stages
    ("tc", 20_000, 416, 416),      # 4 Ka tiles x 2 Nb tiles, 19 splits
    ("tc", 5000, 50, 500),         # 2 Nb tiles of 256, 2 stages
    ("simt", 524_289, 64, 64),     # 512 splits (the cap)
    ("simt", 9000, 37, 70),
]


def _ld(n, kind):
    """Row stride of a view n wide: "al" a multiple of 4 with 4+ padding columns, "odd" an odd stride."""
    return (n + 3) // 4 * 4 + 4 if kind == "al" else n + 1 + n % 2


# (name, A stride kind, B stride kind, C kind, accumulate); C kind "al" / "odd" (odd ldc) / "off" (base one float past a
# 16-byte boundary, ldc % 4 == 0). An odd A or B stride sends tcgen05 products to SIMT, so only SIMT cases run those.
NN_LAYOUTS = [("aligned", "al", "al", "al", False), ("C +=, odd ldb", "al", "odd", "al", True),
              ("odd ldc", "al", "al", "odd", False), ("offset C, C +=", "al", "al", "off", True)]
TN_LAYOUTS = [("aligned", "al", "al", "al", False), ("C +=, odd ldc", "al", "al", "odd", True),
              ("offset C", "al", "al", "off", False)]
SIMT_LAYOUT = ("odd lda, odd ldb", "odd", "odd", "al", True)


def nn_layouts(path):
    return NN_LAYOUTS + ([SIMT_LAYOUT] if path == "simt" else [])


def tn_layouts(path):
    return TN_LAYOUTS + ([SIMT_LAYOUT] if path == "simt" else [])


def nn_kernel(path, m, k, n, lay):
    """Plan of one NN call: the SIMT GEMM or the tcgen05 plan (kernel, tile shape, stages, epilogue ...)."""
    _, a, _, c, acc = lay
    if path == "simt" or (path != "direct" and n > 512) or a != "al":
        return dict(kernel="simt", bands=simt_nn_bands(m), a_vec=a == "al", c_vec=c == "al")
    tc_path = "tc" if path == "direct" else path
    if path != "direct":
        assert gemm_nn_branch(m, n, _ld(k, a), _ld(n, c), acc, 0, tc_path)[0] != "simt"
    return tc_nn_plan(m, n, k, c == "al", acc, 0, tc_path)


def tn_kernel(path, m, ka, nb, lay):
    _, a, b, _, _ = lay
    if path == "simt" or a != "al" or b != "al":
        return dict(kernel="simt", splits=simt_tn_splits(m, ka, nb), a_vec=a == "al")
    return dict(tc_tn_plan(m, ka, nb), kernel="tc")


def test_branch_table_covers_every_class():
    nn = [(path, m, k, n, lay, nn_kernel(path, m, k, n, lay)) for path, m, k, n in NN_CASES for lay in nn_layouts(path)]
    tc = [(p, m, k, n, lay, pl) for p, m, k, n, lay, pl in nn if pl["kernel"] != "simt"]
    # every pipeline depth with every epilogue, at one and at two N tiles; N tiles reach 3
    got = {(pl["n_tiles_n"], pl["stages"], pl["epilogue"]) for *_, pl in tc}
    want = {(1, s, e) for s in (2, 3, 4) for e in ("tma", "row-vec4", "row-scalar")}
    # at two N tiles BN >= 160, so 4 stages never fit and the TMA staging leaves room for 2 only: every other class
    want |= {(2, 2, "tma"), (2, 3, "row-vec4"), (2, 3, "row-scalar"), (2, 2, "row-vec4"), (2, 2, "row-scalar")}
    assert want <= got, want - got
    reachable = {(pl["n_tiles_n"], pl["stages"], pl["epilogue"]) for n in range(257, 513) for c_vec in (True, False)
                 for pl in [tc_nn_plan(1000, n, 64, c_vec)]}
    assert {x for x in reachable if x[0] == 2} <= got
    assert {pl["n_tiles_n"] for *_, pl in tc} >= {1, 2, 3}
    assert all(p == "direct" for p, m, k, n, lay, pl in tc if pl["n_tiles_n"] >= 3)
    assert {pl["BN"] for *_, pl in tc} >= {160, 224, 256}
    # K: < 8, multiple of 32, multiple of 8 only, neither past 32, 9..31; k-blocks >= 3 x stages
    ks = {k for _, m, k, n, lay, pl in tc}
    assert any(k < 8 for k in ks) and any(k % 32 == 0 for k in ks) and any(k % 8 == 0 and k % 32 for k in ks)
    assert any(k % 8 and k > 32 for k in ks) and any(8 < k < 32 for k in ks) and any(k % 32 == 1 for k in ks)
    assert {pl["stages"] for *_, pl in tc if pl["num_kb"] >= 3 * pl["stages"]} == {2, 3, 4}
    # persistent CTAs with 1, 2 and 3 tiles; partial last M tiles
    assert {pl["tiles_per_cta"] for *_, pl in tc} >= {1, 2, 3}
    assert any(m % TC_BM for p, m, k, n, lay, pl in tc) and any(m % TC_BM == 1 for p, m, k, n, lay, pl in tc)
    # pair and cluster kernels at one and two N tiles with an odd M-tile count; with C += the cluster path runs cs = 1
    for kern in ("pair", "cluster"):
        hit = {(pl["n_tiles_n"], pl["m_tiles"] % 2) for *_, pl in tc if pl["kernel"] == kern}
        assert {(1, 1), (2, 1)} <= hit, (kern, hit)
    assert {pl["epilogue"] for *_, pl in tc if pl["kernel"] == "cluster"} == {"tma", "row-scalar"}
    assert 2 * B200_SMS * TC_BM == 37_888 and tc_nn_plan(37_888, 96, 72, True, path="tc-pair")["kernel"] == "pair"
    assert tc_nn_plan(37_760, 96, 72, True, path="tc-pair")["kernel"] == "tc"
    assert tc_nn_plan(B200_SMS * TC_BM, 300, 50, True, path="tc-cluster")["kernel"] == "cluster"
    assert tc_nn_plan(B200_SMS * TC_BM - 128, 300, 50, True, path="tc-cluster")["kernel"] == "tc"
    # SIMT NN: two row bands; vector and scalar A loads; float4 and scalar C stores; odd ldb
    simt = [(p, m, k, n, lay, pl) for p, m, k, n, lay, pl in nn if pl["kernel"] == "simt"]
    assert max(pl["bands"] for *_, pl in simt) == 2 and simt_nn_bands(SIMT_BAND) == 1
    assert {(pl["a_vec"], pl["c_vec"]) for *_, pl in simt} == {(True, True), (True, False), (False, True)}
    assert any(lay[2] == "odd" for *_, lay, pl in simt) and any(n % 4 == 3 for p, m, k, n, lay, pl in simt)
    # TN
    tn = [(path, m, ka, nb, lay, tn_kernel(path, m, ka, nb, lay)) for path, m, ka, nb in TN_CASES for lay in tn_layouts(path)]
    ttc = [pl for *_, pl in tn if pl["kernel"] == "tc"]
    assert {pl["stages"] for pl in ttc} == {2, 3, 4}
    assert any(pl["n_tiles_k"] >= 2 for pl in ttc) and any(ka % 128 == 1 for p, m, ka, nb, lay, pl in tn)
    assert max(pl["n_tiles_n"] for pl in ttc) >= 3
    assert {pl["splits"] == 1 for pl in ttc} == {True, False}
    assert any(pl["splits"] > 1 and pl["last_split_rows"] < 32 for pl in ttc)
    tsimt = [pl for *_, pl in tn if pl["kernel"] == "simt"]
    assert max(pl["splits"] for pl in tsimt) == 512 and simt_tn_splits(511 * 1024, 64, 64) == 511
    assert {pl["a_vec"] for pl in tsimt} == {True, False}


# ---- GPU harness --------------------------------------------------------------------------------------------------
_WORST = {}


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    """Prints (with -s) the largest |err| / bound and the largest block rel-L2 per kernel family."""
    yield
    if _WORST:
        print("\nlargest |err| / bound and block rel-L2 per GEMM family:")
        for fam, (r, b) in sorted(_WORST.items()):
            print(f"  {fam:12s} {r:8.4f} {b:10.3e}")


@pytest.fixture
def gemm_path(monkeypatch):
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


def _dev():
    return torch.device("cuda:0")


def _operand(vals, kind):
    """vals [r, c] (CPU) copied into a view of a NaN-filled device buffer: padding columns, and 5 rows past the view."""
    r, c = vals.shape
    buf = torch.full((r + 5, _ld(c, kind)), float("nan"), device=_dev())
    buf[:r, :c] = vals.to(_dev())
    return buf[:r, :c]


def _out(c0, kind):
    """C0 [m, n] (CPU) in a view of a sentinel-filled buffer: 3 rows above and below, padding columns; "off" starts the
    view one float past a 16-byte boundary. Returns (buffer, view)."""
    m, n = c0.shape
    off = 1 if kind == "off" else 0
    ld = _ld(n + off, "odd" if kind == "odd" else "al")
    buf = torch.full((m + 6, ld), SENTINEL_BITS, dtype=torch.int32, device=_dev()).view(torch.float32)
    view = buf[3:3 + m, off:off + n]
    view.copy_(c0.to(_dev()))
    return buf, view


def _untouched(buf, view):
    """Every float of buf outside view keeps the sentinel's bits."""
    mask = torch.ones(buf.shape, dtype=torch.bool, device=buf.device)
    r0 = (view.data_ptr() - buf.data_ptr()) // 4 // buf.stride(0)
    c0 = (view.data_ptr() - buf.data_ptr()) // 4 % buf.stride(0)
    mask[r0:r0 + view.shape[0], c0:c0 + view.shape[1]] = False
    return bool((buf.view(torch.int32)[mask] == SENTINEL_BITS).all())


def _sample_rows(m, seed):
    if m <= SAMPLE_ABOVE:
        return torch.arange(m)
    t = -(-m // TC_BM)
    g = torch.Generator().manual_seed(seed)
    rows = [torch.arange(0, 2 * TC_BM), torch.arange((t - 2) * TC_BM, m), torch.randint(0, m, (2048,), generator=g)]
    return torch.unique(torch.cat(rows))


def _block_rel_l2(c, ref, rows):
    """Largest rel-L2 over the 128-row x 32-column blocks of the output grid (only the rows given are compared)."""
    n = c.shape[1]
    pad = -n % 32
    e = torch.nn.functional.pad((c - ref) ** 2, (0, pad)).view(len(rows), -1, 32).sum(-1)
    r = torch.nn.functional.pad(ref ** 2, (0, pad)).view(len(rows), -1, 32).sum(-1)
    _, inv = torch.unique(rows // TC_BM, return_inverse=True)
    eb = torch.zeros(int(inv.max()) + 1, e.shape[1], dtype=torch.float64).index_add_(0, inv, e)
    rb = torch.zeros_like(eb).index_add_(0, inv, r)
    return float((eb.sqrt() / rb.sqrt().clamp_min(1e-300)).max())


def _check(family, got, ref, absprod, gamma, c0, rows, what):
    """Element-wise bound and block rel-L2 of got (fp32, CPU) against the fp64 ref on the sampled rows."""
    got = got.double()
    bound = gamma * absprod + (2.0 ** -23 * ref.abs() if c0 is not None else 0.0)
    err = (got - ref).abs()
    assert bool((err <= bound).all()), (what, float((err / bound).max()))
    ratio = float((err / bound.clamp_min(1e-300)).max())
    blk = _block_rel_l2(got if c0 is None else got - c0, ref if c0 is None else ref - c0, rows)
    w = _WORST.get(family, (0.0, 0.0))
    _WORST[family] = (max(w[0], ratio), max(w[1], blk))
    assert blk <= BLOCK_TOL[family], (what, blk)


def _inputs(rows, cols, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(rows, cols, generator=g)


def _call_nn(path, a, b, c, acc):
    from recon_b200 import _lib
    from recon_b200.functional import gemm_nn
    if path != "direct":
        gemm_nn(a, b, out=c, accumulate=acc)
        return
    lib = _lib.load()
    m, k = a.shape
    n = b.shape[1]
    ws = torch.empty(lib.spk_gemm_tc_workspace_floats(n, k), device=_dev())
    _lib.check(lib.spk_gemm_nn_tc_act(_lib.ptr(a), a.stride(0), _lib.ptr(b), b.stride(0), _lib.ptr(c), c.stride(0), m, n,
                                      k, int(acc), 0, _lib.ptr(ws), _lib.stream_ptr()), "gemm_nn_tc_act")


def _nn_family(pl):
    return "nn-" + pl["kernel"]


def _nn_id(case):
    return "-".join(map(str, case))


@pytest.mark.gpu
@pytest.mark.parametrize("case", NN_CASES, ids=_nn_id)
def test_gemm_nn_vs_fp64(case, gemm_path):
    path, m, k, n = case
    gemm_path(path)
    a0, b0 = _inputs(m, k, m + k), _inputs(k, n, n)
    rows = _sample_rows(m, m)
    a64, b64 = a0[rows].double(), b0.double()
    p64, abs64 = a64 @ b64, a64.abs() @ b64.abs()
    for li, lay in enumerate(nn_layouts(path)):
        name, ka, kb, kc, acc = lay
        pl = nn_kernel(path, m, k, n, lay)
        a, b = _operand(a0, ka), _operand(b0, kb)
        c0 = _inputs(m, n, li) if acc else torch.zeros(m, n)
        buf, c = _out(c0, kc)
        _call_nn(path, a, b, c, acc)
        torch.cuda.synchronize()
        what = (name, pl)
        assert _untouched(buf, c), what
        assert bool(torch.isfinite(c).all()), what
        if pl["kernel"] == "simt":
            gamma = (k + 1) * 2.0 ** -24
        else:
            gamma = 3 * 2.0 ** -20 + (3 * math.ceil(k / 8) + 2) * 2.0 ** -23
        c0r = c0[rows].double() if acc else None
        _check(_nn_family(pl), c[rows.to(_dev())].cpu(), p64 + (c0r if acc else 0), abs64, gamma, c0r, rows, what)
        if li == 0:
            buf2, c2 = _out(c0, kc)
            _call_nn(path, a, b, c2, acc)
            assert torch.equal(buf2.view(torch.int32), buf.view(torch.int32)), what
        del a, b, buf, c


@pytest.mark.gpu
@pytest.mark.parametrize("case", NN_CASES, ids=_nn_id)
def test_gemm_nn_nan_reaches_only_its_rows_and_columns(case, gemm_path):
    path, m, k, n = case
    gemm_path(path)
    lay = NN_LAYOUTS[0] if path != "simt" else SIMT_LAYOUT
    pl = nn_kernel(path, m, k, n, lay)
    a0, b0 = _inputs(m, k, m + k + 1), _inputs(k, n, n + 1)
    t = -(-m // TC_BM)
    bad_rows = {0, min(m - 1, TC_BM - 1), (t - 1) * TC_BM, m - 1, min(m - 1, 32 * (m // 64))}
    if m > SIMT_BAND:
        bad_rows |= {SIMT_BAND - 1, SIMT_BAND}
    for i, r in enumerate(sorted(bad_rows)):
        a0[r, (0, k - 1, k // 2)[i % 3]] = float("nan")
    bn = pl.get("BN", 128)                              # SIMT: 128-column tiles
    bad_cols = {c for t0 in range(0, n, bn) for c in (t0, min(n, t0 + bn) - 1)}
    for i, col in enumerate(sorted(bad_cols)):
        b0[(0, k - 1)[i % 2], col] = float("nan")
    a, b = _operand(a0, lay[1]), _operand(b0, lay[2])
    buf, c = _out(torch.zeros(m, n), lay[3])
    _call_nn(path, a, b, c, lay[4])
    torch.cuda.synchronize()
    want = torch.zeros(m, n, dtype=torch.bool, device=_dev())
    want[sorted(bad_rows)] = True
    want[:, sorted(bad_cols)] = True
    assert torch.equal(torch.isnan(c), want), (lay[0], pl)
    assert _untouched(buf, c), (lay[0], pl)


def _call_tn(a, b, c, acc):
    from recon_b200.functional import gemm_tn
    gemm_tn(a, b, out=c, accumulate=acc)


@pytest.mark.gpu
@pytest.mark.parametrize("case", TN_CASES, ids=_nn_id)
def test_gemm_tn_vs_fp64(case, gemm_path):
    path, m, ka, nb = case
    gemm_path(path)
    a0, b0 = _inputs(m, ka, m + ka), _inputs(m, nb, nb)
    a64, b64 = a0.double(), b0.double()
    p64, abs64 = a64.t() @ b64, a64.abs().t() @ b64.abs()
    del a64, b64
    rows = torch.arange(ka)
    for li, lay in enumerate(tn_layouts(path)):
        name, kA, kB, kc, acc = lay
        pl = tn_kernel(path, m, ka, nb, lay)
        a, b = _operand(a0, kA), _operand(b0, kB)
        c0 = _inputs(ka, nb, li) if acc else torch.zeros(ka, nb)
        buf, c = _out(c0, kc)
        _call_tn(a, b, c, acc)
        torch.cuda.synchronize()
        what = (name, pl)
        assert _untouched(buf, c), what
        assert bool(torch.isfinite(c).all()), what
        if pl["kernel"] == "simt":
            gamma = (m + pl["splits"] + 1) * 2.0 ** -24
        else:
            gamma = 3 * 2.0 ** -20 + (3 * math.ceil(m / 8) + pl["splits"] + 2) * 2.0 ** -23
        c0r = c0.double() if acc else None
        _check("tn-" + pl["kernel"], c.cpu(), p64 + (c0r if acc else 0), abs64, gamma, c0r, rows, what)
        if li == 0:
            buf2, c2 = _out(c0, kc)
            _call_tn(a, b, c2, acc)
            assert torch.equal(buf2.view(torch.int32), buf.view(torch.int32)), what


@pytest.mark.gpu
@pytest.mark.parametrize("case", TN_CASES, ids=_nn_id)
def test_gemm_tn_nan_reaches_only_its_rows_and_columns(case, gemm_path):
    path, m, ka, nb = case
    gemm_path(path)
    lay = TN_LAYOUTS[0] if path != "simt" else SIMT_LAYOUT
    pl = tn_kernel(path, m, ka, nb, lay)
    a0, b0 = _inputs(m, ka, m + ka + 1), _inputs(m, nb, nb + 1)
    mps = pl.get("m_per_split", 32)
    at_rows = [0, m - 1, min(m - 1, mps), min(m - 1, mps - 1), min(m - 1, 32 * (m // 64))]
    tk, tb = (128, pl["BN"]) if pl["kernel"] == "tc" else (64, 64)
    bad_rows = sorted({x for t0 in range(0, ka, tk) for x in (t0, min(ka, t0 + tk) - 1)})
    bad_cols = sorted({x for t0 in range(0, nb, tb) for x in (t0, min(nb, t0 + tb) - 1)})
    for i, j in enumerate(bad_rows):
        a0[at_rows[i % len(at_rows)], j] = float("nan")
    for i, j in enumerate(bad_cols):
        b0[at_rows[(i + 2) % len(at_rows)], j] = float("nan")
    a, b = _operand(a0, lay[1]), _operand(b0, lay[2])
    buf, c = _out(torch.zeros(ka, nb), lay[3])
    _call_tn(a, b, c, lay[4])
    torch.cuda.synchronize()
    want = torch.zeros(ka, nb, dtype=torch.bool, device=_dev())
    want[bad_rows] = True
    want[:, bad_cols] = True
    assert torch.equal(torch.isnan(c), want), (lay[0], pl)
    assert _untouched(buf, c), (lay[0], pl)

"""Filtered link-prediction evaluation of the GAT_sep_space variant (entity_ranks / rank_entities with a model_gat that
holds W_ent2rel): candidates are tanh(e . W_ent2rel[r]) per test row's relation r. CPU tests pin the oracle's sep-space
loop (tests/linkpred_sep_oracle.py, through oracle.convkb.conv_only_forward_sep) against its vectorised fp64 form; -m gpu
tests pin the CUDA path, the count kernel's pair-tile heights and the tanh epilogue of gemm_nn."""
import types

import numpy as np
import pytest
import torch

import linkpred_sep_oracle as S
from test_linkpred import _golden_case, _mid_case, _model, _p32, _random_case


def _w_ent2rel(n_rel, d, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n_rel, d, d, generator=g) / d ** 0.5        # e . W_r ~ N(0, 1) for N(0, 1) rows: tanh not saturated


def _gat(w):
    return types.SimpleNamespace(W_ent2rel=w.float().cuda())


# ---- oracle (CPU) --------------------------------------------------------------------------------------
@pytest.mark.parametrize("d,seed", [(12, 0), (40, 1), (12, 2)])
def test_sep_loop_matches_vectorised(d, seed):
    n, n_rel = 40, 3
    p, test, known = _random_case(n, d, n_rel, 150, 16, seed)
    w = _w_ent2rel(n_rel, d, seed).double()
    ue = list(range(0, n, 3)) + list(range(1, n, 3))
    for u in (None, ue):
        rh, rt, _ = S.validation_pred_loop(p, test.numpy(), known.numpy(), n, w, u)
        fh, ft, nh, nt = S.filtered_ranks(p, test, known, n, w, u)
        assert ((torch.as_tensor(rh) - fh).abs() <= nh).all() and ((torch.as_tensor(rt) - ft).abs() <= nt).all()
        assert (fh > 0).sum() > 0


def test_sep_single_relation_reduces_to_gat_oracle():
    """Every test row with relation r: the literal sep-space loop (conv_only_forward_sep) ranks like the literal GAT loop
    (conv_only_forward) on entity table tanh(E W_r), up to near ties (bmm per row against one mm: different roundings)."""
    from oracle import linkpred as O
    n, d, n_rel, r0 = 50, 12, 4, 2
    p, test, known = _random_case(n, d, n_rel, 200, 20, 3)
    test[:, 1] = r0
    w = _w_ent2rel(n_rel, d, 3).double()
    q = dict(p, final_entity_embeddings=torch.tanh(torch.as_tensor(p["final_entity_embeddings"]).double() @ w[r0]))
    sh, st, sm = S.validation_pred_loop(p, test.numpy(), known.numpy(), n, w)
    gh, gt_, gm = O.validation_pred_loop(q, test.numpy(), known.numpy(), n)
    _, _, nh, nt = O.filtered_ranks(q, test, known, n)
    assert ((torch.as_tensor(sh) - torch.as_tensor(gh)).abs() <= nh).all()
    assert ((torch.as_tensor(st) - torch.as_tensor(gt_)).abs() <= nt).all()
    assert sm["n_evaluated"] == gm["n_evaluated"] == len(test) and (sh > 1).any()


# ---- CUDA path -----------------------------------------------------------------------------------------
def _dev():
    return torch.device("cuda:0")


@pytest.mark.gpu
@pytest.mark.parametrize("skip", [False, True])
def test_sep_golden_matches_reference_loop(skip):
    """convkb_sep with its W_ent2rel (N = 120, D = 40, 7 relations, 25 test rows), triples + test triples as the known
    set: ranks equal the literal loop's and the metrics are bit-equal. No kept candidate lies within 2e-7 (relative to
    max(1, |s|)) of a true score (the closest is 3.9e-7 away in fp64), well above the fp32 rounding of these scores."""
    from helpers import load_golden
    from recon_b200 import rank_entities
    p, test, known = _golden_case("convkb_sep")
    w = torch.as_tensor(load_golden("convkb_sep")["W_ent2rel"])
    n = p["final_entity_embeddings"].shape[0]
    ue = np.setdiff1d(np.arange(n), [test[0, 0], test[1, 2]]) if skip else None
    p64, w64 = _p32(p), w.float().double()
    rh, rt, m = rank_entities(_model(p), test, known, ue, model_gat=_gat(w))
    lh, lt, lm = S.validation_pred_loop(p64, test, known, n, w64, ue)
    _, _, nh, nt = S.filtered_ranks(p64, test, known, n, w64, ue, tau_rel=2e-7)
    assert int(nh.sum()) == 0 and int(nt.sum()) == 0
    assert rh.tolist() == lh.tolist() and rt.tolist() == lt.tolist()
    assert m == lm
    if skip:
        assert m["n_evaluated"] < len(test) and rh[0] == 0 and rt[1] == 0


@pytest.mark.gpu
def test_sep_single_relation_equals_gat_path():
    """All rows on relation r: the sep path's ranks are, bit for bit, the GAT path's ranks of a model whose entity table
    is gemm_nn(E, W_r, act=2) (the same P_r, so the same candidate table and the same fp32 chains)."""
    from recon_b200 import entity_ranks
    from recon_b200.functional import gemm_nn
    n, d, n_rel, r0 = 3000, 40, 6, 4
    p, test, known = _mid_case(n, d, n_rel, 12_000, 70, 300, seed=11)
    test[:, 1] = r0
    known = torch.cat((known, test), 0)
    w = _w_ent2rel(n_rel, d, 11)
    sep = entity_ranks(_model(p), test, known, model_gat=_gat(w))
    model = _model(p)
    with torch.no_grad():
        proj = gemm_nn(model.final_entity_embeddings.detach().contiguous(), w[r0].cuda(), act=2)
    model.final_entity_embeddings = torch.nn.Parameter(proj.contiguous())
    gat = entity_ranks(model, test, known)
    assert torch.equal(sep[0], gat[0]) and torch.equal(sep[1], gat[1])
    assert (sep[0] > 1).any() and (sep[1] > 1).any()


def _tile_case(seed):
    """One relation with 300 rows (a full 128-row tile plus a partial one), one with 40, ten with 1-3 rows."""
    n, d, n_rel = 4000, 40, 14
    p, _, known = _mid_case(n, d, n_rel, 20_000, 1, 0, seed=seed)
    g = torch.Generator().manual_seed(seed)
    sizes = [300, 40] + [int(x) for x in torch.randint(1, 4, (10,), generator=g)]
    rel = torch.cat([torch.full((s,), r, dtype=torch.int64) for r, s in enumerate(sizes)])
    t_n = rel.numel()
    test = torch.stack((torch.randint(0, n, (t_n,), generator=g), rel, torch.randint(0, n, (t_n,), generator=g)), 1)
    test = test[torch.randperm(t_n, generator=g)]
    known = torch.cat((known, test[: t_n // 2]), 0)
    return p, test, known, _w_ent2rel(n_rel, d, seed)


@pytest.mark.gpu
@pytest.mark.parametrize("sep", [False, True])
def test_tile_height_invariance(sep):
    """The same ranks, bit for bit, from one call, from per-row calls and from calls on slices of 17, 40, 80, 81, 128 and
    200 rows: each call size picks its own pair-tile height (16 rows up to 80 pairs, else 128), and the counts are
    exact."""
    from recon_b200 import KnownTriples, entity_ranks
    p, test, known, w = _tile_case(13)
    model = _model(p)
    kt = KnownTriples(known, p["final_entity_embeddings"].shape[0], w.shape[0])
    gat = _gat(w) if sep else None
    full = entity_ranks(model, test, kt, model_gat=gat)
    assert (full[0] > 1).any() and (full[1] > 1).any()
    for step in (1, 17, 40, 80, 81, 128, 200):
        parts = [entity_ranks(model, test[i:i + step], kt, model_gat=gat) for i in range(0, test.shape[0], step)]
        assert torch.equal(torch.cat([a for a, _ in parts]), full[0]), step
        assert torch.equal(torch.cat([b for _, b in parts]), full[1]), step


def _check_sep_against_vectorised(p, test, known, w, ue=None):
    from recon_b200 import entity_ranks
    n = p["final_entity_embeddings"].shape[0]
    rh, rt = entity_ranks(_model(p), test, known, ue, model_gat=_gat(w))
    fh, ft, nh, nt = S.filtered_ranks(_p32(p), test, known, n, w.float().double(), ue, device=_dev())
    assert ((rh - fh).abs() <= nh).all(), (rh - fh).abs().max()
    assert ((rt - ft).abs() <= nt).all(), (rt - ft).abs().max()
    return rh, rt, fh, ft


@pytest.mark.gpu
def test_sep_mid_size_with_hub():
    """N = 50k + 37, D = 200, 50 relations, ~500k known triples with a 20k-head (., r0, t0) hub."""
    p, test, known = _mid_case(50_000 + 37, 200, 50, 480_000, 256, 20_000, seed=15)
    rh, rt, fh, ft = _check_sep_against_vectorised(p, test, known, _w_ent2rel(50, 200, 15))
    assert (rh > 0).all() and (rt > 0).all()
    assert (rh == fh).float().mean() > 0.9 and (rt == ft).float().mean() > 0.9


@pytest.mark.gpu
def test_sep_scale_2m_entities():
    """N = 2M, D = 200, 3 relations: the per-relation [N, D] projection and [N, 2D] table pass 2^31 bytes."""
    p, test, known = _mid_case(2_000_000, 200, 3, 2_000_000, 40, 0, seed=16)
    _check_sep_against_vectorised(p, test, known, _w_ent2rel(3, 200, 16))


@pytest.mark.gpu
def test_sep_matches_batch_test_scores():
    """Ranks read off model_conv.batch_test(every candidate triple, model_gat), the product's own sep-space scorer,
    with the known candidates masked, agree within near ties (the two sum in different orders)."""
    from recon_b200 import entity_ranks
    n, d, n_rel = 3000, 40, 5
    p, test, known = _mid_case(n, d, n_rel, 15_000, 12, 200, seed=17)
    w = _w_ent2rel(n_rel, d, 17)
    model, gat = _model(p), _gat(w)
    rh, rt = entity_ranks(model, test, known, model_gat=gat)
    known_set = set(map(tuple, known.tolist()))
    cand = torch.arange(n)
    for side, ranks in ((0, rh), (1, rt)):
        batch = test.repeat_interleave(n, 0)
        batch[:, 0 if side == 0 else 2] = cand.repeat(test.shape[0])
        with torch.no_grad():
            s = model.batch_test(batch.cuda(), gat).view(test.shape[0], n).double().cpu()
        for i, (h, r, t) in enumerate(test.tolist()):
            true = h if side == 0 else t
            mask = torch.tensor([c != true and ((c, r, t) if side == 0 else (h, r, c)) not in known_set
                                 for c in range(n)])
            st = s[i, true]
            want = int(((s[i] > st) & mask).sum()) + 1
            near = int((((s[i] - st).abs() <= 1e-5 * max(1.0, abs(float(st)))) & mask).sum())
            assert abs(int(ranks[i]) - want) <= near, (side, i, int(ranks[i]), want, near)


@pytest.mark.gpu
def test_sep_errors_and_edges():
    from recon_b200 import KnownTriples, entity_ranks, rank_entities
    n, d, n_rel = 2000, 40, 7
    p, test, known = _mid_case(n, d, n_rel, 8000, 60, 200, seed=18)
    model = _model(p)
    kt = KnownTriples(known, n, n_rel)
    w = _w_ent2rel(n_rel, d, 18)
    a = entity_ranks(model, test, kt, model_gat=_gat(w))
    b = entity_ranks(model, test, kt, model_gat=_gat(w))
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    e = entity_ranks(model, torch.zeros(0, 3, dtype=torch.int64), kt, model_gat=_gat(w))
    assert e[0].shape == (0,) and e[1].shape == (0,)
    with pytest.raises(ZeroDivisionError):
        rank_entities(model, torch.zeros(0, 3, dtype=torch.int64), kt, model_gat=_gat(w))
    # every row skipped: zero ranks, no relation pass
    z = entity_ranks(model, test, kt, unique_entities=[], model_gat=_gat(w))
    assert not z[0].any() and not z[1].any()
    for bad_w in (w[:, :, :d - 1], w[:n_rel - 1], w.double()):
        with pytest.raises(ValueError):
            entity_ranks(model, test, kt, model_gat=_gat(bad_w) if bad_w.dtype == torch.float32 else
                         types.SimpleNamespace(W_ent2rel=bad_w.cuda()))
    with pytest.raises(ValueError):
        entity_ranks(model, test, kt, model_gat=types.SimpleNamespace(W_ent2rel=w))          # on the host
    for bad in ([[0, 0, n]], [[-1, 0, 1]], [[0, n_rel, 1]], [[0, -1, 1]]):
        with pytest.raises(IndexError):
            entity_ranks(model, torch.tensor(bad), kt, model_gat=_gat(w))
    with pytest.raises(NotImplementedError, match="GAT_sep_space"):
        entity_ranks(model, test, kt, model_gat=types.SimpleNamespace())


# ---- gemm_nn(act=2): the tanh epilogue -----------------------------------------------------------------
@pytest.fixture(params=["tc", "simt", "tc-pair", "tc-cluster"])
def gemm_path(request, monkeypatch):
    """The tcgen05 3xTF32 GEMM, the exact-fp32 SIMT GEMM, and the two opt-in NN variants (pair-CTA cta_group::2 kernel,
    2-CTA clusters; both off by default, see spk_gemm_tc.cu)."""
    from recon_b200 import functional as SF
    old = SF.USE_TC
    SF.USE_TC = request.param != "simt"
    if request.param == "tc-pair":
        monkeypatch.setenv("SPK_TC_PAIR", "1")
    if request.param == "tc-cluster":
        monkeypatch.setenv("SPK_TC_CLUSTER", "2")
    yield request.param
    SF.USE_TC = old


def _bits(x):
    return x.contiguous().view(torch.int32).cpu()


def _tanh_inplace(x):
    from recon_b200 import _lib
    _lib.check(_lib.load().spk_tanh_fwd(_lib.ptr(x), x.stride(0), x.shape[0], x.shape[1], _lib.stream_ptr()), "tanh_fwd")


@pytest.mark.gpu
@pytest.mark.parametrize("m,k,n", [(1000, 200, 200), (5000, 40, 37), (40_000, 200, 200), (37_991, 64, 96)])
def test_gemm_nn_tanh_epilogue_bit_equal(m, k, n, gemm_path):
    """gemm_nn(act=2) is bit-equal to gemm_nn followed by spk_tanh_fwd: through the TMA-store epilogue (aligned C), the
    per-thread-row epilogue (unaligned C, with and without accumulate; aligned C with accumulate), the SIMT fallback,
    and, at M >= 2 x 148 x 128, the pair-CTA and 2-CTA-cluster kernels. Inputs include huge products, +-inf and NaN."""
    from recon_b200.functional import gemm_nn
    g = torch.Generator().manual_seed(m + k + n)
    a = torch.randn(m, k, generator=g) * 3
    b = torch.randn(k, n, generator=g)
    a[0, :] = 3e38                                   # products overflow to +-inf
    a[1, 0], a[2, 1], a[3, 2] = float("inf"), float("-inf"), float("nan")
    a[4, :] = 1e-30
    a, b = a.cuda(), b.cuda()
    layouts = [("aligned", (n + 3) // 4 * 4), ("unaligned", n + 1 if (n + 1) % 4 else n + 2)]
    for name, ld in layouts:
        for acc in ((False, True) if gemm_path in ("tc", "simt") else (False,)):
            c0 = torch.randn(m, ld, generator=g).cuda()
            ref = c0.clone()[:, :n]
            got = c0.clone()[:, :n]
            gemm_nn(a, b, out=ref, accumulate=acc)
            _tanh_inplace(ref)
            gemm_nn(a, b, out=got, accumulate=acc, act=2)
            assert torch.equal(_bits(got), _bits(ref)), (name, acc)
    assert torch.isnan(got).any() and (got.abs() == 1).any()


@pytest.mark.gpu
def test_gemm_nn_tc_act_rejects_unknown_activation():
    from recon_b200 import _lib
    a, b = torch.randn(256, 8, device=_dev()), torch.randn(8, 16, device=_dev())
    out, ws = torch.empty(256, 16, device=_dev()), torch.empty(4096, device=_dev())
    lib = _lib.load()
    for act in (-1, 3):
        assert lib.spk_gemm_nn_tc_act(_lib.ptr(a), 8, _lib.ptr(b), 16, _lib.ptr(out), 16, 256, 16, 8, 0, act,
                                      _lib.ptr(ws), _lib.stream_ptr()) != 0

"""Filtered link-prediction evaluation (Corpus.get_validation_pred, GAT/create_batch.py:905-1199): entity_ranks /
rank_entities against the oracle's literal restatement of the reference loop (oracle/linkpred.py). CPU tests pin the
oracle on a hand-checked toy and against its vectorised fp64 form; -m gpu tests pin the CUDA path."""
import types

import numpy as np
import pytest
import torch

from helpers import load_golden

KEYS = ["convKB.fc1.weight", "convKB.fc1.bias", "convKB.fc2.weight", "convKB.fc2.bias"]


def _toy():
    """N = 6, D = 2, R = 2. fc1 picks e_h[0] and e_t[1], fc2 adds them: score(h, r, t) = lrelu(E[h,0]) + lrelu(E[t,1]).
    Entity 5 is NaN, so every triple that contains it scores NaN."""
    nan = float("nan")
    ent = torch.tensor([[0.5, 0.2], [0.3, 0.6], [0.8, 0.9], [0.5, 0.4], [0.1, 0.6], [nan, 0.1]], dtype=torch.float64)
    w1 = torch.zeros(2, 6, dtype=torch.float64)
    w1[0, 0] = 1.0                      # out0 = e_h[0]
    w1[1, 5] = 1.0                      # out1 = e_t[1]
    p = {"final_entity_embeddings": ent, "final_relation_embeddings": torch.zeros(2, 2, dtype=torch.float64),
         "convKB.fc1.weight": w1, "convKB.fc1.bias": torch.zeros(2, dtype=torch.float64),
         "convKB.fc2.weight": torch.ones(1, 2, dtype=torch.float64), "convKB.fc2.bias": torch.zeros(1, dtype=torch.float64)}
    test = np.array([[0, 0, 1], [3, 1, 5], [4, 1, 0]])
    known = np.array([[2, 0, 1], [2, 0, 1], [0, 0, 1], [0, 0, 2], [0, 0, 3], [0, 0, 5], [1, 1, 0], [4, 1, 2]])
    return p, test, known, [0, 1, 2, 3, 4]


# row 0 (0,0,1): head side: 2 outscores but is known, 3 ties (not counted), 5 is NaN (counted) -> 2; tail side: 2, 3, 5
#   are known, 4 ties -> 1.  row 1 (3,1,5): skipped without 5 in unique_entities; else its true score is NaN -> 1, 1.
#   row 2 (4,1,0): head side 0, 2, 3, 5 outscore it, 1 is known -> 5; tail side 1, 3, 4, 5 do, 2 is known -> 5.
TOY_HEAD, TOY_TAIL = [2, 0, 5], [1, 0, 5]
TOY_HEAD_ALL, TOY_TAIL_ALL = [2, 1, 5], [1, 1, 5]


def test_toy_hand_checked():
    from oracle import linkpred as O
    p, test, known, ue = _toy()
    rh, rt, m = O.validation_pred_loop(p, test, known, 6, ue)
    assert rh.tolist() == TOY_HEAD and rt.tolist() == TOY_TAIL
    fh, ft, nh, nt = O.filtered_ranks(p, test, known, 6, ue)
    assert fh.tolist() == TOY_HEAD and ft.tolist() == TOY_TAIL
    assert nh.tolist() == [1, 0, 0] and nt.tolist() == [1, 0, 0]           # the exact ties
    assert m["n_evaluated"] == 2
    exp_head = {"hits_at_100": 1.0, "hits_at_10": 1.0, "hits_at_3": 0.5, "hits_at_1": 0.0, "mean_rank": 3.5,
                "mean_recip_rank": (1 / 2 + 1 / 5) / 2}
    exp_tail = {"hits_at_100": 1.0, "hits_at_10": 1.0, "hits_at_3": 0.5, "hits_at_1": 0.5, "mean_rank": 3.0,
                "mean_recip_rank": (1 / 1 + 1 / 5) / 2}
    assert m["head"] == pytest.approx(exp_head) and m["tail"] == pytest.approx(exp_tail)
    assert m["cumulative"] == pytest.approx({k: (exp_head[k] + exp_tail[k]) / 2 for k in exp_head})
    rh, rt, m = O.validation_pred_loop(p, test, known, 6)
    assert rh.tolist() == TOY_HEAD_ALL and rt.tolist() == TOY_TAIL_ALL and m["n_evaluated"] == 3
    fh, ft, _, _ = O.filtered_ranks(p, test, known, 6)
    assert fh.tolist() == TOY_HEAD_ALL and ft.tolist() == TOY_TAIL_ALL


def _random_case(n, d, n_rel, m, t_n, seed):
    from recon_b200.synth import make_triples
    g = torch.Generator().manual_seed(seed)
    fc1 = torch.nn.Linear(3 * d, d).double()
    fc2 = torch.nn.Linear(d, 1).double()
    with torch.no_grad():
        for lin in (fc1, fc2):
            lin.weight.copy_(torch.rand(lin.weight.shape, generator=g, dtype=torch.float64) * 2 - 1)
            lin.bias.copy_(torch.rand(lin.bias.shape, generator=g, dtype=torch.float64) * 2 - 1)
    p = {"final_entity_embeddings": torch.randn(n, d, generator=g, dtype=torch.float64),
         "final_relation_embeddings": torch.randn(n_rel, d, generator=g, dtype=torch.float64),
         "convKB.fc1.weight": fc1.weight.detach() / (3 * d) ** 0.5, "convKB.fc1.bias": fc1.bias.detach(),
         "convKB.fc2.weight": fc2.weight.detach() / d ** 0.5, "convKB.fc2.bias": fc2.bias.detach()}
    known = make_triples(n, m, n_rel, seed=seed)                            # with parallel edges and self loops
    pick = torch.randint(0, m, (t_n,), generator=g)
    test = known[pick].clone()
    test[: t_n // 4] = torch.stack((torch.randint(0, n, (t_n // 4,), generator=g),
                                    torch.randint(0, n_rel, (t_n // 4,), generator=g),
                                    torch.randint(0, n, (t_n // 4,), generator=g)), 1)    # some rows outside the known set
    return p, test, known


@pytest.mark.parametrize("d,seed", [(12, 0), (40, 1), (12, 2)])
def test_loop_matches_vectorised(d, seed):
    from oracle import linkpred as O
    n, n_rel = 40, 3
    p, test, known = _random_case(n, d, n_rel, 150, 16, seed)
    ue = list(range(0, n, 3)) + list(range(1, n, 3))
    for u in (None, ue):
        rh, rt, _ = O.validation_pred_loop(p, test.numpy(), known.numpy(), n, u)
        fh, ft, nh, nt = O.filtered_ranks(p, test, known, n, u)
        assert ((torch.as_tensor(rh) - fh).abs() <= nh).all() and ((torch.as_tensor(rt) - ft).abs() <= nt).all()
        assert (fh > 0).sum() > 0


def test_no_row_evaluated_raises():
    from oracle import linkpred as O
    from recon_b200.linkpred import ranking_metrics
    p, test, known, _ = _toy()
    with pytest.raises(ZeroDivisionError):
        O.validation_pred_loop(p, test, known, 6, unique_entities=[5])
    with pytest.raises(ZeroDivisionError):
        ranking_metrics([])


def test_metrics_match_oracle_bitwise():
    from oracle import linkpred as O
    from recon_b200.linkpred import ranking_metrics
    g = torch.Generator().manual_seed(3)
    ranks = (torch.randint(1, 300, (997,), generator=g)).tolist()
    assert ranking_metrics(ranks) == O.metrics(ranks)


def test_cpu_model_and_sep_space_rejected():
    from recon_b200 import SpKBGATConvOnly, entity_ranks
    m = SpKBGATConvOnly(torch.zeros(6, 10), torch.zeros(2, 10), [2, 4], [2, 4], 0.0, 0.0, 0.2, 0.2, [2, 2], 50)
    with pytest.raises(RuntimeError):
        entity_ranks(m, torch.tensor([[0, 0, 1]]), torch.tensor([[0, 0, 1]]))
    with pytest.raises(NotImplementedError, match="GAT_sep_space"):
        entity_ranks(m, torch.tensor([[0, 0, 1]]), torch.tensor([[0, 0, 1]]), model_gat=types.SimpleNamespace())


# ---- CUDA path ---------------------------------------------------------------------------------------
def _dev():
    return torch.device("cuda:0")


def _model(p):
    """SpKBGATConvOnly on the GPU holding the given fp32 parameters (the unused conv parameters stay default)."""
    from recon_b200 import SpKBGATConvOnly
    d = p["final_entity_embeddings"].shape[1]
    m = SpKBGATConvOnly(torch.zeros(1, 4), torch.zeros(1, 4), [d, d], [d, d], 0.0, 0.0, 0.2, 0.2, [1, 1], 1).to(_dev())
    m.final_entity_embeddings = torch.nn.Parameter(torch.as_tensor(p["final_entity_embeddings"]).float().to(_dev()))
    m.final_relation_embeddings = torch.nn.Parameter(torch.as_tensor(p["final_relation_embeddings"]).float().to(_dev()))
    for k in KEYS:
        mod = m.convKB.fc1 if "fc1" in k else m.convKB.fc2
        setattr(mod, k.split(".")[-1], torch.nn.Parameter(torch.as_tensor(p[k]).float().to(_dev())))
    return m


def _p32(p):
    """The parameters the GPU model holds, as fp64 (the oracle scores what the model scores)."""
    return {k: torch.as_tensor(v).float().double() for k, v in p.items()}


@pytest.mark.gpu
def test_toy_on_gpu():
    from recon_b200 import rank_entities
    from oracle import linkpred as O
    p, test, known, ue = _toy()
    rh, rt, m = rank_entities(_model(p), test, known, ue)
    assert rh.dtype == torch.int64 and rh.tolist() == TOY_HEAD and rt.tolist() == TOY_TAIL
    assert m == O.validation_pred_loop(_p32(p), test, known, 6, ue)[2]
    rh, rt, _ = rank_entities(_model(p), test, known)
    assert rh.tolist() == TOY_HEAD_ALL and rt.tolist() == TOY_TAIL_ALL


def _golden_case(name):
    g = load_golden(name)
    p = {k[len("param."):]: torch.as_tensor(v) for k, v in g.items() if k.startswith("param.")}
    test = g["test_triples"]
    known = np.concatenate((g["triples"], test), 0)
    return p, test, known


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["convkb_small", "convkb_gat", "convkb_sep"])
@pytest.mark.parametrize("skip", [False, True])
def test_golden_params_match_reference_loop(name, skip):
    """The fixture parameters (convkb_sep without its W_ent2rel), their test triples, triples + test triples as the known
    set: ranks equal the literal reference loop's and the metrics are bit-equal. convkb_gat / convkb_sep do hold
    candidates within 1e-5 of a true score (the closest 8.5e-7 apart at |s| ~ 0.08), but none within 2e-7, well above
    the fp32 rounding of these scores, so the comparison is exact."""
    from recon_b200 import rank_entities
    from oracle import linkpred as O
    p, test, known = _golden_case(name)
    n = p["final_entity_embeddings"].shape[0]
    ue = np.setdiff1d(np.arange(n), [test[0, 0], test[1, 2]]) if skip else None
    p64 = _p32(p)
    rh, rt, m = rank_entities(_model(p), test, known, ue)
    lh, lt, lm = O.validation_pred_loop(p64, test, known, n, ue)
    _, _, nh, nt = O.filtered_ranks(p64, test, known, n, ue, tau_rel=2e-7)
    assert int(nh.sum()) == 0 and int(nt.sum()) == 0
    assert rh.tolist() == lh.tolist() and rt.tolist() == lt.tolist()
    assert m == lm
    if skip:
        assert m["n_evaluated"] < len(test) and rh[0] == 0 and rt[1] == 0


def _mid_case(n, d, n_rel, m, t_n, hub, seed):
    g = torch.Generator().manual_seed(seed)
    p = {"final_entity_embeddings": torch.randn(n, d, generator=g),
         "final_relation_embeddings": torch.randn(n_rel, d, generator=g),
         "convKB.fc1.weight": (torch.rand(d, 3 * d, generator=g) * 2 - 1) / (3 * d) ** 0.5,
         "convKB.fc1.bias": torch.rand(d, generator=g) * 0.2 - 0.1,
         "convKB.fc2.weight": (torch.rand(1, d, generator=g) * 2 - 1) / d ** 0.5,
         "convKB.fc2.bias": torch.rand(1, generator=g)}
    known = torch.stack((torch.randint(0, n, (m,), generator=g), torch.randint(0, n_rel, (m,), generator=g),
                         torch.randint(0, n, (m,), generator=g)), 1)
    if hub:                                                                 # (., r0, t0) with `hub` distinct heads
        heads = torch.randperm(n, generator=g)[:hub]
        known = torch.cat((known, torch.stack((heads, torch.zeros_like(heads), torch.full_like(heads, 7)), 1)), 0)
    test = known[torch.randint(0, known.shape[0], (t_n,), generator=g)].clone()
    if hub:
        test[: t_n // 4] = known[m + torch.randint(0, hub, (t_n // 4,), generator=g)]     # rows on the hub
    return p, test, known


def _check_against_vectorised(p, test, known, ue=None):
    from recon_b200 import entity_ranks
    from oracle import linkpred as O
    n = p["final_entity_embeddings"].shape[0]
    rh, rt = entity_ranks(_model(p), test, known, ue)
    fh, ft, nh, nt = O.filtered_ranks(_p32(p), test, known, n, ue, device=_dev())
    assert ((rh - fh).abs() <= nh).all(), (rh - fh).abs().max()
    assert ((rt - ft).abs() <= nt).all(), (rt - ft).abs().max()
    return rh, rt, fh, ft


@pytest.mark.gpu
def test_mid_size_with_hub():
    """N = 50k (not a multiple of the 128-row tile), D = 200, ~500k known triples with a 20k-head (., r0, t0) hub."""
    p, test, known = _mid_case(50_000 + 37, 200, 50, 480_000, 256, 20_000, seed=5)
    rh, rt, fh, ft = _check_against_vectorised(p, test, known)
    assert (rh > 0).all() and (rt > 0).all()
    assert (rh == fh).float().mean() > 0.9 and (rt == ft).float().mean() > 0.9


@pytest.mark.gpu
def test_scale_2m_entities():
    """N = 2M, D = 200: the [N, 2D] candidate table is 3.2 GB, row offsets pass 2^31 bytes."""
    p, test, known = _mid_case(2_000_000, 200, 20, 2_000_000, 64, 0, seed=6)
    _check_against_vectorised(p, test, known)


@pytest.mark.gpu
def test_ties_and_nan():
    from recon_b200 import entity_ranks
    from oracle import linkpred as O
    n, d = 1000, 40
    p, test, known = _mid_case(n, d, 5, 3000, 16, 0, seed=7)
    ent = p["final_entity_embeddings"]
    h0, t0 = int(test[0, 0]), int(test[0, 2])
    copies = [c for c in range(n - 8, n) if c not in (h0, t0)][:5]
    ent[copies] = ent[h0].clone()                               # head-side candidates that tie the true head bitwise
    nan_id = n - 20
    ent[nan_id] = float("nan")
    test[1] = torch.tensor([nan_id, 1, 3])                      # NaN true score on both sides
    test[2:4] = test[2:4].clamp(max=nan_id - 1)
    known = known[(known[:, 0] != nan_id) & (known[:, 2] != nan_id)]
    rh, rt = entity_ranks(_model(p), test, known)
    fh, ft, nh, nt = O.filtered_ranks(_p32(p), test, known, n, device=_dev())
    assert rh[1] == 1 and rt[1] == 1
    assert ((rh - fh).abs() <= nh).all() and ((rt - ft).abs() <= nt).all()
    # the copies are exact ties: on row 0 they are the only near ties, so the rank is exact and ignores them
    assert int(nh[0]) >= len(copies)
    if int(nh[0]) == len(copies):
        assert rh[0] == fh[0]
    # the NaN candidate outscores every finite true score: rows 2, 3 rank below it on both sides
    assert (rh[2:4] >= 2).all() and (rt[2:4] >= 2).all()
    assert ((rh[2:] - fh[2:]).abs() <= nh[2:]).all()


@pytest.mark.gpu
def test_unfiltered_count_matches_score_matrix():
    """With no known triples the count equals the one read off the T x N score matrix that spk_rank_scores writes for
    the same pair vectors (except near ties: the two sum in different orders); filtering only lowers ranks."""
    from recon_b200 import _lib, entity_ranks
    from recon_b200.linkpred import _score_tables
    from recon_b200.convkb import LRELU_SLOPE
    p, test, known = _mid_case(20_000, 200, 30, 200_000, 128, 3000, seed=8)
    model = _model(p)
    empty = torch.zeros(0, 3, dtype=torch.int64)
    uh, ut = entity_ranks(model, test, empty)
    rh, rt = entity_ranks(model, test, known)
    assert (rh <= uh).all() and (rt <= ut).all() and (rh < uh).any()
    lib = _lib.load()
    with torch.no_grad():
        ac, bt, b1, w2 = _score_tables(model)
        d = bt.shape[1]
        a, c = ac[:, :d], ac[:, d:2 * d]
        tri = test.to(_dev())
        b2 = model.convKB.fc2.bias.detach().contiguous()
        for side, ranks in ((0, uh), (1, ut)):
            v = ((c[tri[:, 2]] if side == 0 else a[tri[:, 0]]) + bt[tri[:, 1]]) + b1
            x = (a if side == 0 else c).contiguous()
            true = tri[:, 0] if side == 0 else tri[:, 2]
            s = torch.empty(tri.shape[0], x.shape[0], dtype=torch.float32, device=_dev())
            _lib.check(lib.spk_rank_scores(_lib.ptr(v.contiguous()), d, _lib.ptr(x), x.stride(0), _lib.ptr(w2),
                                           _lib.ptr(b2), LRELU_SLOPE, tri.shape[0], x.shape[0], d, _lib.ptr(s),
                                           s.stride(0), _lib.stream_ptr()), "rank_scores")
            st = s.gather(1, true.unsqueeze(1))
            gt = (s > st) | (torch.isnan(s) & ~torch.isnan(st))
            want = gt.sum(1) + 1
            near = ((s - st).abs() <= 1e-5 * st.abs().clamp(min=1.0)).sum(1) - 1     # minus the true entity itself
            assert ((ranks - want.cpu()).abs() <= near.cpu()).all()
            assert (ranks == want.cpu()).float().mean() > 0.9


@pytest.mark.gpu
def test_determinism_and_edges():
    from recon_b200 import KnownTriples, SpKBGATConvOnly, entity_ranks, rank_entities
    p, test, known = _mid_case(5000, 40, 7, 20_000, 100, 500, seed=9)
    model = _model(p)
    kt = KnownTriples(known, 5000, 7)
    a = entity_ranks(model, test, kt)
    b = entity_ranks(model, test, kt)
    c = entity_ranks(model, test, known)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[0], c[0]) and torch.equal(a[1], c[1])
    assert len(kt) == known.shape[0]
    e = entity_ranks(model, torch.zeros(0, 3, dtype=torch.int64), kt)
    assert e[0].shape == (0,) and e[1].shape == (0,)
    with pytest.raises(ZeroDivisionError):
        rank_entities(model, torch.zeros(0, 3, dtype=torch.int64), kt)
    for bad in ([[0, 0, 5000]], [[-1, 0, 1]], [[0, 7, 1]]):
        with pytest.raises(IndexError):
            entity_ranks(model, torch.tensor(bad), kt)
    with pytest.raises(IndexError):
        KnownTriples(torch.tensor([[0, 0, 5000]]), 5000, 7)
    with pytest.raises(NotImplementedError):
        entity_ranks(model, test, kt, model_gat=types.SimpleNamespace(W_ent2rel=None))
    wide = SpKBGATConvOnly(torch.zeros(4, 4), torch.zeros(2, 4), [260, 520], [260, 520], 0.0, 0.0, 0.2, 0.2, [2, 2],
                           1).to(_dev())
    with pytest.raises(RuntimeError, match="width"):
        entity_ranks(wide, torch.tensor([[0, 0, 1]]), torch.tensor([[0, 0, 1]]))

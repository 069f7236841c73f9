"""TransE margin loss of the GAT_sep_space variant (batch_gat_loss(..., model_gat=)) and the grouped relation-space
projection it runs on (convkb.RelationLayout / PaddedRowsFn / GroupedProjectFn, spk_ent2rel_*, spk_gemm_*_tc_grouped).

CPU (`-m "not gpu"`): the fp64 oracle tests/loss_sep_oracle.py against an independent per-row loop and against
oracle.loss.batch_gat_loss on explicitly projected tables; the sep path refuses CPU tensors.
GPU (`-m gpu`): the grouped projection (forward, dX, dW) and the loss against the fp64 oracle, bit-equality of every group
with the plain tanh GEMM, absent relations, determinism, the error behaviour, launch counts independent of the number of
relations, no host synchronisation, and one training iteration of a sep_space model."""
import types

import pytest
import torch

import loss_sep_oracle as S
from helpers import rel_l2

TOL = 1e-4
TIGHT = 2e-5
PROJ_TOL = 1e-5


def _w(n_rel, d, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n_rel, d, d, generator=g) * (scale / d ** 0.5)      # e . W ~ N(0, scale^2): tanh not saturated


def _tables(n_ent, n_rel, d, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n_ent, d, generator=g), torch.randn(n_rel, d, generator=g)


def _tri(n_ent, n_rel, n_pos, ratio, seed, hub_entity=None, hub_rel=None, rel_corrupt=False):
    from oracle import loss as OL
    tri = OL.make_train_indices(n_ent, n_rel, n_pos, ratio, seed, hub_entity=hub_entity,
                                hub_share=0.5 if hub_entity is not None else 0.0)
    g = torch.Generator().manual_seed(seed + 1000)
    if hub_rel is not None:                          # one relation holds most positives (and so their negatives)
        pick = torch.rand(n_pos, generator=g) < 0.6
        tri[:n_pos][pick, 1] = hub_rel
        tri[n_pos:, 1] = tri[:n_pos, 1].repeat(2 * ratio)
    if rel_corrupt:                                  # oracle/sampler.py also corrupts relations
        k = n_pos * 2 * ratio
        pick = torch.rand(k, generator=g) < 0.3
        tri[n_pos:][pick, 1] = torch.randint(0, n_rel, (int(pick.sum()),), generator=g)
    return tri


# ---- CPU: the oracle ----------------------------------------------------------------------------------------------
def _loop_loss(tri, ent, rel, w, ratio, margin):
    """Independent restatement: a Python loop over rows, row @ W[r] one row at a time."""
    t = tri.shape[0]
    n_pos = t // (2 * ratio + 1)

    def norm(h, r, tl):
        x = torch.tanh(ent[h] @ w[r]) + rel[r] - torch.tanh(ent[tl] @ w[r])
        return x.abs().sum()

    pos = [norm(*tri[i].tolist()) for i in range(n_pos)]
    terms = []
    for k in range(t - n_pos):
        neg = norm(*tri[n_pos + k].tolist())
        terms.append(torch.clamp_min(pos[k % n_pos] - neg + margin, 0))
    return torch.stack(terms).mean()


@pytest.mark.parametrize("d,ratio,seed", [(12, 2, 0), (7, 3, 1), (40, 1, 2)])
def test_oracle_matches_per_row_loop(d, ratio, seed):
    n_ent, n_rel, n_pos = 30, 5, 6
    ent, rel = _tables(n_ent, n_rel, d, seed)
    w = _w(n_rel, d, seed)
    tri = _tri(n_ent, n_rel, n_pos, ratio, seed, rel_corrupt=True)
    args = (tri, ent.double(), rel.double(), w.double(), ratio, 1.0)
    got = S.batch_gat_loss_sep(*args)
    want = _loop_loss(*args)
    assert abs(float(got) - float(want)) <= 1e-12 * max(1.0, abs(float(want)))
    assert float(want) > 0


def test_oracle_reduces_to_plain_loss_on_projected_tables():
    from oracle import loss as OL
    n_ent, n_rel, d, n_pos, ratio = 40, 4, 12, 8, 2
    ent, rel = _tables(n_ent, n_rel, d, 3)
    ent, rel, w = ent.double(), rel.double(), _w(n_rel, d, 3).double()
    tri = _tri(n_ent, n_rel, n_pos, ratio, 3, rel_corrupt=True)
    t = tri.shape[0]
    # explicitly projected table: row i = projected head of triple i, row T + i = its projected tail
    proj = torch.cat((torch.tanh(torch.bmm(ent[tri[:, 0]].unsqueeze(1), w[tri[:, 1]]).squeeze(1)),
                      torch.tanh(torch.bmm(ent[tri[:, 2]].unsqueeze(1), w[tri[:, 1]]).squeeze(1))))
    syn = torch.stack((torch.arange(t), tri[:, 1], torch.arange(t) + t), dim=1)
    got = S.batch_gat_loss_sep(tri, ent, rel, w, ratio, 2.0)
    assert abs(float(got) - float(OL.batch_gat_loss(syn, proj, rel, ratio, 2.0))) <= 1e-13
    # one relation for every row: the projected entity table itself
    tri1 = tri.clone(); tri1[:, 1] = 2
    got1 = S.batch_gat_loss_sep(tri1, ent, rel, w, ratio, 2.0)
    assert abs(float(got1) - float(OL.batch_gat_loss(tri1, torch.tanh(ent @ w[2]), rel, ratio, 2.0))) <= 1e-13


def test_sep_path_raises_without_gpu():
    from recon_b200.loss import batch_gat_loss
    ent, rel = _tables(20, 3, 8, 4)
    tri = _tri(20, 3, 4, 2, 4)
    gat = types.SimpleNamespace(W_ent2rel=_w(3, 8, 4))
    with pytest.raises(RuntimeError):
        batch_gat_loss(torch.nn.MarginRankingLoss(margin=1.0), tri, ent, rel, model_gat=gat)


# ---- GPU: the grouped projection ----------------------------------------------------------------------------------
def _dev():
    return torch.device("cuda:0")


# rows per relation: absent relations, 1, 127, 128, 129, several tiles, and a hub with more than half the rows
GROUP_SIZES = [0, 1, 127, 128, 129, 0, 700, 9000]


def _grouped_case(d, seed, sizes=GROUP_SIZES):
    g = torch.Generator().manual_seed(seed)
    rid = torch.cat([torch.full((c,), r, dtype=torch.int64) for r, c in enumerate(sizes)])
    rid = rid[torch.randperm(rid.numel(), generator=g)]
    rows = torch.randn(rid.numel(), d, generator=g)
    gout = torch.randn(rid.numel(), d, generator=g)
    return rows, rid, _w(len(sizes), d, seed), gout


def _project_gpu(rows, rid, w, gout):
    from recon_b200.convkb import ent2rel_project
    x = rows.to(_dev()).requires_grad_(True)
    wd = w.to(_dev()).requires_grad_(True)
    y = ent2rel_project(x, wd, rid.to(_dev()))
    (y * gout.to(_dev())).sum().backward()
    torch.cuda.synchronize()
    return y.detach(), x.grad, wd.grad


def _project_ref(rows, rid, w, gout):
    from oracle.convkb import ent2rel_project
    x = rows.double().requires_grad_(True)
    wd = w.double().requires_grad_(True)
    y = ent2rel_project(x, wd, rid)
    (y * gout.double()).sum().backward()
    return y.detach(), x.grad, wd.grad


@pytest.mark.gpu
@pytest.mark.parametrize("d", [12, 40, 200])
def test_grouped_projection_vs_fp64(d):
    rows, rid, w, gout = _grouped_case(d, d)
    y, dx, dw = _project_gpu(rows, rid, w, gout)
    ry, rdx, rdw = _project_ref(rows, rid, w, gout)
    assert rel_l2(y, ry) <= PROJ_TOL
    assert rel_l2(dx, rdx) <= PROJ_TOL
    for r, c in enumerate(GROUP_SIZES):
        if c:
            assert rel_l2(dw[r], rdw[r]) <= PROJ_TOL, r
        else:
            assert bool((dw[r] == 0).all()), r
    # the hub relation spans several weight-gradient tasks (8 tiles each)
    from recon_b200.convkb import TILES_PER_TASK
    assert max(GROUP_SIZES) > sum(GROUP_SIZES) / 2 and max(GROUP_SIZES) > 2 * TILES_PER_TASK * 128


@pytest.mark.gpu
@pytest.mark.parametrize("d", [12, 40, 200])
def test_grouped_forward_bit_equal_to_plain_gemm_per_group(d):
    from recon_b200 import _lib
    lib = _lib.load()
    rows, rid, w, gout = _grouped_case(d, d + 1)
    y, _, _ = _project_gpu(rows, rid, w, gout)
    ld = (d + 3) // 4 * 4
    for r, c in enumerate(GROUP_SIZES):
        if not c:
            continue
        sel = (rid == r).nonzero().flatten()
        a = torch.zeros(c, ld, device=_dev())[:, :d]
        a.copy_(rows[sel].to(_dev()))
        b = w[r].to(_dev()).contiguous()
        out = torch.empty(c, ld, device=_dev())[:, :d]
        ws = torch.empty(lib.spk_gemm_tc_workspace_floats(d, d), device=_dev())
        _lib.check(lib.spk_gemm_nn_tc_act(a.data_ptr(), a.stride(0), b.data_ptr(), b.stride(0), out.data_ptr(),
                                          out.stride(0), c, d, d, 0, 2, ws.data_ptr(), _lib.stream_ptr()), "gemm")
        assert torch.equal(y[sel.to(_dev())], out), r


@pytest.mark.gpu
def test_absent_relation_weights_never_read():
    rows, rid, w, gout = _grouped_case(40, 5)
    w = w.clone()
    for r, c in enumerate(GROUP_SIZES):
        if not c:
            w[r].fill_(1e30)
    y, dx, dw = _project_gpu(rows, rid, w, gout)
    assert bool(torch.isfinite(y).all()) and bool(torch.isfinite(dx).all())
    for r, c in enumerate(GROUP_SIZES):
        if c:
            assert bool(torch.isfinite(dw[r]).all())
        else:
            assert bool((dw[r] == 0).all())


def _layout_and_project(rows, rid, w, n_rel):
    from recon_b200.convkb import RelationLayout, PaddedRowsFn, GroupedProjectFn
    lay = RelationLayout(rid, rid.numel(), 1, 1, n_rel)
    x = PaddedRowsFn.apply(rows, lay, None).detach().requires_grad_(True)
    y = GroupedProjectFn.apply(x, w, lay)
    return lay, x, y


@pytest.mark.gpu
def test_projection_launches_do_not_depend_on_relation_count():
    from recon_b200 import _lib
    n_rel, n, d = 300, 6000, 40
    w = _w(n_rel, d, 6).to(_dev()).requires_grad_(True)
    g = torch.Generator().manual_seed(6)
    rows = torch.randn(n, d, generator=g).to(_dev())
    counts = []
    for present in (3, 300):
        rid = (torch.arange(n) % present).to(_dev())              # equal groups of 20 to 2000 rows
        gy = torch.randn(n, d, generator=g)
        torch.cuda.synchronize()
        c0 = _lib.launch_count()
        lay, x, y = _layout_and_project(rows, rid, w, n_rel)
        y.backward(torch.zeros_like(y))
        torch.cuda.synchronize()
        counts.append(_lib.launch_count() - c0)
        del gy
    assert counts[0] == counts[1], counts
    assert counts[0] <= 20, counts


@pytest.mark.gpu
def test_projection_runs_without_host_synchronisation():
    n_rel, n, d = 50, 3000, 40
    g = torch.Generator().manual_seed(7)
    rows = torch.randn(n, d, generator=g).to(_dev())
    rid = torch.randint(0, n_rel, (n,), generator=g).to(_dev())
    w = _w(n_rel, d, 7).to(_dev()).requires_grad_(True)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        lay, x, y = _layout_and_project(rows, rid, w, n_rel)
        y.backward(torch.ones_like(y))
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert bool(torch.isfinite(w.grad).all()) and bool(torch.isfinite(x.grad).all())


# ---- GPU: the loss ------------------------------------------------------------------------------------------------
LOSS_CASES = {
    # name: (n_ent, n_rel, d, n_pos, ratio, margin, extra)
    "refdims": (5000, 40, 200, 600, 2, 5.0, {}),
    "oddwidth_ratio3": (3000, 30, 13, 500, 3, 1.0, {}),
    "hub_entity": (4000, 30, 40, 800, 2, 2.0, {"hub_entity": 7}),
    "hub_relation": (4000, 60, 40, 1500, 2, 2.0, {"hub_rel": 3}),
    "rel_corrupted": (4000, 30, 40, 800, 2, 2.0, {"rel_corrupt": True}),
}


def _loss_inputs(name):
    n_ent, n_rel, d, n_pos, ratio, margin, extra = LOSS_CASES[name]
    seed = sorted(LOSS_CASES).index(name) + 10
    ent, rel = _tables(n_ent, n_rel, d, seed)
    return _tri(n_ent, n_rel, n_pos, ratio, seed, **extra), ent, rel, _w(n_rel, d, seed), ratio, margin


def _loss_gpu(tri, ent, rel, w, ratio, margin):
    from recon_b200.loss import batch_gat_loss
    e = ent.to(_dev()).requires_grad_(True)
    r = rel.to(_dev()).requires_grad_(True)
    wd = w.to(_dev()).requires_grad_(True)
    loss = batch_gat_loss(torch.nn.MarginRankingLoss(margin=margin), tri, e, r, valid_invalid_ratio_gat=ratio,
                          model_gat=types.SimpleNamespace(W_ent2rel=wd))
    loss.backward()
    torch.cuda.synchronize()
    return loss.detach(), e.grad, r.grad, wd.grad


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(LOSS_CASES))
def test_sep_loss_vs_fp64_oracle(name):
    tri, ent, rel, w, ratio, margin = _loss_inputs(name)
    loss, de, dr, dw = _loss_gpu(tri, ent, rel, w, ratio, margin)
    rl, rde, rdr, rdw = S.loss_sep_fwd_bwd(tri, ent.double(), rel.double(), w.double(), ratio, margin)
    assert abs(float(loss) - float(rl)) <= TIGHT * abs(float(rl))
    assert rel_l2(de, rde) <= TOL
    assert rel_l2(dr, rdr) <= TOL
    assert rel_l2(dw, rdw) <= TOL
    absent = torch.ones(w.shape[0], dtype=torch.bool)
    absent[tri[:, 1]] = False
    assert bool((dw[absent.to(_dev())] == 0).all())


@pytest.mark.gpu
def test_sep_loss_is_deterministic():
    tri, ent, rel, w, ratio, margin = _loss_inputs("hub_relation")
    a = _loss_gpu(tri, ent, rel, w, ratio, margin)
    b = _loss_gpu(tri, ent, rel, w, ratio, margin)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


@pytest.mark.gpu
def test_sep_loss_errors():
    from recon_b200.loss import batch_gat_loss
    tri, ent, rel, w, ratio, margin = _loss_inputs("rel_corrupted")
    f = torch.nn.MarginRankingLoss(margin=margin)
    gat = types.SimpleNamespace(W_ent2rel=w.to(_dev()))
    e, r = ent.to(_dev()), rel.to(_dev())
    n_ent, n_rel = ent.shape[0], w.shape[0]
    for col, bad in ((0, n_ent), (2, -1), (1, n_rel), (1, -1)):
        t2 = tri.clone(); t2[5, col] = bad
        with pytest.raises(IndexError):
            batch_gat_loss(f, t2, e, r, valid_invalid_ratio_gat=ratio, model_gat=gat)
    e_nan = e.clone(); e_nan[tri[0, 0]] = float("nan")
    with pytest.raises(AssertionError):
        batch_gat_loss(f, tri, e_nan, r, valid_invalid_ratio_gat=ratio, model_gat=gat)
    with pytest.raises(RuntimeError):
        batch_gat_loss(f, tri[:-1], e, r, valid_invalid_ratio_gat=ratio, model_gat=gat)
    with pytest.raises(RuntimeError):
        batch_gat_loss(f, tri, ent, rel, valid_invalid_ratio_gat=ratio, model_gat=types.SimpleNamespace(W_ent2rel=w))


@pytest.mark.gpu
def test_training_iteration_sep_model_loss_sgd_vs_oracle():
    """One iteration of train_gat for a GAT_sep_space model: forward -> sep loss -> backward -> SGD, against the fp64
    model oracle chained into the fp64 sep loss oracle; every trainable gradient including W_ent2rel."""
    from recon_b200 import SpKBGATModified
    from recon_b200.loss import batch_gat_loss, sgd_step
    from recon_b200.synth import make_kg
    from oracle import ref_torch as O
    from oracle import loss as OL
    n, e, r, f, d, h = 3000, 30000, 20, 50, 100, 2
    edge, etype, nhop = make_kg(n, e, r, 1.1, 3000, seed=21)
    p = O.init_params(n, r, f, d, h, seed=21)
    w = _w(r, d * h, 21, scale=4.0)                 # model outputs are unit rows: e . W ~ N(0, 4 / HD)
    tri = OL.make_train_indices(n, r, 4000, 2, seed=22)
    be = torch.unique(tri[:4000, 0])
    model = SpKBGATModified(p["entity_embeddings"].clone(), p["relation_embeddings"].clone(), [d, 2 * d], [d, 2 * d],
                            0.0, 0.2, [h, h], None, sep_space=True)
    model.load_state_dict(dict(p, W_ent2rel=w))
    model = model.to(_dev())
    out_e, out_r, _ = model(None, be, (edge, etype), nhop)
    loss = batch_gat_loss(torch.nn.MarginRankingLoss(margin=5.0), tri, out_e, out_r, model_gat=model)
    loss.backward()
    loss = loss.detach()
    names = O.trainable_names(p)
    q = {k: (v.double().clone().requires_grad_(True) if k in names else v.double()) for k, v in p.items()}
    w64 = w.double().requires_grad_(True)
    o_e, o_r, _, _ = O.kbgat_forward(q, be, (edge, etype), nhop, 0.2, None, O.seg_sum_index_add)
    ref_loss = S.batch_gat_loss_sep(tri, o_e, o_r, w64, 2, 5.0)
    ref_loss.backward()
    q["W_ent2rel"] = w64
    assert abs(float(loss) - float(ref_loss)) <= TIGHT * abs(float(ref_loss))
    errs = {nm: rel_l2(prm.grad, q[nm].grad) for nm, prm in model.named_parameters()
            if (nm in names or nm == "W_ent2rel") and q[nm].grad is not None}
    assert len(errs) >= 11 and "W_ent2rel" in errs
    bad = {k: v for k, v in errs.items() if not v < TOL}
    assert not bad, bad
    lr = 1e-3
    before = {nm: prm.detach().clone() for nm, prm in model.named_parameters()}
    sgd_step(model.parameters(), lr)
    torch.cuda.synchronize()
    for nm, prm in model.named_parameters():
        if prm.grad is not None:
            want = before[nm].double() - lr * prm.grad.double()
            assert rel_l2(prm, want) <= 1e-6, nm

"""Layer groups at every row-width class and head template the edge kernels are compiled for.

The fused edge kernels (forward, the three backward schedules, the column / relation gathers and the hub-task
finalizes) are instantiated per NCH = ceil(Wd / 128) (float4 chunks per lane, Wd = projected row width in floats,
at most 512) and per head template HT in {1, 2, 4} (H = 3 and H = 4 both run HT = 4), with 2-hop and hub variants on
top. These tests call `functional.attention_group` at one layer geometry per (NCH, HT) pair, at the width boundaries
and at head widths that are not a multiple of 4 (every head chunk then carries pad columns), and compare the outputs
and the gradients of X, Rel, a_h and a_2,h with the fp64 oracle (`oracle.ref_torch.attention_layer`, one call per
head). The graphs reach the hub-row, hub-column and hub-relation tasks, empty rows, self loops, duplicate edges,
2-hop rows and the streaming segment gather; the whole model is checked at the head counts RECON users set.
"""
import json

import pytest
import torch

from helpers import rel_l2

TOL = 1e-4          # project tolerance (gradients)
TIGHT = 2e-5        # what the fp32-exact kernels reach (outputs)
ALPHA = 0.2

# One layer of H heads of width D on F-wide entity rows and Rd-wide relation rows; `elu` is the fused ELU of the
# reference's concat=True layers. Layers with more than 4 heads run as groups of <= 4 (the table below covers the
# geometry of every group).
CASES = [
    # (H, D, F, Rd, elu, note)
    (1, 7, 13, 7, True, "odd head width, narrowest row"),                    # Wd 16   NCH 1
    (1, 124, 50, 50, False, "Wd 128: widest NCH-1 row"),                    # Wd 128  NCH 1
    (2, 13, 1, 1, True, "2 heads, odd width, F = Rd = 1"),                       # Wd 40   NCH 1
    (3, 10, 50, 50, True, "3 heads on the 4-head code"),                    # Wd 40   NCH 1
    (4, 28, 20, 12, False, "4 heads"),                                      # Wd 120  NCH 1
    (1, 132, 50, 50, True, "Wd 136: narrowest NCH-2 row"),                  # Wd 136  NCH 2
    (1, 201, 24, 24, False, "odd width"),                                   # Wd 208  NCH 2
    (2, 100, 50, 50, True, "benchmark layer 1"),                            # Wd 208  NCH 2
    (2, 61, 50, 50, False, "2 heads, odd width"),                           # Wd 136  NCH 2
    (3, 62, 50, 50, True, "3 heads, D % 4 = 2"),                            # Wd 200  NCH 2
    (4, 50, 50, 50, False, "4 heads, D % 4 = 2"),                           # Wd 216  NCH 2
    (1, 300, 60, 40, True, "layer 2 of nheads [3, 3] x 100"),               # Wd 304  NCH 3
    (1, 333, 32, 32, False, "odd width"),                                   # Wd 344  NCH 3
    (2, 150, 50, 50, True, "2 heads, D % 4 = 2"),                           # Wd 312  NCH 3
    (2, 127, 50, 50, False, "2 heads, D % 4 = 3"),                          # Wd 264  NCH 3
    (3, 100, 50, 50, True, "layer 1 of nheads [3, 3] x 100"),               # Wd 304  NCH 3
    (4, 90, 50, 50, False, "4 heads, D % 4 = 2"),                           # Wd 376  NCH 3
    (1, 508, 16, 16, False, "Wd 512: widest row"),                          # Wd 512  NCH 4
    (1, 401, 50, 50, True, "odd width"),                                    # Wd 408  NCH 4
    (2, 250, 50, 50, True, "Wd 512 with 2 heads, D % 4 = 2"),               # Wd 512  NCH 4
    (3, 127, 50, 50, False, "3 heads, D % 4 = 3"),                          # Wd 392  NCH 4
    (4, 100, 50, 50, True, "layer 1 of nheads [4, 4] x 100"),               # Wd 408  NCH 4
    (4, 124, 20, 20, True, "widest 4-head group"),                          # Wd 504  NCH 4
    (5, 60, 50, 50, True, "groups of 4 + 1 heads"),                         # Wd 248 + 64
]

# per case: the (Wd, NCH, HT) of each head group, in group order
EXPECTED_GROUPS = {
    (1, 7): [(16, 1, 1)], (1, 124): [(128, 1, 1)], (2, 13): [(40, 1, 2)], (3, 10): [(40, 1, 4)],
    (4, 28): [(120, 1, 4)], (1, 132): [(136, 2, 1)], (1, 201): [(208, 2, 1)], (2, 100): [(208, 2, 2)],
    (2, 61): [(136, 2, 2)], (3, 62): [(200, 2, 4)], (4, 50): [(216, 2, 4)], (1, 300): [(304, 3, 1)],
    (1, 333): [(344, 3, 1)], (2, 150): [(312, 3, 2)], (2, 127): [(264, 3, 2)], (3, 100): [(304, 3, 4)],
    (4, 90): [(376, 3, 4)], (1, 508): [(512, 4, 1)], (1, 401): [(408, 4, 1)], (2, 250): [(512, 4, 2)],
    (3, 127): [(392, 4, 4)], (4, 100): [(408, 4, 4)], (4, 124): [(504, 4, 4)], (5, 60): [(248, 2, 4), (64, 1, 1)],
}

MASKED = [(4, 100), (3, 100)]                            # also run with a dropout mask (NCH 4 / 3 heads at NCH 3)
SPARSE = [(2, 13), (3, 62), (2, 127), (3, 127)]          # also run on the sparse graph (one case per NCH, D % 4 != 0)


def _case(h, d):
    return next(c for c in CASES if c[:2] == (h, d))


def _groups(h):
    return [min(4, h - g0) for g0 in range(0, h, 4)]


def _nch(wd):
    return (wd // 4 + 31) // 32


def _ht(h):
    return h if h <= 2 else 4


# ---- 1. the geometry table (CPU) ----------------------------------------------------------------------------------
def test_geometry_table_covers_every_kernel_instantiation():
    from recon_b200.functional import Geometry
    seen = set()
    odd_per_nch = set()
    widths = set()
    for H, D, F, Rd, elu, note in CASES:
        got = []
        for hg in _groups(H):
            g = Geometry(hg, D)
            got.append((g.Wd, _nch(g.Wd), _ht(hg)))
            assert g.Dp == (D + 3) // 4 * 4 and g.Wd % 8 == 0 and g.Wd >= hg * g.Dp + hg, (H, D)
            widths.add((hg, D, g.Wd))
        assert got == EXPECTED_GROUPS[(H, D)], (H, D, got)
        for wd, nch, ht in got:
            seen.add((nch, ht))
            if D % 4:
                odd_per_nch.add(nch)
    assert set(EXPECTED_GROUPS) == {c[:2] for c in CASES}
    assert seen == {(n, t) for n in (1, 2, 3, 4) for t in (1, 2, 4)}
    assert odd_per_nch == {1, 2, 3, 4}
    assert any(c[0] == 3 for c in CASES) and any(c[0] > 4 for c in CASES)
    assert {(1, 124, 128), (1, 132, 136), (1, 508, 512), (4, 124, 504)} <= widths
    assert {_nch(EXPECTED_GROUPS[c[:2]][0][0]) for c in CASES if not c[4]} == {1, 2, 3, 4}   # elu off at every NCH
    assert {_nch(EXPECTED_GROUPS[k][0][0]) for k in SPARSE} == {1, 2, 3, 4}
    for h, d in ((1, 509), (4, 125), (2, 253)):
        with pytest.raises(ValueError):
            Geometry(h, d)


# ---- shared harness -------------------------------------------------------------------------------------------------
def dev():
    return torch.device("cuda:0")


def _graph_edges(kind, has2):
    """Caller-order edge lists. "hub": 2000 nodes, 7 relations (every relation segment is a hub), row 3 with ~1500
    in-edges and column 5 with ~1500 entries (both past graph.HUB_THRESH = 512), 64 empty rows, self loops and
    duplicate edges. "sparse": 3000 nodes, 4000 relations, ~2 entries per column and ~2 per relation, so the
    segment gathers request the streaming kernel; one hub row. has2 adds 2-hop rows [s, r1, r2, t]."""
    g = torch.Generator().manual_seed(17 if kind == "hub" else 29)
    ri = lambda hi, n: torch.randint(0, hi, (n,), generator=g)                     # noqa: E731
    if kind == "hub":
        n, r, hub_row, hub_col = 2000, 7, 3, 5
        live = n - 64                                                            # rows live..n-1 get no edges
        rows = torch.cat((ri(live, 8000), torch.full((1500,), hub_row), ri(live, 1500)))
        cols = torch.cat((ri(n, 8000), ri(n, 1500), torch.full((1500,), hub_col)))
        loops = ri(live, 200)
        rows, cols = torch.cat((rows, loops)), torch.cat((cols, loops))
        n2, n2_hub = 2000, 300
    else:
        n, r, hub_row = 3000, 4000, 7
        live = n - 64
        rows = torch.cat((ri(live, 6000), torch.full((600,), hub_row)))
        cols = ri(n, 6600)
        n2, n2_hub = 1000, 100
    etype = ri(r, rows.numel())
    dup = ri(rows.numel(), 300)
    rows, cols, etype = torch.cat((rows, rows[dup])), torch.cat((cols, cols[dup])), torch.cat((etype, etype[dup]))
    perm = torch.randperm(rows.numel(), generator=g)
    edge = torch.stack((rows[perm], cols[perm])).contiguous()
    etype = etype[perm].contiguous()
    nhop = None
    if has2:
        t = torch.cat((ri(live, n2 - n2_hub), torch.full((n2_hub,), hub_row)))
        nhop = torch.stack((ri(n, n2), ri(r, n2), ri(r, n2), t), dim=1)
        nhop = nhop[torch.randperm(n2, generator=g)].contiguous()
    return n, r, edge, etype, nhop


_GRAPHS = {}


def _graph(kind, has2):
    """(n, r, edge, etype, nhop, KGraph) built once per module."""
    if (kind, has2) not in _GRAPHS:
        from recon_b200 import KGraph
        n, r, edge, etype, nhop = _graph_edges(kind, has2)
        kg = KGraph(edge, etype, nhop, n, r, device=dev())
        _GRAPHS[(kind, has2)] = (n, r, edge, etype, nhop, kg)
    return _GRAPHS[(kind, has2)]


def _inputs(case, kind, has2, masked):
    """Seeded fp32 CPU inputs: X, Rel, a_h (xavier_normal, gain 1.414, as GAT/layers.py:100-105), a_2,h, the upstream
    gradient and the [H, E] dropout multipliers in caller edge order (or None)."""
    H, D, F, Rd = case[:4]
    n, r, edge, etype, nhop, _ = _graph(kind, has2)
    e = edge.shape[1] + (nhop.shape[0] if nhop is not None else 0)
    g = torch.Generator().manual_seed(1000 * H + D + 7 * F + 13 * Rd + (1 if has2 else 0))

    def xavier(rows, cols):
        return torch.randn(rows, cols, generator=g) * (1.414 * (2.0 / (rows + cols)) ** 0.5)

    X = torch.randn(n, F, generator=g)
    Rel = torch.randn(r, Rd, generator=g)
    a = [xavier(D, 2 * F + Rd) for _ in range(H)]
    a2 = [xavier(1, D) for _ in range(H)]
    gout = torch.randn(n, H * D, generator=g)
    mask = (torch.rand(H, e, generator=g) >= 0.3).float() / 0.7 if masked else None
    return X, Rel, a, a2, gout, mask


_ORACLE = {}


def _oracle(case, kind, has2, masked):
    """fp64 reference of the layer: out [N, H*D] and the gradients of X, Rel, a_h, a_2,h under the upstream gradient.
    Kept for the few most recent keys (the backward schedules of one case run one after the other)."""
    from oracle import ref_torch as O
    key = (case[:4], case[4], kind, has2, masked)
    if key in _ORACLE:
        return _ORACLE[key]
    n, r, edge, etype, nhop, _ = _graph(kind, has2)
    X, Rel, a, a2, gout, mask = _inputs(case, kind, has2, masked)
    X, Rel = X.double().requires_grad_(True), Rel.double().requires_grad_(True)
    a = [t.double().requires_grad_(True) for t in a]
    a2 = [t.double().requires_grad_(True) for t in a2]
    emb = Rel[etype]
    e_nhop = emb_nhop = None
    if nhop is not None:
        e_nhop = torch.stack((nhop[:, 3], nhop[:, 0]))
        emb_nhop = Rel[nhop[:, 1]] + Rel[nhop[:, 2]]
    outs = [O.attention_layer(X, edge, emb, e_nhop, emb_nhop, a[h], a2[h], ALPHA, case[4],
                              None if mask is None else mask[h].double(), O.seg_sum_index_add)
            for h in range(case[0])]
    out = torch.cat(outs, dim=1)
    grads = torch.autograd.grad(out, [X, Rel] + a + a2, gout.double())
    while len(_ORACLE) >= 3:
        _ORACLE.pop(next(iter(_ORACLE)))
    _ORACLE[key] = (out.detach(), grads)
    return _ORACLE[key]


def _run_layer(case, kind, has2, masked):
    """attention_group forward + backward on the device, twice: (out, grads, nanflag) of the first call and whether
    the second call reproduced every tensor bit for bit."""
    from recon_b200 import functional as SF
    n, r, edge, etype, nhop, kg = _graph(kind, has2)
    X0, Rel0, a0, a20, gout, mask = _inputs(case, kind, has2, masked)
    mask_csr = kg.to_csr_order(mask.to(dev())) if mask is not None else None
    runs = []
    for _ in range(2):
        X = X0.to(dev()).requires_grad_(True)
        Rel = Rel0.to(dev()).requires_grad_(True)
        a = [t.to(dev()).requires_grad_(True) for t in a0]
        a2 = [t.to(dev()).requires_grad_(True) for t in a20]
        nanflag = torch.zeros(1, dtype=torch.int32, device=dev())
        out = SF.attention_group(X, Rel, a, a2, kg, ALPHA, case[4], mask_csr, nanflag)
        grads = torch.autograd.grad(out, [X, Rel] + a + a2, gout.to(dev()))
        runs.append((out.detach(), grads, int(nanflag.item())))
    (out, grads, flag), (out2, grads2, _) = runs
    same = torch.equal(out, out2) and all(torch.equal(x, y) for x, y in zip(grads, grads2))
    return out, grads, flag, same


def _errors(case, got_out, got_grads, ref_out, ref_grads):
    H = case[0]
    errs = {"out": rel_l2(got_out, ref_out), "dX": rel_l2(got_grads[0], ref_grads[0]),
            "dRel": rel_l2(got_grads[1], ref_grads[1])}
    errs["da"] = max(rel_l2(got_grads[2 + h], ref_grads[2 + h]) for h in range(H))
    errs["da2"] = max(rel_l2(got_grads[2 + H + h], ref_grads[2 + H + h]) for h in range(H))
    return errs


def _check(case, kind, has2, masked, record_property):
    out, grads, flag, same = _run_layer(case, kind, has2, masked)
    ref_out, ref_grads = _oracle(case, kind, has2, masked)
    assert out.shape == ref_out.shape == (ref_out.shape[0], case[0] * case[1])
    errs = _errors(case, out, grads, ref_out, ref_grads)
    record_property("rel_l2", json.dumps(errs))
    assert flag == 0, "nanflag set"
    assert errs["out"] < TIGHT, errs
    bad = {k: v for k, v in errs.items() if not v < TOL}
    assert not bad, errs
    assert same, "second call is not bit-identical"
    return errs


@pytest.fixture
def modes():
    """Sets functional.AGG_MODE / BWD_MODE for one test and restores them."""
    from recon_b200 import functional as SF
    old = SF.AGG_MODE, SF.BWD_MODE

    def set_modes(agg, bwd="split"):
        SF.AGG_MODE, SF.BWD_MODE = agg, bwd

    yield set_modes
    SF.AGG_MODE, SF.BWD_MODE = old


# ---- 2. projected layer groups against fp64 --------------------------------------------------------------------------
def _group_params():
    """(case, graph, has2, masked, bwd) with the backward schedules of one oracle key adjacent. "split" falls back to
    "rows" on graphs with 2-hop edges (functional.edge_attn_backward), so has2 runs only "fused" and "rows"."""
    out = []
    keys = [(c, "hub", has2, False) for c in CASES for has2 in (False, True)]
    keys += [(_case(*k), "hub", has2, True) for k in MASKED for has2 in (False, True)]
    keys += [(_case(*k), "sparse", has2, False) for k in SPARSE for has2 in (False, True)]
    for case, kind, has2, masked in keys:
        for bwd in (("fused", "rows") if has2 else ("split", "fused", "rows")):
            nch = EXPECTED_GROUPS[case[:2]][0][1]
            tag = f"H{case[0]}-D{case[1]}-F{case[2]}-R{case[3]}-nch{nch}-{kind}{'-has2' if has2 else ''}" \
                  f"{'-mask' if masked else ''}-{bwd}"
            out.append(pytest.param(case, kind, has2, masked, bwd, id=tag))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("case,kind,has2,masked,bwd", _group_params())
def test_layer_group_matches_fp64(case, kind, has2, masked, bwd, modes, record_property):
    modes("off", bwd)
    *_, kg = _graph(kind, has2)
    if kind == "hub":
        # row, column and relation hub tasks and their finalize kernels all run
        assert kg.row_hubs.n_tasks > 0 and kg.col_hubs.n_tasks > 0 and kg.rel_hubs.n_tasks > 0
        assert kg.rel_hubs.n_hubs == kg.n_rel
    else:
        # functional.seg_gather asks for the streaming kernel here; it serves NCH <= 2, wider rows take the register kernel
        assert kg.row_hubs.n_tasks > 0
        assert kg.csc_row.numel() < 5 * kg.n_cols and kg.rel_row.numel() < 5 * kg.n_rel
    _check(case, kind, has2, masked, record_property)


# ---- 3. aggregate-then-project path at its limits ----------------------------------------------------------------------
AGG_CASES = [
    # (H, D, F, Rd, elu, note)
    (1, 16, 1, 1, True, "F = Rd = 1"),
    (2, 24, 7, 7, True, "F = Rd = 7"),
    (2, 100, 50, 50, True, "benchmark layer 1"),
    (2, 60, 60, 60, False, "F = Rd = 60: widest supported input"),
    (3, 100, 50, 50, True, "2 + 1 head groups"),
    (2, 40, 50, 10, True, "Rd != F: rows backward"),
    (3, 21, 60, 7, False, "2 + 1 head groups, Rd != F"),
    (1, 600, 50, 50, True, "D = 600: past the projected row limit"),
]


def _agg_params():
    out = []
    for c in AGG_CASES:
        for has2 in (False, True):
            out.append(pytest.param(c, "hub", has2, False, id=f"H{c[0]}-D{c[1]}-F{c[2]}-R{c[3]}{'-has2' if has2 else ''}"))
    out.append(pytest.param(AGG_CASES[4], "hub", False, True, id="H3-D100-F50-R50-mask"))
    out.append(pytest.param(AGG_CASES[4], "hub", True, True, id="H3-D100-F50-R50-has2-mask"))
    out.append(pytest.param(AGG_CASES[5], "sparse", False, False, id="H2-D40-F50-R10-sparse"))
    out.append(pytest.param(AGG_CASES[2], "sparse", True, False, id="H2-D100-F50-R50-sparse-has2"))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("case,kind,has2,masked", _agg_params())
def test_aggregate_path_matches_fp64(case, kind, has2, masked, modes, record_property):
    from recon_b200 import functional as SF
    modes("force")
    H, D, F, Rd = case[:4]
    *_, kg = _graph(kind, has2)
    assert SF.use_agg_path(min(H, SF.AGG_MAX_HEADS), F, Rd, D, kg)
    _check(case, kind, has2, masked, record_property)


@pytest.mark.gpu
def test_aggregate_path_is_not_taken_past_60_input_features(modes, record_property):
    """F = 61 is past AggGeometry.supported: even in "force" mode the layer runs on the projected kernels."""
    from recon_b200 import functional as SF
    modes("force")
    case = (2, 32, 61, 61, True, "F = Rd = 61")
    *_, kg = _graph("hub", False)
    assert not SF.use_agg_path(2, 61, 61, 32, kg)
    assert not SF.use_agg_path(2, 60, 61, 32, kg) and not SF.use_agg_path(2, 61, 60, 32, kg)
    _check(case, "hub", False, False, record_property)


@pytest.mark.gpu
def test_wide_heads_need_the_aggregate_path(modes, record_property):
    """H = 1, D = 600: the aggregate path projects after the aggregation (a GEMM, no 512-float row), so it computes the
    layer in "auto" mode as well; with "off" the projected path rejects the width with Geometry's ValueError."""
    from recon_b200 import functional as SF
    case = AGG_CASES[-1]
    assert case[:2] == (1, 600)
    *_, kg = _graph("hub", False)
    modes("auto")
    assert SF.use_agg_path(1, 50, 50, 600, kg)
    _check(case, "hub", False, False, record_property)
    modes("off")
    X, Rel, a, a2, _, _ = _inputs(case, "hub", False, False)
    with pytest.raises(ValueError, match="512-float"):
        SF.attention_group(X.to(dev()), Rel.to(dev()), [t.to(dev()) for t in a], [t.to(dev()) for t in a2], kg,
                           ALPHA, True, None, torch.zeros(1, dtype=torch.int32, device=dev()))


# ---- 4. whole model at ordinary RECON head counts ---------------------------------------------------------------------
@pytest.fixture(params=["auto", "force", "off"])
def agg_path(request):
    from recon_b200 import functional as SF
    old = SF.AGG_MODE
    SF.AGG_MODE = request.param
    yield request.param
    SF.AGG_MODE = old


@pytest.fixture(params=["split", "fused", "rows"])
def bwd_path(request):
    from recon_b200 import functional as SF
    old = SF.BWD_MODE
    SF.BWD_MODE = request.param
    yield request.param
    SF.BWD_MODE = old


MODEL_N, MODEL_E, MODEL_R, MODEL_F = 4000, 40000, 31, 50
_MODEL_ORACLE = {}


def _model_data():
    from recon_b200.synth import make_kg
    return make_kg(MODEL_N, MODEL_E, MODEL_R, 1.1, 4000, seed=21)


def _model_oracle(h, d):
    from oracle import ref_torch as O
    if (h, d) not in _MODEL_ORACLE:
        edge, etype, nhop = _model_data()
        p = O.init_params(MODEL_N, MODEL_R, MODEL_F, d, h, seed=h * 10 + d)
        gen = torch.Generator().manual_seed(h + d)
        ge, gr = torch.randn(MODEL_N, d * h, generator=gen), torch.randn(MODEL_R, d * h, generator=gen)
        be = torch.arange(0, MODEL_N, 3)
        p64 = {k: v.double() for k, v in p.items()}
        ref = O.fwd_bwd(p64, be, (edge, etype), nhop, ALPHA, ge.double(), gr.double(), None, O.seg_sum_index_add)
        _MODEL_ORACLE.clear()
        _MODEL_ORACLE[(h, d)] = (p, ge, gr, be, ref)
    return _MODEL_ORACLE[(h, d)]


@pytest.mark.gpu
@pytest.mark.parametrize("nheads,d", [(3, 100), (4, 100), (5, 21)],
                         ids=["heads3-D100-layer2-D300", "heads4-D100-layer2-D400", "heads5-D21-layer2-D105"])
def test_model_vs_oracle_recon_heads(nheads, d, agg_path, bwd_path, record_property):
    from recon_b200 import SpKBGATModified
    edge, etype, nhop = _model_data()
    p, ge, gr, be, ref = _model_oracle(nheads, d)
    model = SpKBGATModified(p["entity_embeddings"].clone(), p["relation_embeddings"].clone(), [d, nheads * d],
                            [d, nheads * d], 0.0, ALPHA, [nheads, nheads], None)
    model.load_state_dict(p)
    model = model.to(dev())
    out_e, out_r, _ = model(None, be, (edge, etype), nhop)
    ((out_e * ge.to(dev())).sum() + (out_r * gr.to(dev())).sum()).backward()
    errs = {"out_entity": rel_l2(out_e, ref[0]), "out_relation": rel_l2(out_r, ref[1])}
    for nm, prm in model.named_parameters():
        if nm in ref[4]:
            errs["grad." + nm] = rel_l2(prm.grad, ref[4][nm])
    record_property("rel_l2", json.dumps(errs))
    assert len(errs) == 2 + 6 + 2 * nheads         # both outputs, every trainable parameter
    bad = {k: v for k, v in errs.items() if not v < TOL}
    assert not bad, bad
    kg = model.prepare_graph((edge, etype), nhop)
    assert kg.row_hubs.n_hubs > 0 and kg.t2 is not None

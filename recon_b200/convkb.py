"""N4 (SURVEY.md 8f): the ConvKB scoring stage fed by the hot path's output embeddings, on libspkbgat.

  ConvKB            <- GAT/layers.py:12-48     same constructor, parameter names (conv_layer, fc_layer, fc1, fc2) and
                                               forward; the live path is fc2(LeakyReLU(fc1(x))) (the convolution is
                                               commented out in the reference and kept only as parameters)
  SpKBGATConvOnly   <- GAT/models.py:242-304   forward(Corpus_, adj, batch_inputs) / batch_test(batch_inputs); with a
                       GAT_sep_space/models.py:311-339   `model_gat` argument the head / tail rows go through
                                               tanh(e . W_ent2rel[r]) first (relation-space projection)
  ent2rel_project   <- GAT_sep_space/models.py:316-320, GAT_sep_space/main.py:360-377 (RelationLayout + GroupedProjectFn:
                       rows grouped by relation on the device, one grouped tcgen05 GEMM per pass; also the projection of
                       the sep-space TransE loss, loss.batch_gat_loss(..., model_gat=))
  relation_scores / rank_relations <- GAT/create_batch.py:1367-1500 (every test pair scored under every relation)

fc1 over the concatenation [h | r | t] is one tcgen05 GEMM on the gathered rows for training batches (a few thousand
triples); the all-relations ranking uses the re-association fc1([h|r|t]) = W1a e_h + W1b r + W1c e_t + b1, so the T x R
score matrix is one streaming pass (spk_rank_scores) over T pair rows and R relation rows instead of T*R GEMM rows.
No CPU fallback; gradients are deterministic (row sums by sorted segments, fixed-order split GEMMs).
"""
import ctypes as C

import torch
import torch.nn as nn

from . import _lib
from . import functional as SF
from .graph import sort_pairs, _segment_ptr, _key_bits
from .layers import SpecialSpmmFunctionFinal

LRELU_SLOPE = 0.01          # nn.LeakyReLU() default, GAT/layers.py:25


def _gather_concat(pieces, n_out, d):
    """pieces: list of (table [rows, >= d] fp32, index int64 tensor view or None, element stride of the index)."""
    lib = _lib.load()
    dev = pieces[0][0].device
    np_ = len(pieces)
    ldo = (np_ * d + 3) // 4 * 4
    out = torch.empty(n_out, ldo, dtype=torch.float32, device=dev)[:, :np_ * d]
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    src = (C.c_void_p * 3)(); ld = (C.c_int64 * 3)(); idx = (C.c_void_p * 3)(); stride = (C.c_int64 * 3)(); rows = (C.c_int64 * 3)()
    for p, (t, ix, st) in enumerate(pieces):
        assert t.stride(1) == 1 and t.dtype == torch.float32
        src[p] = t.data_ptr(); ld[p] = t.stride(0); rows[p] = t.shape[0]
        idx[p] = ix.data_ptr() if ix is not None else None; stride[p] = st
    _lib.check(lib.spk_gather_concat(src, ld, idx, stride, rows, np_, n_out, d, out.data_ptr(), out.stride(0),
                                     err.data_ptr(), _lib.stream_ptr()), "gather_concat")
    if n_out and int(err.item()):
        raise IndexError("triple index out of range for the embedding tables")
    return out


class GatherRowsFn(torch.autograd.Function):
    """rows = table[idx] (the embedding lookups of GAT/models.py:295-296); backward = deterministic row sums."""

    @staticmethod
    def forward(ctx, table, idx):
        idx = idx.contiguous()
        ctx.save_for_backward(idx)
        ctx.n_rows = table.shape[0]
        t = table if table.stride(1) == 1 else table.contiguous()
        return _gather_concat([(t, idx, 1)], idx.numel(), table.shape[1])

    @staticmethod
    def backward(ctx, g):
        (idx,) = ctx.saved_tensors
        edge = torch.stack((idx, idx), dim=0)
        return SpecialSpmmFunctionFinal.apply(edge, g.contiguous(), ctx.n_rows, idx.numel(), g.shape[1]), None


class MLPHeadFn(torch.autograd.Function):
    """out[b] = fc2(LeakyReLU(H1[b] + fc1.bias)) (GAT/layers.py:44-45) fused into one pass over H1."""

    @staticmethod
    def forward(ctx, H1, b1, w2, b2):
        H1 = H1 if H1.stride(1) == 1 else H1.contiguous()
        b1 = b1.contiguous(); w2 = w2.contiguous(); b2 = b2.contiguous()
        n, d = H1.shape
        out = torch.empty(n, 1, dtype=torch.float32, device=H1.device)
        _lib.check(_lib.load().spk_mlp_head_fwd(_lib.ptr(H1), H1.stride(0), _lib.ptr(b1), _lib.ptr(w2), _lib.ptr(b2),
                                                LRELU_SLOPE, n, d, _lib.ptr(out), _lib.stream_ptr()), "mlp_head_fwd")
        ctx.save_for_backward(H1, b1, w2)
        return out

    @staticmethod
    def backward(ctx, dout):
        H1, b1, w2 = ctx.saved_tensors
        n, d = H1.shape
        dout = dout.contiguous()
        ldp = (d + 3) // 4 * 4
        dH1 = torch.empty(n, ldp, dtype=torch.float32, device=H1.device)[:, :d]
        act = torch.empty(n, ldp, dtype=torch.float32, device=H1.device)[:, :d]
        _lib.check(_lib.load().spk_mlp_head_bwd(_lib.ptr(H1), H1.stride(0), _lib.ptr(b1), _lib.ptr(w2), LRELU_SLOPE,
                                                _lib.ptr(dout), n, d, _lib.ptr(dH1), dH1.stride(0), _lib.ptr(act),
                                                act.stride(0), _lib.stream_ptr()), "mlp_head_bwd")
        ones = torch.ones(n, 1, dtype=torch.float32, device=H1.device)
        db1 = SF.gemm_tn(dH1, ones).reshape(-1) if ctx.needs_input_grad[1] else None          # column sums, fixed order
        dw2 = SF.gemm_tn(act, dout.reshape(n, 1)).reshape(1, -1) if ctx.needs_input_grad[2] else None
        db2 = SF.gemm_tn(dout.reshape(n, 1), ones).reshape(1) if ctx.needs_input_grad[3] else None
        return (dH1 if ctx.needs_input_grad[0] else None), db1, dw2, db2


class TanhFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        y = x.contiguous().clone()
        _lib.check(_lib.load().spk_tanh_fwd(_lib.ptr(y), y.stride(0), y.shape[0], y.shape[1], _lib.stream_ptr()), "tanh_fwd")
        ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, g):
        (y,) = ctx.saved_tensors
        g = g.contiguous()
        d = torch.empty_like(y)
        _lib.check(_lib.load().spk_tanh_bwd(_lib.ptr(y), y.stride(0), _lib.ptr(g), g.stride(0), y.shape[0], y.shape[1],
                                            _lib.ptr(d), d.stride(0), _lib.stream_ptr()), "tanh_bwd")
        return d


TILES_PER_TASK = 8          # a weight-gradient task of the grouped projection: up to 8 x 128 rows of one relation


def _ld4(d):
    return (d + 3) // 4 * 4


class RelationLayout:
    """Rows grouped by relation for the grouped tensor-core projection, built on the device (spk_ent2rel_*).

    Row j (j < reps * n_src) has relation rel[(j % n_src) * stride] (an int64 tensor view). Rows are stably sorted by
    relation; every relation present is one group, padded with zero rows to whole 128-row M tiles, so no tile straddles
    two relations. The host never reads the group count back: buffers are sized for the worst case, min(n_rel, rows)
    groups of 127 pad rows each. `pos[j]` is row j's padded row; `err` is set for a relation id outside [0, n_rel), whose
    row joins no group (so W_ent2rel is never read out of range) and has pos 0."""

    def __init__(self, rel, n_src, reps, stride, n_rel):
        lib = _lib.load()
        dev = rel.device
        n = int(n_src) * int(reps)
        self.n_rows, self.n_rel = n, int(n_rel)
        self.max_groups = max(1, min(self.n_rel, n))
        self.max_tiles = (n + 127 * self.max_groups + 127) // 128
        self.max_rows = 128 * self.max_tiles
        self.max_tasks = min(self.max_tiles, (self.max_tiles + (TILES_PER_TASK - 1) * self.max_groups) // TILES_PER_TASK)
        i32 = dict(dtype=torch.int32, device=dev)
        keys, vals = torch.empty(n, **i32), torch.empty(n, **i32)
        self.err = torch.zeros(1, **i32)
        _lib.check(lib.spk_ent2rel_keys(rel.data_ptr(), stride, n_src, reps, self.n_rel, keys.data_ptr(), vals.data_ptr(),
                                        self.err.data_ptr(), _lib.stream_ptr()), "ent2rel_keys")
        self.keys, self.vals = sort_pairs(keys, vals, _key_bits(self.n_rel + 1))
        self.segptr = _segment_ptr(self.keys, self.n_rel)
        self.rel2group = torch.empty(self.n_rel, **i32)
        self.group_rel = torch.empty(self.max_groups, **i32)
        self.group_tile0 = torch.empty(self.max_groups + 1, **i32)
        self.task_ptr = torch.empty(self.max_groups + 1, **i32)
        self.tile_group = torch.empty(self.max_tiles, **i32)
        self.task_row0 = torch.empty(max(1, self.max_tasks), **i32)
        self.task_row1 = torch.empty(max(1, self.max_tasks), **i32)
        self.counts = torch.empty(3, **i32)                      # groups, M tiles, tasks (device only)
        _lib.check(lib.spk_ent2rel_plan(self.segptr.data_ptr(), self.n_rel, TILES_PER_TASK, self.rel2group.data_ptr(),
                                        self.group_rel.data_ptr(), self.group_tile0.data_ptr(), self.task_ptr.data_ptr(),
                                        self.tile_group.data_ptr(), self.task_row0.data_ptr(), self.task_row1.data_ptr(),
                                        self.counts.data_ptr(), _lib.stream_ptr()), "ent2rel_plan")
        self.pos = torch.empty(n, dtype=torch.int64, device=dev)
        _lib.check(lib.spk_ent2rel_positions(self.keys.data_ptr(), self.vals.data_ptr(), n, self.n_rel,
                                             self.segptr.data_ptr(), self.rel2group.data_ptr(),
                                             self.group_tile0.data_ptr(), self.pos.data_ptr(), _lib.stream_ptr()),
                   "ent2rel_positions")


class PaddedRowsFn(torch.autograd.Function):
    """X[p] = table[ids[j]] at the padded row p = pos[j] of every row j (ids None: table[j]); pad rows are zero.
    Backward: the real rows' gradients back in input order, summed per table row by sorted segments (deterministic)."""

    @staticmethod
    def forward(ctx, table, lay, ids):
        t = table.detach()
        t = t if t.stride(1) == 1 else t.contiguous()
        width = t.shape[1]
        out = torch.empty(lay.max_rows, _ld4(width), dtype=torch.float32, device=t.device)[:, :width]
        _lib.check(_lib.load().spk_ent2rel_gather(_lib.ptr(t), t.stride(0), t.shape[0], _lib.ptr(ids), lay.vals.data_ptr(),
                                                  lay.segptr.data_ptr(), lay.group_rel.data_ptr(),
                                                  lay.group_tile0.data_ptr(), lay.tile_group.data_ptr(),
                                                  lay.counts.data_ptr(), width, lay.max_rows, out.data_ptr(),
                                                  out.stride(0), lay.err.data_ptr(), _lib.stream_ptr()), "ent2rel_gather")
        ctx.lay, ctx.ids, ctx.n_table = lay, ids, t.shape[0]
        return out

    @staticmethod
    def backward(ctx, g):
        lay, ids = ctx.lay, ctx.ids
        g = g if g.stride(1) == 1 else g.contiguous()
        rows = _gather_concat([(g, lay.pos, 1)], lay.n_rows, g.shape[1])
        if ids is None:
            return rows, None, None
        edge = torch.stack((ids, ids), dim=0)
        return SpecialSpmmFunctionFinal.apply(edge, rows, ctx.n_table, ids.numel(), g.shape[1]), None, None


class GroupedProjectFn(torch.autograd.Function):
    """Y = tanh(X_g . W[r_g]) for every group g of a RelationLayout (X padded, pad rows zero -> Y pad rows zero):
    one grouped tcgen05 GEMM with the tanh epilogue. Backward: dZ = dY (1 - Y^2); dX_g = dZ_g . W[r_g]^T (the same
    grouped GEMM reading W untransposed); dW[r] = X_g^T dZ_g as (relation, row chunk) tasks added in task order, exact
    zeros for relations without rows. No host synchronisation and no per-relation launches."""

    @staticmethod
    def forward(ctx, X, W, lay):
        lib = _lib.load()
        w = W.detach()
        w = w if w.is_contiguous() else w.contiguous()
        n_rel, k, n = w.shape
        assert X.shape == (lay.max_rows, k) and X.stride(1) == 1 and n_rel == lay.n_rel
        Y = torch.empty(lay.max_rows, _ld4(n), dtype=torch.float32, device=X.device)[:, :n]
        ws = torch.empty(lib.spk_gemm_nn_tc_grouped_workspace_floats(lay.max_groups, n, k), dtype=torch.float32,
                         device=X.device)
        _lib.check(lib.spk_gemm_nn_tc_grouped(_lib.ptr(X), X.stride(0), lay.max_rows, _lib.ptr(w), k * n, 1, n, n, k,
                                              lay.group_rel.data_ptr(), lay.counts.data_ptr(), lay.max_groups,
                                              lay.tile_group.data_ptr(), Y.data_ptr(), Y.stride(0), 2, ws.data_ptr(),
                                              _lib.stream_ptr()), "gemm_nn_tc_grouped")
        ctx.save_for_backward(X, w, Y)
        ctx.lay = lay
        return Y

    @staticmethod
    def backward(ctx, dY):
        lib = _lib.load()
        X, w, Y = ctx.saved_tensors
        lay = ctx.lay
        n_rel, k, n = w.shape
        dev = X.device
        dY = dY if dY.stride(1) == 1 else dY.contiguous()
        dZ = torch.empty(lay.max_rows, _ld4(n), dtype=torch.float32, device=dev)[:, :n]
        _lib.check(lib.spk_tanh_bwd(Y.data_ptr(), Y.stride(0), dY.data_ptr(), dY.stride(0), lay.max_rows, n,
                                    dZ.data_ptr(), dZ.stride(0), _lib.stream_ptr()), "tanh_bwd")
        dX = dW = None
        if ctx.needs_input_grad[0]:
            dX = torch.empty(lay.max_rows, _ld4(k), dtype=torch.float32, device=dev)[:, :k]
            ws = torch.empty(lib.spk_gemm_nn_tc_grouped_workspace_floats(lay.max_groups, k, n), dtype=torch.float32,
                             device=dev)
            _lib.check(lib.spk_gemm_nn_tc_grouped(dZ.data_ptr(), dZ.stride(0), lay.max_rows, w.data_ptr(), k * n, n, 1, k,
                                                  n, lay.group_rel.data_ptr(), lay.counts.data_ptr(), lay.max_groups,
                                                  lay.tile_group.data_ptr(), dX.data_ptr(), dX.stride(0), 0,
                                                  ws.data_ptr(), _lib.stream_ptr()), "gemm_nn_tc_grouped")
        if ctx.needs_input_grad[1]:
            dW = torch.empty(n_rel, k, n, dtype=torch.float32, device=dev)
            ws = torch.empty(max(1, lib.spk_gemm_tn_tc_grouped_workspace_floats(lay.max_tasks, k, n)),
                             dtype=torch.float32, device=dev)
            _lib.check(lib.spk_gemm_tn_tc_grouped(X.data_ptr(), X.stride(0), dZ.data_ptr(), dZ.stride(0), lay.max_rows,
                                                  k, n, lay.task_row0.data_ptr(), lay.task_row1.data_ptr(),
                                                  lay.counts.data_ptr(), lay.max_tasks, lay.rel2group.data_ptr(),
                                                  lay.task_ptr.data_ptr(), n_rel, dW.data_ptr(), ws.data_ptr(),
                                                  _lib.stream_ptr()), "gemm_tn_tc_grouped")
        return dX, dW, None


def ent2rel_project(rows, w_ent2rel, rel_ids):
    """tanh(rows[b] . W_ent2rel[rel_ids[b]]) (GAT_sep_space/models.py:316-320): rows grouped by relation on the device
    (RelationLayout), one grouped tensor-core GEMM for all relations, results back in input order."""
    rel_ids = rel_ids.to(device=rows.device, dtype=torch.int64).contiguous()
    n = rel_ids.numel()
    if n == 0:
        return rows.new_empty(0, w_ent2rel.shape[2])
    lay = RelationLayout(rel_ids, n, 1, 1, w_ent2rel.shape[0])
    y = GroupedProjectFn.apply(PaddedRowsFn.apply(rows, lay, None), w_ent2rel, lay)
    out = GatherRowsFn.apply(y, lay.pos)
    if int(lay.err.item()):
        raise IndexError("relation id out of range for W_ent2rel")
    return out


class ConvKB(nn.Module):
    """GAT/layers.py:12-48 with the same parameters; forward = fc2(LeakyReLU(fc1(conv_input))) on the library kernels."""

    def __init__(self, input_dim, input_seq_len, in_channels, out_channels, drop_prob, alpha_leaky):
        super().__init__()
        self.conv_layer = nn.Conv2d(in_channels, out_channels, (1, input_seq_len))
        self.dropout = nn.Dropout(drop_prob)
        self.non_linearity = nn.LeakyReLU()
        self.fc_layer = nn.Linear(input_dim * out_channels, 1)
        self.fc1 = nn.Linear(input_dim * 3, input_dim)
        self.nl1 = nn.LeakyReLU()
        self.fc2 = nn.Linear(input_dim, 1)
        nn.init.xavier_uniform_(self.fc_layer.weight, gain=1.414)
        nn.init.xavier_uniform_(self.conv_layer.weight, gain=1.414)

    def forward(self, conv_input):
        if not conv_input.is_cuda:
            raise RuntimeError("recon_b200.ConvKB needs CUDA tensors (no CPU fallback)")
        with torch.cuda.device(conv_input.device):
            h1 = SF.matmul(conv_input, self.fc1.weight.t())                       # layers.py:44 (bias folded into the head)
            return MLPHeadFn.apply(h1, self.fc1.bias, self.fc2.weight, self.fc2.bias)   # layers.py:44-45


class SpKBGATConvOnly(nn.Module):
    """GAT/models.py:242-304 (and its GAT_sep_space variant when `model_gat` is passed): same constructor, parameters
    (final_entity_embeddings, final_relation_embeddings, convKB.*) and forward / batch_test signatures."""

    def __init__(self, initial_entity_emb, initial_relation_emb, entity_out_dim, relation_out_dim,
                 drop_GAT, drop_conv, alpha, alpha_conv, nheads_GAT, conv_out_channels):
        super().__init__()
        self.num_nodes = initial_entity_emb.shape[0]
        self.entity_in_dim = initial_entity_emb.shape[1]
        self.entity_out_dim_1 = entity_out_dim[0]
        self.nheads_GAT_1 = nheads_GAT[0]
        self.entity_out_dim_2 = entity_out_dim[1]
        self.nheads_GAT_2 = nheads_GAT[1]
        self.num_relation = initial_relation_emb.shape[0]
        self.relation_dim = initial_relation_emb.shape[1]
        self.relation_out_dim_1 = relation_out_dim[0]
        self.drop_GAT = drop_GAT
        self.drop_conv = drop_conv
        self.alpha = alpha
        self.alpha_conv = alpha_conv
        self.conv_out_channels = conv_out_channels
        hd = self.entity_out_dim_1 * self.nheads_GAT_1
        self.final_entity_embeddings = nn.Parameter(torch.randn(self.num_nodes, hd))
        self.final_relation_embeddings = nn.Parameter(torch.randn(self.num_relation, hd))
        self.convKB = ConvKB(hd, 3, 1, self.conv_out_channels, self.drop_conv, self.alpha_conv)

    def _conv_input(self, batch_inputs, model_gat):
        ent, rel = self.final_entity_embeddings, self.final_relation_embeddings
        tri = torch.as_tensor(batch_inputs).to(device=ent.device, dtype=torch.int64).contiguous()
        if tri.dim() != 2 or tri.shape[1] != 3:
            raise ValueError("batch_inputs must be [B, 3] (head, relation, tail)")
        d = ent.shape[1]
        grads = torch.is_grad_enabled() and (ent.requires_grad or rel.requires_grad)
        if model_gat is None and not grads:
            # one gather kernel writes [E[h] | Rel[r] | E[t]] (models.py:295-296); the embeddings are frozen during ConvKB
            # training (GAT/main.py:741-742), which is the case this fast path serves
            return _gather_concat([(ent.detach(), tri[:, 0], 3), (rel.detach(), tri[:, 1], 3), (ent.detach(), tri[:, 2], 3)],
                                  tri.shape[0], d)
        h = GatherRowsFn.apply(ent, tri[:, 0].contiguous())
        t = GatherRowsFn.apply(ent, tri[:, 2].contiguous())
        r = GatherRowsFn.apply(rel, tri[:, 1].contiguous())
        if model_gat is not None:                                              # GAT_sep_space/models.py:316-320
            rid = tri[:, 1].contiguous()
            h = ent2rel_project(h, model_gat.W_ent2rel, rid)
            t = ent2rel_project(t, model_gat.W_ent2rel, rid)
        return torch.cat((h, r, t), dim=1)

    def _score(self, batch_inputs, model_gat):
        if not self.final_entity_embeddings.is_cuda:
            raise RuntimeError("recon_b200.SpKBGATConvOnly must live on a CUDA device (no CPU fallback)")
        with torch.cuda.device(self.final_entity_embeddings.device):
            return self.convKB(self._conv_input(batch_inputs, model_gat))

    def forward(self, Corpus_, adj, batch_inputs, model_gat=None):
        return self._score(batch_inputs, model_gat)

    def batch_test(self, batch_inputs, model_gat=None):
        return self._score(batch_inputs, model_gat)


def relation_scores(model_conv, test_triples, num_rels=None, model_gat=None):
    """scores[i, r] = model_conv.batch_test((h_i, r, t_i)) for every relation id r (GAT/create_batch.py:1367-1393, which
    tiles every test triple num_rels times and scores 100 rows per call). Here fc1 is re-associated:
    fc1([e_h | rel_r | e_t]) = (W1a e_h + W1c e_t + b1) + W1b rel_r, so the pair part is one GEMM over the T pairs, the
    relation part one GEMM over the R relations, and the T x R scores one streaming pass. With `model_gat` (sep-space
    variant) the head / tail rows depend on the relation, so each relation is one pass of T-row GEMMs."""
    lib = _lib.load()
    ent, rel = model_conv.final_entity_embeddings.detach(), model_conv.final_relation_embeddings.detach()
    dev = ent.device
    fc1, fc2 = model_conv.convKB.fc1, model_conv.convKB.fc2
    d = ent.shape[1]
    r_all = rel.shape[0] if num_rels is None else int(num_rels)
    tri = torch.as_tensor(test_triples).to(device=dev, dtype=torch.int64).contiguous()
    t_n = tri.shape[0]
    w1 = fc1.weight.detach()                                                # [D, 3D]
    w1a_t, w1b_t, w1c_t = w1[:, :d].t().contiguous(), w1[:, d:2 * d].t().contiguous(), w1[:, 2 * d:].t().contiguous()
    b1, w2, b2 = fc1.bias.detach().contiguous(), fc2.weight.detach().contiguous(), fc2.bias.detach().contiguous()
    scores = torch.empty(t_n, r_all, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev), torch.no_grad():
        if model_gat is None:
            ht = _gather_concat([(ent, tri[:, 0], 3), (ent, tri[:, 2], 3)], t_n, d)           # [T, 2D]
            u = SF.gemm_nn(ht, torch.cat((w1a_t, w1c_t), dim=0))                              # W1a e_h + W1c e_t
            u += b1
            bt = SF.gemm_nn(SF.tc_friendly(rel[:r_all].contiguous()), w1b_t)                  # [R, D]
            _lib.check(lib.spk_rank_scores(_lib.ptr(u), u.stride(0), _lib.ptr(bt), bt.stride(0), _lib.ptr(w2), _lib.ptr(b2),
                                           LRELU_SLOPE, t_n, r_all, d, _lib.ptr(scores), scores.stride(0),
                                           _lib.stream_ptr()), "rank_scores")
        else:
            w = model_gat.W_ent2rel.detach()
            h = SF.tc_friendly(_gather_concat([(ent, tri[:, 0], 3)], t_n, d))
            t = SF.tc_friendly(_gather_concat([(ent, tri[:, 2], 3)], t_n, d))
            col = torch.empty(t_n, 1, dtype=torch.float32, device=dev)
            for r in range(r_all):
                hp = SF.gemm_nn(h, w[r]); tp = SF.gemm_nn(t, w[r])
                for x in (hp, tp):
                    _lib.check(lib.spk_tanh_fwd(_lib.ptr(x), x.stride(0), t_n, d, _lib.stream_ptr()), "tanh_fwd")
                h1 = SF.gemm_nn(hp, w1a_t)
                SF.gemm_nn(tp, w1c_t, out=h1, accumulate=True)
                h1 += rel[r] @ w1b_t                                                         # one row: [D] (host-sized work)
                _lib.check(lib.spk_mlp_head_fwd(_lib.ptr(h1), h1.stride(0), _lib.ptr(b1), _lib.ptr(w2), _lib.ptr(b2),
                                                LRELU_SLOPE, t_n, d, _lib.ptr(col), _lib.stream_ptr()), "mlp_head_fwd")
                scores[:, r] = col[:, 0]
    return scores


def rank_relations(model_conv, test_triples, num_rels=None, model_gat=None):
    """The relation-ranking evaluation of Corpus.get_validation_cnfmat (GAT/create_batch.py:1367-1500): scores of every
    test pair under every relation, sorted descending, then the reference's metrics with its exact bookkeeping
    (predictions per entity pair from the pair's first test row, top max(#actual, 10); ranks looked up in the ordering of
    the last test row, as the reference's loop variable leaves it). Returns (scores, sorted_indices, metrics)."""
    scores = relation_scores(model_conv, test_triples, num_rels, model_gat)
    sorted_indices = torch.sort(scores, dim=-1, descending=True).indices
    tb = torch.as_tensor(test_triples).tolist()
    si = sorted_indices.cpu()
    actual, preds = {}, {}
    for e1, r, e2 in tb:
        actual.setdefault((e1, e2), set()).add(r)
    for i, (e1, _, e2) in enumerate(tb):
        k = (e1, e2)
        if k not in preds:
            preds[k] = set(si[i][:max(len(actual[k]), 10)].tolist())
    last = si[-1].tolist() if tb else []
    pos = {rel: j + 1 for j, rel in enumerate(last)}
    hits, ranks = 0, []
    for k, rels in actual.items():
        hits += len(rels & preds[k])
        ranks.extend(pos[rel] for rel in rels if rel in pos)
    n = max(1, len(ranks))
    metrics = {"hits_at_10": hits, "average_hits_at_10": hits / n, "average_rank": sum(ranks) / n,
               "average_recip_rank": sum(1.0 / x for x in ranks) / n}
    return scores, sorted_indices, metrics

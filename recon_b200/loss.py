"""N1 (SURVEY.md 8f): the training step that follows the hot path in every iteration of the reference.

  * `batch_gat_loss(gat_loss_func, train_indices, entity_embed, relation_embed)` — GAT/main.py:344-376: TransE L1
    distance of the positive and the corrupted triples on the outputs of `SpKBGATModified.forward`,
    `nn.MarginRankingLoss(margin)` with `y = -1`, mean over the `2 * ratio * P` pairs. The reference reads the ratio
    from the global `args.valid_invalid_ratio_gat` (main.py:346); here it is the keyword `valid_invalid_ratio_gat`
    (default 2, main.py:68-69).
  * its backward (the gradient `SpKBGATModified`'s backward consumes) as a deterministic segmented sum over a
    radix-sorted incidence list instead of autograd's `index_put_(accumulate=True)` atomics.
  * with `model_gat=` (the GAT_sep_space variant, GAT_sep_space/main.py:360-377) heads and tails are first projected into
    relation space, tanh(e . W_ent2rel[r]) with each row's own relation: the 2T entity rows are gathered straight into a
    relation-grouped, tile-padded layout, projected by one grouped tcgen05 GEMM (convkb.GroupedProjectFn), and the same
    margin kernels run on the projected table with triples (padded head row, r, padded tail row).
  * `sgd_step(params, lr)` — `torch.optim.SGD(model.parameters(), lr).step()` (main.py:445-446, 524) in one launch.

All arithmetic runs in libspkbgat (`spk_margin_loss_fwd/bwd`, `spk_triple_incidence`, `spk_sort_pairs`,
`spk_sgd_step`); no CPU / PyTorch fallback.
"""
import torch

from . import _lib
from .graph import HubSet, sort_pairs, _segment_ptr, _key_bits


class TripleIncidence:
    """Entity and relation segments of one batch of training triples (int64 [T,3] = head, relation, tail)."""

    def __init__(self, triples, n_ent, n_rel):
        lib = _lib.load()
        dev = triples.device
        t = int(triples.shape[0])
        i32 = dict(dtype=torch.int32, device=dev)
        ek = torch.empty(2 * t, **i32); ev = torch.empty(2 * t, **i32)
        rk = torch.empty(t, **i32); rv = torch.empty(t, **i32)
        err = torch.zeros(1, **i32)
        _lib.check(lib.spk_triple_incidence(_lib.ptr(triples), t, n_ent, n_rel, ek.data_ptr(), ev.data_ptr(),
                                            rk.data_ptr(), rv.data_ptr(), err.data_ptr(), _lib.stream_ptr()),
                   "triple_incidence")
        ek, self.ent_inc = sort_pairs(ek, ev, _key_bits(n_ent))
        rk, self.rel_inc = sort_pairs(rk, rv, _key_bits(n_rel))
        self.ent_ptr = _segment_ptr(ek, n_ent)
        self.rel_ptr = _segment_ptr(rk, n_rel)
        self.ent_hubs = HubSet(self.ent_ptr)
        self.rel_hubs = HubSet(self.rel_ptr)
        # (ids were range-checked by spk_margin_loss_fwd before any backward can run; err stays 0 here)


def _loss_backward(segptr, inc, hubs, coef, sgn, gscale, n_seg, width, mode):
    lib = _lib.load()
    out = torch.empty(n_seg, width, dtype=torch.float32, device=coef.device)
    a = _lib.LossBwdArgs()
    a.segptr = segptr.data_ptr(); a.inc = inc.data_ptr(); a.coef = coef.data_ptr(); a.sgn = sgn.data_ptr()
    a.gscale = gscale.data_ptr(); a.out = out.data_ptr(); a.ldo = out.stride(0)
    a.n_seg = n_seg; a.width = width; a.mode = mode
    ldpart = (width + 3) // 4 * 4
    partial = torch.empty(max(1, hubs.n_tasks), ldpart, dtype=torch.float32, device=coef.device) if hubs.n_tasks else None
    hubs.fill(a.hub, partial, ldpart)
    _lib.check(lib.spk_margin_loss_bwd(a, _lib.stream_ptr()), "margin_loss_bwd")
    return out


class MarginLossFn(torch.autograd.Function):
    """loss = reduce_k clamp_min((||x_pos[k mod P]||_1 - ||x_neg[k]||_1) + margin, 0), x = ent[h] + rel[r] - ent[t]."""

    @staticmethod
    def forward(ctx, entity_embed, relation_embed, train_indices, n_pos, margin, mean):
        lib = _lib.load()
        if not entity_embed.is_cuda:
            raise RuntimeError("recon_b200 ops need CUDA tensors (no CPU fallback)")
        ent = entity_embed.detach()
        rel = relation_embed.detach()
        if ent.stride(1) != 1:
            ent = ent.contiguous()
        if rel.stride(1) != 1:
            rel = rel.contiguous()
        dev = ent.device
        tri = train_indices.to(device=dev, dtype=torch.int64).contiguous()
        t = int(tri.shape[0])
        width = int(ent.shape[1])
        assert rel.shape[1] == width, "entity and relation embeddings must have the same width (main.py:357)"
        w4 = (width + 3) // 4
        norm = torch.empty(t, dtype=torch.float32, device=dev)
        sgn = torch.empty(t, w4, dtype=torch.int32, device=dev)
        coef = torch.empty(t, dtype=torch.float32, device=dev)
        partial = torch.empty(lib.spk_margin_loss_partials(n_pos), dtype=torch.float64, device=dev)
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        err = torch.zeros(1, dtype=torch.int32, device=dev)
        _lib.check(lib.spk_margin_loss_fwd(tri.data_ptr(), t, n_pos, _lib.ptr(ent), ent.stride(0), ent.shape[0],
                                           _lib.ptr(rel), rel.stride(0), rel.shape[0], width, float(margin), int(mean),
                                           norm.data_ptr(), sgn.data_ptr(), coef.data_ptr(), partial.data_ptr(),
                                           loss.data_ptr(), err.data_ptr(), _lib.stream_ptr()), "margin_loss_fwd")
        ctx.tri, ctx.sgn, ctx.coef = tri, sgn, coef
        ctx.shape = (int(ent.shape[0]), int(rel.shape[0]), width)
        ctx.mark_non_differentiable(err)
        return loss.reshape(()), err

    @staticmethod
    def backward(ctx, g, _gerr=None):
        n_ent, n_rel, width = ctx.shape
        inc = TripleIncidence(ctx.tri, n_ent, n_rel)
        gscale = g.detach().to(torch.float32).reshape(1).contiguous()
        d_ent = d_rel = None
        if ctx.needs_input_grad[0]:
            d_ent = _loss_backward(inc.ent_ptr, inc.ent_inc, inc.ent_hubs, ctx.coef, ctx.sgn, gscale, n_ent, width, 0)
        if ctx.needs_input_grad[1]:
            d_rel = _loss_backward(inc.rel_ptr, inc.rel_inc, inc.rel_hubs, ctx.coef, ctx.sgn, gscale, n_rel, width, 1)
        return d_ent, d_rel, None, None, None, None


def _margin_loss_sep(train_indices, entity_embed, relation_embed, w_ent2rel, n_pos, margin, mean):
    """The margin loss of GAT_sep_space/main.py:344-377: x = tanh(e_h W[r]) + rel[r] - tanh(e_t W[r]) per row."""
    from .convkb import RelationLayout, PaddedRowsFn, GroupedProjectFn
    if not (entity_embed.is_cuda and relation_embed.is_cuda and w_ent2rel.is_cuda):
        raise RuntimeError("recon_b200 ops need CUDA tensors (no CPU fallback)")
    dev = entity_embed.device
    with torch.cuda.device(dev):
        tri = train_indices.to(device=dev, dtype=torch.int64).contiguous()
        t = int(tri.shape[0])
        assert w_ent2rel.dim() == 3 and w_ent2rel.shape[1] == entity_embed.shape[1], "W_ent2rel must be [R, HD, HD']"
        lay = RelationLayout(tri[:, 1], t, 2, 3, w_ent2rel.shape[0])     # rows: the T heads, then the T tails
        x = PaddedRowsFn.apply(entity_embed, lay, torch.cat((tri[:, 0], tri[:, 2])))
        y = GroupedProjectFn.apply(x, w_ent2rel, lay)
        syn = torch.stack((lay.pos[:t], tri[:, 1], lay.pos[t:]), dim=1)
        loss, err = MarginLossFn.apply(y, relation_embed, syn, n_pos, margin, mean)
        return loss, err | lay.err


def batch_gat_loss(gat_loss_func, train_indices, entity_embed, relation_embed, valid_invalid_ratio_gat=2, *,
                   model_gat=None):
    """Drop-in for GAT/main.py:344-376. `gat_loss_func` is the reference's `nn.MarginRankingLoss(margin=...)`
    (only its `margin` and `reduction` are read); `train_indices` int64 [T,3], positives first (main.py:348-349).
    `model_gat`: any object with `.W_ent2rel` [R, HD, HD] selects the GAT_sep_space loss (main.py:360-377), whose
    gradient also reaches W_ent2rel (exact zeros for relations without rows)."""
    ratio = int(valid_invalid_ratio_gat)
    t = int(train_indices.shape[0])
    len_pos_triples = int(t / (ratio * 2 + 1))                                    # main.py:345-346
    if len_pos_triples <= 0 or len_pos_triples * (2 * ratio + 1) != t:
        # the reference fails here too: pos_norm [2*ratio*P] and neg_norm [T-P] do not broadcast
        raise RuntimeError(f"batch_gat_loss: {t} triples are not (2*{ratio}+1) x positives")
    margin = float(getattr(gat_loss_func, "margin", gat_loss_func if isinstance(gat_loss_func, (int, float)) else 0.0))
    reduction = getattr(gat_loss_func, "reduction", "mean")
    if reduction not in ("mean", "sum"):
        raise NotImplementedError("batch_gat_loss: reduction must be 'mean' (the reference's) or 'sum'")
    if model_gat is not None:
        loss, err = _margin_loss_sep(train_indices, entity_embed, relation_embed, model_gat.W_ent2rel, len_pos_triples,
                                     margin, reduction == "mean")
    else:
        loss, err = MarginLossFn.apply(entity_embed, relation_embed, train_indices, len_pos_triples, margin,
                                       reduction == "mean")
    if int(err.item()) != 0:                                                      # the reference's gathers (main.py:353-355)
        raise IndexError("train_indices out of range for the entity / relation embedding tables")
    assert not bool(torch.isnan(loss).any()), "batch_gat_loss: NaN loss"          # main.py:374 (the reference syncs here too)
    return loss


def sgd_step(params, lr):
    """`torch.optim.SGD(params, lr=lr).step()` (no momentum / weight decay, as main.py:445-446): p -= lr * p.grad
    for every parameter that has a gradient, 16 tensors per launch."""
    lib = _lib.load()
    todo = [p for p in params if p.grad is not None and p.numel()]
    for p in todo:
        if not p.is_cuda:
            raise RuntimeError("recon_b200 ops need CUDA tensors (no CPU fallback)")
        if not (p.is_contiguous() and p.dtype == torch.float32 and p.grad.dtype == torch.float32):
            raise RuntimeError("sgd_step needs contiguous fp32 parameters")
    for i in range(0, len(todo), 16):
        chunk = todo[i:i + 16]
        grads = [p.grad if p.grad.is_contiguous() else p.grad.contiguous() for p in chunk]
        a = _lib.SgdArgs()
        for j, (p, g) in enumerate(zip(chunk, grads)):
            a.param[j] = p.data_ptr(); a.grad[j] = g.data_ptr(); a.numel[j] = p.numel()
        a.count = len(chunk); a.lr = float(lr)
        _lib.check(lib.spk_sgd_step(a, _lib.stream_ptr()), "sgd_step")

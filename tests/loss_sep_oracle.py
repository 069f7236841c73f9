"""CPU oracle of the GAT_sep_space TransE loss (GAT_sep_space/main.py:344-377) -- TEST INFRASTRUCTURE, NOT PRODUCT.

The reference tree is not needed to run it: it is the composition of two oracles already pinned to the reference,
oracle.convkb.ent2rel_project (pinned by tests/golden/convkb_sep.npz, written by the reference's own sep-space classes)
and the L1 / margin steps of oracle.loss.batch_gat_loss (pinned by tests/golden/loss_*.npz), written out as one function
so that it can be read against GAT_sep_space/main.py line by line.
"""
import torch

from oracle.convkb import ent2rel_project


def batch_gat_loss_sep(train_indices, entity_embed, relation_embed, w_ent2rel, ratio, margin):
    """GAT_sep_space/main.py:344-377 with args.valid_invalid_ratio_gat = ratio, gat_loss_func = MarginRankingLoss(margin)
    and model_gat.W_ent2rel = w_ent2rel."""
    t = train_indices.shape[0]
    n_pos = int(t / (int(ratio) * 2 + 1))                                  # main.py:345-346
    pos, neg = train_indices[:n_pos], train_indices[n_pos:]                # main.py:348-349
    pos = pos.repeat(int(ratio) * 2, 1)                                    # main.py:351

    def l1(tri):                                                           # main.py:353-365 with the projection
        r = tri[:, 1]                                                      # of main.py:360-377
        src = ent2rel_project(entity_embed[tri[:, 0]], w_ent2rel, r)
        tail = ent2rel_project(entity_embed[tri[:, 2]], w_ent2rel, r)
        x = src + relation_embed[r] - tail
        return x.abs().sum(dim=1)

    pos_norm, neg_norm = l1(pos), l1(neg)
    y = -torch.ones(int(ratio * 2) * n_pos, dtype=pos_norm.dtype)         # main.py:367-370
    loss = torch.clamp_min(-y * (pos_norm - neg_norm) + margin, 0).mean()  # nn.MarginRankingLoss, main.py:372
    assert not torch.isnan(loss).any()                                     # main.py:374
    return loss


def loss_sep_fwd_bwd(train_indices, entity_embed, relation_embed, w_ent2rel, ratio, margin):
    """Returns (loss, d entity_embed, d relation_embed, d W_ent2rel)."""
    ent = entity_embed.detach().clone().requires_grad_(True)
    rel = relation_embed.detach().clone().requires_grad_(True)
    w = w_ent2rel.detach().clone().requires_grad_(True)
    loss = batch_gat_loss_sep(train_indices, ent, rel, w, ratio, margin)
    loss.backward()
    return loss.detach(), ent.grad, rel.grad, w.grad

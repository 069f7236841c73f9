"""Oracle for the GAT_sep_space filtered link-prediction evaluation -- TEST INFRASTRUCTURE, NOT PRODUCT.

In the sep-space variant (GAT_sep_space/models.py:311-339) the head and tail rows of a triple with relation r are
tanh(e . W_ent2rel[r]); the relation row is not projected. Restated twice, on top of oracle/linkpred.py:
  * validation_pred_loop  the reference loop of Corpus.get_validation_pred literally, as oracle.linkpred restates it for the
                          GAT variant, but scoring through oracle.convkb.conv_only_forward_sep (pinned to the reference by
                          tests/golden/convkb_sep.npz) in fp64, with the same stable descending sort;
  * filtered_ranks        vectorised fp64: the rows of relation r are exactly the GAT-variant evaluation with entity table
                          tanh(E W_r), so every distinct relation among the test rows is one oracle.linkpred.filtered_ranks
                          call on that table (one table in memory at a time); near ties are counted as there.
Only tests/ and profiles/ may import this module.
"""
import numpy as np
import torch

from oracle.convkb import conv_only_forward_sep
from oracle.linkpred import filtered_ranks as _gat_filtered_ranks
from oracle.linkpred import metrics


def validation_pred_loop(p, test_triples, known_triples, n_entities, w_ent2rel, unique_entities=None):
    """p: parameter dict of SpKBGATConvOnly, w_ent2rel [R, D, D], both used in fp64. Returns (ranks_head, ranks_tail) as
    int64 numpy arrays [T] (0 = skipped row) and the metrics dict {"head", "tail", "cumulative", "n_evaluated"}."""
    p64 = {k: torch.as_tensor(v).double() for k, v in p.items()}
    w64 = torch.as_tensor(w_ent2rel).double()
    test = np.asarray(test_triples, dtype=np.int64)
    valid_triples_dict = {tuple(int(x) for x in row): 1 for row in np.asarray(known_triples, dtype=np.int64)}
    ue = None if unique_entities is None else set(int(x) for x in unique_entities)
    entity_list = list(range(n_entities))
    ranks_head, ranks_tail = [], []
    out_head = np.zeros(len(test), dtype=np.int64)
    out_tail = np.zeros(len(test), dtype=np.int64)
    for i in range(len(test)):
        if ue is not None and (int(test[i, 0]) not in ue or int(test[i, 2]) not in ue):
            continue
        new_x_batch_head = np.tile(test[i, :], (n_entities, 1))
        new_x_batch_tail = np.tile(test[i, :], (n_entities, 1))
        new_x_batch_head[:, 0] = entity_list
        new_x_batch_tail[:, 2] = entity_list
        last_index_head = [j for j in range(n_entities) if tuple(int(x) for x in new_x_batch_head[j]) in valid_triples_dict]
        last_index_tail = [j for j in range(n_entities) if tuple(int(x) for x in new_x_batch_tail[j]) in valid_triples_dict]
        new_x_batch_head = np.insert(np.delete(new_x_batch_head, last_index_head, axis=0), 0, test[i], axis=0)
        new_x_batch_tail = np.insert(np.delete(new_x_batch_tail, last_index_tail, axis=0), 0, test[i], axis=0)
        for batch, ranks, out in ((new_x_batch_head, ranks_head, out_head), (new_x_batch_tail, ranks_tail, out_tail)):
            with torch.no_grad():
                scores = conv_only_forward_sep(p64, torch.as_tensor(batch), w64).view(-1)
            sorted_indices = torch.sort(scores, dim=-1, descending=True, stable=True).indices
            rank = int(np.where(sorted_indices.numpy() == 0)[0][0]) + 1
            ranks.append(rank)
            out[i] = rank
    head, tail = metrics(ranks_head), metrics(ranks_tail)
    cumulative = {k: (head[k] + tail[k]) / 2 for k in head}
    return out_head, out_tail, {"head": head, "tail": tail, "cumulative": cumulative, "n_evaluated": len(ranks_head)}


def filtered_ranks(p, test_triples, known_triples, n_entities, w_ent2rel, unique_entities=None, device="cpu",
                   chunk_elems=1 << 27, tau_rel=1e-5):
    """Vectorised fp64 sep-space filtered ranks: (ranks_head, ranks_tail, near_head, near_tail), int64 CPU tensors [T]
    (0 for a skipped row), with the near-tie counts of oracle.linkpred.filtered_ranks."""
    dev = torch.device(device)
    ent = torch.as_tensor(p["final_entity_embeddings"]).to(dev, torch.float64)
    w = torch.as_tensor(w_ent2rel).to(dev, torch.float64)
    tri = torch.as_tensor(test_triples).to(torch.int64).reshape(-1, 3).cpu()
    known = torch.as_tensor(known_triples).to(dev, torch.int64).reshape(-1, 3)
    out = [torch.zeros(tri.shape[0], dtype=torch.int64) for _ in range(4)]
    for r in torch.unique(tri[:, 1]).tolist():
        rows = (tri[:, 1] == r).nonzero().flatten()
        p_r = dict(p, final_entity_embeddings=torch.tanh(ent @ w[r]))
        res = _gat_filtered_ranks(p_r, tri[rows].to(dev), known, n_entities, unique_entities, device=dev,
                                  chunk_elems=chunk_elems, tau_rel=tau_rel)
        for o, x in zip(out, res):
            o[rows] = x
    return tuple(out)

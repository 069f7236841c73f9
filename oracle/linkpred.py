"""Oracle for the filtered link-prediction evaluation -- TEST INFRASTRUCTURE, NOT PRODUCT.

Restates Corpus.get_validation_pred (GAT/create_batch.py:905-1199, the GAT variant, SURVEY.md 2.1 row 6) twice:
  * validation_pred_loop  the reference loop literally: np.tile over the N entities, a per-row Python filter against the
                          known set, np.delete, np.insert of the test triple at index 0, scores through
                          oracle.convkb.conv_only_forward in fp64, a descending sort and the position of index 0. The sort
                          is torch.sort(stable=True) (NaN sorts as the largest value), so exact ties with the test triple
                          do not count against it; the reference's unstable CUDA sort may order such ties either way.
  * filtered_ranks        an independent vectorised fp64 form, chunked over candidates, on any device; it also reports
                          per row the kept candidates whose score lies within tau = 1e-5 * max(1, |s_true|) of the true
                          score ("near ties"; tau_rel sets the 1e-5), the only places where an fp32 evaluation may
                          legitimately rank differently.
The per-row scores are oracle.convkb.conv_only_forward, which tests/golden/convkb_*.npz pin to the reference's batch_test.
Only tests/ (and profiles/) may import this module.
"""
import numpy as np
import torch

from .convkb import conv_only_forward


def metrics(ranks):
    """The reference's per-side numbers over the rank list in row order, in Python floats (ZeroDivisionError if empty)."""
    n = len(ranks)
    return {"hits_at_100": sum(1 for x in ranks if x <= 100) / n, "hits_at_10": sum(1 for x in ranks if x <= 10) / n,
            "hits_at_3": sum(1 for x in ranks if x <= 3) / n, "hits_at_1": sum(1 for x in ranks if x == 1) / n,
            "mean_rank": sum(ranks) / n, "mean_recip_rank": sum(1.0 / x for x in ranks) / n}


def validation_pred_loop(p, test_triples, known_triples, n_entities, unique_entities=None):
    """p: parameter dict of SpKBGATConvOnly (final_*_embeddings, convKB.fc1.*, convKB.fc2.*), used in fp64.
    Returns (ranks_head, ranks_tail) as int64 numpy arrays [T] (0 = skipped row) and the metrics dict
    {"head", "tail", "cumulative", "n_evaluated"}."""
    p64 = {k: torch.as_tensor(v).double() for k, v in p.items()}
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
        last_index_head, last_index_tail = [], []
        for tmp_index in range(len(new_x_batch_head)):
            temp_triple_head = (int(new_x_batch_head[tmp_index][0]), int(new_x_batch_head[tmp_index][1]),
                                int(new_x_batch_head[tmp_index][2]))
            if temp_triple_head in valid_triples_dict:
                last_index_head.append(tmp_index)
            temp_triple_tail = (int(new_x_batch_tail[tmp_index][0]), int(new_x_batch_tail[tmp_index][1]),
                                int(new_x_batch_tail[tmp_index][2]))
            if temp_triple_tail in valid_triples_dict:
                last_index_tail.append(tmp_index)
        new_x_batch_head = np.delete(new_x_batch_head, last_index_head, axis=0)
        new_x_batch_tail = np.delete(new_x_batch_tail, last_index_tail, axis=0)
        new_x_batch_head = np.insert(new_x_batch_head, 0, test[i], axis=0)
        new_x_batch_tail = np.insert(new_x_batch_tail, 0, test[i], axis=0)
        for batch, ranks, out in ((new_x_batch_head, ranks_head, out_head), (new_x_batch_tail, ranks_tail, out_tail)):
            with torch.no_grad():
                scores = conv_only_forward(p64, torch.as_tensor(batch)).view(-1)
            sorted_indices = torch.sort(scores, dim=-1, descending=True, stable=True).indices
            rank = int(np.where(sorted_indices.numpy() == 0)[0][0]) + 1
            ranks.append(rank)
            out[i] = rank
    head, tail = metrics(ranks_head), metrics(ranks_tail)
    cumulative = {k: (head[k] + tail[k]) / 2 for k in head}
    return out_head, out_tail, {"head": head, "tail": tail, "cumulative": cumulative, "n_evaluated": len(ranks_head)}


def _gt(a, b):
    return (a > b) | (torch.isnan(a) & ~torch.isnan(b))


def filtered_ranks(p, test_triples, known_triples, n_entities, unique_entities=None, device="cpu", chunk_elems=1 << 27,
                   tau_rel=1e-5):
    """Vectorised fp64 filtered ranks. Returns (ranks_head, ranks_tail, near_head, near_tail), int64 CPU tensors [T]
    (rank 0 and near 0 for a skipped row); near counts the kept candidates within tau_rel * max(1, |s_true|)."""
    dev = torch.device(device)
    ent = torch.as_tensor(p["final_entity_embeddings"]).to(dev, torch.float64)
    rel = torch.as_tensor(p["final_relation_embeddings"]).to(dev, torch.float64)
    w1 = torch.as_tensor(p["convKB.fc1.weight"]).to(dev, torch.float64)
    b1 = torch.as_tensor(p["convKB.fc1.bias"]).to(dev, torch.float64)
    w2 = torch.as_tensor(p["convKB.fc2.weight"]).to(dev, torch.float64).reshape(-1)
    b2 = torch.as_tensor(p["convKB.fc2.bias"]).to(dev, torch.float64).reshape(())
    n, d = ent.shape
    n_rel = rel.shape[0]
    a_tab, c_tab = ent @ w1[:, :d].t(), ent @ w1[:, 2 * d:].t()
    bt = rel @ w1[:, d:2 * d].t()
    tri = torch.as_tensor(test_triples).to(dev, torch.int64).reshape(-1, 3)
    t_n = tri.shape[0]
    h, r, t = tri[:, 0], tri[:, 1], tri[:, 2]
    keep = torch.ones(t_n, dtype=torch.bool, device=dev)
    if unique_entities is not None:
        ue = torch.as_tensor(list(unique_entities) if not isinstance(unique_entities, torch.Tensor) else unique_entities)
        ue = ue.to(dev, torch.int64).reshape(-1)
        keep = torch.isin(h, ue) & torch.isin(t, ue)
    kn = torch.as_tensor(known_triples).to(dev, torch.int64).reshape(-1, 3)
    known_keys = torch.unique((kn[:, 0] * n_rel + kn[:, 1]) * n + kn[:, 2])        # sorted, distinct
    out = []
    for side in (0, 1):
        v = (c_tab[t] if side == 0 else a_tab[h]) + bt[r] + b1                    # [T, D]
        x_tab = a_tab if side == 0 else c_tab
        true = h if side == 0 else t
        s_true = torch.nn.functional.leaky_relu(x_tab[true] + v) @ w2 + b2
        tau = tau_rel * torch.clamp(s_true.abs(), min=1.0)
        cnt = torch.zeros(t_n, dtype=torch.int64, device=dev)
        near = torch.zeros(t_n, dtype=torch.int64, device=dev)
        step = max(1, chunk_elems // max(1, t_n * d))
        for c0 in range(0, n, step):
            c = torch.arange(c0, min(n, c0 + step), device=dev)
            s = torch.nn.functional.leaky_relu(x_tab[c].unsqueeze(0) + v.unsqueeze(1)) @ w2 + b2       # [T, chunk]
            if side == 0:
                keys = (c.unsqueeze(0) * n_rel + r.unsqueeze(1)) * n + t.unsqueeze(1)
            else:
                keys = (h.unsqueeze(1) * n_rel + r.unsqueeze(1)) * n + c.unsqueeze(0)
            pos = torch.searchsorted(known_keys, keys).clamp_(max=max(0, known_keys.numel() - 1))
            is_known = (known_keys[pos] == keys) if known_keys.numel() else torch.zeros_like(keys, dtype=torch.bool)
            kept = ~is_known & (c.unsqueeze(0) != true.unsqueeze(1))
            cnt += (kept & _gt(s, s_true.unsqueeze(1))).sum(1)
            near += (kept & ((s - s_true.unsqueeze(1)).abs() <= tau.unsqueeze(1))).sum(1)
        out.append((torch.where(keep, cnt + 1, 0).cpu(), torch.where(keep, near, 0).cpu()))
    return out[0][0], out[1][0], out[0][1], out[1][1]

"""ConvKB link-prediction evaluation on the device: filtered entity ranks, MR, MRR and Hits@k.

  KnownTriples        <- valid_triples_dict            GAT/create_batch.py:82-83 (train + validation + test)
  entity_ranks /      <- Corpus.get_validation_pred    GAT/create_batch.py:905-1199 (SURVEY.md 2.1 row 6)
  rank_entities

For every test row (h, r, t) the reference tiles the triple over all N entities, drops the candidates (c, r, t) resp.
(h, r, c) that are known triples, puts the test triple first, scores the rows with batch_test and takes the position of
row 0 after a descending sort. Here the same rank is a count, computed without the T x N score matrix:
  * one tensor-core GEMM gives [A | C] = E . [W1a^T | W1c^T], and Bt = Rel . W1b^T (the re-association of
    relation_scores), so every candidate score is s_c = b2 + sum_d w2[d] * lrelu(X[c, d] + v_i[d]) with X = A or C;
  * spk_linkpred_count streams all N candidate rows past tiles of pair vectors and counts, per row, the candidates that
    outscore the test triple; spk_linkpred_filter walks each row's range of sorted known-triple keys and takes back the
    known candidates it counted. Both compute a score as the same sequential fp32 chain, so they agree bit for bit.
GAT_sep_space (`model_gat` with a W_ent2rel [R, D, D]): the head and tail rows are projected, tanh(e . W_ent2rel[r]),
so the candidate table depends on the relation. The kept rows are grouped by relation and every group is one pass of
the same kernels against its own table: P_r = tanh(E . W_ent2rel[r]) (one GEMM, tanh in its epilogue), then
AC_r = P_r . [W1a^T | W1c^T] (one GEMM); the relation row is not projected, so Bt is shared. Small groups take the
count kernel's narrow pair tiles.
Ties: rank = 1 + #{kept candidates c != true : s_c > s_true}, where NaN counts as larger than any number (torch.sort's
order). That is the position of the test triple under a STABLE descending sort: an exact tie with the true score does not
count against it. The reference uses an unstable CUDA sort and may place exact ties either way.
Not covered: raw (unfiltered) ranks.
"""
import torch

from . import _lib
from . import functional as SF
from .convkb import LRELU_SLOPE
from .nhop import _stable_order

MAX_WIDTH = 512             # embedding widths spk_linkpred_* accept


def _sorted_keys(tri, n_entities, n_relations, err):
    """Keys (h*R + r)*N + t of int64 [M,3] triples sorted (h, r, t)-lexicographically, as TripleSampler builds its
    valid_keys: stable LSD order over (t, r, h), then spk_triple_keys. Repeated triples keep repeated keys."""
    m = int(tri.shape[0])
    if m:
        order = _stable_order([tri[:, 2].contiguous(), tri[:, 1].contiguous(), tri[:, 0].contiguous()], tri.device)
        tri = tri.index_select(0, order).contiguous()
    keys = torch.empty(m, dtype=torch.int64, device=tri.device)
    _lib.check(_lib.load().spk_triple_keys(_lib.ptr(tri) if m else None, m, n_entities, n_relations, _lib.ptr(keys),
                                           _lib.ptr(err), _lib.stream_ptr()), "triple_keys")
    return keys


class KnownTriples:
    """The filter set of the evaluation (the reference's valid_triples_dict): int [M,3] (head, rel, tail) triples, usually
    train + validation + test; repeats are harmless. Holds two sorted key arrays on the device: `tail_keys` over
    (h, r, t), where the known tails of (h, r, .) form one key range, and `head_keys` over the column-swapped (t, r, h),
    where the known heads of (., r, t) do. Build it once and evaluate every epoch against it."""

    def __init__(self, triples, n_entities, n_relations, device=None):
        lib = _lib.load()                                                  # noqa: F841  (raises if the library is missing)
        tri = torch.as_tensor(triples)
        if device is None:
            device = tri.device if tri.is_cuda else torch.device("cuda", torch.cuda.current_device())
        tri = tri.to(device=device, dtype=torch.int64).reshape(-1, 3).contiguous()
        self.device = torch.device(device)
        self.n_entities, self.n_relations = int(n_entities), int(n_relations)
        err = torch.zeros(1, dtype=torch.int32, device=device)
        with torch.cuda.device(self.device):
            self.tail_keys = _sorted_keys(tri, self.n_entities, self.n_relations, err)
            self.head_keys = _sorted_keys(tri[:, [2, 1, 0]].contiguous(), self.n_entities, self.n_relations, err)
        if tri.shape[0] and int(err.item()):
            raise IndexError("known triples: entity / relation id out of range")

    def __len__(self):
        return int(self.tail_keys.numel())


def _head_weights(model_conv):
    """W_ac = [W1a^T | W1c^T] [D, 2D], Bt = Rel . W1b^T [R, D], b1, w2 of a SpKBGATConvOnly, all on its device."""
    ent, rel = model_conv.final_entity_embeddings.detach(), model_conv.final_relation_embeddings.detach()
    fc1, fc2 = model_conv.convKB.fc1, model_conv.convKB.fc2
    d = ent.shape[1]
    w1 = fc1.weight.detach()                                                # [D, 3D] = [W1a | W1b | W1c]
    w_ac = torch.cat((w1[:, :d].t(), w1[:, 2 * d:].t()), dim=1).contiguous()  # [D, 2D]
    bt = SF.gemm_nn(SF.tc_friendly(rel.contiguous()), w1[:, d:2 * d].t().contiguous())
    return w_ac, bt, fc1.bias.detach().contiguous(), fc2.weight.detach().reshape(-1).contiguous()


def _score_tables(model_conv):
    """AC = [A | C] [N, 2D] (one GEMM), Bt [R, D], b1, w2 of a SpKBGATConvOnly, all on its device."""
    w_ac, bt, b1, w2 = _head_weights(model_conv)
    ac = SF.gemm_nn(SF.tc_friendly(model_conv.final_entity_embeddings.detach().contiguous()), w_ac)
    return ac, bt, b1, w2


def _pair_buffers(t_n, d, dev):
    """Per side (head, tail): pair vectors V [T, D padded to 16 B], s_true, true_id, count."""
    ldv = (d + 3) // 4 * 4
    return [(torch.empty(t_n, ldv, dtype=torch.float32, device=dev), torch.empty(t_n, dtype=torch.float32, device=dev),
             torch.empty(t_n, dtype=torch.int32, device=dev), torch.empty(t_n, dtype=torch.int32, device=dev))
            for _ in range(2)]


def _count_and_filter(lib, ac, bt, b1, w2, d, tri, keep, known, work, err, bufs, lo=0):
    """spk_linkpred_count + spk_linkpred_filter, both sides, for the rows of tri [T, 3] against one candidate table
    AC, into rows lo .. lo + T of the _pair_buffers bufs. work: int64 [>= 3T + 1]. Stream-ordered, no synchronisation."""
    n_ent, n_rel = ac.shape[0], bt.shape[0]
    t_n = int(tri.shape[0])
    for side, keys in ((0, known.head_keys), (1, known.tail_keys)):
        v, s_true, true_id, count = (x[lo:lo + t_n] for x in bufs[side])
        _lib.check(lib.spk_linkpred_count(_lib.ptr(ac), ac.stride(0), n_ent, _lib.ptr(bt), bt.stride(0), n_rel,
                                          _lib.ptr(b1), _lib.ptr(w2), LRELU_SLOPE, d, _lib.ptr(tri), _lib.ptr(keep),
                                          t_n, side, _lib.ptr(v), v.stride(0), _lib.ptr(s_true), _lib.ptr(true_id),
                                          _lib.ptr(count), _lib.ptr(err), _lib.stream_ptr()), "linkpred_count")
        _lib.check(lib.spk_linkpred_filter(_lib.ptr(ac), ac.stride(0), n_ent, n_rel, _lib.ptr(w2), LRELU_SLOPE, d,
                                           _lib.ptr(tri), t_n, side, _lib.ptr(v), v.stride(0), _lib.ptr(s_true),
                                           _lib.ptr(true_id), _lib.ptr(keys) if keys.numel() else None, keys.numel(),
                                           _lib.ptr(work), _lib.ptr(count), _lib.ptr(err), _lib.stream_ptr()),
                   "linkpred_filter")


def _ranks(bufs):
    """(head, tail) int64 ranks of filled _pair_buffers: 1 + count, 0 for a skipped row."""
    return [torch.where(true_id >= 0, count.to(torch.int64) + 1, 0) for _, _, true_id, count in bufs]


def _sep_ranks(lib, model_conv, w_ent2rel, tri, keep, known, err):
    """Ranks (head, tail) of the GAT_sep_space variant, int64 [T] on the device in input order (0: skipped). The kept rows
    are sorted stably by relation; each relation present is one pass of _count_and_filter over its contiguous group
    against AC_r = tanh(E . W_ent2rel[r]) . [W1a^T | W1c^T], built in two reused buffers. One host synchronisation (the
    group sizes and the id check). Raises IndexError for an out-of-range id before any W_ent2rel row is read."""
    ent = model_conv.final_entity_embeddings.detach()
    dev = ent.device
    n_ent, d = ent.shape
    n_rel = w_ent2rel.shape[0]
    t_n = int(tri.shape[0])
    h, r, t = tri[:, 0], tri[:, 1], tri[:, 2]
    bad = ((h < 0) | (h >= n_ent) | (t < 0) | (t >= n_ent) | (r < 0) | (r >= n_rel)).any()
    kept = torch.ones(t_n, dtype=torch.bool, device=dev) if keep is None else keep.bool()
    rk = torch.where(kept & (r >= 0) & (r < n_rel), r, n_rel)               # skipped rows sort last, into no group
    order = torch.sort(rk, stable=True).indices
    counts = torch.bincount(rk, minlength=n_rel + 1)
    host = torch.cat((counts, bad.view(1).to(torch.int64))).cpu()           # synchronisation 1
    if int(host[-1]):
        raise IndexError("test triples: entity / relation id out of range")
    counts = host[:n_rel].tolist()
    n_kept = sum(counts)
    out = [torch.zeros(t_n, dtype=torch.int64, device=dev) for _ in range(2)]
    if n_kept == 0:
        return out
    order = order[:n_kept]
    tri_s = tri.index_select(0, order).contiguous()
    w_ac, bt, b1, w2 = _head_weights(model_conv)
    e_op = SF.tc_friendly(ent.contiguous())
    ldp, ldac = (d + 3) // 4 * 4, (2 * d + 3) // 4 * 4                      # 16 B rows: TMA-stored, TMA-read
    p_buf = torch.empty(n_ent, ldp, dtype=torch.float32, device=dev)[:, :d]
    ac = torch.empty(n_ent, ldac, dtype=torch.float32, device=dev)[:, :2 * d]
    work = torch.empty(3 * max(counts) + 1, dtype=torch.int64, device=dev)
    bufs = _pair_buffers(n_kept, d, dev)
    lo = 0
    for rel_id, c in enumerate(counts):
        if not c:
            continue
        SF.gemm_nn(e_op, w_ent2rel[rel_id], out=p_buf, act=2)                # P_r = tanh(E . W_r)
        SF.gemm_nn(p_buf, w_ac, out=ac)                                     # AC_r = P_r . [W1a^T | W1c^T]
        _count_and_filter(lib, ac, bt, b1, w2, d, tri_s[lo:lo + c], None, known, work, err, bufs, lo)
        lo += c
    for side, rk_s in enumerate(_ranks(bufs)):
        out[side][order] = rk_s
    return out


def entity_ranks(model_conv, test_triples, known, unique_entities=None, model_gat=None):
    """Filtered head and tail ranks of Corpus.get_validation_pred (GAT/create_batch.py:905-1199) for a SpKBGATConvOnly.
    test_triples: int [T,3] (head, rel, tail); known: a KnownTriples or an int [M,3] tensor of the known triples;
    unique_entities (optional): a row whose head or tail is not in it is skipped, as in the reference;
    model_gat (optional): the GAT_sep_space variant, whose W_ent2rel (fp32 [R, D, D] on the model's device) projects the
    head and tail rows as SpKBGATConvOnly.batch_test(..., model_gat) does.
    Returns (ranks_head, ranks_tail), int64 [T] on the host, 0 for a skipped row. One host synchronisation, two with
    model_gat (the relation group sizes are read back before the per-relation passes).
    Ties: see the module docstring (position under a stable descending sort; NaN sorts as the largest score)."""
    w_ent2rel = None
    if model_gat is not None:
        w_ent2rel = getattr(model_gat, "W_ent2rel", None)
        if not isinstance(w_ent2rel, torch.Tensor):
            raise NotImplementedError("entity_ranks: a GAT_sep_space model_gat needs its W_ent2rel tensor "
                                      "(candidates projected by tanh(e . W_ent2rel[r]))")
    ent = model_conv.final_entity_embeddings
    if not ent.is_cuda:
        raise RuntimeError("recon_b200.entity_ranks needs a model on a CUDA device (no CPU fallback)")
    lib = _lib.load()
    dev = ent.device
    n_ent, d = ent.shape
    n_rel = model_conv.final_relation_embeddings.shape[0]
    if w_ent2rel is not None:
        w_ent2rel = w_ent2rel.detach()
        if (w_ent2rel.dtype != torch.float32 or w_ent2rel.device != dev
                or tuple(w_ent2rel.shape) != (n_rel, d, d)):
            raise ValueError(f"model_gat.W_ent2rel must be float32 [{n_rel}, {d}, {d}] on {dev}, got "
                             f"{w_ent2rel.dtype} {tuple(w_ent2rel.shape)} on {w_ent2rel.device}")
        w_ent2rel = w_ent2rel.contiguous()
    if not isinstance(known, KnownTriples):
        known = KnownTriples(known, n_ent, n_rel, device=dev)
    if (known.n_entities, known.n_relations) != (n_ent, n_rel) or known.device != dev:
        raise ValueError("known triples were built for another entity / relation count or device")
    tri = torch.as_tensor(test_triples).to(device=dev, dtype=torch.int64)
    if tri.dim() != 2 or tri.shape[1] != 3:
        raise ValueError("test_triples must be [T, 3] (head, relation, tail)")
    tri = tri.contiguous()
    t_n = int(tri.shape[0])
    if t_n == 0:
        empty = torch.zeros(0, dtype=torch.int64)
        return empty, empty.clone()
    with torch.cuda.device(dev), torch.no_grad():
        keep = None
        if unique_entities is not None:
            ue = unique_entities
            if not isinstance(ue, torch.Tensor):
                ue = torch.as_tensor(list(ue), dtype=torch.int64)
            ue = ue.to(device=dev, dtype=torch.int64).reshape(-1)
            keep = (torch.isin(tri[:, 0], ue) & torch.isin(tri[:, 2], ue)).to(torch.uint8).contiguous()
        err = torch.zeros(1, dtype=torch.int32, device=dev)
        if w_ent2rel is None:
            ac, bt, b1, w2 = _score_tables(model_conv)
            work = torch.empty(3 * t_n + 1, dtype=torch.int64, device=dev)
            bufs = _pair_buffers(t_n, d, dev)
            _count_and_filter(lib, ac, bt, b1, w2, d, tri, keep, known, work, err, bufs)
            ranks = _ranks(bufs)
        else:
            ranks = _sep_ranks(lib, model_conv, w_ent2rel, tri, keep, known, err)
        host = torch.cat((ranks[0], ranks[1], err.to(torch.int64))).cpu()          # the (last) synchronisation
    if int(host[-1]):
        raise IndexError("test triples: entity / relation id out of range")
    return host[:t_n].clone(), host[t_n:2 * t_n].clone()


def ranking_metrics(ranks):
    """Hits@100/10/3/1, mean rank and mean reciprocal rank of a list of ranks, summed in list order in Python floats
    (GAT/create_batch.py:1150-1199). An empty list raises ZeroDivisionError, as the reference does."""
    n = len(ranks)
    return {"hits_at_100": sum(1 for x in ranks if x <= 100) / n, "hits_at_10": sum(1 for x in ranks if x <= 10) / n,
            "hits_at_3": sum(1 for x in ranks if x <= 3) / n, "hits_at_1": sum(1 for x in ranks if x == 1) / n,
            "mean_rank": sum(ranks) / n, "mean_recip_rank": sum(1.0 / x for x in ranks) / n}


def rank_entities(model_conv, test_triples, known, unique_entities=None, model_gat=None):
    """The evaluation of Corpus.get_validation_pred: entity_ranks plus the reference's metrics per side, and their
    average ("cumulative"; the reference's one-iteration outer loop makes its averaged numbers these same values).
    Returns (ranks_head, ranks_tail, metrics) with metrics = {"head": {...}, "tail": {...}, "cumulative": {...},
    "n_evaluated": n}. Raises ZeroDivisionError when no row is evaluated."""
    rh, rt = entity_ranks(model_conv, test_triples, known, unique_entities, model_gat)
    head = ranking_metrics([x for x in rh.tolist() if x > 0])
    tail = ranking_metrics([x for x in rt.tolist() if x > 0])
    cumulative = {k: (head[k] + tail[k]) / 2 for k in head}
    return rh, rt, {"head": head, "tail": tail, "cumulative": cumulative, "n_evaluated": int((rh > 0).sum())}

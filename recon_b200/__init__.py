"""recon_b200 -- B200-native (sm_100a) implementation of RECON's KBGAT sparse triple-attention hot path.

Drop-in for the reference's `GAT/layers.py` + `GAT/models.py` module surface:
    from recon_b200 import SpKBGATModified, SpGAT, SpGraphAttentionLayer, SpecialSpmmFunctionFinal, ConvKB
The steps right after the hot path (SURVEY.md 8f) live in `recon_b200.loss` (batch_gat_loss, sgd_step),
`recon_b200.export` (save_embed, load_embed, save_model, save_ent2rel), `recon_b200.sampler` (TripleSampler) and
`recon_b200.convkb` (ConvKB, SpKBGATConvOnly, the W_ent2rel projection and the relation-ranking evaluation) and
`recon_b200.linkpred` (KnownTriples, entity_ranks, rank_entities: the filtered link-prediction evaluation).
All compute runs in libspkbgat.so (hand-written CUDA behind the C ABI of include/spkbgat.h);
there is no CPU or PyTorch-eager fallback.
"""
from .graph import KGraph, triples_to_adj                                                   # noqa: F401
from .layers import (SpecialSpmmFunctionFinal, SpecialSpmmFinal,           # noqa: F401
                     SpGraphAttentionLayer, ConvKB)
from .models import SpGAT, SpKBGATModified                                  # noqa: F401
from .convkb import SpKBGATConvOnly, ent2rel_project, relation_scores, rank_relations   # noqa: F401
from .linkpred import KnownTriples, entity_ranks, rank_entities                          # noqa: F401

__all__ = ["KGraph", "triples_to_adj", "SpecialSpmmFunctionFinal", "SpecialSpmmFinal", "SpGraphAttentionLayer", "ConvKB",
           "SpGAT", "SpKBGATModified", "SpKBGATConvOnly", "ent2rel_project", "relation_scores", "rank_relations",
           "KnownTriples", "entity_ranks", "rank_entities"]

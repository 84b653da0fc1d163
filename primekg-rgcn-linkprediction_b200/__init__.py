"""B200-native (sm_100a) RGCN message-passing hot path for PrimeKG link prediction.

A from-scratch implementation of the one hot path of arnold117/PrimeKG-RGCN-LinkPrediction
(reference src/models/rgcn.py): hand-written CUDA kernels behind a C ABI
(``include/rgcn_b200.h`` -> ``csrc/librgcn_b200.so``), bound with ctypes, behind the reference's own
``nn.Module`` API.  No CPU fallback: see ``oracle/`` for the CPU restatement used by the tests.
"""
from .conv import RGCNConv, default_mode
from .graph import RelGraph, clear_graph_cache, get_graph, graph_from_state, graph_state, register_graph
from .graphed import GraphedTrainStep
from .rank import KnownTriples, rank_true_tails, ranking_metrics, score_all_pairs, topk_all_pairs
from .modules import DrugDiseaseModel, DrugDiseaseRGCN, LinkPredictor
from .sampler import NegativeSampler, RelationConstraints
from .optim import FusedAdam, FusedAdamW

__all__ = ["RGCNConv", "DrugDiseaseRGCN", "LinkPredictor", "DrugDiseaseModel", "RelGraph", "get_graph",
           "clear_graph_cache", "default_mode", "GraphedTrainStep", "graph_state", "graph_from_state", "register_graph", "KnownTriples", "rank_true_tails", "ranking_metrics", "score_all_pairs", "topk_all_pairs",
           "NegativeSampler", "RelationConstraints", "FusedAdam", "FusedAdamW"]
__version__ = "0.1.0"

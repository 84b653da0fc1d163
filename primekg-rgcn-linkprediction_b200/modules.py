"""The reference's model trio on the sm_100a kernels — same constructor arguments, attribute names,
state-dict keys, method set and error behaviour as reference src/models/rgcn.py:

    DrugDiseaseRGCN  (:21-142)   node_embeddings, conv1, conv2, dropout
    LinkPredictor    (:145-243)  relation_embeddings, dropout
    DrugDiseaseModel (:246-415)  encoder, decoder; forward / predict / predict_all_tails / get_embeddings

so that src/train.py, src/evaluate.py and the analysis scripts of the reference run unchanged on top
(`from models.rgcn import DrugDiseaseModel`).  State-dict keys: encoder.node_embeddings.weight,
encoder.conv{1,2}.{weight,[comp],root,bias}, decoder.relation_embeddings.weight — 2,078,208
parameters at the defaults (reference results/results.json:29).
"""
from __future__ import annotations

import os
from typing import Optional

import torch
import torch.nn as nn

from . import autograph
from . import ops
from . import rowsparse
from .conv import RGCNConv
from .graph import get_graph


def sparse_forward_enabled() -> bool:
    """Listed-rows forward of the last layer in ``DrugDiseaseModel``'s training call (it needs the row-sparse backward)."""
    return os.environ.get("PRIMEKG_RGCN_SPARSE_FWD", "1") != "0" and rowsparse.enabled()


def _need_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"{what}: this is the B200 (sm_100a) implementation and has no CPU path; "
                           "move the model and its inputs to a CUDA device")


class DrugDiseaseRGCN(nn.Module):
    """RGCN encoder: Embedding(N, d_e) -> RGCNConv -> ReLU -> Dropout -> RGCNConv (reference :51-130).
    ``num_layers`` > 2 appends further ReLU/Dropout/RGCNConv(hidden, hidden) stages (the extension
    pattern of reference guide/MODEL_ARCHITECTURE.md:245-249; used by the 3-layer 10 M-node config)."""

    def __init__(self, num_nodes: int, num_relations: int, embedding_dim: int = 64, hidden_dim: int = 128,
                 dropout: float = 0.5, num_bases: Optional[int] = None, num_layers: int = 2,
                 num_blocks: Optional[int] = None, aggr: str = "mean"):
        super().__init__()
        self.num_nodes = num_nodes
        self.num_relations = num_relations
        self.embedding_dim = embedding_dim
        self.hidden_dim = hidden_dim
        # construction order = the reference's, so a seeded init draws the same random stream
        self.node_embeddings = nn.Embedding(num_nodes, embedding_dim)
        dec = dict(num_bases=num_bases, num_blocks=num_blocks, aggr=aggr)       # aggr: every layer's aggregation
        self.conv1 = RGCNConv(embedding_dim, hidden_dim, num_relations, **dec)
        self.conv2 = RGCNConv(hidden_dim, hidden_dim, num_relations, **dec)
        if num_layers > 2:
            self.extra_convs = nn.ModuleList(
                RGCNConv(hidden_dim, hidden_dim, num_relations, **dec) for _ in range(num_layers - 2))
        self.dropout = nn.Dropout(dropout)
        self._eval_cache = None
        self._register_load_state_dict_pre_hook(self._drop_cache_on_load)
        self._init_embeddings()

    def _init_embeddings(self) -> None:
        nn.init.xavier_uniform_(self.node_embeddings.weight)

    def _eval_key(self):
        """Identity of an eval-mode encoding besides the graph object: every parameter's storage + in-place version
        (optimizer steps, ``load_state_dict`` and ``.to()`` all change one of them).  Writes that bypass the version
        counter (``p.data`` tricks, raw-pointer or graph-replayed updates) are covered by the cache's LIFETIME instead:
        it is dropped by every ``train()`` <-> ``eval()`` switch, ``.to()`` / ``_apply``, ``load_state_dict`` and
        ``invalidate_eval_cache()``, so it only ever spans one evaluation phase."""
        ps = tuple((p.data_ptr(), p._version, str(p.device)) for p in self.parameters())
        modes = tuple(c.mode for c in self._layers())
        return (ps, modes, os.environ.get("PRIMEKG_RGCN_MODE", ""), os.environ.get("PRIMEKG_RGCN_BASIS_FORM", ""))

    def invalidate_eval_cache(self) -> None:
        """Forget the cached eval-mode encoding (call after changing parameters behind autograd's back)."""
        self._eval_cache = None

    def train(self, mode: bool = True):
        if bool(mode) != self.training:          # a real switch (the reference's predict / get_embeddings call eval() on
            self._eval_cache = None              # every use): also frees the [N, hidden] tensor for the training epochs
        return super().train(mode)

    def _apply(self, fn, *args, **kwargs):
        self._eval_cache = None
        return super()._apply(fn, *args, **kwargs)

    def _drop_cache_on_load(self, *args, **kwargs) -> None:
        # (a pre-hook, not a load_state_dict override: a PARENT's load_state_dict reaches this module through
        # _load_from_state_dict, which runs the hook)
        self._eval_cache = None

    def _layers(self):
        yield self.conv1
        yield self.conv2
        if hasattr(self, "extra_convs"):
            yield from self.extra_convs

    def forward(self, edge_index: torch.Tensor, edge_type: torch.Tensor,
                node_indices: Optional[torch.Tensor] = None) -> torch.Tensor:
        return self._encode(edge_index, edge_type, node_indices)

    def _encode(self, edge_index, edge_type, node_indices=None, read_rows=None) -> torch.Tensor:
        """``read_rows`` = (head, tail): the caller — ``DrugDiseaseModel``'s training call — reads ONLY these rows of the
        result (``node_embeddings[head]``, ``[tail]``, reference :325-326).  The last layer then walks and transforms the
        listed rows alone (``PRIMEKG_RGCN_SPARSE_FWD=0`` or ``PRIMEKG_RGCN_SPARSE_BWD=0``: all rows); every other row of
        the returned matrix is UNDEFINED, which is why only the model's own forward uses this form."""
        x = self.node_embeddings.weight if node_indices is None else self.node_embeddings(node_indices)
        _need_cuda(x, "DrugDiseaseRGCN.forward")
        graph = get_graph(edge_index, edge_type, x.size(0), self.num_relations)
        # The reference's ranking evaluation re-encodes the full graph for every batch of test edges with unchanged
        # weights (src/evaluate.py:251-254: 16 identical passes per evaluation).  In eval mode without autograd the
        # result is a pure function of (graph, parameters): keep the last one and hand it back while neither changed.
        cacheable = not self.training and not torch.is_grad_enabled() and node_indices is None
        if cacheable:
            key = self._eval_key()
            hit = self._eval_cache          # (key, graph — a strong reference, so its id can never be recycled —, x, version)
            if hit is not None and hit[1] is graph and hit[0] == key and hit[2]._version == hit[3]:
                return hit[2]
        layers = list(self._layers())
        listed = None
        if read_rows is not None and not cacheable and node_indices is None and sparse_forward_enabled():
            head, tail = read_rows
            if 0 < 2 * head.numel() <= rowsparse.MAX_FRACTION * x.size(0) and head.numel() == tail.numel():
                listed = ops.rows_list_build(head, tail, x.size(0))
        in_scale = None         # 1 / (1 - p) of the fused ReLU / dropout that produced x (None: x is not such an output)
        for li, conv in enumerate(layers):
            last = li == len(layers) - 1
            # ReLU and (in training) dropout live in the layer's GEMM epilogue; p == 1 keeps nn.Dropout's all-zero output
            p = self.dropout.p if (self.training and not last) else 0.0
            x = conv.forward_graph(x, graph, relu=not last, dropout_p=p if p < 1.0 else 0.0, in_mask_scale=in_scale,
                                   listed=listed if last else None)
            in_scale = 1.0 / (1.0 - p) if (not last and p < 1.0) else None
            if not last and p >= 1.0:
                x = self.dropout(x)
        if cacheable:
            self._eval_cache = (key, graph, x, x._version)
        return x

    def get_node_embeddings(self, node_indices: torch.Tensor) -> torch.Tensor:
        return self.node_embeddings(node_indices)


class _DistMultGather(torch.autograd.Function):
    """score[p] = <emb[head[p]], r_p, emb[tail[p]]> with the row gathers fused into the kernel."""

    @staticmethod
    def forward(ctx, emb, head, tail, rel, rel_table, rel_rows, rel_scale):
        ctx.save_for_backward(emb, head, tail, rel, rel_table, rel_rows, rel_scale)
        return ops.distmult_fwd(emb, emb, head, tail, rel, rel_table, rel_rows, rel_scale)

    @staticmethod
    def backward(ctx, g):
        emb, head, tail, rel, rel_table, rel_rows, rel_scale = ctx.saved_tensors
        g_emb, _, g_tab, g_rows = ops.distmult_bwd(emb, emb, head, tail, rel, rel_table, rel_rows, g,
                                                   ctx.needs_input_grad[4], rel_scale)
        if not ctx.needs_input_grad[0]:
            return None, None, None, None, g_tab, g_rows, None
        # g_emb is zero outside the head / tail rows: tell the last encoder layer (rowsparse.py)
        rowsparse.announce(g_emb, torch.cat([head.reshape(-1), tail.reshape(-1)]).to(torch.int64))
        return g_emb, None, None, None, g_tab, g_rows, None


class _DistMultRows(torch.autograd.Function):
    """score[p] = <head_emb[p], r_p, tail_emb[p]> on rows the caller already gathered."""

    @staticmethod
    def forward(ctx, head_emb, tail_emb, rel, rel_table, rel_rows, rel_scale):
        ctx.save_for_backward(head_emb, tail_emb, rel, rel_table, rel_rows, rel_scale)
        return ops.distmult_fwd(head_emb, tail_emb, None, None, rel, rel_table, rel_rows, rel_scale)

    @staticmethod
    def backward(ctx, g):
        head_emb, tail_emb, rel, rel_table, rel_rows, rel_scale = ctx.saved_tensors
        g_h, g_t, g_tab, g_rows = ops.distmult_bwd(head_emb, tail_emb, None, None, rel, rel_table, rel_rows, g,
                                                   ctx.needs_input_grad[3], rel_scale)
        return g_h, g_t, None, g_tab, g_rows, None


class LinkPredictor(nn.Module):
    """DistMult decoder (reference :165-243): score(h, r, t) = sum_k h_k r_k t_k."""

    def __init__(self, num_relations: int, embedding_dim: int, dropout: float = 0.0):
        super().__init__()
        self.num_relations = num_relations
        self.embedding_dim = embedding_dim
        self.relation_embeddings = nn.Embedding(num_relations, embedding_dim)
        self.dropout = nn.Dropout(dropout)
        self._init_embeddings()

    def _init_embeddings(self) -> None:
        nn.init.xavier_uniform_(self.relation_embeddings.weight)

    def _relation_operand(self, relation_types):
        """(rel_table, rel_scale).  The kernel gathers relation rows from the table itself; when dropout is
        active (reference :207-208) the per-pair mask / (1 - p) is drawn from torch's generator, as
        nn.Dropout does, and applied inside the kernel."""
        table = self.relation_embeddings.weight
        p = self.dropout.p
        if self.training and p > 0:
            if p >= 1:
                return table, torch.zeros(relation_types.numel(), table.size(1), device=table.device)
            scale = torch.empty(relation_types.numel(), table.size(1), device=table.device).bernoulli_(1 - p)
            return table, scale.div_(1 - p)
        return table, None

    def forward(self, head_embeddings: torch.Tensor, tail_embeddings: torch.Tensor,
                relation_types: torch.Tensor) -> torch.Tensor:
        _need_cuda(head_embeddings, "LinkPredictor.forward")
        table, scale = self._relation_operand(relation_types)
        return _DistMultRows.apply(head_embeddings, tail_embeddings, relation_types, table, None, scale)

    def score_pairs(self, node_embeddings: torch.Tensor, head_indices: torch.Tensor, tail_indices: torch.Tensor,
                    relation_types: torch.Tensor) -> torch.Tensor:
        """Fused form of ``forward(emb[head], emb[tail], rel)`` (reference :325-329)."""
        _need_cuda(node_embeddings, "LinkPredictor.score_pairs")
        p = self.dropout.p if self.training else 0.0
        if p >= 1.0:
            table, scale = self._relation_operand(relation_types)
            return _DistMultGather.apply(node_embeddings, head_indices, tail_indices, relation_types, table, None, scale)
        # the fused kernels' scores-only form: relation dropout by counter-based mask (no mask tensor, no extra launches)
        seed, ctr = self._dropout_rng(node_embeddings.device) if p > 0 else (0, None)
        return ops.pair_scores(node_embeddings, self.relation_embeddings.weight, head_indices, tail_indices,
                               relation_types, p, seed, ctr)

    def score_all_tails(self, head_embeddings: torch.Tensor, relation_types: torch.Tensor,
                        all_tail_embeddings: torch.Tensor) -> torch.Tensor:
        """(h * r) @ T^T -> [batch, num_entities] (reference :234-241; no dropout here, as there)."""
        _need_cuda(head_embeddings, "LinkPredictor.score_all_tails")
        return _ScoreAllTails.apply(head_embeddings, self.relation_embeddings.weight, relation_types,
                                    all_tail_embeddings)

    def _dropout_rng(self, device):
        """(seed, device counter) of the fused loss's relation dropout; the seed comes from torch's generator on first use."""
        st = getattr(self, "_drop_rng", None)
        if st is None or st[1].device != device:
            st = self._drop_rng = (int(torch.randint(0, 2 ** 31 - 1, (1,)).item()), ops.rng_counter(device))
        return st

    def link_loss(self, node_embeddings: torch.Tensor, head_indices: torch.Tensor, tail_indices: torch.Tensor,
                  relation_types: torch.Tensor, labels: torch.Tensor):
        """(loss, scores, n_correct): ``score_pairs`` + ``BCEWithLogitsLoss`` + the sigmoid > 0.5 accuracy count of the
        reference's training step (src/train.py:291-300, :321-322) in one kernel pair; both extra outputs are device
        tensors, so a caller can log them without the two ``.item()`` syncs per step."""
        _need_cuda(node_embeddings, "LinkPredictor.link_loss")
        p = self.dropout.p if self.training else 0.0
        if p >= 1.0:
            scores = self.score_pairs(node_embeddings, head_indices, tail_indices, relation_types)
            loss, correct = ops.bce_with_logits(scores, labels, with_accuracy=True)
            return loss, scores, correct
        seed, ctr = self._dropout_rng(node_embeddings.device) if p > 0 else (0, None)
        return ops.link_loss(node_embeddings, self.relation_embeddings.weight, head_indices, tail_indices, relation_types,
                             labels, p, seed, ctr)

    def rank_tails(self, node_embeddings: torch.Tensor, head_indices: torch.Tensor, relation_types: torch.Tensor,
                   tail_indices: torch.Tensor, filter=None):
        """(rank, ties) of the true tails among all entities — the fused form of ``score_all_tails`` + the per-row
        ``argsort`` loop of reference src/evaluate.py:260-276.  ``filter`` (a ``KnownTriples``): filtered ranks, the
        other known tails of each (head, relation) left out."""
        from .rank import rank_true_tails
        return rank_true_tails(node_embeddings, self.relation_embeddings.weight, head_indices, relation_types,
                               tail_indices, filter=filter)


class _ScoreAllTails(torch.autograd.Function):
    """scores = (h * r[rel]) @ T^T through the all-pairs kernel; the (never hot) backward uses three library GEMMs."""

    @staticmethod
    def forward(ctx, h, table, rel, T):
        from .rank import _prep, scores_from_rows
        hr = _prep(h, None, table, rel, False)
        ctx.save_for_backward(h, table, rel, T)
        return scores_from_rows(hr, T)

    @staticmethod
    def backward(ctx, g):
        h, table, rel, T = ctx.saved_tensors
        r = table[rel]
        g_hr = g @ T                                  # [B, d]
        g_h = g_hr * r if ctx.needs_input_grad[0] else None
        g_table = None
        if ctx.needs_input_grad[1]:
            g_table = torch.zeros_like(table).index_add_(0, rel, g_hr * h)
        g_T = g.t() @ (h * r) if ctx.needs_input_grad[3] else None
        return g_h, g_table, None, g_T


class DrugDiseaseModel(nn.Module):
    """Encoder + decoder (reference :267-415)."""

    def __init__(self, num_nodes: int, num_relations: int, embedding_dim: int = 64, hidden_dim: int = 128,
                 dropout: float = 0.5, decoder_dropout: float = 0.0, num_bases: Optional[int] = None,
                 num_layers: int = 2, num_blocks: Optional[int] = None, aggr: str = "mean"):
        super().__init__()
        self.num_nodes = num_nodes
        self.num_relations = num_relations
        self.hidden_dim = hidden_dim
        self.encoder = DrugDiseaseRGCN(num_nodes=num_nodes, num_relations=num_relations,
                                       embedding_dim=embedding_dim, hidden_dim=hidden_dim, dropout=dropout,
                                       num_bases=num_bases, num_layers=num_layers, num_blocks=num_blocks, aggr=aggr)
        self.decoder = LinkPredictor(num_relations=num_relations, embedding_dim=hidden_dim, dropout=decoder_dropout)

    def forward(self, edge_index, edge_type, head_indices, tail_indices, relation_types) -> torch.Tensor:
        # training calls that repeat (same graph tensors, batch size, parameters) replay two captured CUDA graphs —
        # forward, backward — behind this very signature (autograph.py): the reference's loop is bound by the host
        fn = autograph.lookup(self, edge_index, edge_type, head_indices, tail_indices, relation_types)
        if fn is not None:
            return fn(head_indices, tail_indices, relation_types)
        return self._forward_eager(edge_index, edge_type, head_indices, tail_indices, relation_types)

    def _forward_eager(self, edge_index, edge_type, head_indices, tail_indices, relation_types) -> torch.Tensor:
        node_embeddings = self._encode_for(edge_index, edge_type, head_indices, tail_indices)
        return self.decoder.score_pairs(node_embeddings, head_indices, tail_indices, relation_types)

    def _encode_for(self, edge_index, edge_type, head_indices, tail_indices) -> torch.Tensor:
        """Encoder output for a decoder that reads rows ``head`` / ``tail`` only (reference :325-326): with autograd on
        (a training step) the last layer computes just those rows; eval / no-grad calls keep the full, cached matrix."""
        if torch.is_grad_enabled() and head_indices.is_cuda and head_indices.numel() == tail_indices.numel():
            return self.encoder._encode(edge_index, edge_type, None, (head_indices, tail_indices))
        return self.encoder(edge_index, edge_type)

    def invalidate_graphs(self) -> None:
        """Drop the captured training-call graphs (autograph.py), e.g. before freeing the graph tensors."""
        autograph.invalidate(self)

    def link_loss(self, edge_index, edge_type, head_indices, tail_indices, relation_types, labels):
        """Encoder + fused decoder / loss / accuracy: the whole of src/train.py:291-300 and :321-322 -> (loss, scores,
        n_correct), all on the device."""
        node_embeddings = self._encode_for(edge_index, edge_type, head_indices, tail_indices)
        return self.decoder.link_loss(node_embeddings, head_indices, tail_indices, relation_types, labels)

    def predict(self, edge_index, edge_type, head_indices, tail_indices, relation_types) -> torch.Tensor:
        self.eval()
        with torch.no_grad():
            return self.forward(edge_index, edge_type, head_indices, tail_indices, relation_types)

    def predict_all_tails(self, edge_index, edge_type, head_indices, relation_types) -> torch.Tensor:
        self.eval()
        with torch.no_grad():
            emb = self.encoder(edge_index, edge_type)
            return self.decoder.score_all_tails(emb[head_indices], relation_types, emb)

    def get_embeddings(self, edge_index, edge_type) -> torch.Tensor:
        self.eval()
        with torch.no_grad():
            return self.encoder(edge_index, edge_type)

"""CPU oracle of RGCNConv(aggr=, root_weight=, bias=) — TEST INFRASTRUCTURE ONLY.

Restates PyG's loop path as ``oracle/rgcn_ref.py`` does for the mean (parity unpinned: PyG is not installed): per
relation r, ``h_r = aggr_{j in N_r(i)} x_j`` with torch's own ops — ``index_add_`` for the sum (and the mean, divided by
the clamped count), and, for 'max', ``x.new_zeros(..).scatter_reduce_(0, idx, src, 'amax', include_self=False)``, which
is what PyG's ``utils.scatter`` runs without torch-scatter — then ``h_r @ W_r``; after the loop ``x @ root`` if root
exists and ``bias`` if bias exists.  The max oracle's autograd is torch's, ties and the zero initial value included.
Parameter layout and init order are PyG's: weight, comp, root, bias, absent ones registered as None.
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn as nn

from oracle import rgcn_ref as O

ALIASES = {"mean": "mean", "add": "sum", "sum": "sum", "max": "max"}


def aggregate_ref(x: torch.Tensor, src: torch.Tensor, dst: torch.Tensor, n: int, aggr: str) -> torch.Tensor:
    """h[i] = aggr_{e: dst[e] == i} x[src[e]]  (an empty neighbourhood gives 0)."""
    aggr = ALIASES[aggr]
    xj = x.index_select(0, src)
    if aggr == "max":
        return x.new_zeros(n, x.size(1)).scatter_reduce_(0, dst.unsqueeze(1).expand_as(xj), xj, "amax",
                                                          include_self=False)
    s = x.new_zeros(n, x.size(1)).index_add_(0, dst, xj)
    if aggr == "sum":
        return s
    cnt = x.new_zeros(n).index_add_(0, dst, x.new_ones(dst.numel())).clamp_(min=1)
    return s / cnt.unsqueeze(1)


def rgcn_conv_aggr_ref(x, edge_index, edge_type, weight, root: Optional[torch.Tensor], bias: Optional[torch.Tensor],
                       aggr: str = "mean", comp=None) -> torch.Tensor:
    """RGCNConv(aggr=aggr).forward, PyG's loop path; ``weight`` dense [R, in, out] (or bases with ``comp``)."""
    N = x.size(0)
    W = weight if comp is None else (comp @ weight.view(weight.size(0), -1)).view(comp.size(0), weight.size(1),
                                                                                   weight.size(2))
    out = x.new_zeros(N, W.size(2))
    for r in range(W.size(0)):
        m = edge_type == r
        out = out + aggregate_ref(x, edge_index[0][m], edge_index[1][m], N, aggr) @ W[r]
    if root is not None:
        out = out + x @ root
    if bias is not None:
        out = out + bias
    return out


class RGCNConvAggrRef(nn.Module):
    """Parameter layout and init order of PyG's RGCNConv(in, out, R, num_bases, num_blocks, aggr, root_weight,
    is_sorted, bias)."""

    def __init__(self, in_channels, out_channels, num_relations, num_bases=None, num_blocks=None, aggr="mean",
                 root_weight=True, is_sorted=False, bias=True):
        super().__init__()
        self.aggr = aggr
        if num_bases is not None:
            self.weight = nn.Parameter(torch.empty(num_bases, in_channels, out_channels))
            self.comp = nn.Parameter(torch.empty(num_relations, num_bases))
        elif num_blocks is not None:
            self.weight = nn.Parameter(torch.empty(num_relations, num_blocks, in_channels // num_blocks,
                                                   out_channels // num_blocks))
            self.register_parameter("comp", None)
        else:
            self.weight = nn.Parameter(torch.empty(num_relations, in_channels, out_channels))
            self.register_parameter("comp", None)
        if root_weight:
            self.root = nn.Parameter(torch.empty(in_channels, out_channels))
        else:
            self.register_parameter("root", None)
        if bias:
            self.bias = nn.Parameter(torch.empty(out_channels))
        else:
            self.register_parameter("bias", None)
        O.glorot_(self.weight)
        O.glorot_(self.comp)
        O.glorot_(self.root)
        if self.bias is not None:
            with torch.no_grad():
                self.bias.zero_()

    def forward(self, x, edge_index, edge_type):
        if self.weight.dim() == 4:
            from blocks_oracle import expand_blocks
            W = expand_blocks(self.weight)
        else:
            W = self.weight
        return rgcn_conv_aggr_ref(x, edge_index, edge_type, W, self.root, self.bias, self.aggr, self.comp)


class ModelAggrRef(nn.Module):
    """The reference model (Embedding -> conv -> ReLU -> conv, DistMult decoder) with every layer's aggregation set."""

    def __init__(self, num_nodes, num_relations, embedding_dim=64, hidden_dim=128, aggr="mean"):
        super().__init__()
        self.encoder = nn.Module()
        self.encoder.node_embeddings = nn.Embedding(num_nodes, embedding_dim)
        self.encoder.conv1 = RGCNConvAggrRef(embedding_dim, hidden_dim, num_relations, aggr=aggr)
        self.encoder.conv2 = RGCNConvAggrRef(hidden_dim, hidden_dim, num_relations, aggr=aggr)
        self.decoder = O.DecoderRef(num_relations, hidden_dim)

    def forward(self, edge_index, edge_type, heads, tails, rels):
        x = self.encoder.node_embeddings.weight
        x = torch.relu(self.encoder.conv1(x, edge_index, edge_type))
        x = self.encoder.conv2(x, edge_index, edge_type)
        return self.decoder(x[heads], x[tails], rels)

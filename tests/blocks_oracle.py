"""CPU oracle of the block-diagonal relation weights, RGCNConv(num_blocks=nb) — TEST INFRASTRUCTURE ONLY.

Restates PyG's ``rgcn_conv.py`` block path as ``oracle/rgcn_ref.py`` restates its loop path (parity unpinned: PyG is
not installed): per relation r, the per-(destination, relation) mean ``h``, then
``einsum('abc,bcd->abd', h.view(-1, nb, bi), weight[r])`` added as ``[N, out]``; then ``x @ root + bias``.
Parameter layout and init order are PyG's: ``weight [R, nb, in/nb, out/nb]``, ``comp`` = None, ``root``, ``bias``,
glorot with the fans of the last two dims.  The dense formulation ``rgcn_conv_dense_ref`` of the oracle, run on the
expanded block-diagonal matrix (``expand_blocks``), is the independent cross-check.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from oracle import rgcn_ref as O


def expand_blocks(weight: torch.Tensor) -> torch.Tensor:
    """[R, nb, bi, bo] -> [R, nb * bi, nb * bo]: W_r = blockdiag(weight[r, 0], .., weight[r, nb - 1])."""
    return torch.stack([torch.block_diag(*weight[r].unbind(0)) for r in range(weight.size(0))])


def diag_blocks(W: torch.Tensor, nb: int) -> torch.Tensor:
    """Inverse of ``expand_blocks`` on the diagonal: [R, nb * bi, nb * bo] -> [R, nb, bi, bo]."""
    R, d_in, d_out = W.shape
    bi, bo = d_in // nb, d_out // nb
    return torch.stack([W[:, k * bi:(k + 1) * bi, k * bo:(k + 1) * bo] for k in range(nb)], 1)


def rgcn_conv_blocks_ref(x, edge_index, edge_type, weight, root, bias):
    """RGCNConv(num_blocks=nb).forward, PyG's loop path with the block-diagonal contraction."""
    N = x.size(0)
    R, nb, bi, bo = weight.shape
    out = torch.zeros(N, nb * bo, dtype=x.dtype, device=x.device)
    for r in range(R):
        m = edge_type == r
        src, dst = edge_index[0][m], edge_index[1][m]
        s = torch.zeros(N, x.size(1), dtype=x.dtype, device=x.device).index_add_(0, dst, x.index_select(0, src))
        cnt = torch.zeros(N, dtype=x.dtype, device=x.device).index_add_(
            0, dst, torch.ones(dst.numel(), dtype=x.dtype, device=x.device)).clamp_(min=1)
        h = (s / cnt.unsqueeze(1)).view(-1, nb, bi)
        h = torch.einsum("abc,bcd->abd", h, weight[r])
        out = out + h.contiguous().view(-1, nb * bo)
    return out + x @ root + bias


class RGCNConvBlocksRef(nn.Module):
    """Parameter layout and init order of PyG's RGCNConv(num_blocks=nb): weight, comp (None), root, bias."""

    def __init__(self, in_channels, out_channels, num_relations, num_blocks):
        super().__init__()
        if in_channels % num_blocks or out_channels % num_blocks:
            raise ValueError("channels must be divisible by the number of blocks")
        self.in_channels, self.out_channels = in_channels, out_channels
        self.num_relations, self.num_blocks = num_relations, num_blocks
        self.weight = nn.Parameter(torch.empty(num_relations, num_blocks, in_channels // num_blocks,
                                               out_channels // num_blocks))
        self.register_parameter("comp", None)
        self.root = nn.Parameter(torch.empty(in_channels, out_channels))
        self.bias = nn.Parameter(torch.empty(out_channels))
        self.reset_parameters()

    def reset_parameters(self):
        O.glorot_(self.weight)
        O.glorot_(self.comp)
        O.glorot_(self.root)
        self.bias.data.zero_()

    def forward(self, x, edge_index, edge_type):
        assert edge_type is not None
        return rgcn_conv_blocks_ref(x, edge_index, edge_type, self.weight, self.root, self.bias)


class EncoderBlocksRef(O.EncoderRef):
    """``oracle.rgcn_ref.EncoderRef`` (same construction order, same forward) with block-diagonal convolutions."""

    def __init__(self, num_nodes, num_relations, embedding_dim=64, hidden_dim=128, dropout=0.5, num_blocks=4,
                 num_layers=2):
        nn.Module.__init__(self)
        self.node_embeddings = nn.Embedding(num_nodes, embedding_dim)
        self.conv1 = RGCNConvBlocksRef(embedding_dim, hidden_dim, num_relations, num_blocks)
        self.conv2 = RGCNConvBlocksRef(hidden_dim, hidden_dim, num_relations, num_blocks)
        self.extra = nn.ModuleList(
            [RGCNConvBlocksRef(hidden_dim, hidden_dim, num_relations, num_blocks) for _ in range(num_layers - 2)])
        self.dropout = nn.Dropout(dropout)
        nn.init.xavier_uniform_(self.node_embeddings.weight)


class ModelBlocksRef(O.ModelRef):
    """``oracle.rgcn_ref.ModelRef`` with block-diagonal convolutions."""

    def __init__(self, num_nodes, num_relations, embedding_dim=64, hidden_dim=128, dropout=0.5, decoder_dropout=0.0,
                 num_blocks=4, num_layers=2):
        nn.Module.__init__(self)
        self.encoder = EncoderBlocksRef(num_nodes, num_relations, embedding_dim, hidden_dim, dropout, num_blocks,
                                        num_layers)
        self.decoder = O.DecoderRef(num_relations, hidden_dim, decoder_dropout)

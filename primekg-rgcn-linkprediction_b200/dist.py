"""Destination-range partitioned RGCN for graphs too large for one GPU (SURVEY.md §8e, BASELINE.json cfg5).

The reference has no distributed code (no ``torch.distributed`` import anywhere); this is the scale-out of its
full-batch path.  One process per GPU:

* nodes are cut into P contiguous destination ranges balanced by IN-EDGE count (hubs!); rank p owns rows [lo_p, hi_p)
  of every feature matrix and of the embedding table, and the CSR slice of the edges whose destination it owns;
* per layer forward: all-gather of the input-feature shards (NCCL over NVLink) -> every rank holds all source rows
  -> purely local aggregation + tensor-core transform of its own rows;
* per layer backward: the local transposed-CSR gather yields a full-length partial grad-X (contributions to remote
  sources) -> reduce-scatter (sum) back to the owners — the exact transpose of the all-gather;
* weight / root / bias gradients: all-reduce (sum); the embedding-table gradient stays sharded.

Shards are padded to a common row count ``max_n`` so the collectives are the fixed-size tensor variants; node ids are
relabelled once to the padded id space  pid = owner * max_n + (node - lo_owner).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Tuple

import torch
import torch.distributed as dist
import torch.nn as nn

from .conv import RGCNConv, _RGCNLayerFn, default_mode
from .graph import RelGraph


# ---------------------------------------------------------------------------------------------------
# partition plan (pure index arithmetic: runs on CPU or GPU tensors)
# ---------------------------------------------------------------------------------------------------
@dataclass
class PartitionPlan:
    bounds: List[int]          # P + 1 node boundaries, bounds[p] <= node < bounds[p+1] is owned by p
    max_n: int                 # padded shard size

    @property
    def world(self) -> int:
        return len(self.bounds) - 1

    def size(self, p: int) -> int:
        return self.bounds[p + 1] - self.bounds[p]

    def to_padded(self, nodes: torch.Tensor) -> torch.Tensor:
        """global node id -> padded id  owner * max_n + (node - lo_owner)."""
        b = torch.tensor(self.bounds[1:-1], dtype=nodes.dtype, device=nodes.device)
        owner = torch.bucketize(nodes, b, right=True)
        lo = torch.tensor(self.bounds[:-1], dtype=nodes.dtype, device=nodes.device)
        return owner * self.max_n + (nodes - lo[owner])


def plan_partition(dst: torch.Tensor, num_nodes: int, world: int) -> PartitionPlan:
    """Contiguous destination ranges with (nearly) equal in-edge counts.  Deterministic: every rank computes the same
    plan from the same destination array."""
    deg = torch.bincount(dst, minlength=num_nodes)
    csum = torch.cumsum(deg, 0)
    E = int(csum[-1]) if num_nodes else 0
    bounds = [0]
    for p in range(1, world):
        target = (E * p + world - 1) // world
        b = int(torch.searchsorted(csum, torch.tensor(target, dtype=csum.dtype, device=csum.device)).item()) + 1
        b = min(max(b, bounds[-1]), num_nodes)       # monotone, in range (a rank may own 0 rows on tiny graphs)
        bounds.append(b)
    bounds.append(num_nodes)
    max_n = max(bounds[p + 1] - bounds[p] for p in range(world))
    max_n = (max(max_n, 1) + 3) // 4 * 4
    return PartitionPlan(bounds, max_n)


def local_edges(edge_index: torch.Tensor, edge_type: torch.Tensor, plan: PartitionPlan, rank: int
                ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """(src in padded ids, dst local to the shard, rel) of the edges whose destination this rank owns; edge order kept."""
    lo, hi = plan.bounds[rank], plan.bounds[rank + 1]
    m = (edge_index[1] >= lo) & (edge_index[1] < hi)
    src = plan.to_padded(edge_index[0][m])
    return src, edge_index[1][m] - lo, edge_type[m]


# ---------------------------------------------------------------------------------------------------
# collectives with autograd (NCCL on GPUs; gloo in the CPU tests)
# ---------------------------------------------------------------------------------------------------
def _all_gather_rows(x: torch.Tensor, world: int) -> torch.Tensor:
    out = torch.empty(world * x.size(0), x.size(1), dtype=x.dtype, device=x.device)
    if dist.get_backend() == "nccl":
        dist.all_gather_into_tensor(out, x.contiguous())
    else:
        dist.all_gather(list(out.chunk(world, 0)), x.contiguous())
    return out


def _reduce_scatter_rows(g: torch.Tensor, world: int, rank: int) -> torch.Tensor:
    n = g.size(0) // world
    if dist.get_backend() == "nccl":
        out = torch.empty(n, g.size(1), dtype=g.dtype, device=g.device)
        dist.reduce_scatter_tensor(out, g.contiguous(), op=dist.ReduceOp.SUM)
        return out
    g = g.contiguous().clone()
    dist.all_reduce(g, op=dist.ReduceOp.SUM)
    return g[rank * n:(rank + 1) * n].clone()


class AllGatherRows(torch.autograd.Function):
    """[max_n, d] shard -> [P * max_n, d]; backward = reduce-scatter (sum) of the full-length gradient."""

    @staticmethod
    def forward(ctx, x):
        ctx.world, ctx.rank = dist.get_world_size(), dist.get_rank()
        return _all_gather_rows(x, ctx.world)

    @staticmethod
    def backward(ctx, g):
        return _reduce_scatter_rows(g, ctx.world, ctx.rank)


class AllReduceGrad(torch.autograd.Function):
    """Identity forward; backward all-reduces (sums) the gradient — wraps the replicated weights."""

    @staticmethod
    def forward(ctx, w):
        return w.view_as(w)

    @staticmethod
    def backward(ctx, g):
        g = g.contiguous().clone()
        dist.all_reduce(g, op=dist.ReduceOp.SUM)
        return g


# ---------------------------------------------------------------------------------------------------
# the partitioned encoder
# ---------------------------------------------------------------------------------------------------
class PartitionedRGCN(nn.Module):
    """Encoder of the reference (Embedding -> [RGCNConv -> ReLU -> Dropout] x (L-1) -> RGCNConv, src/models/rgcn.py:97-130)
    over a destination-range shard.  ``forward()`` returns this rank's rows ``[max_n, hidden]`` (rows past the
    shard's true size are padding).  Weights are replicated (same seed on every rank), the table is sharded."""

    def __init__(self, plan: PartitionPlan, rank: int, num_relations: int, embedding_dim: int = 64,
                 hidden_dim: int = 128, dropout: float = 0.5, num_bases: Optional[int] = None, num_layers: int = 2,
                 seed: int = 42):
        super().__init__()
        self.plan, self.rank, self.num_relations = plan, rank, num_relations
        self.n_local = plan.size(rank)
        g = torch.Generator().manual_seed(seed)
        dims = [embedding_dim] + [hidden_dim] * num_layers
        self.convs = nn.ModuleList(RGCNConv(dims[i], dims[i + 1], num_relations, num_bases=num_bases)
                                   for i in range(num_layers))
        for conv in self.convs:                       # identical replicated weights on every rank
            for prm in (conv.weight, conv.comp, conv.root):
                if prm is not None:
                    a = (6.0 / (prm.size(-2) + prm.size(-1))) ** 0.5
                    with torch.no_grad():
                        prm.copy_((torch.rand(prm.shape, generator=g) * 2 - 1) * a)
        # the shard's rows of the Xavier-initialised table; padding rows are zero and never gathered
        table = torch.zeros(plan.max_n, embedding_dim)
        a = (6.0 / (sum(plan.size(p) for p in range(plan.world)) + embedding_dim)) ** 0.5
        gs = torch.Generator().manual_seed(seed + 1 + rank)
        table[: self.n_local] = (torch.rand(self.n_local, embedding_dim, generator=gs) * 2 - 1) * a
        self.node_embeddings = nn.Parameter(table)
        self.dropout = nn.Dropout(dropout)
        self.graph: Optional[RelGraph] = None

    def set_graph(self, graph) -> None:
        """``graph``: RelGraph over the local edges (n_dst = max_n rows, n_src = P * max_n padded source ids)."""
        self.graph = graph

    def build_graph(self, edge_index: torch.Tensor, edge_type: torch.Tensor) -> None:
        src, dst, rel = local_edges(edge_index, edge_type, self.plan, self.rank)
        self.set_graph(RelGraph(src, dst, rel, self.plan.max_n, self.plan.world * self.plan.max_n, self.num_relations))

    def forward(self) -> torch.Tensor:
        x = self.node_embeddings
        last = len(self.convs) - 1
        for li, conv in enumerate(self.convs):
            x_full = AllGatherRows.apply(x)                                  # NCCL all-gather over NVLink
            W = AllReduceGrad.apply(conv.relation_weights())
            root, bias = AllReduceGrad.apply(conv.root), AllReduceGrad.apply(conv.bias)
            p = self.dropout.p if (self.training and li != last) else 0.0
            drop = conv.dropout_state(p, x.device) if 0.0 < p < 1.0 else None
            # the mask is keyed by global node id, as on one GPU (padding rows share ids with the next shard's first rows:
            # harmless, no edge and no decoder reads a padding row)
            x = _RGCNLayerFn.apply(x_full, x, W, root, bias, self.graph, li != last, conv.mode or default_mode(), drop,
                                   None, None, self.plan.bounds[self.rank])
            if li != last and p > 0.0 and drop is None:
                x = self.dropout(x)
        return x


def gather_embeddings(x_local: torch.Tensor) -> torch.Tensor:
    """All ranks' output shards -> [P * max_n, hidden] in padded id order (for the decoder / evaluation)."""
    return AllGatherRows.apply(x_local)


class PartitionedModel(nn.Module):
    """Encoder shard + replicated DistMult decoder (reference src/models/rgcn.py:300-331 on P GPUs).

    ``forward(heads, tails, rels)`` takes THIS RANK'S slice of the batch in global node ids and returns its scores;
    with ``loss = local_sum / global_batch`` on every rank the reduce-scatter in backward sums exactly the right
    gradient.  Call ``allreduce_decoder_grads()`` after ``backward()`` (the conv weights are reduced in-graph)."""

    def __init__(self, plan: PartitionPlan, rank: int, num_relations: int, embedding_dim: int = 64,
                 hidden_dim: int = 128, dropout: float = 0.5, decoder_dropout: float = 0.0,
                 num_bases: Optional[int] = None, num_layers: int = 2, seed: int = 42):
        super().__init__()
        from .modules import LinkPredictor
        self.plan = plan
        self.encoder = PartitionedRGCN(plan, rank, num_relations, embedding_dim, hidden_dim, dropout, num_bases,
                                       num_layers, seed)
        state = torch.random.get_rng_state()
        torch.manual_seed(seed + 12345)                       # identical decoder on every rank
        self.decoder = LinkPredictor(num_relations, hidden_dim, decoder_dropout)
        torch.random.set_rng_state(state)

    def forward(self, heads: torch.Tensor, tails: torch.Tensor, rels: torch.Tensor) -> torch.Tensor:
        emb = gather_embeddings(self.encoder())               # [P * max_n, hidden], padded id order
        return self.decoder.score_pairs(emb, self.plan.to_padded(heads), self.plan.to_padded(tails), rels)

    def allreduce_decoder_grads(self) -> None:
        for p in self.decoder.parameters():
            if p.grad is not None:
                dist.all_reduce(p.grad, op=dist.ReduceOp.SUM)

"""Destination-range partitioned RGCN whose exchange steps are done by OUR kernels over peer-mapped memory
(NVLink loads / stores) instead of collective-library calls — the fused form of ``dist.py`` (SURVEY.md §8e).

Per layer, forward (rank p owns rows [lo_p, hi_p), padded to ``max_n``):

    X_full (all rows, this rank's copy)  --aggregate-->  H  --tcgen05 transform, epilogue stores each finished
    tile into the row slot of EVERY rank's next X_full over NVLink-->  [barrier]

so the all-gather of the next layer's input is the transform's own epilogue and overlaps its MMA main loop tile by
tile; only a device-side barrier separates the layers.  Backward:

    [barrier]  pull this rank's rows of every rank's full-length partial grad-X over NVLink, sum in RANK ORDER,
    add the local root-term gradient, apply the ReLU / dropout mask and emit the bf16 planes G + bias-gradient
    partials (one kernel = reduce-scatter + mask + operand conversion)  ->  dgrad  ->  transposed-CSR gather into
    this rank's partial buffer  ->  wgrad

Weight gradients are all-reduced once per step as one flat NCCL call (plumbing).  Two halves of one peer buffer
alternate between layers; the per-layer barrier is what makes the reuse safe (a rank can only be one layer ahead).
The encoder's OUTPUT lives in a third, dedicated region and every forward starts with a barrier, so a fast rank can
never overwrite what a slow rank's decoder is still reading (forward-only loops included).  The output is valid until
the next forward; only one forward may be outstanding per backward (checked: ``_Exchange.generation``).
Everything is deterministic: fixed reduction orders everywhere, no atomics.

The NCCL form in ``dist.py`` (all-gather / reduce-scatter / all-reduce with autograd) stays as the baseline this
is measured against and as the form the CPU (gloo) tests exercise.
"""
from __future__ import annotations

from typing import List, Optional

import torch
import torch.distributed as dist
import torch.nn as nn

import os

from . import ops, rowsparse
from .conv import default_mode
from .dist import PartitionPlan, PartitionedRGCN
from .peer import PeerBuffer


def sparse_last_layer() -> bool:
    """Row-sparse backward of the last layer in the partitioned path (``PRIMEKG_RGCN_SPARSE_BWD=0`` turns it off)."""
    return os.environ.get("PRIMEKG_RGCN_SPARSE_BWD", "1") != "0"


def push_after_transform() -> bool:
    """A/B switch (``RGCN_PEER_PUSH=1``): the all-gather of a layer's output as a separate row push after the transform
    instead of peer stores from its epilogue."""
    return os.environ.get("RGCN_PEER_PUSH", "0") == "1"


def listed_last_layer() -> bool:
    """Listed-rows forward of the last layer (``PRIMEKG_RGCN_SPARSE_FWD=0`` or ``PRIMEKG_RGCN_SPARSE_BWD=0``: all rows)."""
    return sparse_last_layer() and os.environ.get("PRIMEKG_RGCN_SPARSE_FWD", "1") != "0" and ops.prepared_weights()


class _Exchange:
    """The two peer buffers (features forward, partial gradients backward), each cut into two halves."""

    def __init__(self, plan: PartitionPlan, rank: int, dims: List[int], device: torch.device):
        self.rank, self.world = rank, plan.world
        self.n_total = plan.world * plan.max_n
        self.max_n = plan.max_n
        self.row0 = rank * plan.max_n
        self.node0 = plan.bounds[rank]                      # global id of this shard's first node
        self.half = self.n_total * max(dims)               # floats per half
        self.half = (self.half + 63) // 64 * 64
        # features: two halves that alternate between the layers + a DEDICATED region for the encoder's output, so the
        # tensor a forward returns is never a buffer the next forward's initial push stores into
        self.x = PeerBuffer(3 * self.half * 4, device)
        self.g = PeerBuffer(2 * self.half * 4, device)
        self.n_layers = len(dims) - 1
        self.generation = 0                                # bumped by every forward; a backward checks it is the latest

    def _x_off(self, k: int) -> int:
        return 2 * self.half if k == self.n_layers else (k % 2) * self.half

    def x_view(self, k: int, d: int) -> torch.Tensor:
        return self.x.view(self.n_total, d, self._x_off(k))

    def g_view(self, k: int, d: int) -> torch.Tensor:
        return self.g.view(self.n_total, d, (k % 2) * self.half)

    def x_ptrs(self, k: int) -> List[int]:
        return self.x.peer_ptrs(self._x_off(k))

    def g_ptrs(self, k: int) -> List[int]:
        return self.g.peer_ptrs((k % 2) * self.half)


class _FusedEncoderFn(torch.autograd.Function):
    """(table shard, W_1, root_1, bias_1, ..., W_L, root_L, bias_L) -> all ranks' final embeddings [P * max_n, H]
    (this rank's copy; rows in padded id order).  Its gradient is the full-length PARTIAL gradient of this rank."""

    @staticmethod
    def forward(ctx, ex: _Exchange, graph, mode: str, drops, read_ids, x0, *params):
        """``read_ids`` (int64 padded global ids, even length, or None): the rows THIS rank's decoder will read; with it
        the last layer computes — and sends to every rank — only the rows some rank reads."""
        L = len(params) // 3
        n, row0 = ex.max_n, ex.row0
        x0 = x0.contiguous()
        if L != ex.n_layers:
            raise ValueError("the exchange buffers were sized for another number of layers")
        ex.generation += 1
        # every rank must be done with the PREVIOUS call's buffers (its decoder reading the output region, its last layer
        # reading half (L-1) % 2) before anybody stores into them again: in training the backward's barriers imply it, in
        # forward-only loops (evaluation) nothing else does
        ex.x.barrier()
        ops.p2p_push_rows(x0, ex.x_ptrs(0), row0, x0.size(1))
        ex.x.barrier()
        listed = None
        if read_ids is not None and read_ids.numel() > 0 and read_ids.numel() % 2 == 0 and \
                ex.world * read_ids.numel() <= rowsparse.MAX_FRACTION * n:
            # every rank's list (a few kilobytes; plumbing): a rank computes the rows of ITS shard that anybody reads;
            # the others are parked on local row 0 as invalid entries (never walked, never stored)
            mine = read_ids.to(torch.int64).contiguous()
            all_ids = torch.empty(ex.world * mine.numel(), dtype=torch.int64, device=mine.device)
            if ex.world > 1:
                dist.all_gather_into_tensor(all_ids, mine)
            else:
                all_ids = mine
            inside = (all_ids >= row0) & (all_ids < row0 + n)
            local = torch.where(inside, all_ids - row0, torch.full_like(all_ids, -1))
            half = local.numel() // 2
            listed = ops.rows_list_build(local[:half], local[half:], n) + (all_ids, mine)
        saved, outs, wps = [], [], []
        for l in range(L):
            W, root, bias = params[3 * l: 3 * l + 3]
            R, d_in, d_out = W.shape
            K1, K2 = R * d_in, d_in
            x_full = ex.x_view(l, d_in)
            p_drop, seed, ctr = drops[l] if drops[l] is not None else (0.0, 0, None)
            last = l == L - 1
            # aggregate -> planes -> transform whose epilogue also stores every tile into all ranks' next buffer
            rows_l, slot_l = listed[:2] if (last and listed is not None) else (None, None)
            push_after = rows_l is None and push_after_transform()
            # the dropout mask is keyed by global node id (ex.node0), as on one GPU; padding rows share ids with the next
            # shard's first rows, which is harmless: no edge and no decoder reads a padding row
            out, A, wp = ops.layer_fwd(graph, x_full, x_full[row0:row0 + n], W.reshape(K1, d_out), root, bias, not last, mode,
                                       p_drop, seed, ctr, peer_out=None if push_after else ex.x_ptrs(l + 1), peer_row0=row0,
                                       peer_ld=d_out, rows=rows_l, slot=slot_l, dropout_row0=ex.node0)
            if push_after:
                # all-gather as a separate push of whole rows (512-byte bursts per warp) instead of the epilogue's 64-byte
                # pieces: no overlap with the MMA main loop, but a far better NVLink packet mix
                ops.p2p_push_rows(out, ex.x_ptrs(l + 1), row0, d_out)
            ex.x.barrier()
            saved += [A[0], A[1], W, root]
            wps.append(wp)
            outs.append(None if last else out)          # post-ReLU/dropout output = the backward mask
        ctx.ex, ctx.graph, ctx.mode, ctx.L = ex, graph, mode, L
        ctx.listed = listed
        ctx.generation = ex.generation
        ctx.w_planes = wps
        ctx.p_drops = [d[0] if d is not None else 0.0 for d in drops]
        ctx.d0 = x0.size(1)
        ctx.save_for_backward(*saved, *[o for o in outs if o is not None])
        d_last = params[3 * (L - 1)].shape[2]
        out = ex.x_view(L, d_last)
        if listed is not None:
            rowsparse.mark_listed_output(out)       # the decoder's backward may leave the unlisted gradient rows undefined
        else:
            rowsparse.unmark_listed_output()
        return out

    @staticmethod
    def backward(ctx, g_full):
        ex, graph, mode, L = ctx.ex, ctx.graph, ctx.mode, ctx.L
        if ctx.generation != ex.generation:
            # the returned embeddings (saved by the decoder for ITS backward) live in the peer buffer and a later forward
            # has rewritten them through raw pointers, which autograd's version counters cannot see
            raise RuntimeError("FusedPartitionedRGCN: backward of a forward that is no longer the latest one; only one "
                               "forward may be outstanding per backward (clone the output to keep it across forwards)")
        n, row0 = ex.max_n, ex.row0
        t = ctx.saved_tensors
        masks = list(t[4 * L:])
        dev = g_full.device
        d_last = t[4 * (L - 1) + 2].shape[2]
        if ctx.listed is not None:
            # only the rows some rank's decoder read can carry a gradient, and only those are pulled: zero them in the peer
            # visible buffer, then copy this rank's own rows (g_full is undefined elsewhere) — kilobytes instead of N x d
            all_ids, mine = ctx.listed[2:]
            gv = ex.g_view(L, d_last)
            gv.index_fill_(0, all_ids, 0.0)
            gv.index_copy_(0, mine, g_full.index_select(0, mine))       # (a repeated id carries the same row)
        else:
            ex.g_view(L, d_last).copy_(g_full)          # this rank's partial gradient of ALL rows, peer visible
        # The loss reads 2 * batch rows of the output (src/models/rgcn.py:325-326): every rank's g_full is zero outside the
        # rows ITS slice of the batch names (the decoder's backward announces them, rowsparse.py).  With all ranks' lists
        # the LAST layer's backward runs row-sparse, like the one-GPU model: a pull of the listed rows only (kilobytes
        # instead of this rank's shard of every rank's buffer) and dgrad / walk / wgrad over <= 2 * batch compact rows.
        sparse_rows = slot_fwd = None
        claimed = rowsparse.claim(g_full) if sparse_last_layer() else None
        if ctx.listed is not None:
            # the forward computed the listed rows only (the same all-ranks list, already local): its compact planes are
            # the weight gradient's operand, its slot map serves the compaction
            sparse_rows, slot_fwd = ctx.listed[:2]
        elif claimed is not None:
            mine_rows = claimed[0]                                          # padded global ids, 2 * local batch entries
            all_rows = torch.empty(ex.world * mine_rows.numel(), dtype=torch.int64, device=dev)
            if ex.world > 1:
                dist.all_gather_into_tensor(all_rows, mine_rows.contiguous())
            else:
                all_rows = mine_rows
            inside = (all_rows >= row0) & (all_rows < row0 + n)
            # rows of other shards are replaced by local row 0: listing a row that nobody's loss touches is harmless, its
            # pulled gradient is exactly zero (fixed list length: no host synchronisation)
            sparse_rows = torch.where(inside, all_rows - row0, torch.zeros_like(all_rows))
        ex.g.barrier()
        extra = None
        grads = [None] * (3 * L)
        for l in range(L - 1, -1, -1):
            A_hi, A_lo, W, root = t[4 * l: 4 * l + 4]
            R, d_in, d_out = W.shape
            K1, K2 = R * d_in, d_in
            mask = masks[l] if l < L - 1 else None
            Wf = W.reshape(K1, d_out)
            if l == L - 1 and sparse_rows is not None:
                g_local = torch.empty(n, d_out, dtype=torch.float32, device=dev)      # only the listed rows are read
                ops.p2p_pull_rows(ex.g_ptrs(l + 1), row0, d_out, sparse_rows, g_local)
                _, gA_c, gWf, groot, gb, slot = ops.layer_bwd(
                    graph, g_local, None, 1.0, (A_hi, A_lo), Wf, root, d_in, mode, need_x=True, add_root_term=False,
                    need_w=True, need_b=True, gx_out=ex.g_view(l, d_in), rows=sparse_rows, w_planes=ctx.w_planes[l],
                    return_compact=True, slot=slot_fwd, a_compact=slot_fwd is not None)
                # root-term gradient of this rank's rows: the compact rows scattered back (unlisted rows read the zero row)
                extra = gA_c[:, K1:].index_select(0, slot.long())
                grads[3 * l: 3 * l + 3] = [gWf.view(R, d_in, d_out), groot, gb]
                ex.g.barrier()
                continue
            G = ops.alloc_planes(n, d_out, mode, dev)
            # reduce-scatter by pull + root-term gradient + ReLU/dropout mask + operand conversion, one kernel
            _, colsum = ops.p2p_reduce_split(ex.g_ptrs(l + 1), row0, d_out, n, d_out, dev, extra=extra, relu_mask=mask,
                                             mask_scale=1.0 / (1.0 - ctx.p_drops[l]), planes=G, colsum=True)
            gA = ops.transform_dgrad(G, d_out, Wf, root, mode, w_planes=ctx.w_planes[l])
            ops.aggregate_bwd(graph, gA, d_in, init=None, out=ex.g_view(l, d_in))
            extra = gA[:, K1:]
            gWf, groot, gb = ops.transform_wgrad((A_hi, A_lo), K1, K2, G, d_out, colsum, mode)
            grads[3 * l: 3 * l + 3] = [gWf.view(R, d_in, d_out), groot, gb]
            ex.g.barrier()
        gx0, _ = ops.p2p_reduce_split(ex.g_ptrs(0), row0, ctx.d0, n, ctx.d0, dev, extra=extra, want_fp32=True)
        # replicated weights: one flat all-reduce (sum) for all layers
        flat = torch.cat([g.reshape(-1) for g in grads])
        dist.all_reduce(flat, op=dist.ReduceOp.SUM)
        off = 0
        for i, g in enumerate(grads):
            grads[i] = flat[off: off + g.numel()].view_as(g)
            off += g.numel()
        return (None, None, None, None, None, gx0, *grads)


class FusedPartitionedRGCN(PartitionedRGCN):
    """``PartitionedRGCN`` (same parameters, same plan, same graph shard) with the peer-memory exchange.
    ``forward()`` returns ALL ranks' output rows ``[P * max_n, hidden]`` (padded id order) — the final all-gather is
    the last transform's epilogue too."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self._ex: Optional[_Exchange] = None

    def _exchange(self) -> _Exchange:
        if self._ex is None:
            dims = [self.convs[0].in_channels] + [c.out_channels for c in self.convs]
            self._ex = _Exchange(self.plan, self.rank, dims, self.node_embeddings.device)
        return self._ex

    def forward(self, read_ids: Optional[torch.Tensor] = None) -> torch.Tensor:
        """``read_ids`` (padded global ids, e.g. ``cat(heads, tails)`` of this rank's batch): the caller reads ONLY these
        rows of the result; with autograd on the last layer then computes and exchanges just the rows some rank reads
        (every other row of the returned matrix is undefined)."""
        if not self.node_embeddings.is_cuda:
            raise RuntimeError("FusedPartitionedRGCN needs CUDA devices with peer access; dist.PartitionedRGCN is the "
                               "collective-library form")
        last = len(self.convs) - 1
        params, drops = [], []
        for li, conv in enumerate(self.convs):
            params += [conv.relation_weights(), conv.root, conv.bias]
            p = self.dropout.p if (self.training and li != last) else 0.0
            if p >= 1.0:
                raise ValueError("fused dropout needs p < 1")
            drops.append(conv.dropout_state(p, self.node_embeddings.device) if p > 0.0 else None)
        mode = self.convs[0].mode or default_mode()
        if read_ids is not None and not (torch.is_grad_enabled() and listed_last_layer()):
            read_ids = None
        return _FusedEncoderFn.apply(self._exchange(), self.graph, mode, drops, read_ids, self.node_embeddings, *params)


class FusedPartitionedModel(nn.Module):
    """Encoder shard with peer-memory exchange + replicated DistMult decoder; the interface of ``dist.PartitionedModel``."""

    def __init__(self, plan: PartitionPlan, rank: int, num_relations: int, embedding_dim: int = 64,
                 hidden_dim: int = 128, dropout: float = 0.5, decoder_dropout: float = 0.0,
                 num_bases: Optional[int] = None, num_layers: int = 2, seed: int = 42):
        super().__init__()
        from .modules import LinkPredictor
        self.plan = plan
        self.encoder = FusedPartitionedRGCN(plan, rank, num_relations, embedding_dim, hidden_dim, dropout, num_bases,
                                            num_layers, seed)
        state = torch.random.get_rng_state()
        torch.manual_seed(seed + 12345)                       # identical decoder on every rank
        self.decoder = LinkPredictor(num_relations, hidden_dim, decoder_dropout)
        torch.random.set_rng_state(state)

    def forward(self, heads: torch.Tensor, tails: torch.Tensor, rels: torch.Tensor) -> torch.Tensor:
        h, t = self.plan.to_padded(heads), self.plan.to_padded(tails)
        emb = self.encoder(torch.cat([h.reshape(-1), t.reshape(-1)]))       # [P * max_n, hidden], padded id order
        return self.decoder.score_pairs(emb, h, t, rels)

    def allreduce_decoder_grads(self) -> None:
        for p in self.decoder.parameters():
            if p.grad is not None:
                dist.all_reduce(p.grad, op=dist.ReduceOp.SUM)

"""RGCNConv operator: PyG-compatible module over the sm_100a kernels.

Replaces ``torch_geometric.nn.RGCNConv`` as the reference uses it (import src/models/rgcn.py:17,
construction :72-85, calls :123 and :128): same constructor arguments, parameter names, shapes,
initialisation (PyG ``glorot`` / zeros, in PyG's order) and ``forward(x, edge_index, edge_type)``.

    x'_i = root^T x_i + bias + sum_r (1 / |N_r(i)|) sum_{j in N_r(i)} W_r^T x_j        (mean per (dst, relation))

Formulation: aggregate first (gather width d_in <= d_out, like the reference), then ONE dense
contraction over the concatenated K = (R+1) * d_in.  Backward runs the mirrored gather over the
transposed CSR (deterministic, no atomics) and the dense dgrad / wgrad contractions.
"""
from __future__ import annotations

import math
import os
from typing import Optional

import torch
import torch.nn as nn

from . import ops, rowsparse
from .graph import RelGraph, get_graph


MODES = ("fp32", "bf16")


def default_mode() -> str:
    m = os.environ.get("PRIMEKG_RGCN_MODE", "fp32").lower()
    if m not in MODES:
        raise ValueError(f"PRIMEKG_RGCN_MODE must be one of {MODES}, got {m!r}")
    return m


class _RGCNLayerFn(torch.autograd.Function):
    """out = [relu]( H(x) @ Wf + x @ root + bias ),  Wf = W.view(R * d_in, d_out).

    Data flow (all on hand-written sm_100a kernels):
      forward : aggregate_fwd writes H as bf16 planes into A[:, :R*d_in]; split_planes writes x into A[:, R*d_in:];
                transform_fwd (tcgen05) = A @ [Wf ; root] + bias (, ReLU).
      backward: split_planes(gO, relu mask) -> G planes + bias-gradient partials; transform_dgrad -> gA;
                aggregate_bwd over the transposed CSR -> grad x; transform_wgrad (split-K tcgen05) -> grad W, root, bias.
    """

    @staticmethod
    def forward(ctx, x_src, x_root, W, root, bias, graph: RelGraph, relu: bool, mode: str, drop=None, in_mask_scale=None,
                listed=None, dropout_row0: int = 0):
        """x_src [n_src, d_in]: rows the edges gather from; x_root [n_dst, d_in]: the rows being updated (self-loop
        term).  On one GPU they are the same tensor; on a destination-range shard x_src is the all-gathered matrix.
        ``dropout_row0``: global node id of row 0 of x_root (a shard's first node), which keys the dropout mask."""
        R, d_in, d_out = W.shape
        shared = x_src.data_ptr() == x_root.data_ptr() and x_src.shape == x_root.shape
        x_src = x_src.contiguous()
        x_root = x_src if shared else x_root.contiguous()
        if x_root.size(0) != graph.n_dst:
            raise ValueError(f"x has {x_root.size(0)} rows, the graph updates {graph.n_dst}")
        # drop = (p, seed, device counter): ReLU + dropout fused into the GEMM epilogue (reference :124-125)
        p_drop, seed, ctr = drop if drop is not None else (0.0, 0, None)
        # bf16-transform mode: the walk gathers a bf16 copy of x — left by the previous layer's epilogue (hand-over in
        # rowsparse.py) or made here (the embedding table) — and a ReLU layer leaves the copy of ITS output for the next one
        x16 = None
        use16 = mode == "bf16" and shared and ops.bf16_gather() and ops.prepared_weights()
        if use16 and d_in % 8 == 0:
            x16 = rowsparse.claim_bf16(x_src)
            if x16 is None:
                x16 = ops.to_bf16(x_src.detach())
        want16 = bool(use16 and relu and d_out % 8 == 0)
        # listed = (rows, slot): only these output rows will be read (the decoder's head / tail rows): walk and transform
        # them alone; the planes come back compact, in list order — what the row-sparse backward wants
        ctx.listed = listed if (listed is not None and shared and p_drop == 0.0 and not want16) else None
        rows_l, slot_l = ctx.listed if ctx.listed is not None else (None, None)
        # the row offset keys the dropout mask and nothing else: handed on only where it changes the result
        row0 = {"dropout_row0": dropout_row0} if (p_drop > 0.0 and dropout_row0) else {}
        res = ops.layer_fwd(graph, x_src, x_root, W.reshape(R * d_in, d_out), root, bias, relu, mode, p_drop, seed, ctr,
                            x_bf16=x16, want_out_bf16=want16, rows=rows_l, slot=slot_l, **row0)
        out, A, wp = res[:3]
        if ctx.listed is not None:
            rowsparse.mark_listed_output(out)
        else:
            rowsparse.unmark_listed_output()
        if want16 and res[3] is not None:
            rowsparse.announce_bf16(out, res[3])
        ctx.graph, ctx.relu, ctx.mode, ctx.shared, ctx.p_drop = graph, relu, mode, shared, p_drop
        ctx.w_planes = wp               # the weights as bf16 planes (converted once): the backward's dgrad reads them
        # in_mask_scale: x is the fused ReLU (+ dropout) output of the layer upstream, whose backward will want this
        # layer's input gradient masked by x > 0 and scaled — the backward walk can write that directly (rowsparse.py)
        ctx.in_mask_scale = in_mask_scale if (shared and in_mask_scale is not None) else None
        ctx.x_is_param = bool(shared and x_src.is_leaf and x_src.requires_grad)     # e.g. the embedding table
        ctx.save_for_backward(A[0], A[1], W, root, out if relu else None, x_src if ctx.in_mask_scale is not None else None)
        return out

    @staticmethod
    def backward(ctx, gO):
        A_hi, A_lo, W, root, out, x_in = ctx.saved_tensors
        graph, mode = ctx.graph, ctx.mode
        R, d_in, d_out = W.shape
        K1 = R * d_in
        need_src, need_root_x, need_W, need_root, need_b = ctx.needs_input_grad[:5]
        need_w_any = need_W or need_root or need_b
        need_x = need_src or need_root_x
        # gO zero outside a short, announced row list (the decoder's backward, rowsparse.py): compact backward
        rows = slot = None
        a_compact = False
        if ctx.listed is not None:
            # the forward computed the listed rows only (the others were never defined, nothing may flow into them): the
            # compaction of gO runs over the forward's own list, and its compact planes are the weight gradient's operand
            rowsparse.claim(gO)
            rows, slot = ctx.listed
            a_compact = True
        elif out is None and ctx.shared and graph.n_src == graph.n_dst:
            claimed = rowsparse.claim(gO)
            if claimed is not None:
                rows, slot = claimed
        # out is zero exactly where ReLU or the fused dropout killed the element: one mask serves both
        mask_scale = 1.0 / (1.0 - ctx.p_drop)
        # the downstream layer's walk may have left this layer's masked output gradient as planes already
        g_ready = rowsparse.claim_planes(gO, out, mask_scale, mode) if (out is not None and rows is None) else None
        next_mask = (x_in, ctx.in_mask_scale) if (x_in is not None and need_x and rowsparse.planes_enabled()) else None
        res = ops.layer_bwd(
            graph, gO.contiguous(), out, mask_scale, (A_hi, A_lo), W.reshape(K1, d_out), root, d_in, mode,
            need_x=need_x, add_root_term=ctx.shared, need_w=need_w_any, need_b=need_w_any, rows=rows, g_ready=g_ready,
            next_mask=next_mask, slot=slot, w_planes=ctx.w_planes, a_compact=a_compact,
            gx_out=ops.param_grad(graph.n_src, d_in, device=gO.device) if (need_x and ctx.x_is_param) else None)
        gx, gA, gWf, groot, gb = res[:5]
        if next_mask is not None:
            rowsparse.announce_planes(gx, x_in, ctx.in_mask_scale, mode, res[5])
        gx_src = gx_root = None
        if need_x:
            if ctx.shared:
                gx_src = gx
            else:
                gx_src = gx if need_src else None             # full-length partial, reduced by the caller
                gx_root = gA[:, K1:]
        gW = gWf.view(R, d_in, d_out) if gWf is not None else None
        return gx_src, gx_root, gW, groot, gb, None, None, None, None, None, None, None


class _RGCNBasisLayerFn(torch.autograd.Function):
    """Basis-decomposed layer in the B-accumulator ("Z") form:  out = [relu]( [Z | x] @ [V_1; ..; V_B; root] + bias ),
    Z_b = sum_r comp[r, b] * H_r(x)  — the same function as ``_RGCNLayerFn`` with W_r = sum_b comp[r, b] V_b, but the
    [N, R * d_in] matrix of per-relation means never exists: K shrinks from (R+1) d_in to (B+1) d_in.

      forward : aggregate_fwd(comp) mixes the relations in registers and writes Z as planes; transform_fwd over K = (B+1) d_in.
      backward: G = gO * mask (planes + fp32);  P = x @ [V_1 .. V_B] (for the coefficient gradient);
                mirrored aggregation over the transposed CSR: T_b[j] = sum_r comp[r, b] sum_{e: j->i, r} w_e G[i]
                with gc[r, b] = sum_j <S_r[j], P_b[j]> as a side output;
                grad x = [T | G] @ [V_1^T; ..; V_B^T; root^T];   grad [V; root] = [Z | x]^T @ G (split-K wgrad).
    Gather width in backward is d_out, so the layer picks this form only when d_out <= d_in."""

    @staticmethod
    def forward(ctx, x, V, comp, root, bias, graph: RelGraph, relu: bool, mode: str, drop=None):
        B, d_in, d_out = V.shape
        x = x.contiguous()
        if graph.n_src != graph.n_dst or x.size(0) != graph.n_dst:
            raise ValueError("the basis (Z) form works on an unpartitioned graph")
        K1, K2 = B * d_in, d_in
        A = ops.alloc_planes(graph.n_dst, K1 + K2, mode, x.device)
        ops.aggregate_fwd(graph, x, comp=comp, planes=A)
        ops.split_planes(x, A, col0=K1)
        p_drop, seed, ctr = drop if drop is not None else (0.0, 0, None)
        out = ops.transform_fwd(A, K1, K2, V.reshape(K1, d_out), root, bias, relu, mode, p_drop, seed, ctr)
        ctx.graph, ctx.relu, ctx.mode, ctx.p_drop = graph, relu, mode, p_drop
        ctx.save_for_backward(A[0], A[1], V, comp, root, out if relu else None)
        return out

    @staticmethod
    def backward(ctx, gO):
        A_hi, A_lo, V, comp, root, out = ctx.saved_tensors
        graph, mode = ctx.graph, ctx.mode
        B, d_in, d_out = V.shape
        K1, K2 = B * d_in, d_in
        n = graph.n_dst
        gO = gO.contiguous()
        need_x, need_V, need_comp, need_root, need_b = ctx.needs_input_grad[:5]
        # A' = [T | G] as planes; G is formed once (mask, dropout scale), also kept in fp32 for the mirrored gather
        Ap = ops.alloc_planes(n, (B + 1) * d_out, mode, gO.device)
        Gp = (Ap[0][:, B * d_out:], None if Ap[1] is None else Ap[1][:, B * d_out:])
        Gf = torch.empty(n, d_out, dtype=torch.float32, device=gO.device) if (need_x or need_comp) else None
        colsum = ops.split_planes(gO, Ap, col0=B * d_out, relu_mask=out, colsum=need_b or need_V or need_root,
                                  mask_scale=1.0 / (1.0 - ctx.p_drop), out_f32=Gf)
        gx = gV = gcomp = groot = gb = None
        if need_x or need_comp:
            P = None
            if need_comp:
                # P[i, b*d_out:(b+1)*d_out] = x[i] @ V_b : one GEMM over the x planes saved inside A
                Vcat = V.detach().permute(1, 0, 2).reshape(d_in, B * d_out).contiguous()
                Xp = (A_hi[:, K1:], None if A_lo is None else A_lo[:, K1:])
                P = ops.transform_fwd(Xp, d_in, 0, Vcat, None, None, False, mode)
            res = ops.aggregate_fwd(graph, Gf, comp=comp, planes=Ap, transposed=True, dot_p=P)
            if need_comp:
                gcomp = res[1]
            if need_x:
                Wt = V.detach().transpose(1, 2).reshape(B * d_out, d_in).contiguous()
                gx = ops.transform_fwd(Ap, B * d_out, d_out, Wt, root.detach().t().contiguous(), None, False, mode)
        if need_V or need_root or need_b:
            gVf, groot, gb = ops.transform_wgrad((A_hi, A_lo), K1, K2, Gp, d_out, colsum, mode)
            gV = gVf.view(B, d_in, d_out)
        return gx, gV, gcomp, groot, gb, None, None, None, None


def basis_form() -> str:
    f = os.environ.get("PRIMEKG_RGCN_BASIS_FORM", "auto").lower()
    if f not in ("auto", "z", "w"):
        raise ValueError("PRIMEKG_RGCN_BASIS_FORM must be auto, z (B accumulators) or w (materialised W_r)")
    return f


def _glorot_(t: Optional[torch.Tensor]) -> None:
    # torch_geometric.nn.inits.glorot: fans are the LAST TWO dims (not nn.init.xavier_uniform_'s)
    if t is not None:
        a = math.sqrt(6.0 / (t.size(-2) + t.size(-1)))
        with torch.no_grad():
            t.uniform_(-a, a)               # (not t.data.uniform_: in-place writes must bump the version counter)


class RGCNConv(nn.Module):
    def __init__(self, in_channels: int, out_channels: int, num_relations: int, num_bases: Optional[int] = None,
                 mode: Optional[str] = None):
        super().__init__()
        if in_channels % 4 or out_channels % 4:
            raise ValueError("the sm_100a kernels need channel counts that are multiples of 4")
        self.in_channels, self.out_channels = in_channels, out_channels
        self.num_relations, self.num_bases = num_relations, num_bases
        self.mode = mode
        self._drop_ctr, self._drop_seed = None, 0
        if num_bases is not None:
            self.weight = nn.Parameter(torch.empty(num_bases, in_channels, out_channels))
            self.comp = nn.Parameter(torch.empty(num_relations, num_bases))
        else:
            self.weight = nn.Parameter(torch.empty(num_relations, in_channels, out_channels))
            self.register_parameter("comp", None)
        self.root = nn.Parameter(torch.empty(in_channels, out_channels))
        self.bias = nn.Parameter(torch.empty(out_channels))
        self.reset_parameters()

    def reset_parameters(self) -> None:
        _glorot_(self.weight)
        _glorot_(self.comp)
        _glorot_(self.root)
        with torch.no_grad():
            self.bias.zero_()

    def relation_weights(self) -> torch.Tensor:
        """[R, d_in, d_out]; with bases W_r = sum_b comp[r, b] V_b (differentiable)."""
        if self.comp is None:
            return self.weight
        B = self.weight.size(0)
        if self.weight.is_cuda and B <= 16 and self.num_relations <= 64:
            return ops.basis_combine(self.comp, self.weight)          # our kernels (csrc/basis.cu), forward and backward
        return (self.comp @ self.weight.view(B, -1)).view(self.num_relations, self.in_channels, self.out_channels)

    def dropout_state(self, p: float, device):
        """(p, seed, counter) for the fused ReLU + dropout epilogue.  The seed is drawn from torch's generator the
        first time dropout is used (so ``torch.manual_seed`` makes runs repeatable); the device-side counter is
        advanced by every call, also under CUDA-graph replay."""
        if not (0.0 <= p < 1.0):
            raise ValueError("fused dropout needs 0 <= p < 1")
        ctr = self._drop_ctr
        if ctr is None or ctr.device != device:
            self._drop_seed = int(torch.randint(0, 2 ** 31 - 1, (1,)).item())
            ctr = self._drop_ctr = ops.dropout_counter(device)
        return (float(p), self._drop_seed, ctr)

    def forward_graph(self, x: torch.Tensor, graph: RelGraph, relu: bool = False, dropout_p: float = 0.0,
                      in_mask_scale: Optional[float] = None, listed=None) -> torch.Tensor:
        """``dropout_p`` > 0 (training): ReLU and dropout are applied in the transform's epilogue (needs relu=True).
        ``in_mask_scale``: ``x`` is the fused ReLU / dropout output of the previous layer (whose 1 / (1 - p) this is).
        ``listed`` = (rows, slot) from ``ops.rows_list_build``: the caller reads ONLY these rows of the result (the last
        layer under a link-prediction decoder, reference src/models/rgcn.py:325-326); every other row is left undefined."""
        if x.dim() != 2 or x.size(1) != self.in_channels:
            raise ValueError(f"x must be [N, {self.in_channels}]")
        if graph.R != self.num_relations:
            raise ValueError("graph and layer disagree on the number of relations")
        if dropout_p > 0.0 and not relu:
            raise ValueError("the fused dropout follows the fused ReLU; use nn.Dropout for other placements")
        drop = self.dropout_state(dropout_p, x.device) if dropout_p > 0.0 else None
        if self._use_z_form(graph):
            return _RGCNBasisLayerFn.apply(x, self.weight, self.comp, self.root, self.bias, graph, relu,
                                           self.mode or default_mode(), drop)
        if listed is not None and (relu or dropout_p > 0.0 or not ops.prepared_weights() or not rowsparse.enabled()):
            listed = None
        return _RGCNLayerFn.apply(x, x, self.relation_weights(), self.root, self.bias, graph, relu,
                                  self.mode or default_mode(), drop, in_mask_scale, listed)

    def _use_z_form(self, graph: RelGraph) -> bool:
        """B-accumulator form of the basis decomposition (``PRIMEKG_RGCN_BASIS_FORM=z``).  It halves the layer's
        memory (no [N, R * d_in] operand: 4.8 GB instead of 10.4 GB for a cfg3 step) and shrinks every GEMM by
        (R+1)/(B+1), but the coefficient gradient then costs B dot products per (row, relation) segment inside the
        mirrored gather; measured on cfg3 the two forms are within 5 % of each other, so ``auto`` keeps the
        materialised-W_r form and the Z form is the choice when memory is the limit."""
        if self.comp is None or graph.n_src != graph.n_dst or self.num_bases > 8:
            return False
        return basis_form() == "z"

    def forward(self, x: torch.Tensor, edge_index: torch.Tensor, edge_type: torch.Tensor) -> torch.Tensor:
        if edge_type is None:
            raise ValueError("edge_type is required")
        if not x.is_cuda:
            raise RuntimeError("RGCNConv (B200) needs CUDA tensors: there is no CPU implementation of this path")
        graph = get_graph(edge_index, edge_type, x.size(0), self.num_relations)
        return self.forward_graph(x, graph)

    def extra_repr(self) -> str:
        return (f"{self.in_channels}, {self.out_channels}, num_relations={self.num_relations}, "
                f"num_bases={self.num_bases}")

"""Thin host wrappers: one Python function per C-ABI entry point of ``include/rgcn_b200.h``.

Every function launches hand-written sm_100a kernels on torch's current stream and returns
torch tensors; nothing here computes on the CPU or through another library.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib
from .graph import RelGraph, _ptr, _stream, _stream_id


class GradArena:
    """One flat fp32 buffer that the backward kernels write the PARAMETER gradients into (weight, root, bias of every
    layer, the embedding-table gradient, the relation-table gradient), in call order.  A data-parallel caller then
    all-reduces ONE tensor instead of eight: measured on 2 / 4 B200s, 63 / 70 us against 107 / 124 us for the same
    9.2 MB as a coalesced group.  ``GraphedTrainStep(flat_grads="arena")`` activates it; every step starts with
    ``reset()`` and takes the same slices, so the addresses are static under CUDA-graph capture."""

    def __init__(self, numel: int, device, buf: Optional[torch.Tensor] = None):
        """``buf``: use this flat fp32 tensor (e.g. the peer-visible input of ``peer.PeerAllReduce``) as the storage."""
        if buf is not None and (buf.dtype != torch.float32 or buf.dim() != 1 or buf.numel() < int(numel)):
            raise ValueError("arena storage must be a flat float32 tensor of at least numel entries")
        self.buf = torch.zeros(int(numel), dtype=torch.float32, device=device) if buf is None else buf
        self.off = 0

    def reset(self) -> None:
        self.off = 0

    def take(self, *shape) -> Optional[torch.Tensor]:
        n = 1
        for s in shape:
            n *= int(s)
        pad = (n + 63) // 64 * 64                  # keeps every slice 256-byte aligned
        if self.off + pad > self.buf.numel():
            return None                            # not sized for this gradient: the caller allocates as usual
        t = self.buf[self.off:self.off + n].view(*shape)
        self.off += pad
        return t

    @property
    def used(self) -> torch.Tensor:
        return self.buf[:self.off]


_ARENA: Optional[GradArena] = None


def set_grad_arena(arena: Optional[GradArena]) -> None:
    global _ARENA
    _ARENA = arena


def param_grad(*shape, device) -> torch.Tensor:
    """Storage for a parameter gradient: a slice of the active arena, else a fresh tensor."""
    if _ARENA is not None and _ARENA.buf.device == device:
        t = _ARENA.take(*shape)
        if t is not None:
            return t
    return torch.empty(*shape, dtype=torch.float32, device=device)


def _f32c(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: the RGCN B200 path has no CPU implementation")
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32, got {t.dtype}")
    if t.dim() != 2:
        raise ValueError(f"{name} must be 2-D")
    if t.stride(1) != 1 or t.stride(0) % 4 != 0 or t.data_ptr() % 16 != 0:
        t = t.contiguous()
    return t


def aggregate_fwd(g: RelGraph, x: torch.Tensor, out_bf16: bool = False, comp: Optional[torch.Tensor] = None,
                  planes=None, transposed: bool = False, dot_p: Optional[torch.Tensor] = None,
                  x_root: Optional[torch.Tensor] = None):
    """H[i, r*d:(r+1)*d] = mean_{j in N_r(i)} x[j]  (or the basis-mixed Z when ``comp`` [R, B] is given).

    ``planes=(hi, lo_or_None)``: write the result as bf16 planes (the tensor-core operand format) into the first
    R*d (or B*d) columns of the given row-major bf16 tensors instead of allocating an fp32 / bf16 matrix.
    ``transposed``: walk the (src, rel) CSR with its 1/count edge weights instead — with ``comp`` and x = the masked
    output gradient this is the mirrored backward of the basis form.  ``dot_p`` [rows, B*d] (needs ``comp``):
    also return gc[r, b] = sum_i <h_r[i], dot_p[i, b]> (the gradient of ``comp``) -> (H, gc).
    ``x_root`` [rows, d] (unmixed form, needs ``planes`` / an output R+1 blocks wide): appended as block R of every
    output row — the operand [H | X] of the transform in one kernel."""
    lib = _lib.load()
    x = _f32c(x, "x")
    ori = g.bwd if transposed else g.fwd
    n_in, n_out = (g.n_dst, g.n_src) if transposed else (g.n_src, g.n_dst)
    if x.size(0) != n_in:
        raise ValueError(f"x has {x.size(0)} rows, the graph gathers from {n_in}")
    d = x.size(1)
    if d % 4 != 0 or d > 1024:
        raise ValueError("feature width must be a multiple of 4 and at most 1024")
    blocks = g.R if comp is None else int(comp.size(1))
    if comp is not None:
        comp = comp.detach().to(torch.float32).contiguous()
        if comp.size(0) != g.R:
            raise ValueError("comp must have one row per relation")
    ws = ori.workspace(d)
    if planes is not None:
        hi, lo = planes
        if hi.dtype != torch.bfloat16 or hi.size(0) != n_out or hi.size(1) < blocks * d or hi.stride(1) != 1:
            raise ValueError("planes must be bf16 [rows, >= blocks*d] row-major")
        H, H_lo, mode = hi, lo, (2 if lo is not None else 1)
    else:
        H = torch.empty(n_out, blocks * d, dtype=torch.bfloat16 if out_bf16 else torch.float32, device=x.device)
        H_lo, mode = None, int(out_bf16)
    if x_root is not None:
        x_root = _f32c(x_root, "x_root")
        if comp is not None or x_root.size(0) != n_out or x_root.size(1) != d or H.size(1) < (blocks + 1) * d:
            raise ValueError("x_root needs the unmixed form, [rows, d] and an output of R+1 blocks")
    gc_part = None
    if dot_p is not None:
        if comp is None:
            raise ValueError("dot_p needs comp")
        dot_p = _f32c(dot_p, "dot_p")
        if dot_p.size(0) != n_out or dot_p.size(1) < blocks * d:
            raise ValueError("dot_p must be [rows, >= B*d]")
        nb = lib.rgcn_aggregate_blocks(ori.ref, d)
        gc_part = torch.empty(max(nb, 1), g.R * blocks, dtype=torch.float32, device=x.device)
    _lib.check(lib.rgcn_aggregate_fwd(ori.ref, _ptr(x), x.stride(0), d, _ptr(comp), 0 if comp is None else blocks,
                                      _ptr(H), _ptr(H_lo), H.stride(0), mode, _ptr(dot_p),
                                      0 if dot_p is None else dot_p.stride(0), _ptr(gc_part), _ptr(x_root),
                                      0 if x_root is None else x_root.stride(0), _ptr(ws),
                                      0 if ws is None else ws.numel() * 4, _stream(x.device)), "rgcn_aggregate_fwd")
    if dot_p is None:
        return H
    return H, reduce_partials(gc_part).view(g.R, blocks)


def reduce_partials(part: torch.Tensor) -> torch.Tensor:
    """Column sums of a [n_part, n_cols] fp32 partial buffer in a fixed order (n_cols padded to a multiple of 4)."""
    lib = _lib.load()
    n, c = part.shape
    if c % 4:
        pad = torch.zeros(n, (c + 3) // 4 * 4, dtype=torch.float32, device=part.device)
        pad[:, :c] = part
        part = pad
    out = torch.empty(part.size(1), dtype=torch.float32, device=part.device)
    _lib.check(lib.rgcn_reduce_partials(_ptr(part), n, part.size(1), _ptr(out), _stream(part.device)),
               "rgcn_reduce_partials")
    return out[:c]


def aggregate_bwd(g: RelGraph, gH: torch.Tensor, d: int, init: Optional[torch.Tensor] = None,
                  out: Optional[torch.Tensor] = None, slot: Optional[torch.Tensor] = None,
                  zero_row: int = -1, masked=None) -> torch.Tensor:
    """gX[j] = init[j] + sum_r sum_{(j->i, r)} gH[i, r*d:(r+1)*d] / max(|N_r(i)|, 1)  over the transposed CSR.
    ``out``: write into this [n_src, d] fp32 tensor (e.g. a peer-visible buffer) instead of allocating.
    ``slot`` (int32 [n_dst]) + ``zero_row``: gH (and init) hold only the listed rows; node i lives in row slot[i], every
    other node maps to the all-zero row ``zero_row`` (``rgcn_aggregate_bwd_rows``).
    ``masked`` = (mask [n_src, d], scale, (hi, lo | None), colsum | None): second output, gX masked / scaled as bf16
    planes + per-block column sums (``rgcn_masked_planes_out``)."""
    lib = _lib.load()
    gH = _f32c(gH, "gH")
    rows_form = slot is not None
    if rows_form:
        if slot.dtype != torch.int32 or slot.numel() != g.n_dst or not (0 <= zero_row < gH.size(0)) or \
                (init is not None and g.n_src != g.n_dst):
            raise ValueError("slot must be int32 [n_dst] and zero_row a row of gH (init needs n_src == n_dst)")
        slot = slot.contiguous()
    if (not rows_form and gH.size(0) != g.n_dst) or gH.size(1) < g.R * d:
        raise ValueError("gH must be [n_dst, >= R*d]")
    if init is not None:
        init = _f32c(init, "init")
        if init.size(0) != (gH.size(0) if rows_form else g.n_src) or init.size(1) < d:
            raise ValueError("init must be [n_src, >= d]")
    if out is None:
        gX = torch.empty(g.n_src, d, dtype=torch.float32, device=gH.device)
    else:
        gX = out
        if gX.dtype != torch.float32 or gX.shape != (g.n_src, d) or gX.stride(1) != 1 or gX.stride(0) % 4:
            raise ValueError("out must be a row-major float32 [n_src, d] tensor")
    ws = g.bwd.workspace(d)
    mp = None if masked is None else C.byref(masked_planes_struct(*masked))
    if rows_form:
        _lib.check(lib.rgcn_aggregate_bwd_rows(g.bwd.ref, _ptr(gH), gH.stride(0), d, _ptr(slot), int(zero_row), _ptr(init),
                                               0 if init is None else init.stride(0), _ptr(gX), gX.stride(0), mp, _ptr(ws),
                                               0 if ws is None else ws.numel() * 4, _stream(gH.device)),
                   "rgcn_aggregate_bwd_rows")
        return gX
    _lib.check(lib.rgcn_aggregate_bwd(g.bwd.ref, _ptr(gH), gH.stride(0), d, _ptr(init),
                                      0 if init is None else init.stride(0), _ptr(gX), gX.stride(0), mp, _ptr(ws),
                                      0 if ws is None else ws.numel() * 4, _stream(gH.device)), "rgcn_aggregate_bwd")
    return gX


def aggregate_max_fwd(g: RelGraph, x: torch.Tensor, planes, x_root: Optional[torch.Tensor] = None):
    """Max aggregation (``rgcn_aggregate_max_fwd``): writes H[i, r] = max_{j in N_r(i)} x[j] (0 for an empty segment) as
    bf16 planes into the first R*d columns of ``planes`` = (hi, lo | None), x_root appended as block R when given, and
    returns (Hmax, Hcnt) fp32 [n_dst, R*d]: the maxima and the tie counts the backward divides by."""
    lib = _lib.load()
    x = _f32c(x, "x")
    if x.size(0) != g.n_src:
        raise ValueError(f"x has {x.size(0)} rows, the graph gathers from {g.n_src}")
    d = x.size(1)
    hi, lo = planes
    if hi.dtype != torch.bfloat16 or hi.size(0) != g.n_dst or hi.stride(1) != 1 or \
            hi.size(1) < (g.R + (x_root is not None)) * d:
        raise ValueError("planes must be bf16 [n_dst, >= R*d (+ d with x_root)] row-major")
    if x_root is not None:
        x_root = _f32c(x_root, "x_root")
        if x_root.shape != (g.n_dst, d):
            raise ValueError("x_root must be [n_dst, d]")
    Hmax = torch.empty(g.n_dst, g.R * d, dtype=torch.float32, device=x.device)
    Hcnt = torch.empty_like(Hmax)
    ws = g.fwd.workspace(2 * d)                    # (max, ties) chunk partials of the hub segments
    _lib.check(lib.rgcn_aggregate_max_fwd(g.fwd.ref, _ptr(x), x.stride(0), d, _ptr(hi), _ptr(lo), hi.stride(0),
                                          2 if lo is not None else 1, _ptr(x_root), 0 if x_root is None else x_root.stride(0),
                                          _ptr(Hmax), _ptr(Hcnt), Hmax.stride(0), _ptr(ws), 0 if ws is None else ws.numel() * 4,
                                          _stream(x.device)), "rgcn_aggregate_max_fwd")
    return Hmax, Hcnt


def aggregate_max_bwd(g: RelGraph, gH: torch.Tensor, Hmax: torch.Tensor, Hcnt: torch.Tensor, x: torch.Tensor,
                      init: Optional[torch.Tensor] = None) -> torch.Tensor:
    """gX[j] = init[j] + sum_r sum_{(j->i, r)} [x[j] == Hmax[i, r]] gH[i, r] / Hcnt[i, r] over the transposed CSR
    (``rgcn_aggregate_max_bwd``; deterministic; NaN where Hmax is NaN, as torch's backward gives)."""
    lib = _lib.load()
    gH, x = _f32c(gH, "gH"), _f32c(x, "x")
    d = x.size(1)
    if gH.size(0) != g.n_dst or gH.size(1) < g.R * d or Hmax.shape != (g.n_dst, g.R * d) or Hcnt.shape != Hmax.shape:
        raise ValueError("gH, Hmax and Hcnt must be [n_dst, R*d]")
    if x.size(0) != g.n_src:
        raise ValueError("x must be the layer input [n_src, d]")
    if init is not None:
        init = _f32c(init, "init")
        if init.size(0) != g.n_src or init.size(1) < d:
            raise ValueError("init must be [n_src, >= d]")
    gX = torch.empty(g.n_src, d, dtype=torch.float32, device=x.device)
    ws = g.bwd.workspace(d)
    _lib.check(lib.rgcn_aggregate_max_bwd(g.bwd.ref, _ptr(gH), gH.stride(0), _ptr(Hmax), _ptr(Hcnt), Hmax.stride(0),
                                          _ptr(x), x.stride(0), d, _ptr(init), 0 if init is None else init.stride(0),
                                          _ptr(gX), gX.stride(0), _ptr(ws), 0 if ws is None else ws.numel() * 4,
                                          _stream(x.device)), "rgcn_aggregate_max_bwd")
    return gX


def masked_planes_struct(mask: torch.Tensor, scale: float, planes, colsum: Optional[torch.Tensor]):
    """``rgcn_masked_planes_out`` for (mask, scale, (hi, lo | None), colsum | None); the tensors must outlive the call."""
    if _f32c(mask, "mask") is not mask:
        raise ValueError("mask must be a 16-byte aligned row-major float32 matrix")
    hi, lo = planes
    if hi.dtype != torch.bfloat16 or hi.stride(1) != 1 or hi.shape[0] != mask.shape[0] or hi.shape[1] < mask.shape[1]:
        raise ValueError("masked planes must be bf16 row-major [rows, >= d]")
    return _lib.MaskedPlanesOut(mask.data_ptr(), mask.stride(0), float(scale), hi.data_ptr(), _dp(lo), hi.stride(0), _dp(colsum))


def _idx(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor")
    return t.to(torch.int64).contiguous()


def check_pairs(head, tail, rel, n_nodes: int, n_rel: int) -> None:
    """Raise IndexError on an out-of-range pair (synchronises; used outside the training hot loop)."""
    lib = _lib.load()
    flag = torch.zeros(1, dtype=torch.int32, device=head.device)
    _lib.check(lib.rgcn_check_pairs(_ptr(head), _ptr(tail), _ptr(rel), head.numel(), n_nodes, n_rel, _ptr(flag),
                                    _stream(head.device)), "rgcn_check_pairs")
    if int(flag.item()):
        raise IndexError("head/tail/relation index out of range")


def _rows(t, name):
    return None if t is None else _f32c(t, name).contiguous()


def distmult_fwd(emb_h: torch.Tensor, emb_t: torch.Tensor, head, tail, rel, rel_table: Optional[torch.Tensor],
                 rel_rows: Optional[torch.Tensor], rel_scale: Optional[torch.Tensor] = None) -> torch.Tensor:
    """score[p] = sum_k emb_h[hp, k] * r_p[k] * emb_t[tp, k]; hp = head[p] (or p when head is None)."""
    lib = _lib.load()
    emb_h, emb_t = _f32c(emb_h, "head embeddings"), _f32c(emb_t, "tail embeddings")
    head = None if head is None else _idx(head, "head")
    tail = None if tail is None else _idx(tail, "tail")
    rel = None if rel is None else _idx(rel, "rel")
    n = head.numel() if head is not None else emb_h.size(0)
    d = emb_h.size(1)
    if emb_t.size(1) != d:
        raise ValueError("head and tail embeddings differ in width")
    rel_rows, rel_table = _rows(rel_rows, "rel_rows"), _rows(rel_table, "rel_table")
    rel_scale = _rows(rel_scale, "rel_scale")
    score = torch.empty(n, dtype=torch.float32, device=emb_h.device)
    _lib.check(lib.rgcn_distmult_fwd(_ptr(emb_h), emb_h.stride(0), _ptr(emb_t), emb_t.stride(0), _ptr(head),
                                     _ptr(tail), _ptr(rel), _ptr(rel_table), _ptr(rel_rows), _ptr(rel_scale), n, d,
                                     _ptr(score),
                                     _stream(emb_h.device)), "rgcn_distmult_fwd")
    return score


def distmult_bwd(emb_h, emb_t, head, tail, rel, rel_table, rel_rows, g_score, need_rel_table_grad: bool,
                 rel_scale=None):
    """Returns (g_h, g_t, g_rel_table | None, g_rel_rows | None).  With index arrays and emb_h is emb_t the
    two row gradients are accumulated into ONE dense [N, d] buffer (returned as g_h, g_t = None)."""
    lib = _lib.load()
    shared = emb_h is emb_t and head is not None and tail is not None
    emb_h = _f32c(emb_h, "head embeddings")
    emb_t = emb_h if shared else _f32c(emb_t, "tail embeddings")
    head = None if head is None else _idx(head, "head")
    tail = None if tail is None else _idx(tail, "tail")
    rel = None if rel is None else _idx(rel, "rel")
    g_score = g_score.to(torch.float32).contiguous()
    n = g_score.numel()
    d = emb_h.size(1)
    dev = emb_h.device
    mk = torch.zeros if head is not None else torch.empty
    g_h = mk(emb_h.size(0), d, dtype=torch.float32, device=dev)
    if shared:
        g_t = g_h
    else:
        mk = torch.zeros if tail is not None else torch.empty
        g_t = mk(emb_t.size(0), d, dtype=torch.float32, device=dev)
    rel_rows, rel_table = _rows(rel_rows, "rel_rows"), _rows(rel_table, "rel_table")
    g_rows = torch.empty(n, d, dtype=torch.float32, device=dev) if rel_rows is not None else None
    g_tab = torch.zeros_like(rel_table) if (rel_rows is None and need_rel_table_grad) else None
    rel_scale = _rows(rel_scale, "rel_scale")
    _lib.check(lib.rgcn_distmult_bwd(_ptr(emb_h), emb_h.stride(0), _ptr(emb_t), emb_t.stride(0), _ptr(head),
                                     _ptr(tail), _ptr(rel), _ptr(rel_table), _ptr(rel_rows), _ptr(rel_scale),
                                     _ptr(g_score), n, d,
                                     _ptr(g_h), g_h.stride(0), _ptr(g_t), g_t.stride(0), _ptr(g_tab), _ptr(g_rows),
                                     _stream(dev)), "rgcn_distmult_bwd")
    return g_h, (None if shared else g_t), g_tab, g_rows


# ---- relational transform on the tensor cores -------------------------------------------------------
_WS = {}


def _workspace(device, nbytes: int) -> torch.Tensor:
    """Per-device scratch reused by every transform call (all calls are ordered on one stream)."""
    key = (device, _stream_id(device))
    ws = _WS.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(int(nbytes * 1.25) + 4096, dtype=torch.uint8, device=device)
        _WS[key] = ws
    return ws


def _mode_id(mode: str) -> int:
    if mode == "fp32":
        return 0
    if mode == "bf16":
        return 1
    raise ValueError(f"mode must be 'fp32' or 'bf16', got {mode!r}")


def _w2d(w: torch.Tensor, name: str) -> torch.Tensor:
    if not w.is_cuda or w.dtype != torch.float32:
        raise TypeError(f"{name} must be a CUDA float32 tensor")
    return w.detach().contiguous()


def alloc_planes(rows: int, cols: int, mode: str, device):
    """(hi, lo | None): bf16 row-major [rows, ld] with ld padded to a multiple of 8 (TMA stride alignment)."""
    ld = (cols + 7) // 8 * 8
    hi = torch.empty(rows, ld, dtype=torch.bfloat16, device=device)
    lo = torch.empty(rows, ld, dtype=torch.bfloat16, device=device) if mode == "fp32" else None
    if ld != cols:
        hi = hi[:, :cols]
        lo = None if lo is None else lo[:, :cols]
    return hi, lo


def split_planes(x: torch.Tensor, planes, col0: int = 0, relu_mask: Optional[torch.Tensor] = None,
                 colsum: bool = False, mask_scale: float = 1.0, out_f32: Optional[torch.Tensor] = None):
    """Write fp32 ``x`` [rows, cols] into columns [col0, col0+cols) of the bf16 planes (hi [, lo]); optionally zero
    where relu_mask <= 0 (and multiply the rest by ``mask_scale``, the 1 / (1 - p) of a fused dropout) and return the
    per-block column-sum partials [nblocks, cols] of the masked values."""
    lib = _lib.load()
    x = _f32c(x, "x")
    rows, cols = x.shape
    hi, lo = planes
    if relu_mask is not None:
        relu_mask = _f32c(relu_mask, "relu_mask")
    part = None
    if colsum:
        nb = lib.rgcn_split_planes_blocks(rows, cols)
        # no rows: the kernel writes no partial, so the one row handed on must be zero (a sum over nothing)
        part = (torch.empty if nb > 0 else torch.zeros)(max(nb, 1), cols, dtype=torch.float32, device=x.device)
    hi_v = hi[:, col0:col0 + cols]
    lo_v = None if lo is None else lo[:, col0:col0 + cols]
    _lib.check(lib.rgcn_split_planes(_ptr(x), x.stride(0), _ptr(relu_mask), 0 if relu_mask is None else relu_mask.stride(0),
                                     rows, cols, _ptr(hi_v), _ptr(lo_v), hi.stride(0), _ptr(part), float(mask_scale),
                                     _ptr(out_f32), 0 if out_f32 is None else out_f32.stride(0), _stream(x.device)),
               "rgcn_split_planes")
    return part


def dropout_counter(device) -> torch.Tensor:
    """Device-side step counter of the fused dropout (uint64 stored as int64 [1]); advanced by every layer call."""
    return torch.zeros(1, dtype=torch.int64, device=device)


def _ptr_array(ptrs):
    """HOST array of device pointers (the ``*_host`` arguments of the C ABI)."""
    return (C.c_void_p * len(ptrs))(*[int(a) for a in ptrs])


def transform_fwd(planes, K1: int, K2: int, W1: torch.Tensor, W2: Optional[torch.Tensor],
                  bias: Optional[torch.Tensor], relu: bool, mode: str, dropout_p: float = 0.0,
                  dropout_seed: int = 0, dropout_ctr: Optional[torch.Tensor] = None, peer_out=None,
                  peer_row0: int = 0, peer_ld: int = 0) -> torch.Tensor:
    """out = A @ [W1 ; W2] + bias (, ReLU (, dropout)) with A given as bf16 planes [n, K1 + K2] — tcgen05 kernel.
    ``peer_out``: device pointers of other GPUs' (peer-mapped) feature buffers [*, peer_ld]; the epilogue also stores
    every tile into rows ``peer_row0 + i`` of each of them (fused all-gather)."""
    lib = _lib.load()
    hi, lo = planes
    n = hi.size(0)
    W1 = _w2d(W1, "W1")
    d_out = W1.size(-1)
    if W2 is not None:
        W2 = _w2d(W2, "W2")
    if W1.numel() != K1 * d_out or (K2 and W2.numel() != K2 * d_out) or hi.size(1) < K1 + K2:
        raise ValueError("weight shapes do not match the operands")
    if bias is not None:
        bias = bias.detach().contiguous()
    out = torch.empty(n, d_out, dtype=torch.float32, device=hi.device)
    nb = lib.rgcn_transform_workspace_bytes(n, K1 + K2, d_out)
    ws = _workspace(hi.device, nb)
    _lib.check(lib.rgcn_transform_fwd(_ptr(hi), _ptr(lo), hi.stride(0), K1, K2, _ptr(W1), _ptr(W2), _ptr(bias),
                                      int(relu), n, d_out, _ptr(out), out.stride(0), _mode_id(mode), float(dropout_p),
                                      int(dropout_seed) & 0xFFFFFFFF, _ptr(dropout_ctr if dropout_p > 0 else None),
                                      _ptr_array(peer_out) if peer_out else None, len(peer_out) if peer_out else 0,
                                      int(peer_row0), int(peer_ld),
                                      _ptr(ws), ws.numel(), _stream(hi.device)), "rgcn_transform_fwd")
    return out


def prepare_weights(W1: torch.Tensor, W2: Optional[torch.Tensor], mode: str, dropout_ctr: Optional[torch.Tensor] = None
                    ) -> torch.Tensor:
    """bf16 hi (, lo) planes of the row-major block [W1; W2] ([K1 + K2, d_out]) — ``rgcn_prepare_weights``; the buffer
    serves ``transform_fwd(..., w_planes=)`` (MN-major operand) and ``transform_dgrad(..., w_planes=)`` (K-major)."""
    lib = _lib.load()
    W1 = _w2d(W1, "W1")
    d_out = W1.size(-1)
    K1 = W1.numel() // d_out
    K2 = 0
    if W2 is not None:
        W2 = _w2d(W2, "W2")
        K2 = W2.numel() // d_out
    wp = torch.empty(weight_planes_bytes(K1 + K2, d_out), dtype=torch.uint8, device=W1.device)
    _lib.check(lib.rgcn_prepare_weights(_ptr(W1), K1, _ptr(W2), K2, d_out, _mode_id(mode), _ptr(wp), _ptr(dropout_ctr),
                                        _stream(W1.device)), "rgcn_prepare_weights")
    return wp


def transform_fwd_w(planes, K: int, w_planes: torch.Tensor, d_out: int, bias: Optional[torch.Tensor], relu: bool, mode: str,
                    dropout_p: float = 0.0, dropout_seed: int = 0, dropout_ctr: Optional[torch.Tensor] = None,
                    row_offset: int = 0, out: Optional[torch.Tensor] = None, out_bf16: Optional[torch.Tensor] = None
                    ) -> torch.Tensor:
    """out = A @ W + bias (, ReLU (, dropout)) with the weights already converted (``prepare_weights``): the tcgen05 kernel
    alone, B read MN-major.  ``row_offset``: global row of A's row 0 (row-chunked calls draw one consistent dropout mask)."""
    lib = _lib.load()
    hi, lo = planes
    n = hi.size(0)
    if bias is not None:
        bias = bias.detach().contiguous()
    if out is None:
        out = torch.empty(n, d_out, dtype=torch.float32, device=hi.device)
    _lib.check(lib.rgcn_transform_fwd_w(_ptr(hi), _ptr(lo), hi.stride(0), K, _ptr(w_planes), _ptr(bias), int(relu), n, d_out,
                                        _ptr(out), out.stride(0), _mode_id(mode), float(dropout_p),
                                        int(dropout_seed) & 0xFFFFFFFF, _ptr(dropout_ctr if dropout_p > 0 else None),
                                        int(row_offset), None, 0, 0, 0, _ptr(out_bf16),
                                        0 if out_bf16 is None else out_bf16.stride(0), _stream(hi.device)), "rgcn_transform_fwd_w")
    return out


def transform_dgrad(g_planes, d_out: int, W1: torch.Tensor, W2: Optional[torch.Tensor], mode: str,
                    w_planes: Optional[torch.Tensor] = None) -> torch.Tensor:
    """gA = G @ [W1 ; W2]^T  -> [n, K1 + K2]; G given as bf16 planes [n, d_out].  ``w_planes``: the weights as converted
    by ``prepare_weights`` / ``layer_fwd`` (skips the conversion kernel)."""
    lib = _lib.load()
    hi, lo = g_planes
    n = hi.size(0)
    W1 = _w2d(W1, "W1")
    K1 = W1.numel() // d_out
    K2 = 0
    if W2 is not None:
        W2 = _w2d(W2, "W2")
        K2 = W2.numel() // d_out
    gA = torch.empty(n, K1 + K2, dtype=torch.float32, device=hi.device)
    if w_planes is not None:
        _lib.check(lib.rgcn_transform_dgrad_w(_ptr(hi), _ptr(lo), hi.stride(0), d_out, _ptr(w_planes), K1 + K2, n, _ptr(gA),
                                              gA.stride(0), _mode_id(mode), _stream(hi.device)), "rgcn_transform_dgrad_w")
        return gA
    nb = lib.rgcn_transform_workspace_bytes(n, K1 + K2, d_out)
    ws = _workspace(hi.device, nb)
    _lib.check(lib.rgcn_transform_dgrad(_ptr(hi), _ptr(lo), hi.stride(0), d_out, _ptr(W1), K1, _ptr(W2), K2, n,
                                        _ptr(gA), gA.stride(0), _mode_id(mode), _ptr(ws), ws.numel(),
                                        _stream(hi.device)), "rgcn_transform_dgrad")
    return gA


def transform_wgrad(a_planes, K1: int, K2: int, g_planes, d_out: int, colsum_partial: Optional[torch.Tensor], mode: str):
    """(gW1 [K1, d_out], gW2 [K2, d_out] | None, gbias [d_out] | None) = A^T @ G, sum of the column-sum partials."""
    lib = _lib.load()
    ahi, alo = a_planes
    ghi, glo = g_planes
    n = ahi.size(0)
    dev = ahi.device
    gW1 = torch.empty(K1, d_out, dtype=torch.float32, device=dev)
    gW2 = torch.empty(K2, d_out, dtype=torch.float32, device=dev) if K2 else None
    gb = torch.empty(d_out, dtype=torch.float32, device=dev) if colsum_partial is not None else None
    nb = lib.rgcn_transform_workspace_bytes(n, K1 + K2, d_out)
    ws = _workspace(dev, nb)
    _lib.check(lib.rgcn_transform_wgrad(_ptr(ahi), _ptr(alo), ahi.stride(0), K1, K2, _ptr(ghi), _ptr(glo), ghi.stride(0),
                                        d_out, n, _ptr(colsum_partial),
                                        0 if colsum_partial is None else colsum_partial.size(0), _ptr(gW1), _ptr(gW2),
                                        _ptr(gb), _mode_id(mode), _ptr(ws), ws.numel(), _stream(dev)),
               "rgcn_transform_wgrad")
    return gW1, gW2, gb


# ---- one layer per foreign call ---------------------------------------------------------------------
_WS_BYTES = {}
_WP_BYTES = {}


def bf16_gather() -> bool:
    """bf16-transform mode: gather a bf16 copy of the layer input (``PRIMEKG_RGCN_BF16_GATHER=0``: gather fp32 as round 1)."""
    import os
    return os.environ.get("PRIMEKG_RGCN_BF16_GATHER", "1") != "0"


def to_bf16(x: torch.Tensor) -> torch.Tensor:
    """bf16 copy of an fp32 matrix by our conversion kernel (row stride padded to a multiple of 8)."""
    x = _f32c(x, "x")
    hi, _ = alloc_planes(x.size(0), x.size(1), "bf16", x.device)
    split_planes(x, (hi, None))
    return hi


def prepared_weights() -> bool:
    """Weights converted once per layer call and shared by forward and dgrad (``PRIMEKG_RGCN_PREPARED_WEIGHTS=0``: the
    round-1 form, one conversion per GEMM)."""
    import os
    return os.environ.get("PRIMEKG_RGCN_PREPARED_WEIGHTS", "1") != "0"


def weight_planes_bytes(K: int, d_out: int) -> int:
    key = (int(K), int(d_out))
    nb = _WP_BYTES.get(key)
    if nb is None:
        nb = _WP_BYTES[key] = int(_lib.load().rgcn_weight_planes_bytes(int(K), int(d_out)))
    return nb


def _gemm_workspace(device, n: int, K: int, d_out: int) -> torch.Tensor:
    key = (n, K, d_out)
    nb = _WS_BYTES.get(key)
    if nb is None:
        nb = _WS_BYTES[key] = int(_lib.load().rgcn_transform_workspace_bytes(n, K, d_out))
    return _workspace(device, nb)


MARK_SOURCES_RATIO = 64      # rows of the graph per list entry from which the row-sparse walk marks its sources first (cfg3, ratio 32:
                             # most rows are marked anyway and the marked variant costs 7 %; a partitioned shard: ratio 300+)


def mark_sources() -> bool:
    import os
    return os.environ.get("RGCN_MARK_SOURCES", "1") != "0"


def _dp(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def layer_fwd(g: RelGraph, x_src: torch.Tensor, x_root: torch.Tensor, W2d: torch.Tensor, root: torch.Tensor,
              bias: torch.Tensor, relu: bool, mode: str, dropout_p: float = 0.0, dropout_seed: int = 0,
              dropout_ctr: Optional[torch.Tensor] = None, peer_out=None, peer_row0: int = 0, peer_ld: int = 0,
              pipeline: int = 0, x_bf16: Optional[torch.Tensor] = None, want_out_bf16: bool = False,
              rows: Optional[torch.Tensor] = None, slot: Optional[torch.Tensor] = None, dropout_row0: int = 0):
    """aggregate -> operand planes -> tensor-core transform of one layer in ONE C call (``rgcn_layer_fwd``).
    bf16 mode: ``x_bf16`` = a bf16 copy of x (the walk gathers it: half the bytes); ``want_out_bf16``: also return the
    layer output rounded to bf16 as a fourth result (the next layer's ``x_bf16``).
    Returns (out [n_dst, d_out], (A_hi, A_lo | None), w_planes | None): ``w_planes`` = the layer's weights as bf16 planes,
    converted once by the call; hand it to ``layer_bwd`` (its dgrad then skips the conversion).
    ``pipeline``: 0 = the library decides whether the walk of row chunk c + 1 runs under the transform of chunk c (it does
    not: measured slower; RGCN_PIPELINE=1 opts in), 1 = never, 2 = always.
    ``rows`` (int64 device list from ``rows_list_build``, with its ``slot`` map): the LISTED-ROWS form — only these rows of
    the output are computed (``out`` is uninitialised elsewhere) and the returned planes are compact
    [rows_compact_size(len(rows)), K] in list order; pass them to ``layer_bwd(..., rows=, slot=, a_compact=True)``.
    ``dropout_row0``: the layer-output row that row 0 of ``out`` is, for the dropout mask only — a destination-range
    shard passes its first node's global id, so every node draws the mask it draws on one GPU."""
    lib = _lib.load()
    x_src = _f32c(x_src, "x")
    x_root = x_src if x_root is x_src else _f32c(x_root, "x_root")
    if x_src.size(0) != g.n_src or x_root.size(0) != g.n_dst:
        raise ValueError(f"x has {x_src.size(0)} / {x_root.size(0)} rows, the graph gathers from {g.n_src} and updates {g.n_dst}")
    d_in = x_src.size(1)
    if d_in % 4 or d_in > 1024:
        raise ValueError("feature width must be a multiple of 4 and at most 1024")
    W2d, root = _w2d(W2d, "weight"), _w2d(root, "root")
    bias = bias.detach().contiguous()
    d_out = W2d.size(-1)
    K = (g.R + 1) * d_in
    if W2d.numel() != g.R * d_in * d_out or root.numel() != d_in * d_out:
        raise ValueError("weight shapes do not match the operands")
    dev = x_src.device
    listed = rows is not None
    if listed:
        if not prepared_weights() or dropout_p > 0 or want_out_bf16:
            raise ValueError("the listed-rows forward needs prepared weights and excludes dropout and the bf16 output copy")
        if rows.dtype != torch.int64 or rows.dim() != 1 or not rows.is_contiguous() or rows.numel() == 0:
            raise ValueError("rows must be a non-empty contiguous int64 list (rows_list_build)")
        if slot is None or slot.dtype != torch.int32 or slot.numel() != g.n_dst or not slot.is_contiguous():
            raise ValueError("slot must be the contiguous int32 [n_dst] map of rows_list_build")
    n_a = int(lib.rgcn_rows_compact_size(rows.numel())) if listed else g.n_dst
    A = alloc_planes(n_a, K, mode, dev)
    out = torch.empty(g.n_dst, d_out, dtype=torch.float32, device=dev)
    aws = g.fwd.workspace(d_in)
    gws = _gemm_workspace(dev, g.n_dst, K, d_out)
    peers = _ptr_array(peer_out) if peer_out else None
    # the layer's weights as bf16 planes, converted once by the call and kept for the backward's dgrad
    wp = torch.empty(weight_planes_bytes(K, d_out), dtype=torch.uint8, device=dev) if prepared_weights() else None
    use16 = mode == "bf16" and wp is not None and x_root is x_src
    if x_bf16 is not None and (not use16 or x_bf16.dtype != torch.bfloat16 or x_bf16.shape != x_src.shape or d_in % 8
                               or x_bf16.stride(1) != 1 or x_bf16.stride(0) % 8 or x_bf16.data_ptr() % 16):
        x_bf16 = None
    out16 = torch.empty(g.n_dst, d_out, dtype=torch.bfloat16, device=dev) if (want_out_bf16 and use16) else None
    args = _lib.LayerFwdArgs(
        g.fwd.ptr, x_src.data_ptr(), x_src.stride(0), x_root.data_ptr(), x_root.stride(0), d_in, d_out, int(relu),
        _mode_id(mode), W2d.data_ptr(), root.data_ptr(), bias.data_ptr(), float(dropout_p), int(dropout_seed) & 0xFFFFFFFF,
        _dp(dropout_ctr) if dropout_p > 0 else None, A[0].data_ptr(), _dp(A[1]), A[0].stride(0), out.data_ptr(),
        out.stride(0), C.cast(peers, C.c_void_p) if peers is not None else None, len(peer_out) if peer_out else 0,
        int(peer_row0), int(peer_ld), _dp(aws), 0 if aws is None else aws.numel() * 4, gws.data_ptr(), gws.numel(),
        _dp(wp), 0 if wp is None else wp.numel(), int(pipeline),
        _dp(x_bf16), 0 if x_bf16 is None else x_bf16.stride(0), _dp(out16), 0 if out16 is None else out16.stride(0),
        _dp(rows), rows.numel() if listed else 0, _dp(slot) if listed else None, int(dropout_row0))
    _lib.check(lib.rgcn_layer_fwd(C.byref(args), _stream(dev)), "rgcn_layer_fwd")
    if want_out_bf16:
        return out, A, wp, out16
    return out, A, wp


def layer_bwd(g: RelGraph, gO: torch.Tensor, relu_mask: Optional[torch.Tensor], mask_scale: float, planes, W2d: torch.Tensor,
              root: torch.Tensor, d_in: int, mode: str, need_x: bool, add_root_term: bool, need_w: bool, need_b: bool,
              gx_out: Optional[torch.Tensor] = None, rows: Optional[torch.Tensor] = None, g_ready=None, next_mask=None,
              slot: Optional[torch.Tensor] = None, w_planes: Optional[torch.Tensor] = None, return_compact: bool = False,
              a_compact: bool = False, scratch_w: bool = False):
    """split(gO, mask) -> dgrad -> transposed gather -> wgrad of one layer in ONE C call (``rgcn_layer_bwd``).
    Returns (g_x | None, gA | None, gW2d | None, g_root | None, g_bias | None); ``gA[:, R*d_in:]`` is the root-term
    gradient (already inside g_x when ``add_root_term``).
    ``rows`` (int64 device list, duplicates allowed): the caller guarantees gO is zero outside these rows; the backward
    then runs on the compacted rows (csrc/rowsparse.cu) with the same results, and gA comes back compact (``None`` here).
    ``slot`` (int32 [n]): the node -> first-position map of ``rows``, already built by the decoder's backward.
    ``return_compact`` (row-sparse form): return the compact gA [m_c + 1, K] (row m_c = zeros) instead of None and append
    the slot map to the result — a shard (add_root_term=False) reads its root-term gradient rows from it.
    ``a_compact`` (row-sparse form): ``planes`` are the compact planes of the listed-rows forward over this very list.
    ``g_ready`` = ((G_hi, G_lo | None), colsum [n, d_out]): this layer's masked output gradient as planes, already written
    by the downstream layer (skips the split pass).  ``next_mask`` = (mask [n_src, d_in], scale): also produce g_x masked
    for the upstream layer; the result gains a sixth entry ((hi, lo | None), colsum).
    ``scratch_w``: the weight is an intermediate (``is_grad_scratch``), its gradient a plain tensor outside the arena."""
    lib = _lib.load()
    gO = _f32c(gO, "gO")
    if relu_mask is not None:
        relu_mask = _f32c(relu_mask, "relu_mask")
    W2d, root = _w2d(W2d, "weight"), _w2d(root, "root")
    n, d_out = gO.shape
    if n != g.n_dst:
        raise ValueError("gO must have one row per destination")
    K1 = g.R * d_in
    K = K1 + d_in
    dev = gO.device
    A_hi, A_lo = planes
    sparse = rows is not None
    if sparse:
        if relu_mask is not None or (add_root_term and g.n_src != g.n_dst):
            raise ValueError("the row-sparse backward serves a layer without ReLU; on a destination-range shard "
                             "(n_src != n_dst) the root term stays separate (add_root_term=False)")
        rows = _idx(rows, "rows").reshape(-1)
        m = int(lib.rgcn_rows_compact_size(rows.numel()))
    else:
        m = n
    if g_ready is not None:
        if sparse or g_ready[0][0].shape != (n, d_out) or (mode == "fp32") != (g_ready[0][1] is not None):
            raise ValueError("g_ready does not match this layer")
        G, colsum_ready = g_ready
    else:
        G = alloc_planes(m, d_out, mode, dev)
    colsum = None
    if g_ready is not None:
        colsum = colsum_ready
    elif need_b:
        nb = lib.rgcn_rows_compact_blocks(rows.numel()) if sparse else lib.rgcn_split_planes_blocks(n, d_out)
        colsum = torch.empty(max(int(nb), 1), d_out, dtype=torch.float32, device=dev)
    gA = torch.empty(m + (1 if sparse else 0), K, dtype=torch.float32, device=dev) if need_x else None
    gx = None
    if need_x:
        gx = gx_out if gx_out is not None else torch.empty(g.n_src, d_in, dtype=torch.float32, device=dev)
    gW = None
    if need_w:
        gW = torch.empty(K1, d_out, dtype=torch.float32, device=dev) if scratch_w else param_grad(K1, d_out, device=dev)
    groot = param_grad(d_in, d_out, device=dev) if need_w else None
    gb = param_grad(d_out, device=dev) if (need_w and need_b) else None
    slot_ready = bool(sparse and slot is not None)
    if slot_ready and (slot.dtype != torch.int32 or slot.numel() != n or not slot.is_contiguous()):
        raise ValueError("slot must be a contiguous int32 [n_dst] tensor")
    if not slot_ready:
        slot = torch.empty(n, dtype=torch.int32, device=dev) if sparse else None
    if a_compact and (not sparse or A_hi.size(0) != m):
        raise ValueError("a_compact needs the row list of the listed-rows forward that made the planes")
    Ac = alloc_planes(m, K, mode, dev) if (sparse and need_w and not a_compact) else (None, None)
    nxt = nxt_struct = None
    if next_mask is not None and need_x:
        nmask, nscale = next_mask
        if nmask.shape != (g.n_src, d_in):
            raise ValueError("next_mask must be [n_src, d_in]")
        nplanes = alloc_planes(g.n_src, d_in, mode, dev)
        ncs = torch.empty(max(int(lib.rgcn_aggregate_row_blocks(g.bwd.ref, d_in)), 1), d_in, dtype=torch.float32, device=dev)
        nxt = (nplanes, ncs)
        nxt_struct = masked_planes_struct(nmask, nscale, nplanes, ncs)
    aws = g.bwd.workspace(d_in)
    gws = _gemm_workspace(dev, m, K, d_out)
    # graphs much larger than the row list: the walk skips the sources without an edge into a listed row
    src_flag = None
    if sparse and need_x and next_mask is None and g.n_src >= MARK_SOURCES_RATIO * rows.numel() and mark_sources():
        src_flag = torch.empty(g.n_src, dtype=torch.uint8, device=dev)
    args = _lib.LayerBwdArgs(
        g.bwd.ptr, gO.data_ptr(), gO.stride(0), _dp(relu_mask), 0 if relu_mask is None else relu_mask.stride(0),
        float(mask_scale), n, d_in, d_out, _mode_id(mode), int(add_root_term), W2d.data_ptr(), root.data_ptr(),
        A_hi.data_ptr(), _dp(A_lo), A_hi.stride(0), G[0].data_ptr(), _dp(G[1]), G[0].stride(0),
        _dp(colsum if (gb is not None and colsum is not None) else None),
        _dp(gA), 0 if gA is None else gA.stride(0), _dp(gx), 0 if gx is None else gx.stride(0), _dp(gW), _dp(groot), _dp(gb),
        _dp(aws), 0 if aws is None else aws.numel() * 4, gws.data_ptr(), gws.numel(),
        _dp(rows), 0 if rows is None else rows.numel(), _dp(slot), _dp(Ac[0]), _dp(Ac[1]),
        0 if Ac[0] is None else Ac[0].stride(0),
        C.pointer(nxt_struct) if nxt_struct is not None else None, int(g_ready is not None),
        0 if g_ready is None else colsum.size(0), int(slot_ready), _dp(w_planes), int(bool(a_compact)),
        g.fwd.ptr if src_flag is not None else None, _dp(src_flag))
    _lib.check(lib.rgcn_layer_bwd(C.byref(args), _stream(dev)), "rgcn_layer_bwd")
    if sparse and return_compact:
        return gx, gA, gW, groot, gb, slot
    if next_mask is not None:
        return gx, (None if sparse else gA), gW, groot, gb, nxt
    return gx, (None if sparse else gA), gW, groot, gb


def rows_list_build(head: torch.Tensor, tail: torch.Tensor, n_nodes: int):
    """(rows int64 [2 n], slot int32 [n_nodes]) of a link-prediction batch — ``rgcn_rows_list_build``: heads then tails
    (out-of-range indices parked on row 0), slot = node -> first list position or rows_compact_size(2 n)."""
    lib = _lib.load()
    head, tail = _idx(head, "head").reshape(-1), _idx(tail, "tail").reshape(-1)
    n = head.numel()
    if tail.numel() != n or n == 0:
        raise ValueError("head and tail must be non-empty and equally long")
    rows = torch.empty(2 * n, dtype=torch.int64, device=head.device)
    slot = torch.empty(int(n_nodes), dtype=torch.int32, device=head.device)
    _lib.check(lib.rgcn_rows_list_build(_ptr(head), _ptr(tail), n, int(n_nodes), _ptr(rows), _ptr(slot), _stream(head.device)),
               "rgcn_rows_list_build")
    return rows, slot


# ---- peer-memory exchange (destination-range partition over the GPUs of one NVSwitch domain) -----------
def p2p_push_rows(src: torch.Tensor, dst_ptrs, row0: int, ld_dst: int) -> None:
    """dst_q[row0 + i, :] = src[i, :] for every peer-mapped destination buffer (all-gather by push)."""
    lib = _lib.load()
    src = _f32c(src, "src")
    _lib.check(lib.rgcn_p2p_push_rows(_ptr(src), src.stride(0), src.size(0), src.size(1), _ptr_array(dst_ptrs),
                                      len(dst_ptrs), int(row0), int(ld_dst), _stream(src.device)), "rgcn_p2p_push_rows")


def p2p_pull_rows(part_ptrs, row0: int, ld_part: int, rows: torch.Tensor, out: torch.Tensor) -> None:
    """out[rows[c], :] = sum_q part_q[row0 + rows[c], :] (rank order) for the listed local rows only (reduce-scatter of a
    row-sparse gradient by pull); the other rows of ``out`` are left untouched."""
    lib = _lib.load()
    rows = _idx(rows, "rows").reshape(-1)
    out = _f32c(out, "out")
    _lib.check(lib.rgcn_p2p_pull_rows(_ptr_array(part_ptrs), len(part_ptrs), int(row0), int(ld_part), _ptr(rows), rows.numel(),
                                      out.size(0), out.size(1), _ptr(out), out.stride(0), _stream(out.device)),
               "rgcn_p2p_pull_rows")


def p2p_reduce_split(part_ptrs, row0: int, ld_part: int, rows: int, cols: int, device,
                     extra: Optional[torch.Tensor] = None, relu_mask: Optional[torch.Tensor] = None,
                     mask_scale: float = 1.0, want_fp32: bool = False, planes=None, colsum: bool = False):
    """v = extra + sum_q part_q[row0 : row0 + rows] (rank order), masked like ``split_planes``; returns
    (fp32 tensor | None, column-sum partials | None) and fills ``planes`` when given (reduce-scatter by pull)."""
    lib = _lib.load()
    if extra is not None:
        extra = _f32c(extra, "extra")
    if relu_mask is not None:
        relu_mask = _f32c(relu_mask, "relu_mask")
    out = torch.empty(rows, cols, dtype=torch.float32, device=device) if want_fp32 else None
    hi, lo = planes if planes is not None else (None, None)
    part = None
    if colsum:
        nb = lib.rgcn_split_planes_blocks(rows, cols)
        part = (torch.empty if nb > 0 else torch.zeros)(max(nb, 1), cols, dtype=torch.float32, device=device)
    _lib.check(lib.rgcn_p2p_reduce_split(_ptr_array(part_ptrs), len(part_ptrs), int(row0), int(ld_part), _ptr(extra),
                                         0 if extra is None else extra.stride(0), _ptr(relu_mask),
                                         0 if relu_mask is None else relu_mask.stride(0), float(mask_scale), rows, cols,
                                         _ptr(out), cols, _ptr(hi), _ptr(lo), 0 if hi is None else hi.stride(0),
                                         _ptr(part), _stream(device)), "rgcn_p2p_reduce_split")
    return out, part


# ---- fused BCE-with-logits (the loss of reference src/train.py:139, :300) ------------------------------
class _BCEWithLogits(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, labels):
        lib = _lib.load()
        logits = logits.contiguous()
        labels = labels.to(torch.float32).contiguous()
        loss = torch.empty((), dtype=torch.float32, device=logits.device)
        correct = torch.empty((), dtype=torch.int32, device=logits.device)
        _lib.check(lib.rgcn_bce_logits_fwd(_ptr(logits), _ptr(labels), logits.numel(), _ptr(loss), _ptr(correct),
                                           _stream(logits.device)), "rgcn_bce_logits_fwd")
        ctx.save_for_backward(logits, labels)
        ctx.mark_non_differentiable(correct)
        return loss, correct

    @staticmethod
    def backward(ctx, g_loss, _g_correct):
        lib = _lib.load()
        logits, labels = ctx.saved_tensors
        g = torch.empty_like(logits)
        g_loss = g_loss.to(torch.float32).contiguous()
        _lib.check(lib.rgcn_bce_logits_bwd(_ptr(logits), _ptr(labels), logits.numel(), _ptr(g_loss), _ptr(g),
                                           _stream(logits.device)), "rgcn_bce_logits_bwd")
        return g, None


def bce_with_logits(logits: torch.Tensor, labels: torch.Tensor, with_accuracy: bool = False):
    """Mean binary cross-entropy on logits in one kernel (+ the number of correct sigmoid > 0.5 predictions)."""
    if not logits.is_cuda or logits.dtype != torch.float32 or logits.dim() != 1:
        raise ValueError("bce_with_logits expects a 1-D float32 CUDA tensor of logits")
    loss, correct = _BCEWithLogits.apply(logits, labels)
    return (loss, correct) if with_accuracy else loss


# ---- fused tail of the training step (SURVEY §8f row 2; reference src/train.py:276-300, :321-322) --------------------
def rng_counter(device) -> torch.Tensor:
    """Device-side step counter of a counter-based RNG stream (uint64 stored as int64 [1])."""
    return torch.zeros(1, dtype=torch.int64, device=device)


def link_batch(pos_head: torch.Tensor, pos_tail: torch.Tensor, pos_rel: torch.Tensor, num_nodes: int, num_neg: int,
               seed: int, counter: torch.Tensor, out=None):
    """(heads, tails, rels, labels) = positives followed by ``num_neg`` corruptions each (``rgcn_link_batch``).
    ``out``: four preallocated tensors (e.g. the static buffers of a captured step)."""
    lib = _lib.load()
    ph, pt, pr = _idx(pos_head, "pos_head"), _idx(pos_tail, "pos_tail"), _idx(pos_rel, "pos_rel")
    h, t, r, y = out = _link_batch_out(ph, num_neg, out)
    _lib.check(lib.rgcn_link_batch(_ptr(ph), _ptr(pt), _ptr(pr), ph.numel(), int(num_neg), int(num_nodes),
                                   int(seed) & 0xFFFFFFFF, _ptr(counter), _ptr(h), _ptr(t), _ptr(r), _ptr(y),
                                   _stream(ph.device)), "rgcn_link_batch")
    return out


def _link_batch_out(ph: torch.Tensor, num_neg: int, out):
    tot = ph.numel() * (1 + num_neg)
    dev = ph.device
    if out is None:
        out = (torch.empty(tot, dtype=torch.int64, device=dev), torch.empty(tot, dtype=torch.int64, device=dev),
               torch.empty(tot, dtype=torch.int64, device=dev), torch.empty(tot, dtype=torch.float32, device=dev))
    h, t, r, y = out
    if not (h.numel() == t.numel() == r.numel() == y.numel() == tot and h.dtype == t.dtype == r.dtype == torch.int64
            and y.dtype == torch.float32 and all(x.is_contiguous() for x in out)):
        raise ValueError("out must be (int64, int64, int64, float32) contiguous tensors of n_pos * (1 + num_neg) entries")
    return out


def link_batch_ex(pos_head: torch.Tensor, pos_tail: torch.Tensor, pos_rel: torch.Tensor, num_nodes: int, num_neg: int,
                  seed: int, counter: torch.Tensor, out=None, *, num_rel: int = 0,
                  head_prob: Optional[torch.Tensor] = None, filter=None, constraints=None, max_tries: int = 1,
                  exhausted: Optional[torch.Tensor] = None, ticket: Optional[torch.Tensor] = None):
    """``link_batch`` with the tables of ``rgcn_link_batch_ex``, all device tensors: ``head_prob`` float32 [num_rel];
    ``filter`` = (keys int64, tails int32) of a ``KnownTriples``; ``constraints`` = (head_offsets int64 [num_rel + 1],
    head_nodes int32, tail_offsets, tail_nodes); ``exhausted`` int64 [1], incremented per negative that kept a rejected
    draw; ``ticket`` int32 [1], zero before the first call: one thread per output entry instead of one block.  The
    tables' contents are not checked here (``NegativeSampler`` checks them once at construction)."""
    lib = _lib.load()
    ph, pt, pr = _idx(pos_head, "pos_head"), _idx(pos_tail, "pos_tail"), _idx(pos_rel, "pos_rel")
    h, t, r, y = out = _link_batch_out(ph, num_neg, out)
    fk, ft = filter if filter is not None else (None, None)
    ho, hn, to, tn = constraints if constraints is not None else (None, None, None, None)
    a = _lib.LinkBatchArgs(
        pos_head=_ptr(ph), pos_tail=_ptr(pt), pos_rel=_ptr(pr), n_pos=ph.numel(), num_neg=int(num_neg),
        num_rel=int(num_rel), num_nodes=int(num_nodes), seed=int(seed) & 0xFFFFFFFF, max_tries=int(max_tries),
        counter=_ptr(counter), heads=_ptr(h), tails=_ptr(t), rels=_ptr(r), labels=_ptr(y), head_prob=_ptr(head_prob),
        filter_keys=_ptr(fk), filter_tails=_ptr(ft), n_filter=0 if fk is None else fk.numel(),
        head_offsets=_ptr(ho), head_nodes=_ptr(hn), tail_offsets=_ptr(to), tail_nodes=_ptr(tn),
        exhausted=_ptr(exhausted), ticket=_ptr(ticket))
    _lib.check(lib.rgcn_link_batch_ex(C.byref(a), _stream(ph.device)), "rgcn_link_batch_ex")
    return out


_LINK_WS = {}
_PAIR_STATUS = {}


def _link_workspace(device, n_pairs: int) -> torch.Tensor:
    """Zero-initialised partial / ticket buffer of the fused loss kernel (the kernel leaves the ticket at zero).
    One buffer per (device, STREAM, batch size): two streams issuing the same batch size never share a ticket."""
    key = (str(device), _stream_id(device), int(n_pairs))
    ws = _LINK_WS.get(key)
    if ws is None:
        ws = torch.zeros(int(_lib.load().rgcn_link_loss_workspace_bytes(n_pairs)), dtype=torch.uint8, device=device)
        _LINK_WS[key] = ws
    return ws


def pair_status(device) -> torch.Tensor:
    """Device flag (int32 [1]) the fused decoder kernels set when they meet an out-of-range head / tail / relation index
    (the pair is skipped: NaN score and loss, no gradient).  Polled by ``raise_on_bad_pairs``."""
    key = str(device)
    st = _PAIR_STATUS.get(key)
    if st is None:
        st = _PAIR_STATUS[key] = torch.zeros(1, dtype=torch.int32, device=device)
    return st


def raise_on_bad_pairs(device=None) -> None:
    """Raise IndexError if any fused decoder call since the last check met an out-of-range index (synchronises).  The
    reference's ``node_embeddings[idx]`` / ``nn.Embedding`` raise a device-side assert in the same situation; here the
    kernels skip the pair and the check is lazy: ``GraphedTrainStep`` polls after its warm-up steps, the modules poll on
    every call when ``PRIMEKG_RGCN_CHECK_PAIRS=1``, and a NaN loss is the always-visible symptom."""
    for key, st in list(_PAIR_STATUS.items()):
        if device is not None and key != str(device):
            continue
        if int(st.item()):
            st.zero_()
            raise IndexError("head / tail / relation index out of range in a link-prediction batch "
                             "(the offending pairs were skipped: NaN score, no gradient)")


def _check_pairs_now() -> bool:
    import os
    return os.environ.get("PRIMEKG_RGCN_CHECK_PAIRS", "0") == "1"


def _link_bwd(ctx_p_drop, ctx_seed, emb, rel_table, head, tail, rel, labels, score, state, g_loss, g_score, need_emb,
              need_tab):
    """Deterministic backward of the fused decoder (``rgcn_link_loss_bwd_rows``): returns (g_emb | None, g_tab | None)
    and announces the row list + slot map to the last encoder layer's row-sparse backward."""
    from . import rowsparse
    lib = _lib.load()
    dev = emb.device
    n, d, n_nodes, n_rel = head.numel(), emb.size(1), emb.size(0), rel_table.size(0)
    g_emb = torch.empty(n_nodes, d, dtype=torch.float32, device=dev)        # every row written exactly once by the kernel
    # ... unless emb is the output of a listed-rows last layer, whose backward reads the listed rows of g_emb alone
    listed_only = need_emb and rowsparse.is_listed_output(emb)
    g_tab = param_grad(*rel_table.shape, device=dev) if need_tab else None
    slot = torch.empty(n_nodes, dtype=torch.int32, device=dev)
    rows = torch.empty(2 * n, dtype=torch.int64, device=dev)
    ws = _workspace(dev, int(lib.rgcn_link_bwd_rows_workspace_bytes(n, n_rel, d)))     # position / pair contributions
    _lib.check(lib.rgcn_link_loss_bwd_rows(_ptr(emb), emb.stride(0), _ptr(head), _ptr(tail), _ptr(rel), _ptr(rel_table),
                                           _ptr(labels), _ptr(score), _ptr(g_loss), _ptr(g_score), n, d, ctx_p_drop,
                                           ctx_seed & 0xFFFFFFFF, _ptr(state), n_nodes, n_rel, _ptr(g_emb), g_emb.stride(0),
                                           _ptr(g_tab), _ptr(slot), _ptr(rows), _ptr(pair_status(dev)), int(listed_only), _ptr(ws),
                                           0 if ws is None else ws.numel(), _stream(dev)), "rgcn_link_loss_bwd_rows")
    if not need_emb:
        return None, g_tab
    rowsparse.announce(g_emb, rows, slot)                   # zero outside the head / tail rows
    return g_emb, g_tab


class _LinkLoss(torch.autograd.Function):
    """(loss, scores, n_correct) = BCEWithLogits(DistMult(emb[head], rel_table[rel] (dropout), emb[tail]), labels)."""

    @staticmethod
    def forward(ctx, emb, rel_table, head, tail, rel, labels, p_drop, seed, counter):
        lib = _lib.load()
        emb = _f32c(emb, "node embeddings")
        rel_table = _f32c(rel_table, "relation table").contiguous()
        head, tail, rel = _idx(head, "head"), _idx(tail, "tail"), _idx(rel, "rel")
        labels = labels.to(torch.float32).contiguous()
        n, d, dev = head.numel(), emb.size(1), emb.device
        if rel_table.size(1) != d or not (tail.numel() == rel.numel() == labels.numel() == n):
            raise ValueError("link_loss: shapes disagree")
        score = torch.empty(n, dtype=torch.float32, device=dev)
        loss = torch.empty((), dtype=torch.float32, device=dev)
        correct = torch.empty((), dtype=torch.int32, device=dev)
        state = torch.empty(1, dtype=torch.int64, device=dev) if p_drop > 0 else None
        ws = _link_workspace(dev, n)
        _lib.check(lib.rgcn_link_loss_fwd(_ptr(emb), emb.stride(0), _ptr(head), _ptr(tail), _ptr(rel), _ptr(rel_table),
                                          _ptr(labels), n, d, float(p_drop), int(seed) & 0xFFFFFFFF,
                                          _ptr(counter if p_drop > 0 else None), _ptr(state), _ptr(score), _ptr(loss),
                                          _ptr(correct), emb.size(0), rel_table.size(0), _ptr(pair_status(dev)),
                                          _ptr(ws), ws.numel(), _stream(dev)), "rgcn_link_loss_fwd")
        if _check_pairs_now():
            raise_on_bad_pairs(dev)
        ctx.save_for_backward(emb, rel_table, head, tail, rel, labels, score, state)
        ctx.p_drop, ctx.seed = float(p_drop), int(seed)
        ctx.mark_non_differentiable(score, correct)
        ctx.set_materialize_grads(False)          # no zero-filled gradients for the two non-differentiable outputs
        return loss, score, correct

    @staticmethod
    def backward(ctx, g_loss, _gs, _gc):
        emb, rel_table, head, tail, rel, labels, score, state = ctx.saved_tensors
        if g_loss is None:
            return (None,) * 9
        g_loss = g_loss.to(torch.float32).contiguous()
        g_emb, g_tab = _link_bwd(ctx.p_drop, ctx.seed, emb, rel_table, head, tail, rel, labels, score, state, g_loss, None,
                                 ctx.needs_input_grad[0], ctx.needs_input_grad[1])
        return g_emb, g_tab, None, None, None, None, None, None, None


def link_loss(emb, rel_table, head, tail, rel, labels, p_drop: float = 0.0, seed: int = 0, counter=None):
    """Fused decoder + loss of the training step; returns (loss, scores, n_correct)."""
    if not emb.is_cuda:
        raise RuntimeError("link_loss needs CUDA tensors: there is no CPU implementation of this path")
    if p_drop > 0 and counter is None:
        raise ValueError("link_loss: dropout needs a device counter (ops.rng_counter)")
    return _LinkLoss.apply(emb, rel_table, head, tail, rel, labels, float(p_drop), int(seed), counter)


# ---- basis decomposition of the relation weights (RGCNConv(num_bases = B)) -------------------------------------------
class _BasisCombine(torch.autograd.Function):
    """W[r] = sum_b comp[r, b] V[b]  ([R, in, out] from comp [R, B] and V [B, in, out]) and its backward, on our kernels
    (``rgcn_basis_combine`` / ``_bwd``) instead of a library matmul."""

    @staticmethod
    def forward(ctx, comp, V):
        lib = _lib.load()
        comp_c = comp.detach().to(torch.float32).contiguous()
        V_c = V.detach().to(torch.float32).contiguous()
        R, B = comp_c.shape
        io = V_c[0].numel()
        W = torch.empty(R, *V_c.shape[1:], dtype=torch.float32, device=V.device)
        _lib.check(lib.rgcn_basis_combine(_ptr(comp_c), _ptr(V_c), R, B, io, _ptr(W), _stream(V.device)), "rgcn_basis_combine")
        ctx.save_for_backward(comp_c, V_c)
        return W

    @staticmethod
    def backward(ctx, gW):
        lib = _lib.load()
        comp, V = ctx.saved_tensors
        R, B = comp.shape
        gW = gW.to(torch.float32).contiguous()
        g_comp = param_grad(R, B, device=V.device) if ctx.needs_input_grad[0] else None
        g_V = param_grad(*V.shape, device=V.device) if ctx.needs_input_grad[1] else None
        _lib.check(lib.rgcn_basis_combine_bwd(_ptr(comp), _ptr(V), _ptr(gW), R, B, V[0].numel(), _ptr(g_V), _ptr(g_comp),
                                              _stream(V.device)), "rgcn_basis_combine_bwd")
        return g_comp, g_V


def basis_combine(comp: torch.Tensor, V: torch.Tensor) -> torch.Tensor:
    if not V.is_cuda:
        raise RuntimeError("basis_combine needs CUDA tensors: there is no CPU implementation of this path")
    if comp.size(0) > 64 or comp.size(1) > 16 or V[0].numel() % 4:
        raise ValueError("basis_combine handles up to 64 relations, 16 bases and in * out a multiple of 4")
    return _BasisCombine.apply(comp, V)


# ---- block-diagonal relation weights (RGCNConv(num_blocks = nb)) -----------------------------------------------------
class _BlockDiag(torch.autograd.Function):
    """W [R, nb * bi, nb * bo] = blockdiag(blocks[r, 0], .., blocks[r, nb - 1]) from blocks [R, nb, bi, bo], and its
    backward (the diagonal blocks of the dense gradient), on ``rgcn_block_diag_expand`` / ``_gather``."""

    @staticmethod
    def forward(ctx, blocks):
        lib = _lib.load()
        b = blocks.detach().contiguous()
        R, nb, bi, bo = b.shape
        W = torch.empty(R, nb * bi, nb * bo, dtype=torch.float32, device=b.device)
        _lib.check(lib.rgcn_block_diag_expand(_ptr(b), R, nb, bi, bo, _ptr(W), _stream(b.device)), "rgcn_block_diag_expand")
        ctx.shape = (R, nb, bi, bo)
        return W

    @staticmethod
    def backward(ctx, gW):
        lib = _lib.load()
        R, nb, bi, bo = ctx.shape
        gW = gW.to(torch.float32).contiguous()
        g = param_grad(R, nb, bi, bo, device=gW.device)
        _lib.check(lib.rgcn_block_diag_gather(_ptr(gW), R, nb, bi, bo, _ptr(g), _stream(gW.device)), "rgcn_block_diag_gather")
        return g


def block_diag_weights(blocks: torch.Tensor) -> torch.Tensor:
    """The dense [R, in, out] relation weights of a block-diagonal layer (differentiable).  The layer's backward writes
    the dense weight gradient into scratch, not into the gradient arena: only the compact block gradient is a parameter
    gradient (``is_grad_scratch``)."""
    if not blocks.is_cuda:
        raise RuntimeError("block_diag_weights needs CUDA tensors: there is no CPU implementation of this path")
    if blocks.dim() != 4 or blocks.dtype != torch.float32:
        raise ValueError("blocks must be a float32 [R, num_blocks, in / num_blocks, out / num_blocks] tensor")
    W = _BlockDiag.apply(blocks)
    W._rgcn_grad_scratch = True
    return W


def is_grad_scratch(W: torch.Tensor) -> bool:
    """True for weights whose gradient is an intermediate (e.g. ``block_diag_weights``): a backward kernel writes it
    into a plain tensor instead of a slice of the gradient arena, which is sized for the parameters alone."""
    return bool(getattr(W, "_rgcn_grad_scratch", False))


class _PairScores(torch.autograd.Function):
    """scores[p] = <emb[head[p]], dropout(rel_table[rel[p]]), emb[tail[p]]> — ``LinkPredictor.score_pairs`` on the fused
    kernels' scores-only form: the relation dropout (reference src/models/rgcn.py:207-208) is the counter-based mask the
    backward regenerates, so no mask tensor and no ``bernoulli`` / ``div`` launches."""

    @staticmethod
    def forward(ctx, emb, rel_table, head, tail, rel, p_drop, seed, counter):
        lib = _lib.load()
        emb = _f32c(emb, "node embeddings")
        rel_table = _f32c(rel_table, "relation table").contiguous()
        head, tail, rel = _idx(head, "head"), _idx(tail, "tail"), _idx(rel, "rel")
        n, d, dev = head.numel(), emb.size(1), emb.device
        if rel_table.size(1) != d or not (tail.numel() == rel.numel() == n):
            raise ValueError("score_pairs: shapes disagree")
        score = torch.empty(n, dtype=torch.float32, device=dev)
        state = torch.empty(1, dtype=torch.int64, device=dev) if p_drop > 0 else None
        if n:
            ws = _link_workspace(dev, n)
            _lib.check(lib.rgcn_link_loss_fwd(_ptr(emb), emb.stride(0), _ptr(head), _ptr(tail), _ptr(rel), _ptr(rel_table),
                                              None, n, d, float(p_drop), int(seed) & 0xFFFFFFFF,
                                              _ptr(counter if p_drop > 0 else None), _ptr(state), _ptr(score), None, None,
                                              emb.size(0), rel_table.size(0), _ptr(pair_status(dev)),
                                              _ptr(ws), ws.numel(), _stream(dev)), "rgcn_link_loss_fwd")
            if _check_pairs_now():
                raise_on_bad_pairs(dev)
        ctx.save_for_backward(emb, rel_table, head, tail, rel, state)
        ctx.p_drop, ctx.seed = float(p_drop), int(seed)
        return score

    @staticmethod
    def backward(ctx, g_score):
        emb, rel_table, head, tail, rel, state = ctx.saved_tensors
        g_score = g_score.to(torch.float32).contiguous()
        if head.numel() == 0:
            return (torch.zeros_like(emb) if ctx.needs_input_grad[0] else None,
                    torch.zeros_like(rel_table) if ctx.needs_input_grad[1] else None, None, None, None, None, None, None)
        g_emb, g_tab = _link_bwd(ctx.p_drop, ctx.seed, emb, rel_table, head, tail, rel, None, None, state, None, g_score,
                                 ctx.needs_input_grad[0], ctx.needs_input_grad[1])
        return g_emb, g_tab, None, None, None, None, None, None


def pair_scores(emb, rel_table, head, tail, rel, p_drop: float = 0.0, seed: int = 0, counter=None) -> torch.Tensor:
    if not emb.is_cuda:
        raise RuntimeError("score_pairs needs CUDA tensors: there is no CPU implementation of this path")
    if p_drop > 0 and counter is None:
        raise ValueError("pair_scores: dropout needs a device counter (ops.rng_counter)")
    return _PairScores.apply(emb, rel_table, head, tail, rel, float(p_drop), int(seed), counter)


# ---- measurement aid ---------------------------------------------------------------------------------------------------
def probe_gather(table: torch.Tensor, idx: Optional[torch.Tensor], n_idx: Optional[int] = None, blocks_per_sm: int = 4) -> None:
    """The aggregation's row-gather pattern alone (``rgcn_probe_gather``): sums ``table[idx[i]]`` (``idx`` int32, or rows
    in order when None) — bench.py times it to measure the L2 / HBM gather ceilings on the box it runs on."""
    lib = _lib.load()
    table = _f32c(table, "table")
    if idx is not None and (idx.dtype != torch.int32 or not idx.is_contiguous()):
        raise ValueError("idx must be a contiguous int32 tensor")
    n = int(idx.numel() if idx is not None else (n_idx or table.size(0)))
    sink = _workspace(table.device, int(lib.rgcn_probe_gather_sink_floats(blocks_per_sm)) * 4 + 64)
    sp = (sink.data_ptr() + 15) // 16 * 16
    _lib.check(lib.rgcn_probe_gather(_ptr(table), table.stride(0), table.size(0), table.size(1), _ptr(idx), n,
                                     int(blocks_per_sm), C.c_void_p(sp), _stream(table.device)), "rgcn_probe_gather")

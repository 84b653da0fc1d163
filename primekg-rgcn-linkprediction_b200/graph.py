"""Device-resident relational graph: (dst, rel) CSR + (src, rel) transposed CSR + hub plans.

Built once per ``(edge_index, edge_type)`` pair by ``rgcn_csr_build`` / ``rgcn_hub_plan`` and cached:
the reference passes the SAME tensor objects on every step (src/train.py:130-135, :291-293, :389-391;
src/evaluate.py:251-254), so the cache hits on every call after the first.

HBM layout (all int32 / fp32, contiguous):
    rowptr   [n_dst * R + 1]   col   [E]   perm   [E]        keyed dst * R + rel
    rowptr_t [n_src * R + 1]   row_t [E]   perm_t [E]  w_t [E]   keyed src * R + rel
    inv_cnt  [n_dst * R]       1 / max(|N_r(i)|, 1)
    hub_keys / hub_chunk_ptr / chunk_table   per orientation (segments > hub_threshold() edges, cut into 128-edge chunks)
    row_order [n_rows]         rows by decreasing edge count, the order the lane groups take them
"""
from __future__ import annotations

import ctypes as C
import os
import weakref
from collections import OrderedDict
from typing import Optional

import torch

from . import _lib


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream_id(device) -> int:
    """torch's current stream on ``device`` as a raw handle (the direct binding is several times cheaper than building a
    ``torch.cuda.Stream`` object; the eager step makes ~10 such calls and is bound by the host)."""
    if _raw_stream is not None:
        idx = device.index if isinstance(device, torch.device) else torch.device(device).index
        if idx is None:
            idx = torch.cuda.current_device()
        return int(_raw_stream(idx))
    return int(torch.cuda.current_stream(device).cuda_stream)


def _stream(device) -> C.c_void_p:
    return C.c_void_p(_stream_id(device))


def hub_threshold() -> int:
    """Segments longer than this go through the chunk path (``PRIMEKG_RGCN_HUB_THRESHOLD``).  Measured on the B200
    (cfg2 / cfg3 aggregation, profiles/r1_agg_threshold_order_ab.txt): 128 beats 64 and 32 — the chunk path costs
    more than the shorter serial walks save."""
    t = int(os.environ.get("PRIMEKG_RGCN_HUB_THRESHOLD", "128"))
    if t < 1:
        raise ValueError("PRIMEKG_RGCN_HUB_THRESHOLD must be positive")
    return t


ORDER_CHUNK_ROWS = 8192      # rows per block of the chunk-wise row order (64 row tiles of the transform)


class _Orientation:
    """One CSR orientation + its hub plan, and the ``rgcn_csr_t`` handed to the kernels."""

    def __init__(self, rowptr, idx, w, n_rows, R, E):
        self.rowptr, self.idx, self.w = rowptr, idx, w
        self.n_rows, self.R, self.E = int(n_rows), int(R), int(E)
        self.hub_keys = self.hub_chunk_ptr = self.chunk_table = self.row_order = None
        self.n_hubs = self.n_chunks = 0
        self.threshold = hub_threshold()
        self._plan_hubs()
        order = os.environ.get("PRIMEKG_RGCN_ROW_ORDER", "auto")
        if order not in ("auto", "degree", "none"):
            raise ValueError("PRIMEKG_RGCN_ROW_ORDER must be auto, degree or none")
        # measured: +6-8 % on the L2-resident cfg2 aggregation, -3 % on cfg3 whose feature matrix does not fit the L2
        # (index order keeps neighbouring rows' gathers close) => by default only for graphs up to 64 k rows
        self.order_chunk_rows = 0
        if self.n_rows > 1 and (order == "degree" or (order == "auto" and self.n_rows <= 65536)):
            # rows by decreasing edge count (stable): blocks get rows of similar length, the longest walks start first
            ends = rowptr[self.R::self.R]
            deg = (ends - rowptr[:-1:self.R][: ends.numel()]).to(torch.int64)
            if self.n_rows >= 2 * ORDER_CHUNK_ROWS:
                # ... inside consecutive blocks of ORDER_CHUNK_ROWS rows, so that every block's rows stay a contiguous
                # range: rgcn_layer_fwd walks block c + 1 while the transform of block c runs (csrc/layer.cu)
                self.order_chunk_rows = ORDER_CHUNK_ROWS
                block = torch.arange(self.n_rows, device=deg.device, dtype=torch.int64) // ORDER_CHUNK_ROWS
                key = block * (int(deg.max()) + 1) + (int(deg.max()) - deg)
                self.row_order = torch.argsort(key, stable=True).to(torch.int32).contiguous()
            else:
                self.row_order = torch.argsort(deg, descending=True, stable=True).to(torch.int32).contiguous()
        self.struct = _lib.CsrStruct(
            _ptr(rowptr), _ptr(idx), _ptr(w), self.n_rows, self.E, self.R, self.n_hubs, self.n_chunks, self.threshold,
            _ptr(self.hub_keys), _ptr(self.hub_chunk_ptr), _ptr(self.chunk_table), _ptr(self.row_order),
            self.order_chunk_rows)
        self.ref = C.byref(self.struct)
        self.ptr = C.pointer(self.struct)          # for struct fields of type POINTER(rgcn_csr_t)
        self._ws = {}

    def _plan_hubs(self):
        lib = _lib.load()
        dev = self.rowptr.device
        cap = self.E // self.threshold + 1
        n_keys = self.n_rows * self.R
        hub_keys = torch.empty(cap, dtype=torch.int32, device=dev)
        chunk_ptr = torch.empty(cap + 1, dtype=torch.int32, device=dev)
        ws_bytes = lib.rgcn_hub_plan_workspace_bytes(n_keys, cap)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        nh, nc = C.c_int32(0), C.c_int32(0)
        _lib.check(lib.rgcn_hub_plan(_ptr(self.rowptr), n_keys, self.threshold, _ptr(hub_keys), _ptr(chunk_ptr), cap,
                                     C.byref(nh), C.byref(nc), _ptr(ws), ws_bytes, _stream(dev)), "rgcn_hub_plan")
        self.n_hubs, self.n_chunks = int(nh.value), int(nc.value)
        if self.n_hubs:
            self.hub_keys = hub_keys[: self.n_hubs].clone()
            self.hub_chunk_ptr = chunk_ptr[: self.n_hubs + 1].clone()
            self.chunk_table = torch.empty(self.n_chunks, 4, dtype=torch.int32, device=dev)
            _lib.check(lib.rgcn_hub_chunk_table(_ptr(self.hub_keys), _ptr(self.hub_chunk_ptr), self.n_hubs, self.R,
                                                _ptr(self.chunk_table), _stream(dev)), "rgcn_hub_chunk_table")

    def workspace(self, d: int) -> Optional[torch.Tensor]:
        """Chunk-partial buffer for feature width d (kept; sized n_chunks * d floats)."""
        if self.n_chunks == 0:
            return None
        ws = self._ws.get(d)
        if ws is None:
            ws = torch.empty(self.n_chunks * d + 64, dtype=torch.float32, device=self.rowptr.device)
            self._ws[d] = ws
        return ws


class RelGraph:
    """The preprocessed graph.  ``n_dst`` rows are aggregated into, ``n_src`` rows are gathered from
    (equal on one GPU; a destination-range shard has n_dst < n_src)."""

    def __init__(self, src: torch.Tensor, dst: torch.Tensor, rel: torch.Tensor, n_dst: int, n_src: int,
                 num_relations: int):
        lib = _lib.load()
        if not src.is_cuda:
            raise RuntimeError("RelGraph needs CUDA tensors: the RGCN B200 path has no CPU implementation")
        _lib.check(lib.rgcn_check_device(), "rgcn_check_device")
        src, dst, rel = (t.contiguous().to(torch.int64) for t in (src, dst, rel))
        E = int(rel.numel())
        if src.numel() != E or dst.numel() != E:
            raise ValueError("edge_index and edge_type disagree on the number of edges")
        dev = src.device
        R = int(num_relations)
        self.n_dst, self.n_src, self.R, self.E, self.device = int(n_dst), int(n_src), R, E, dev
        i32 = dict(dtype=torch.int32, device=dev)
        self.rowptr = torch.empty(n_dst * R + 1, **i32)
        self.rowptr_t = torch.empty(n_src * R + 1, **i32)
        self.col, self.perm = torch.empty(E, **i32), torch.empty(E, **i32)
        self.row_t, self.perm_t = torch.empty(E, **i32), torch.empty(E, **i32)
        self.inv_cnt = torch.empty(n_dst * R, dtype=torch.float32, device=dev)
        self.w_t = torch.empty(E, dtype=torch.float32, device=dev)
        status = torch.zeros(4, dtype=torch.int32, device=dev)
        ws_bytes = lib.rgcn_csr_build_workspace_bytes(E, n_dst, n_src, R)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            _lib.check(lib.rgcn_csr_build(
                _ptr(src), _ptr(dst), _ptr(rel), E, n_dst, n_src, R,
                _ptr(self.rowptr), _ptr(self.col), _ptr(self.perm),
                _ptr(self.rowptr_t), _ptr(self.row_t), _ptr(self.perm_t),
                _ptr(self.inv_cnt), _ptr(self.w_t), _ptr(status), _ptr(ws), ws_bytes, _stream(dev)),
                "rgcn_csr_build")
            st = status.cpu().tolist()          # one-off synchronisation per graph
            if st[0]:
                what = [n for b, n in ((1, "source index"), (2, "destination index"), (4, "edge_type")) if st[0] & b]
                raise IndexError(f"graph has out-of-range {', '.join(what)} "
                                 f"(n_src={n_src}, n_dst={n_dst}, num_relations={R})")
            self.max_seg, self.max_seg_t = st[2], st[3]
            self.fwd = _Orientation(self.rowptr, self.col, None, n_dst, R, E)
            self.bwd = _Orientation(self.rowptr_t, self.row_t, self.w_t, n_src, R, E)
        del ws

    def for_aggr(self, aggr: str) -> "RelGraph":
        """The graph as the layer kernels see it for aggregation ``aggr``: itself for 'mean' and 'max'; for 'sum' a view
        (made once, kept) whose two orientations carry unit edge weights.  The weighted walks then compute the plain
        segment sum: fma(1, v, s) rounds exactly like s + v, so the forward equals index_add_ in edge order, and the
        transposed walk is the sum's backward."""
        if aggr != "sum":
            return self
        views = self.__dict__.setdefault("_views", {})
        v = views.get(aggr)
        if v is None:
            v = RelGraph.__new__(RelGraph)
            v.__dict__.update({k: val for k, val in self.__dict__.items() if k != "_views"})
            ones = torch.ones(max(self.E, 1), dtype=torch.float32, device=self.device)
            with torch.cuda.device(self.device):
                v.fwd = _Orientation(self.rowptr, self.col, ones, self.n_dst, self.R, self.E)
                v.bwd = _Orientation(self.rowptr_t, self.row_t, ones, self.n_src, self.R, self.E)
            v.unit_w = ones
            views[aggr] = v
        return v

    @classmethod
    def from_edges(cls, edge_index: torch.Tensor, edge_type: torch.Tensor, num_nodes: int, num_relations: int):
        if edge_index.dim() != 2 or edge_index.size(0) != 2:
            raise ValueError("edge_index must have shape [2, E]")
        if edge_type is None:
            raise ValueError("edge_type is required")          # PyG asserts the same
        return cls(edge_index[0], edge_index[1], edge_type, num_nodes, num_nodes, num_relations)


# ---- cache keyed on tensor identity -------------------------------------------------------------
_CACHE: "OrderedDict[tuple, tuple]" = OrderedDict()
_CACHE_MAX = 8


def get_graph(edge_index: torch.Tensor, edge_type: torch.Tensor, num_nodes: int, num_relations: int) -> RelGraph:
    """Cached ``RelGraph`` for this ``(edge_index, edge_type)`` pair.

    An entry is valid only while the tensors it was built from are alive and unmodified
    (weak references + ``_version``), so a recycled allocation can never alias a stale graph."""
    key = (edge_index.data_ptr(), edge_type.data_ptr(), tuple(edge_index.shape), edge_index.stride(),
           str(edge_index.device), int(num_nodes), int(num_relations))
    hit = _CACHE.get(key)
    if hit is not None:
        g, r_ei, r_et, v_ei, v_et = hit
        if r_ei() is not None and r_et() is not None and edge_index._version == v_ei and edge_type._version == v_et:
            _CACHE.move_to_end(key)
            return g
        del _CACHE[key]
    g = RelGraph.from_edges(edge_index, edge_type, num_nodes, num_relations)
    _CACHE[key] = (g, weakref.ref(edge_index), weakref.ref(edge_type), edge_index._version, edge_type._version)
    while len(_CACHE) > _CACHE_MAX:
        _CACHE.popitem(last=False)
    return g


def clear_graph_cache() -> None:
    _CACHE.clear()


# ---- on-disk form (SURVEY.md §8f-4) ---------------------------------------------------------------
def graph_state(g: RelGraph) -> dict:
    """Plain dict of CPU tensors / ints with the preprocessed CSR + CSR^T, to be stored next to ``edge_index`` in the
    reference's ``data/processed/*.pt`` files (its loaders read keys by name and ignore extras: src/train.py:130-135),
    so later runs skip the sort."""
    keys = ("rowptr", "col", "perm", "rowptr_t", "row_t", "perm_t", "inv_cnt", "w_t")
    out = {f"csr_{k}": getattr(g, k).cpu() for k in keys}
    out.update(csr_n_dst=g.n_dst, csr_n_src=g.n_src, csr_num_relations=g.R, csr_num_edges=g.E,
               csr_max_seg=g.max_seg, csr_max_seg_t=g.max_seg_t, csr_format=1)
    return out


def graph_from_state(state: dict, device) -> RelGraph:
    """Rebuild a ``RelGraph`` on ``device`` from ``graph_state`` output (only the hub plan is recomputed)."""
    if state.get("csr_format") != 1:
        raise ValueError("unknown CSR format")
    g = RelGraph.__new__(RelGraph)
    _lib.check(_lib.load().rgcn_check_device(), "rgcn_check_device")
    g.n_dst, g.n_src, g.R, g.E = (int(state[k]) for k in ("csr_n_dst", "csr_n_src", "csr_num_relations", "csr_num_edges"))
    g.device = torch.device(device)
    for k in ("rowptr", "col", "perm", "rowptr_t", "row_t", "perm_t", "inv_cnt", "w_t"):
        setattr(g, k, state[f"csr_{k}"].to(g.device).contiguous())
    if g.rowptr.numel() != g.n_dst * g.R + 1 or g.col.numel() != g.E or int(g.rowptr[-1]) != g.E:
        raise ValueError("inconsistent CSR state")
    g.max_seg, g.max_seg_t = int(state["csr_max_seg"]), int(state["csr_max_seg_t"])
    with torch.cuda.device(g.device):
        g.fwd = _Orientation(g.rowptr, g.col, None, g.n_dst, g.R, g.E)
        g.bwd = _Orientation(g.rowptr_t, g.row_t, g.w_t, g.n_src, g.R, g.E)
    return g


def register_graph(edge_index: torch.Tensor, edge_type: torch.Tensor, g: RelGraph) -> None:
    """Seed the identity cache so ``model(edge_index, edge_type, ...)`` uses a pre-built / loaded graph."""
    key = (edge_index.data_ptr(), edge_type.data_ptr(), tuple(edge_index.shape), edge_index.stride(),
           str(edge_index.device), int(g.n_src), int(g.R))
    _CACHE[key] = (g, weakref.ref(edge_index), weakref.ref(edge_type), edge_index._version, edge_type._version)

"""TEST INFRASTRUCTURE: CPU stand-ins for the C-ABI wrappers in ``ops.py`` so the host-side plumbing above the
kernels (the partition plan, padded relabelling, collectives with autograd, layer wiring) can be exercised with
``gloo`` on a machine without a GPU.  Same formulas as oracle/rgcn_ref.py; never imported by the product."""
import torch


class CpuGraph:
    """Stand-in for graph.RelGraph: keeps the local edge list (src may live in a larger, padded id space)."""

    def __init__(self, src, dst, rel, n_dst, n_src, R):
        self.src, self.dst, self.rel = src.long(), dst.long(), rel.long()
        self.n_dst, self.n_src, self.R, self.E = int(n_dst), int(n_src), int(R), int(rel.numel())
        key = self.dst * R + self.rel
        self.cnt = torch.bincount(key, minlength=self.n_dst * R).clamp(min=1).to(torch.float32).view(self.n_dst, R)


def alloc_planes(rows, cols, mode, device):
    return torch.zeros(rows, cols), None


def aggregate_fwd(g, x, out_bf16=False, comp=None, planes=None):
    d = x.size(1)
    H = planes[0] if planes is not None else torch.zeros(g.n_dst, g.R * d)
    for r in range(g.R):
        m = g.rel == r
        s = torch.zeros(g.n_dst, d).index_add_(0, g.dst[m], x[g.src[m]])
        H[:, r * d:(r + 1) * d] = s / g.cnt[:, r:r + 1]
    return H


def split_planes(x, planes, col0=0, relu_mask=None, colsum=False, mask_scale=1.0):
    v = x if relu_mask is None else x * (relu_mask > 0) * mask_scale
    planes[0][:, col0:col0 + x.size(1)] = v
    return v.sum(0, keepdim=True) if colsum else None


def transform_fwd(planes, K1, K2, W1, W2, bias, relu, mode, dropout_p=0.0, dropout_seed=0, dropout_ctr=None):
    assert dropout_p == 0.0, "the CPU stand-in has no fused dropout"
    W = W1.reshape(K1, -1) if W2 is None else torch.cat([W1.reshape(K1, -1), W2], 0)
    out = planes[0][:, :K1 + K2] @ W.detach() + bias.detach()
    return out.clamp(min=0) if relu else out


def transform_dgrad(g_planes, d_out, W1, W2, mode):
    W = W1.reshape(-1, d_out) if W2 is None else torch.cat([W1.reshape(-1, d_out), W2], 0)
    return g_planes[0] @ W.detach().t()


def transform_wgrad(a_planes, K1, K2, g_planes, d_out, colsum_partial, mode):
    gW = a_planes[0][:, :K1 + K2].t() @ g_planes[0]
    return gW[:K1].contiguous(), (gW[K1:].contiguous() if K2 else None), (
        None if colsum_partial is None else colsum_partial.sum(0))


def aggregate_bwd(g, gH, d, init=None):
    gx = torch.zeros(g.n_src, d)
    if init is not None:
        gx[: init.size(0)] += init[:, :d]
    for r in range(g.R):
        m = g.rel == r
        contrib = gH[g.dst[m], r * d:(r + 1) * d] / g.cnt[g.dst[m], r:r + 1]
        gx.index_add_(0, g.src[m], contrib)
    return gx


def layer_fwd(g, x_src, x_root, W2d, root, bias, relu, mode, dropout_p=0.0, dropout_seed=0, dropout_ctr=None,
              peer_out=None, peer_row0=0, peer_ld=0, pipeline=0, x_bf16=None, want_out_bf16=False, rows=None, slot=None,
              dropout_row0=0):
    assert not peer_out and not want_out_bf16 and rows is None          # (the listed-rows forward needs CUDA index tensors)
    d_in = x_src.size(1)
    K1 = g.R * d_in
    A = alloc_planes(g.n_dst, K1 + d_in, mode, None)
    aggregate_fwd(g, x_src.detach(), planes=A)
    split_planes(x_root.detach(), A, col0=K1)
    out = transform_fwd(A, K1, d_in, W2d, root, bias, relu, mode)
    if dropout_p > 0.0:
        # the fused ReLU + dropout epilogue with the kernels' counter-based mask (the counter is advanced before the
        # transform reads it), keyed by the global row dropout_row0 + i; the backward needs no mask tensor (the output is
        # zero exactly where ReLU or dropout killed the element)
        from test_gpu_gemm_conformance import drop_keep, drop_scale
        dropout_ctr += 1
        keep = drop_keep(out.size(0), int(dropout_row0), out.size(1), dropout_p, int(dropout_seed), int(dropout_ctr),
                         device=out.device)
        out = torch.where(keep, out * drop_scale(dropout_p), 0.0)
    return out, A, None


def layer_bwd(g, gO, relu_mask, mask_scale, planes, W2d, root, d_in, mode, need_x, add_root_term, need_w, need_b,
              gx_out=None, rows=None, g_ready=None, next_mask=None, slot=None, w_planes=None, a_compact=False):
    assert g_ready is None and next_mask is None and not a_compact
    d_out = gO.size(1)
    K1 = g.R * d_in
    G = alloc_planes(gO.size(0), d_out, mode, None)
    colsum = split_planes(gO, G, relu_mask=relu_mask, colsum=True, mask_scale=mask_scale)
    gx = gA = gW = groot = gb = None
    if need_x:
        gA = transform_dgrad(G, d_out, W2d, root, mode)
        gx = aggregate_bwd(g, gA, d_in, init=gA[:, K1:] if add_root_term else None)
    if need_w:
        gW, groot, gb = transform_wgrad(planes, K1, d_in, G, d_out, colsum if need_b else None, mode)
    return gx, gA, gW, groot, gb


# ---- the rest of the product's kernel entry points, for running the WHOLE module trio on a CPU-only machine ----------
_GRAPHS = {}


def get_graph(edge_index, edge_type, num_nodes, num_relations):
    if edge_type is None:
        raise ValueError("edge_type is required")
    key = (edge_index.data_ptr(), edge_type.data_ptr(), tuple(edge_index.shape), edge_index._version, int(num_nodes))
    g = _GRAPHS.get(key)
    if g is None:
        if edge_index.numel() and (int(edge_index.min()) < 0 or int(edge_index.max()) >= num_nodes):
            raise IndexError("graph has out-of-range node index")
        if len(_GRAPHS) > 8:
            _GRAPHS.clear()
        g = _GRAPHS[key] = CpuGraph(edge_index[0], edge_index[1], edge_type, num_nodes, num_nodes, num_relations)
        g._keep = (edge_index, edge_type)
    return g


def pair_scores(emb, rel_table, head, tail, rel, p_drop=0.0, seed=0, counter=None):
    r = rel_table[rel]
    if p_drop > 0.0:
        r = torch.nn.functional.dropout(r, p_drop, True)
    return (emb[head] * r * emb[tail]).sum(1)


def link_loss(emb, rel_table, head, tail, rel, labels, p_drop=0.0, seed=0, counter=None):
    s = pair_scores(emb, rel_table, head, tail, rel, p_drop)
    loss = torch.nn.functional.binary_cross_entropy_with_logits(s, labels)
    return loss, s.detach(), ((torch.sigmoid(s.detach()) > 0.5).float() == labels).sum().to(torch.int32)


def rank_prep(emb, idx, rel_table, rel, normalize):
    a = emb.detach() if idx is None else emb.detach()[idx]
    if rel is not None:
        a = a * rel_table.detach()[rel]
    return a / a.norm(dim=1, keepdim=True) if normalize else a


def scores_from_rows(A, B, b_idx=None, alpha=1.0, beta=0.0, method="tc"):
    Bm = B.detach() if b_idx is None else B.detach()[b_idx]
    return alpha * (A.detach() @ Bm.t()) + beta


def install_full(monkeypatch, pkg):
    """Patch EVERY device entry point the module trio reaches (``ops``, the graph cache, the CUDA guards, the all-pairs
    helpers) with the CPU stand-ins, through ``monkeypatch`` so the patches are undone after the test."""
    from primekg_rgcn_linkprediction_b200 import conv, graph, modules, ops, rank
    for name in ("alloc_planes", "aggregate_fwd", "split_planes", "transform_fwd", "transform_dgrad",
                 "transform_wgrad", "aggregate_bwd", "layer_fwd", "layer_bwd", "pair_scores", "link_loss"):
        monkeypatch.setattr(ops, name, globals()[name])
    for mod in (graph, conv, modules):
        monkeypatch.setattr(mod, "get_graph", get_graph)
    monkeypatch.setattr(modules, "_need_cuda", lambda t, what: None)
    monkeypatch.setattr(rank, "_prep", rank_prep)
    monkeypatch.setattr(rank, "scores_from_rows", scores_from_rows)
    _GRAPHS.clear()


def install(monkeypatch_target):
    """Replace the kernel wrappers in ``ops`` (module object) by the CPU stand-ins."""
    for name in ("alloc_planes", "aggregate_fwd", "split_planes", "transform_fwd", "transform_dgrad",
                 "transform_wgrad", "aggregate_bwd", "layer_fwd", "layer_bwd"):
        setattr(monkeypatch_target, name, globals()[name])

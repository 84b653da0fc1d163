"""The destination-range partitioned layer on ONE GPU with P emulated ranks (P distinct local buffers stand in for the
peer-mapped ones): every kernel runs on a real shard — a rectangular CSR (n_dst = max_n, n_src = P * max_n, padded
source ids), the transform epilogue storing into P buffers at peer_row0 = p * max_n, a transposed walk writing a
partial g_x over all P * max_n rows without the root term, and the pull-reduce / pull-rows exchange kernels over P
distinct partials — against the whole-graph layer and a float64 restatement.

* Forward: ``local_edges`` keeps the edge order, so every (row, relation) segment of a shard sums the same terms in the
  same order as the whole graph: shard outputs and operand planes must equal the whole-graph layer's rows BIT FOR BIT,
  under every schedule.  The planes also lie within ``(len + 2) * 2^-24 * sum|x| / len + split * |H|`` of a float64 mean
  (split = 2^-16 for the hi + lo pair of the fp32 mode, 2^-8 for the bf16 hi plane).
  Schedule 3 (the fused walk + transform kernel, opt-in) is the exception: it splits each row tile's edge stream into
  equal shares per producer warp wherever that cuts a row, so a row's fp32 rounding depends on the other rows of its
  tile, and a shard's tiles hold other rows than the whole graph's.  There shard and whole graph must agree within twice
  the float64 bound of the layer output, and the shard's planes lie within the bound above.
* Backward: per-element bounds built from the float64 sum of |terms| through dgrad (``2^-14 + (3 d_out + 3) * 2^-23``
  in fp32, ``2^-7 + 2^-14 + (d_out + 3) * 2^-23`` in bf16: two rounded operands per product and the tensor core's
  adder), the walk and the reduction over ranks (one 2^-24 per added term); a wrong row fails, not just a wrong norm.
* Dropout: the fused mask is keyed by the global node id (``dropout_row0``), so shard p's rows draw the masks of the
  one-GPU layer and not those of shard 0's rows.

The worst error-to-bound ratio of each family is printed when the module finishes (``pytest -s``).
"""
import pytest
import torch

from test_gpu_gemm_conformance import drop_keep, drop_scale

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
U = 2.0 ** -24
E23 = 2.0 ** -23
HUB_CHUNK = 128                               # kHubChunk of csrc/common.cuh
MODES = ["fp32", "bf16"]
CASES = [  # (graph, P, d_in, d_out)
    ("primekg", 2, 64, 128),                  # max_n >= 16,384: chunk-wise row order, pipelined chunks
    ("primekg", 8, 128, 256),
    ("skewed", 3, 256, 64),                   # a third of the edges into one node: uneven ranges, hub segments
    ("tiny", 8, 64, 64),                      # ranks that own no row
]
SEED, CTR0 = 0x5EED1234, (1 << 32) * 3 + 17

_WORST = {}


@pytest.fixture(scope="module")
def ops(lib_built):
    from primekg_rgcn_linkprediction_b200 import ops
    return ops


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for fam in sorted(_WORST):
        print(f"\n[partition shards] {fam}: worst |err| / bound = {_WORST[fam]:.3g}", end="")
    print()


# ---- graphs, shards, inputs -------------------------------------------------------------------------------------------
_GRAPHS = {}


def _graph(name):
    from primekg_rgcn_linkprediction_b200 import synth
    if name == "primekg":
        kg = synth.primekg_subgraph(150_000, seed=3)
        return kg.edge_index, kg.edge_type, kg.num_nodes, kg.num_relations
    if name == "skewed":
        kg = synth.uniform_kg(6000, 60_000, 4, seed=5)
        ei = kg.edge_index.clone()
        ei[1, ::3] = 3
        return ei, kg.edge_type, kg.num_nodes, kg.num_relations
    kg = synth.uniform_kg(10, 40, 2, seed=6)
    ei = kg.edge_index.clone()
    ei[1, ::2] = 0
    return ei, kg.edge_type, kg.num_nodes, kg.num_relations


class _Setup:
    """Whole graph + the P shards of one partition, built once per (graph, P)."""

    def __init__(self, name, P):
        import primekg_rgcn_linkprediction_b200 as pkg
        from primekg_rgcn_linkprediction_b200 import dist as D
        ei, et, N, R = _graph(name)
        self.ei, self.et = ei.to(DEV), et.to(DEV)
        self.N, self.R, self.P = N, R, P
        self.plan = D.plan_partition(self.ei[1], N, P)
        self.max_n = self.plan.max_n
        self.whole = pkg.RelGraph.from_edges(self.ei, self.et, N, R)
        self.local = [D.local_edges(self.ei, self.et, self.plan, p) for p in range(P)]
        self.shards = [pkg.RelGraph(s, d, r, self.max_n, P * self.max_n, R) for s, d, r in self.local]
        self.pid = self.plan.to_padded(torch.arange(N, device=DEV))

    def rng(self, p):
        return self.plan.bounds[p], self.plan.bounds[p + 1]


def _setup(name, P):
    key = (name, P)
    if key not in _GRAPHS:
        _GRAPHS[key] = _Setup(name, P)
    return _GRAPHS[key]


def _gen(seed):
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    return g


def _rows_scaled(n, d, g):
    """normal values with row scales over 2^-4 .. 2^4 and 30 % exact zeros (a ReLU output)."""
    x = torch.randn(n, d, generator=g, device=DEV) * torch.exp2(torch.randint(-4, 5, (n, 1), generator=g, device=DEV).float())
    return torch.where(torch.rand(n, d, generator=g, device=DEV) < 0.3, 0.0, x)


def _inputs(S, d_in, d_out, seed):
    g = _gen(seed)
    x = _rows_scaled(S.N, d_in, g)
    # padding rows: finite garbage no edge may read (a previous layer's relu(bias) lands there in the model)
    x_full = torch.full((S.P * S.max_n, d_in), 7777.0, device=DEV) + torch.randn(S.P * S.max_n, d_in, generator=g, device=DEV)
    x_full[S.pid] = x
    W = torch.randn(S.R * d_in, d_out, generator=g, device=DEV) * d_in ** -0.5
    root = torch.randn(d_in, d_out, generator=g, device=DEV) * d_in ** -0.5
    b = torch.randn(d_out, generator=g, device=DEV) * 0.1
    return x, x_full, W, root, b


# ---- checks -------------------------------------------------------------------------------------------------------------
def _bits(got, want, what):
    bad = ~((got == want) | (got.isnan() & want.isnan()))
    if bool(bad.any()):
        i = int(bad.flatten().nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements differ; first at flat index {i}: got "
                             f"{float(got.flatten()[i])!r}, want {float(want.flatten()[i])!r}")


def _check(fam, got, ref, bound, what):
    err = (got.double() - ref).abs()
    bad = ~(err <= bound)                                # NaN fails
    pos = bound > 0
    worst = float((err[pos] / bound[pos]).max()) if bool(pos.any()) else 0.0
    _WORST[fam] = max(_WORST.get(fam, 0.0), worst)
    if bool(bad.any()):
        i = int(bad.flatten().nonzero()[0])
        raise AssertionError(f"{fam} {what}: {int(bad.sum())} of {bad.numel()} elements outside the bound; first at flat "
                             f"index {i} (row {i // got.size(-1)}): got {float(got.flatten()[i])!r}, ref "
                             f"{float(ref.flatten()[i])!r}, bound {float(bound.flatten()[i]):.3g}")


def _split_rel(mode):
    return 2.0 ** -16 if mode == "fp32" else 2.0 ** -8


def _plane_value(A, rows, cols):
    hi, lo = A
    v = hi[rows, :cols].double()
    return v if lo is None else v + lo[rows, :cols].double()


def _agg64(x64, src, dst, rel, n, R):
    """float64 per-(row, relation) means of x and of |x|, and the segment lengths [n, R]."""
    d = x64.size(1)
    key = dst * R + rel
    cnt = torch.bincount(key, minlength=n * R)
    c = cnt.clamp(min=1).double()[:, None]
    H = torch.zeros(n * R, d, dtype=torch.float64, device=DEV).index_add_(0, key, x64[src]) / c
    S = torch.zeros(n * R, d, dtype=torch.float64, device=DEV).index_add_(0, key, x64[src].abs()) / c
    return H.view(n, R * d), S.view(n, R * d), cnt.view(n, R)


# =========================================================================================================================
# a. the shard CSR against a rectangular restatement of oracle.csr_oracle
# =========================================================================================================================
def _csr_rect(major, minor, rel, n_major, R):
    key = major * R + rel
    perm = torch.sort(key, stable=True).indices
    cnt = torch.bincount(key, minlength=n_major * R)
    rowptr = torch.zeros(n_major * R + 1, dtype=torch.int64, device=DEV)
    rowptr[1:] = torch.cumsum(cnt, 0)
    return rowptr, minor[perm], perm, cnt


def _check_orientation(ori, rowptr, R, what):
    from primekg_rgcn_linkprediction_b200.graph import ORDER_CHUNK_ROWS
    seg = rowptr[1:] - rowptr[:-1]
    hubs = (seg > ori.threshold).nonzero().flatten()
    assert ori.n_hubs == hubs.numel(), what
    if hubs.numel():
        assert torch.equal(ori.hub_keys.long(), hubs), what
        chunks = (seg[hubs] + HUB_CHUNK - 1) // HUB_CHUNK
        ptr = torch.zeros(hubs.numel() + 1, dtype=torch.int64, device=DEV)
        ptr[1:] = torch.cumsum(chunks, 0)
        assert torch.equal(ori.hub_chunk_ptr.long(), ptr), what
        assert ori.n_chunks == int(ptr[-1]), what
    else:
        assert ori.n_chunks == 0, what
    n = ori.n_rows
    if ori.row_order is None:
        return
    order = ori.row_order.long()
    pos = torch.arange(n, device=DEV)
    assert torch.equal(torch.sort(order).values, pos), what + ": row_order is not a permutation"
    deg = seg.view(n, R).sum(1)[order]
    if ori.order_chunk_rows > 0:
        assert ori.order_chunk_rows == ORDER_CHUNK_ROWS
        assert torch.equal(order // ORDER_CHUNK_ROWS, pos // ORDER_CHUNK_ROWS), what + ": a block left its rows"
        same = (pos[1:] // ORDER_CHUNK_ROWS) == (pos[:-1] // ORDER_CHUNK_ROWS)
        assert bool(torch.all(deg[1:][same] <= deg[:-1][same])), what
    else:
        assert bool(torch.all(deg[1:] <= deg[:-1])), what


@pytest.mark.parametrize("name,P", sorted({(c[0], c[1]) for c in CASES}))
def test_shard_csr(ops, name, P):
    S = _setup(name, P)
    assert S.plan.bounds[0] == 0 and S.plan.bounds[-1] == S.N
    sizes = [S.plan.size(p) for p in range(P)]
    if name == "primekg" and P == 2:
        assert S.max_n >= 16_384 and all(g.fwd.order_chunk_rows > 0 for g in S.shards)
    if name == "tiny":
        assert min(sizes) == 0
    assert any(s < S.max_n for s in sizes)                # padding rows
    for p, (g, (src, dst, rel)) in enumerate(zip(S.shards, S.local)):
        what = f"{name} P={P} rank {p}"
        n_dst, n_src, R = S.max_n, P * S.max_n, S.R
        assert (g.n_dst, g.n_src, g.E) == (n_dst, n_src, src.numel())
        rowptr, col, perm, cnt = _csr_rect(dst, src, rel, n_dst, R)
        rowptr_t, row_t, perm_t, _ = _csr_rect(src, dst, rel, n_src, R)
        for got, want, k in ((g.rowptr, rowptr, "rowptr"), (g.col, col, "col"), (g.perm, perm, "perm"),
                             (g.rowptr_t, rowptr_t, "rowptr_t"), (g.row_t, row_t, "row_t"), (g.perm_t, perm_t, "perm_t")):
            assert torch.equal(got.long(), want), f"{what}: {k}"
        inv = 1.0 / cnt.clamp(min=1).float()
        assert torch.equal(g.inv_cnt, inv), what
        assert torch.equal(g.w_t, inv[(dst * R + rel)[perm_t]]), what
        _check_orientation(g.fwd, rowptr, R, what + " fwd")
        _check_orientation(g.bwd, rowptr_t, R, what + " bwd")


# =========================================================================================================================
# b. forward: shard rows == whole-graph rows, bitwise; peer stores; listed form
# =========================================================================================================================
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name,P,d_in,d_out", CASES)
def test_shard_forward(ops, name, P, d_in, d_out, mode):
    S = _setup(name, P)
    x, x_full, W, root, b = _inputs(S, d_in, d_out, seed=P * 1000 + d_in + d_out)
    K1, K = S.R * d_in, (S.R + 1) * d_in
    x64 = x.double()
    _, SH, _ = _agg64(x64, S.ei[0], S.ei[1], S.et, S.N, S.R)
    S_out = torch.cat([SH, x64.abs()], 1) @ torch.cat([W, root], 0).double().abs()     # sum |terms| of each output
    for sched in (1, 2, 3):
        out_w, A_w, _ = ops.layer_fwd(S.whole, x, x, W, root, b, True, mode, pipeline=sched)
        for p in range(P):
            lo, hi = S.rng(p)
            m, row0 = hi - lo, p * S.max_n
            bufs = [torch.full((P * S.max_n, d_out), float("nan"), device=DEV) for _ in range(P)]
            out, A, _ = ops.layer_fwd(S.shards[p], x_full, x_full[row0:row0 + S.max_n], W, root, b, True, mode,
                                      peer_out=[t.data_ptr() for t in bufs], peer_row0=row0, peer_ld=d_out, pipeline=sched)
            torch.cuda.synchronize()
            what = f"{name} P={P} {mode} schedule {sched} rank {p}"
            if sched != 3:
                _bits(out[:m], out_w[lo:hi], what + ": output")
                _bits(A[0][:m, :K], A_w[0][lo:hi, :K], what + ": hi plane")
                if mode == "fp32":
                    _bits(A[1][:m, :K], A_w[1][lo:hi, :K], what + ": lo plane")
            elif m:
                # the fused kernel cuts each row tile's edge stream into equal shares per producer warp, whatever rows
                # that splits, and sums a cut row from its pieces: the fp32 rounding of a row depends on the other rows
                # of its tile, which differ between a shard and the whole graph.  Both sides lie within the float64 bound.
                rel = _split_rel(mode) + (S.whole.max_seg + 2) * U + ((3 * K if mode == "fp32" else K) + 3) * E23
                _check(f"forward schedule 3 {mode}", out[:m], out_w[lo:hi].double(),
                       2 * rel * S_out[lo:hi] + 2 * U * b.double().abs(), what + ": output against the whole graph")
            for q, t in enumerate(bufs):
                _bits(t[row0:row0 + S.max_n], out, f"{what}: peer buffer {q}")
                assert bool(t[:row0].isnan().all()) and bool(t[row0 + S.max_n:].isnan().all()), \
                    f"{what}: peer buffer {q} written outside rows [{row0}, {row0 + S.max_n})"
            if sched != 2 and m:
                # the operand planes against a float64 aggregation of x over this shard's edges (global node ids)
                src, dst, rel = S.local[p]
                H, Sx, cnt = _agg64(x_full.double(), src, dst, rel, S.max_n, S.R)
                seg = cnt[:m].repeat_interleave(d_in, 1).double()
                bound = (seg + 2) * U * Sx[:m] + _split_rel(mode) * H[:m].abs()
                _check(f"forward planes {mode}", _plane_value(A, slice(0, m), K1), H[:m], bound, what)
                xr = x64[lo:hi]
                _check(f"forward planes {mode}", _plane_value((A[0][:, K1:], None if A[1] is None else A[1][:, K1:]),
                                                              slice(0, m), d_in), xr, _split_rel(mode) * xr.abs(), what + " root block")
    # listed form: an all-ranks list (duplicates included) with the other shards' entries parked as -1; only this
    # shard's listed rows are computed and stored into the peers
    out_w, _, _ = ops.layer_fwd(S.whole, x, x, W, root, b, False, mode)
    g = _gen(P + d_out)
    ids = S.pid[torch.randint(0, S.N, (2 * max(S.N // 7, 4),), generator=g, device=DEV)]
    ids[1] = ids[0]
    for p in range(P):
        lo, hi = S.rng(p)
        row0 = p * S.max_n
        local = torch.where((ids >= row0) & (ids < row0 + S.max_n), ids - row0, torch.full_like(ids, -1))
        half = local.numel() // 2
        rows, slot = ops.rows_list_build(local[:half], local[half:], S.max_n)
        bufs = [torch.full((P * S.max_n, d_out), float("nan"), device=DEV) for _ in range(P)]
        ops.layer_fwd(S.shards[p], x_full, x_full[row0:row0 + S.max_n], W, root, b, False, mode,
                      peer_out=[t.data_ptr() for t in bufs], peer_row0=row0, peer_ld=d_out, rows=rows, slot=slot)
        torch.cuda.synchronize()
        mine = local[local >= 0].unique()
        want = torch.full((P * S.max_n, d_out), float("nan"), device=DEV)
        want[row0 + mine] = out_w[lo + mine]
        for q, t in enumerate(bufs):
            _bits(t, want, f"{name} P={P} {mode} listed rank {p}: peer buffer {q}")


# =========================================================================================================================
# c. backward: transposed walk into P partials, pull-reduce over ranks, weight gradients summed over shards
# =========================================================================================================================
def _prod_rel(mode):
    """relative error of a product of two operands as the tensor core sees them: hi + lo (2^-16 each, lo * lo dropped)
    in the fp32 mode, one bf16 rounding (2^-8) each in the bf16 mode."""
    return 2.0 ** -14 if mode == "fp32" else 2.0 ** -7 + 2.0 ** -14


def _gemm_rel(mode, k):
    return _prod_rel(mode) + ((3 * k if mode == "fp32" else k) + 3) * E23


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name,P,d_in,d_out", CASES)
def test_shard_backward(ops, name, P, d_in, d_out, mode):
    S = _setup(name, P)
    x, x_full, W, root, b = _inputs(S, d_in, d_out, seed=P * 2000 + d_in + d_out)
    R, N, n, K1 = S.R, S.N, S.max_n, S.R * d_in
    K = K1 + d_in
    g = _gen(P * 3 + d_in)
    # the ReLU + dropout output of the whole-graph layer is the mask of the layer's output gradient
    ctr = torch.tensor([CTR0], dtype=torch.int64, device=DEV)
    out_w, A_w, _ = ops.layer_fwd(S.whole, x, x, W, root, b, True, mode, 0.5, SEED, ctr)
    gO = _rows_scaled(N, d_out, g)
    x_scale = 2.0                                       # the upstream layer's dropout scale (x is its masked output)
    parts = [torch.full((P * n, d_in), float("nan"), device=DEV) for _ in range(P)]
    gAs, gW64, groot64, gb64 = [], 0.0, 0.0, 0.0
    for p in range(P):
        lo, hi = S.rng(p)
        row0 = p * n
        _, A, wp = ops.layer_fwd(S.shards[p], x_full, x_full[row0:row0 + n], W, root, b, True, mode, pipeline=1)
        gO_p = torch.zeros(n, d_out, device=DEV)
        gO_p[:hi - lo] = gO[lo:hi]
        mask_p = torch.zeros(n, d_out, device=DEV)
        mask_p[:hi - lo] = out_w[lo:hi]
        gx, gA, gW, groot, gb = ops.layer_bwd(S.shards[p], gO_p, mask_p, drop_scale(0.5), A, W, root, d_in, mode,
                                              need_x=True, add_root_term=False, need_w=True, need_b=True, gx_out=parts[p],
                                              w_planes=wp)
        assert gx is parts[p]
        gAs.append(gA)
        gW64, groot64, gb64 = gW64 + gW.double(), groot64 + groot.double(), gb64 + gb.double()
    torch.cuda.synchronize()
    for p in range(P):
        assert not bool(parts[p].isnan().any()), f"rank {p}: the walk left rows of its partial unwritten"
    # float64 restatement of the whole-graph layer's backward
    Wcat = torch.cat([W, root], 0).double()
    G = gO.double() * (out_w > 0) * float(drop_scale(0.5))
    gA64, SgA = G @ Wcat.t(), G.abs() @ Wcat.abs().t()
    src, dst, rel = S.ei[0], S.ei[1], S.et
    key = dst * R + rel
    inv = 1.0 / torch.bincount(key, minlength=N * R).clamp(min=1).double()
    # edge j -> i of relation r carries inv_cnt[i, r] * gA[i, r d_in : (r + 1) d_in] back to j
    flat = dst[:, None] * K + rel[:, None] * d_in + torch.arange(d_in, device=DEV)[None, :]
    term, Sterm = gA64.reshape(-1)[flat] * inv[key][:, None], SgA.reshape(-1)[flat] * inv[key][:, None]
    gx64 = torch.zeros(N, d_in, dtype=torch.float64, device=DEV).index_add_(0, src, term) + gA64[:, K1:]
    Sgx = torch.zeros(N, d_in, dtype=torch.float64, device=DEV).index_add_(0, src, Sterm) + SgA[:, K1:]
    keep_x = (x > 0).double() * x_scale
    gx64, Sgx = gx64 * keep_x, Sgx * keep_x
    deg_src = torch.bincount(src, minlength=N).double()[:, None]
    bound_gx = Sgx * (_gemm_rel(mode, d_out) + (deg_src + P + 4) * U)
    for p in range(P):
        lo, hi = S.rng(p)
        m, row0 = hi - lo, p * n
        planes = ops.alloc_planes(n, d_in, mode, DEV)
        v, part = ops.p2p_reduce_split([t.data_ptr() for t in parts], row0, d_in, n, d_in, torch.device(DEV),
                                       extra=gAs[p][:, K1:], relu_mask=x_full[row0:row0 + n], mask_scale=x_scale,
                                       want_fp32=True, planes=planes, colsum=True)
        torch.cuda.synchronize()
        what = f"{name} P={P} {mode} rank {p}"
        _check(f"backward g_x {mode}", v[:m], gx64[lo:hi], bound_gx[lo:hi], what)
        assert bool((v[m:] == 0).all()), f"{what}: padding rows got a gradient"
        hi16 = v.to(torch.bfloat16)
        _bits(planes[0], hi16, what + ": reduce-split hi plane")
        if mode == "fp32":
            _bits(planes[1], (v - hi16.float()).to(torch.bfloat16), what + ": reduce-split lo plane")
        cs = v.double().sum(0)
        _check(f"backward colsum {mode}", part.sum(0), cs, (n + part.size(0) + 2) * U * v.double().abs().sum(0) + 1e-300,
               what + " column sums")
    # weight, root and bias gradients summed over the shards against the whole graph's A^T G
    H, SH, cnt = _agg64(x.double(), src, dst, rel, N, R)
    A64, SA = torch.cat([H, x.double()], 1), torch.cat([SH, x.double().abs()], 1)
    gWc64, SgW = A64.t() @ G, SA.t() @ G.abs()
    bound_w = SgW * (_prod_rel(mode) + (S.whole.max_seg + 2) * U + (3 * n + 3 if mode == "fp32" else n + 3) * E23 + (P + 2) * U)
    _check(f"backward weight {mode}", gW64, gWc64[:K1], bound_w[:K1], f"{name} P={P} weight")
    _check(f"backward weight {mode}", groot64, gWc64[K1:], bound_w[K1:], f"{name} P={P} root")
    _check(f"backward bias {mode}", gb64, G.sum(0), (n + 64 + P) * U * G.abs().sum(0) + 1e-300, f"{name} P={P} bias")


@pytest.mark.parametrize("name,P", [("primekg", 2), ("skewed", 3), ("tiny", 8)])
def test_pull_rows_over_ranks(ops, name, P):
    """Row-sparse last layer: an all-ranks list with duplicates and other shards' rows parked on local row 0; the listed
    rows get the sum of the P partials, every other row of ``out`` stays untouched."""
    S = _setup(name, P)
    n, d = S.max_n, 128
    g = _gen(P * 11)
    parts = [_rows_scaled(P * n, d, g) for _ in range(P)]
    ids = S.pid[torch.randint(0, S.N, (max(S.N // 5, 6),), generator=g, device=DEV)]
    ids[1] = ids[0]
    ref = torch.stack([t.double() for t in parts]).sum(0)
    Sref = torch.stack([t.double().abs() for t in parts]).sum(0)
    for p in range(P):
        row0 = p * n
        inside = (ids >= row0) & (ids < row0 + n)
        local = torch.where(inside, ids - row0, torch.zeros_like(ids))
        out = torch.full((n, d), float("nan"), device=DEV)
        ops.p2p_pull_rows([t.data_ptr() for t in parts], row0, d, local, out)
        torch.cuda.synchronize()
        listed = local.unique()
        _check("pull rows", out[listed], ref[row0 + listed], (P + 1) * U * Sref[row0 + listed], f"{name} P={P} rank {p}")
        rest = torch.ones(n, dtype=torch.bool, device=DEV)
        rest[listed] = False
        assert bool(out[rest].isnan().all()), f"{name} P={P} rank {p}: pull_rows wrote an unlisted row"


# =========================================================================================================================
# d. the fused dropout keyed by global node id
# =========================================================================================================================
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name,P,d_in,d_out", CASES)
def test_shard_dropout_keyed_by_global_node(ops, name, P, d_in, d_out, mode):
    """One (seed, counter) on every shard, as in the partitioned models: shard rows equal the whole-graph layer's rows
    bit for bit (schedule 3: the same keep pattern), their keep pattern is the ported hash at row offset bounds[p], and
    node bounds[p] + i does not repeat the mask of node i."""
    S = _setup(name, P)
    x, x_full, W, root, _ = _inputs(S, d_in, d_out, seed=P * 3000 + d_in + d_out)
    b = torch.full((d_out,), 4096.0, device=DEV)         # every pre-dropout value > 0: out != 0 exactly where kept
    p_drop, scale = 0.5, drop_scale(0.5)
    for sched in (1, 2, 3):
        plain, _, _ = ops.layer_fwd(S.whole, x, x, W, root, b, True, mode, pipeline=sched)
        assert bool((plain > 0).all())
        ctr = torch.tensor([CTR0], dtype=torch.int64, device=DEV)
        out_w, _, _ = ops.layer_fwd(S.whole, x, x, W, root, b, True, mode, p_drop, SEED, ctr, pipeline=sched)
        kept = []
        for p in range(P):
            lo, hi = S.rng(p)
            row0 = p * S.max_n
            x_root = x_full[row0:row0 + S.max_n]
            mine, _, _ = ops.layer_fwd(S.shards[p], x_full, x_root, W, root, b, True, mode, pipeline=sched)
            ctr = torch.tensor([CTR0], dtype=torch.int64, device=DEV)
            out, _, _ = ops.layer_fwd(S.shards[p], x_full, x_root, W, root, b, True, mode, p_drop, SEED, ctr,
                                      pipeline=sched, dropout_row0=lo)
            torch.cuda.synchronize()
            what = f"{name} P={P} {mode} schedule {sched} rank {p}"
            assert int(ctr) == CTR0 + 1
            if sched != 3:                                # (schedule 3: see the module docstring)
                _bits(out[:hi - lo], out_w[lo:hi], what + ": output")
            keep = drop_keep(hi - lo, lo, d_out, p_drop, SEED, CTR0 + 1)
            _bits(out[:hi - lo], torch.where(keep, mine[:hi - lo] * scale, 0.0), what + ": keep pattern")
            if sched == 3:
                _bits((out[:hi - lo] != 0).float(), (out_w[lo:hi] != 0).float(), what + ": the whole graph's keep pattern")
            kept.append(out[:hi - lo] != 0)
        m0 = kept[0].size(0)
        for p in range(1, P):
            m = min(m0, kept[p].size(0))
            if m * d_out >= 4096:
                agree = float((kept[p][:m] == kept[0][:m]).float().mean())
                assert 0.45 < agree < 0.55, f"{name} P={P} schedule {sched}: rank {p} repeats rank 0's masks ({agree:.3f})"

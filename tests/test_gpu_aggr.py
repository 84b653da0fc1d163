"""RGCNConv(aggr='sum' / 'max', root_weight=False, bias=False) on the B200 against the CPU oracle of PyG's loop path.

Sum runs the mean's weighted walks with unit weights (the bits of index_add_ in edge order below the hub threshold);
max runs its own walks (csrc/aggregate_max.cu), exact in fp32 — ties, exact-zero maxima, empty and all-negative
segments, NaN.  Layers, the models (autograph, captured step with FusedAdam and the arena, eval cache, ranking) and the
partitioned models at world size 1 are checked around them.
"""
import os
import socket

import pytest
import torch
import torch.nn.functional as F

from aggr_oracle import ModelAggrRef, RGCNConvAggrRef, aggregate_ref, rgcn_conv_aggr_ref
from test_gpu_parity import DEV, graphs, _close_by_scale

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg(lib_built):
    return lib_built


def _hub_graph():
    """Segments longer than the hub threshold (128): 40 destinations with 300 to 700 in-edges of one relation, plus
    isolated nodes (empty segments)."""
    g = torch.Generator().manual_seed(11)
    N, R = 3000, 2
    dst = torch.cat([torch.full((300 + 10 * k,), k) for k in range(40)])
    src = torch.randint(0, N, (dst.numel(),), generator=g)
    et = torch.randint(0, R, (dst.numel(),), generator=g) * (dst % 2)
    return torch.stack([src, dst]), et, N, R


def _graph(name):
    return _hub_graph() if name == "hubs" else graphs()[name]


def _ref_blocks(x, ei, et, N, R, aggr):
    return torch.cat([aggregate_ref(x, ei[0][et == r], ei[1][et == r], N, aggr) for r in range(R)], 1)


# ---- the walks -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["val_fixture", "primekg_100k", "hubs", "ragged"])
@pytest.mark.parametrize("d", [4, 16, 64, 256])
def test_sum_walk_is_index_add(pkg, name, d):
    from primekg_rgcn_linkprediction_b200 import ops
    ei, et, N, R = _graph(name)
    if N * R * d > 60_000_000:
        pytest.skip("oracle too slow at this size")
    x = torch.randn(N, d, generator=torch.Generator().manual_seed(d))
    g = pkg.RelGraph.from_edges(ei.to(DEV), et.to(DEV), N, R).for_aggr("sum")
    H = ops.aggregate_fwd(g, x.to(DEV)).cpu()
    want = _ref_blocks(x, ei, et, N, R, "sum")
    # hub segments (up to 700 edges here) are summed in chunks: another order, sums of up to ~50 in magnitude
    torch.testing.assert_close(H, want, rtol=1e-5, atol=5e-4)
    cnt = (g.rowptr[1:] - g.rowptr[:-1]).cpu().view(N, R)
    small = (cnt <= g.fwd.threshold)[:, :, None].expand(N, R, d).reshape(N, R * d)
    assert torch.equal(H[small], want[small])             # serial segments: index_add_'s bits
    if name == "hubs":
        assert int((cnt > g.fwd.threshold).sum()) > 0


@pytest.mark.parametrize("name", ["val_fixture", "primekg_100k", "hubs", "ragged"])
@pytest.mark.parametrize("d", [4, 64, 256])
@pytest.mark.parametrize("inputs", ["small_ints", "relu", "negative"])
def test_max_walk_is_exact(pkg, name, d, inputs):
    from primekg_rgcn_linkprediction_b200 import ops
    ei, et, N, R = _graph(name)
    if N * R * d > 60_000_000:
        pytest.skip("oracle too slow at this size")
    gen = torch.Generator().manual_seed(d + 1)
    x = {"small_ints": torch.randint(-3, 4, (N, d), generator=gen).float(),
         "relu": torch.relu(torch.randn(N, d, generator=gen)),
         "negative": -torch.rand(N, d, generator=gen) - 0.5}[inputs]
    g = pkg.RelGraph.from_edges(ei.to(DEV), et.to(DEV), N, R)
    A = ops.alloc_planes(N, (R + 1) * d, "fp32", DEV)
    xd = x.to(DEV)
    Hmax, Hcnt = ops.aggregate_max_fwd(g, xd, A, x_root=xd)
    want = _ref_blocks(x, ei, et, N, R, "max")
    assert torch.equal(Hmax.cpu(), want)
    hi, lo = A[0][:, : R * d].float(), A[1][:, : R * d].float()
    torch.testing.assert_close((hi + lo).cpu(), want, rtol=2 ** -16, atol=0)
    assert torch.equal(A[0][:, R * d:].cpu(), x.to(torch.bfloat16))
    cnt = (g.rowptr[1:] - g.rowptr[:-1]).cpu().view(N, R)
    empty = (cnt == 0)[:, :, None].expand(N, R, d).reshape(N, R * d)
    assert torch.equal(Hmax.cpu()[empty], torch.zeros(int(empty.sum())))
    if inputs == "negative":
        assert bool((Hmax.cpu()[~empty] < 0).all())        # all-negative segments give their max, not 0


def test_max_walk_propagates_nan(pkg):
    from primekg_rgcn_linkprediction_b200 import ops
    ei, et, N, R = graphs()["ragged"]
    x = torch.randn(N, 8)
    x[1, 3] = float("nan")
    g = pkg.RelGraph.from_edges(ei.to(DEV), et.to(DEV), N, R)
    A = ops.alloc_planes(N, R * 8, "fp32", DEV)
    Hmax, _ = ops.aggregate_max_fwd(g, x.to(DEV), A)
    want = _ref_blocks(x, ei, et, N, R, "max")
    assert torch.equal(torch.isnan(Hmax.cpu()), torch.isnan(want)) and bool(torch.isnan(want).any())
    ok = ~torch.isnan(want)
    assert torch.equal(Hmax.cpu()[ok], want[ok])


def test_max_backward_nan_segments_match_torch(pkg):
    """A segment whose maximum is NaN gives every source a NaN gradient in torch (zero mask times gH / 0)."""
    from primekg_rgcn_linkprediction_b200 import ops
    ei, et, N, R = graphs()["ragged"]
    d = 8
    x = torch.randn(N, d, dtype=torch.float64)
    x[1, 3] = float("nan")
    g = pkg.RelGraph.from_edges(ei.to(DEV), et.to(DEV), N, R)
    A = ops.alloc_planes(N, R * d, "fp32", DEV)
    xd = x.float().to(DEV)
    Hmax, Hcnt = ops.aggregate_max_fwd(g, xd, A)
    gH = torch.randn(N, R * d, dtype=torch.float64)
    got = ops.aggregate_max_bwd(g, gH.float().to(DEV), Hmax, Hcnt, xd).cpu()
    x64 = x.clone().requires_grad_()
    (_ref_blocks(x64, ei, et, N, R, "max") * gH).sum().backward()
    want = x64.grad.float()
    assert bool(torch.isnan(want).any())
    assert torch.equal(torch.isnan(got), torch.isnan(want))
    ok = ~torch.isnan(want)
    torch.testing.assert_close(got[ok], want[ok], rtol=1e-6, atol=1e-6)


# ---- layers --------------------------------------------------------------------------------------------------------
def _layer_case(pkg, name, d_in, d_out, aggr, mode, root_weight, bias, inputs, seed=5):
    ei, et, N, R = _graph(name)
    torch.manual_seed(seed)
    conv = pkg.RGCNConv(d_in, d_out, R, aggr=aggr, root_weight=root_weight, bias=bias).to(DEV)
    conv.mode = mode
    if conv.bias is not None:
        with torch.no_grad():
            conv.bias.normal_()
    gen = torch.Generator().manual_seed(seed + 1)
    x = {"small_ints": torch.randint(-2, 3, (N, d_in), generator=gen).float(),
         "relu": torch.relu(torch.randn(N, d_in, generator=gen)),
         "randn": torch.randn(N, d_in, generator=gen)}[inputs]
    coef = torch.randn(N, d_out, generator=gen)
    return ei, et, N, R, conv, x, coef


def _check_layer(pkg, conv, ei, et, N, R, x, coef, mode, relu=False, p=0.0):
    g = pkg.RelGraph.from_edges(ei.to(DEV), et.to(DEV), N, R)
    xd = x.to(DEV).requires_grad_()
    out = conv.forward_graph(xd, g, relu=relu, dropout_p=p)
    (out * coef.to(DEV)).sum().backward()
    x64 = x.double().requires_grad_()
    prm = {k: v.detach().cpu().double().requires_grad_() for k, v in conv.named_parameters()}
    ref = rgcn_conv_aggr_ref(x64, ei, et, prm["weight"], prm.get("root"), prm.get("bias"), conv.aggr)
    if relu:
        # the device's own ReLU (and dropout) pattern: an output within rounding of 0 may fall on either side of the kink
        ref = ref * (out.detach().cpu() > 0) / (1.0 - p)
    (ref * coef.double()).sum().backward()
    tol = dict(rtol=1e-4, atol=2e-5) if mode == "fp32" else dict(rtol=3e-2, atol=2e-2)
    _close_by_scale(out.detach().cpu(), ref.detach().float(), "out", **tol)
    _close_by_scale(xd.grad.cpu(), x64.grad.float(), "grad x", **tol)
    for k, v in conv.named_parameters():
        _close_by_scale(v.grad.cpu(), prm[k].grad.float(), f"grad {k}", **tol)
    for k in ("root", "bias"):
        assert (getattr(conv, k) is None) == (k not in prm)
    return out.detach(), xd.grad.detach()


@pytest.mark.parametrize("name", ["val_fixture", "hubs", "ragged"])
@pytest.mark.parametrize("d_in,d_out", [(4, 8), (64, 64), (256, 128)])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("epilogue", ["none", "relu", "relu_dropout"])
def test_sum_layer_against_oracle(pkg, name, d_in, d_out, mode, epilogue):
    ei, et, N, R, conv, x, coef = _layer_case(pkg, name, d_in, d_out, "add", mode, True, True, "randn")
    _check_layer(pkg, conv, ei, et, N, R, x, coef, mode, epilogue != "none", 0.3 if epilogue == "relu_dropout" else 0.0)


@pytest.mark.parametrize("name", ["val_fixture", "hubs", "ragged"])
@pytest.mark.parametrize("d_in,d_out", [(4, 8), (64, 64), (256, 128)])
@pytest.mark.parametrize("inputs", ["small_ints", "relu"])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("p", [0.0, 0.3])
def test_max_layer_against_oracle(pkg, name, d_in, d_out, inputs, mode, p):
    ei, et, N, R, conv, x, coef = _layer_case(pkg, name, d_in, d_out, "max", mode, True, True, inputs)
    out, gx = _check_layer(pkg, conv, ei, et, N, R, x, coef, mode, relu=True, p=p)
    if p == 0.0:
        # two runs, the same bits
        conv.zero_grad()
        out2, gx2 = _check_layer(pkg, conv, ei, et, N, R, x, coef, mode, relu=True)
        assert torch.equal(out, out2) and torch.equal(gx, gx2)


@pytest.mark.parametrize("aggr", ["mean", "sum", "max"])
@pytest.mark.parametrize("root_weight,bias", [(False, True), (True, False), (False, False)])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("decomp", [None, "bases", "blocks"])
def test_no_root_no_bias_against_oracle(pkg, aggr, root_weight, bias, mode, decomp):
    ei, et, N, R = graphs()["val_fixture"]
    torch.manual_seed(1)
    kw = {"bases": dict(num_bases=2), "blocks": dict(num_blocks=4), None: {}}[decomp]
    conv = pkg.RGCNConv(64, 32, R, aggr=aggr, root_weight=root_weight, bias=bias, **kw).to(DEV)
    conv.mode = mode
    gen = torch.Generator().manual_seed(2)
    x = torch.relu(torch.randn(N, 64, generator=gen))
    coef = torch.randn(N, 32, generator=gen)
    g = pkg.RelGraph.from_edges(ei.to(DEV), et.to(DEV), N, R)
    xd = x.to(DEV).requires_grad_()
    out = conv.forward_graph(xd, g, relu=True, dropout_p=0.0)
    (out * coef.to(DEV)).sum().backward()
    oracle = RGCNConvAggrRef(64, 32, R, aggr=aggr, root_weight=root_weight, bias=bias, **kw).double()
    oracle.load_state_dict(conv.state_dict(), strict=True)
    x64 = x.double().requires_grad_()
    ref = oracle(x64, ei, et)
    ref = ref * (out.detach().cpu() > 0)                   # the device's ReLU pattern (outputs within rounding of 0)
    (ref * coef.double()).sum().backward()
    tol = dict(rtol=1e-4, atol=2e-5) if mode == "fp32" else dict(rtol=3e-2, atol=2e-2)
    _close_by_scale(out.detach().cpu(), ref.detach().float(), "out", **tol)
    _close_by_scale(xd.grad.cpu(), x64.grad.float(), "grad x", **tol)
    assert [k for k, _ in conv.named_parameters()] == [k for k, _ in oracle.named_parameters()]
    for (k, p), (_, q) in zip(conv.named_parameters(), oracle.named_parameters()):
        _close_by_scale(p.grad.cpu(), q.grad.float(), f"grad {k}", **tol)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_sum_basis_z_form_against_oracle(pkg, monkeypatch, mode):
    monkeypatch.setenv("PRIMEKG_RGCN_BASIS_FORM", "z")
    ei, et, N, R = graphs()["val_fixture"]
    torch.manual_seed(3)
    conv = pkg.RGCNConv(64, 32, R, num_bases=3, aggr="sum").to(DEV)
    conv.mode = mode
    g = pkg.RelGraph.from_edges(ei.to(DEV), et.to(DEV), N, R)
    assert conv._use_z_form(g.for_aggr("sum"))
    gen = torch.Generator().manual_seed(4)
    x, coef = torch.randn(N, 64, generator=gen), torch.randn(N, 32, generator=gen)
    xd = x.to(DEV).requires_grad_()
    out = conv.forward_graph(xd, g, relu=False)
    (out * coef.to(DEV)).sum().backward()
    prm = {k: v.detach().cpu().double().requires_grad_() for k, v in conv.named_parameters()}
    x64 = x.double().requires_grad_()
    ref = rgcn_conv_aggr_ref(x64, ei, et, prm["weight"], prm["root"], prm["bias"], "sum", comp=prm["comp"])
    (ref * coef.double()).sum().backward()
    tol = dict(rtol=1e-4, atol=2e-5) if mode == "fp32" else dict(rtol=3e-2, atol=2e-2)
    _close_by_scale(out.detach().cpu(), ref.detach().float(), "out", **tol)
    _close_by_scale(xd.grad.cpu(), x64.grad.float(), "grad x", **tol)
    for k, v in conv.named_parameters():
        _close_by_scale(v.grad.cpu(), prm[k].grad.float(), f"grad {k}", **tol)


# ---- models --------------------------------------------------------------------------------------------------------
def _model(pkg, kg, aggr, mode="fp32", seed=0, dropout=0.0, **kw):
    torch.manual_seed(seed)
    m = pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, 64, 128, dropout=dropout, decoder_dropout=0.0,
                             aggr=aggr, **kw).to(DEV)
    for c in m.encoder._layers():
        c.mode = mode
    return m


@pytest.mark.parametrize("aggr", ["sum", "max"])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_model_trains_like_the_oracle_model(pkg, monkeypatch, aggr, mode):
    """Three SGD steps of the model's training call against the fp64 oracle model.  A sum model runs the listed last
    layer (the row-sparse backward claims the decoder's gradient) and, in bf16 mode, the bf16 gather."""
    monkeypatch.setenv("PRIMEKG_RGCN_AUTOGRAPH", "0")
    from primekg_rgcn_linkprediction_b200 import ops, rowsparse, synth
    kg = synth.primekg_subgraph(20_000, seed=5)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    batches = [[v.to(DEV) for v in synth.link_batch(kg, 256, seed=2 + i)] for i in range(3)]
    m = _model(pkg, kg, aggr, mode)
    ref = ModelAggrRef(kg.num_nodes, kg.num_relations, 64, 128, aggr=aggr).double()
    ref.load_state_dict(m.state_dict())
    ref.to(DEV)
    m.train()
    gathers16 = []
    to_bf16 = ops.to_bf16
    monkeypatch.setattr(ops, "to_bf16", lambda x: gathers16.append(x.shape) or to_bf16(x))
    claimed0 = rowsparse.stats["claimed"]
    lr = 0.05
    tol = 1e-4 if mode == "fp32" else 3e-2
    for step, (h, t, r, y) in enumerate(batches):
        m.zero_grad(); ref.zero_grad()
        loss = F.binary_cross_entropy_with_logits(m(ei, et, h, t, r), y)
        loss.backward()
        rl = F.binary_cross_entropy_with_logits(ref(ei, et, h, t, r), y.double())
        rl.backward()
        assert abs(float(loss) - float(rl)) <= tol * max(1.0, abs(float(rl))), (float(loss), float(rl))
        for (k, p), q in zip(m.named_parameters(), ref.parameters()):
            err = float((p.grad.double() - q.grad).norm() / (q.grad.norm() + 1e-30))
            # bf16 operands: 5 % on the first step; the two models' parameters then drift apart by bf16 rounding per update
            assert err < (1e-3 if mode == "fp32" else (5e-2 if step == 0 else 1e-1)), (step, k, err)
        with torch.no_grad():
            for p, q in zip(m.parameters(), ref.parameters()):
                p -= lr * p.grad
                q -= lr * q.grad
    if aggr == "sum":
        assert rowsparse.stats["claimed"] - claimed0 == len(batches)       # the listed last layer ran
        assert bool(gathers16) == (mode == "bf16")                         # the bf16 gather ran


@pytest.mark.parametrize("aggr", ["sum", "max"])
def test_models_train_captured_with_fused_adam_and_arena(pkg, monkeypatch, aggr):
    from primekg_rgcn_linkprediction_b200 import synth
    kg = synth.primekg_subgraph(20_000, seed=5)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    batches = [[v.to(DEV) for v in synth.link_batch(kg, 256, seed=10 + i)] for i in range(4)]
    m = _model(pkg, kg, aggr, dropout=0.5)
    m.train()
    opt = pkg.FusedAdam(m.parameters(), lr=1e-2, max_grad_norm=1.0)
    step = pkg.GraphedTrainStep(m, ei, et, batch_size=512, optimizer=opt, flat_grads="arena")
    before = [p.detach().clone() for p in m.parameters()]
    losses = [float(step(*batches[i % 4])) for i in range(16)]
    assert all(l == l and abs(l) < 1e6 for l in losses), losses
    assert all(not torch.equal(a, p.detach()) for a, p in zip(before, m.parameters()))     # every parameter trained
    # the model(...) autograph path of the reference's loop
    monkeypatch.setenv("PRIMEKG_RGCN_AUTOGRAPH", "1")
    h, t, r, y = batches[0]
    ls = []
    for _ in range(4):
        m.zero_grad()
        loss = F.binary_cross_entropy_with_logits(m(ei, et, h, t, r), y)
        loss.backward()
        ls.append(float(loss))
    assert all(l == l for l in ls)
    # eval cache and ranking
    m.eval()
    with torch.no_grad():
        e1 = m.encoder(ei, et)
        e2 = m.encoder(ei, et)
        assert e1 is e2
        from primekg_rgcn_linkprediction_b200 import rank
        rk, _ = rank.rank_true_tails(e1, m.decoder.relation_embeddings.weight, h[:64], r[:64], t[:64])
        assert int(rk.min()) >= 1 and int(rk.max()) <= kg.num_nodes


def test_explicit_mean_is_bit_identical_to_the_default(pkg, monkeypatch):
    monkeypatch.setenv("PRIMEKG_RGCN_AUTOGRAPH", "0")
    from primekg_rgcn_linkprediction_b200 import synth
    kg = synth.primekg_subgraph(20_000, seed=5)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    h, t, r, y = [v.to(DEV) for v in synth.link_batch(kg, 256, seed=2)]
    outs = []
    for aggr in (None, "mean"):
        torch.manual_seed(0)
        kw = {} if aggr is None else {"aggr": aggr}
        m = pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, 64, 128, dropout=0.5, **kw).to(DEV)
        m.train()
        torch.manual_seed(1)
        loss = F.binary_cross_entropy_with_logits(m(ei, et, h, t, r), y)
        loss.backward()
        outs.append((loss.detach(), [p.grad.clone() for p in m.parameters()]))
    assert torch.equal(outs[0][0], outs[1][0])
    assert all(torch.equal(a, b) for a, b in zip(outs[0][1], outs[1][1]))


@pytest.fixture(scope="module")
def pg(lib_built):
    import torch.distributed as dist
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device(DEV))
    yield lib_built
    dist.destroy_process_group()


@pytest.mark.parametrize("kind", ["fused", "nccl"])
def test_partitioned_sum_model_matches_single_gpu(pg, monkeypatch, kind):
    import primekg_rgcn_linkprediction_b200 as pkg
    from primekg_rgcn_linkprediction_b200 import dist as D
    from primekg_rgcn_linkprediction_b200 import dist_fused as DF
    from primekg_rgcn_linkprediction_b200 import synth
    monkeypatch.setenv("PRIMEKG_RGCN_AUTOGRAPH", "0")
    torch.manual_seed(0)
    N, R, d_e, H, B = 5000, 5, 64, 128, 512
    kg = synth.uniform_kg(N, 60_000, R, seed=3)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    plan = D.plan_partition(ei[1], N, 1)
    cls = DF.FusedPartitionedModel if kind == "fused" else D.PartitionedModel
    mp = cls(plan, 0, R, d_e, H, dropout=0.0, seed=5, aggr="sum").to(DEV)
    mp.encoder.build_graph(ei, et)
    mp.train()
    heads = torch.randint(0, N, (B,), device=DEV)
    tails = torch.randint(0, N, (B,), device=DEV)
    rels = torch.randint(0, R, (B,), device=DEV)
    labels = (torch.rand(B, device=DEV) < 0.5).float()
    s = mp(heads, tails, rels)
    loss = F.binary_cross_entropy_with_logits(s, labels)
    loss.backward()
    ref = pkg.DrugDiseaseModel(N, R, d_e, H, dropout=0.0, decoder_dropout=0.0, aggr="sum").to(DEV)
    with torch.no_grad():
        ref.encoder.node_embeddings.weight.copy_(mp.encoder.node_embeddings[:N])
        for mine, theirs in zip(mp.encoder.convs, ref.encoder._layers()):
            theirs.weight.copy_(mine.weight); theirs.root.copy_(mine.root); theirs.bias.copy_(mine.bias)
        ref.decoder.relation_embeddings.weight.copy_(mp.decoder.relation_embeddings.weight)
    ref.train()
    rs = ref(ei, et, heads, tails, rels)
    rloss = F.binary_cross_entropy_with_logits(rs, labels)
    rloss.backward()
    torch.testing.assert_close(s.detach(), rs.detach(), rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(mp.encoder.node_embeddings.grad[:N], ref.encoder.node_embeddings.weight.grad,
                               rtol=1e-3, atol=1e-6)
    for mine, theirs in zip(mp.encoder.convs, ref.encoder._layers()):
        for a, b in ((mine.weight, theirs.weight), (mine.root, theirs.root), (mine.bias, theirs.bias)):
            assert float((a.grad - b.grad).norm() / (b.grad.norm() + 1e-30)) < 1e-4

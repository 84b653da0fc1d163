"""Block-diagonal relation weights, RGCNConv(num_blocks=nb), on the B200.

The layer materialises W_r = blockdiag(weight[r, 0], .., weight[r, nb - 1]) (``rgcn_block_diag_expand``) and runs the
unchanged layer kernels; zeros split into bf16 planes as exact zeros, so a block layer gives THE SAME BITS as the dense
layer whose ``weight`` holds the expanded matrix, and its weight gradient is the diagonal blocks of that layer's weight
gradient (``rgcn_block_diag_gather``: copies only).  Around that: the cfg3-size layer against the CPU oracle's
statement of PyG's block path, the model paths (listed last layer, eval cache, ranking, determinism), the captured
training step with the fused optimizer and the gradient arena, the partitioned models at world size 1, and training.
"""
import os
import socket

import pytest
import torch
import torch.nn.functional as F

from blocks_oracle import ModelBlocksRef, RGCNConvBlocksRef, diag_blocks, expand_blocks
from test_gpu_parity import DEV, graphs, _close_by_scale

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg(lib_built):
    return lib_built


def _block_and_dense(pkg, d_in, d_out, R, nb, mode, seed=3):
    torch.manual_seed(seed)
    blk = pkg.RGCNConv(d_in, d_out, R, num_blocks=nb).to(DEV)
    dense = pkg.RGCNConv(d_in, d_out, R).to(DEV)
    with torch.no_grad():
        blk.bias.normal_()                                            # a non-zero bias reaches the epilogue
        dense.weight.copy_(expand_blocks(blk.weight.detach()))
        dense.root.copy_(blk.root)
        dense.bias.copy_(blk.bias)
    blk.mode = dense.mode = mode
    return blk, dense


# ------------------------------------------------------------------------------------------------
# (1) bit-identity with the dense layer
@pytest.mark.parametrize("epilogue", ["none", "relu_dropout"])
@pytest.mark.parametrize("graph", ["val_fixture", "primekg_100k"])
@pytest.mark.parametrize("d_in,d_out,nb", [(64, 64, 1), (64, 128, 2), (64, 256, 4), (64, 256, 16), (128, 64, 16),
                                           (32, 32, 16), (48, 24, 4)])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_block_layer_is_bit_identical_to_the_expanded_dense_layer(pkg, mode, d_in, d_out, nb, graph, epilogue):
    ei, et, N, R = graphs()[graph]
    g = pkg.RelGraph.from_edges(ei.to(DEV), et.to(DEV), N, R)
    blk, dense = _block_and_dense(pkg, d_in, d_out, R, nb, mode)
    gen = torch.Generator(device=DEV).manual_seed(9)
    x = torch.randn(N, d_in, device=DEV, generator=gen).requires_grad_()
    xd = x.detach().clone().requires_grad_()
    coef = torch.randn(N, d_out, device=DEV, generator=gen)
    relu = epilogue != "none"
    p = 0.3 if relu else 0.0
    ob = blk.forward_graph(x, g, relu=relu, dropout_p=p)
    if relu:
        # the dense layer draws the same dropout stream: the block layer's seed, its counter before the call above
        dense._drop_seed, dense._drop_ctr = blk._drop_seed, blk._drop_ctr - 1
    od = dense.forward_graph(xd, g, relu=relu, dropout_p=p)
    assert torch.equal(ob, od)
    (ob * coef).sum().backward()
    (od * coef).sum().backward()
    assert torch.equal(x.grad, xd.grad)
    assert torch.equal(blk.root.grad, dense.root.grad)
    assert torch.equal(blk.bias.grad, dense.bias.grad)
    assert blk.weight.grad.shape == blk.weight.shape
    assert torch.equal(blk.weight.grad, diag_blocks(dense.weight.grad, nb))


def test_expand_and_gather_kernels_against_torch(pkg):
    from primekg_rgcn_linkprediction_b200 import ops
    for R, nb, bi, bo in ((30, 4, 16, 64), (3, 16, 4, 16), (5, 16, 2, 2), (2, 4, 12, 6), (1, 1, 4, 4), (7, 3, 5, 3)):
        w = torch.randn(R, nb, bi, bo, device=DEV).requires_grad_()
        W = ops.block_diag_weights(w)
        assert ops.is_grad_scratch(W)
        assert torch.equal(W, expand_blocks(w.detach()))          # zeros included
        gW = torch.randn_like(W)
        W.backward(gW)
        assert torch.equal(w.grad, diag_blocks(gW, nb))


# ------------------------------------------------------------------------------------------------
# (2) against the oracle at cfg3 size
def test_cfg3_full_size_block_layer_forward_backward(pkg):
    """cfg3 graph (129,375 nodes / ~8.1 M edges / 30 relations), one 64 -> 256 layer with 4 blocks, forward and backward
    against the oracle's statement of PyG's block path run on the same device (fp32 mode, rtol 1e-4)."""
    from primekg_rgcn_linkprediction_b200 import synth
    kg = synth.primekg_full()
    torch.manual_seed(3)
    conv = pkg.RGCNConv(64, 256, 30, num_blocks=4).to(DEV)
    conv.mode = "fp32"
    ref = RGCNConvBlocksRef(64, 256, 30, 4).to(DEV)
    ref.load_state_dict(conv.state_dict())
    x = (torch.randn(kg.num_nodes, 64, device=DEV) * 0.5).requires_grad_()
    xr = x.detach().clone().requires_grad_()
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    coef = torch.randn(kg.num_nodes, 256, device=DEV)
    out = conv(x, ei, et)
    (out * coef).sum().backward()
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        want = ref(xr, ei, et)
        (want * coef).sum().backward()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    torch.testing.assert_close(out.detach(), want.detach(), rtol=1e-4, atol=1e-4 * float(want.detach().abs().max()))
    for got, exp, name in ((x.grad, xr.grad, "x"), (conv.weight.grad, ref.weight.grad, "weight"),
                           (conv.root.grad, ref.root.grad, "root"), (conv.bias.grad, ref.bias.grad, "bias")):
        rel = float((got - exp).norm() / (exp.norm() + 1e-30))
        assert rel < 1e-4, (name, rel)


# ------------------------------------------------------------------------------------------------
# (3) model paths on cfg1
_CFG1 = None


def _cfg1():
    global _CFG1
    if _CFG1 is None:
        from primekg_rgcn_linkprediction_b200 import synth
        kg = synth.primekg_subgraph()
        _CFG1 = (kg, [t.to(DEV) for t in synth.link_batch(kg, 1024)])
    return _CFG1


def _block_model(pkg, kg, mode="fp32", seed=0, dropout=0.0):
    torch.manual_seed(seed)
    m = pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, 64, 128, dropout=dropout, decoder_dropout=0.0,
                             num_blocks=4).to(DEV)
    for c in m.encoder._layers():
        c.mode = mode
    return m


def _train_call(pkg, monkeypatch, listed: bool, mode):
    from primekg_rgcn_linkprediction_b200 import rowsparse
    monkeypatch.setenv("PRIMEKG_RGCN_SPARSE_FWD", "1" if listed else "0")
    monkeypatch.setenv("PRIMEKG_RGCN_SPARSE_BWD", "1")
    monkeypatch.setenv("PRIMEKG_RGCN_AUTOGRAPH", "0")
    monkeypatch.setattr(rowsparse, "MAX_FRACTION", 1e9)
    rowsparse.clear()
    kg, (h, t, r, y) = _cfg1()
    m = _block_model(pkg, kg, mode)
    m.train()
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    scores = m(ei, et, h, t, r)
    F.binary_cross_entropy_with_logits(scores, y).backward()
    return scores.detach().clone(), {k: p.grad.clone() for k, p in m.named_parameters()}


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_listed_last_layer_equals_dense_forward(pkg, monkeypatch, mode):
    s1, g1 = _train_call(pkg, monkeypatch, True, mode)
    s0, g0 = _train_call(pkg, monkeypatch, False, mode)
    assert torch.equal(s1, s0)
    for k in g0:
        _close_by_scale(g1[k], g0[k], k, rtol=1e-4, atol=2e-5)
    s2, g2 = _train_call(pkg, monkeypatch, True, mode)                 # a second run: the same bits
    assert torch.equal(s2, s1)
    for k in g1:
        assert torch.equal(g2[k], g1[k]), k


def test_block_model_eval_cache_and_ranking(pkg):
    from primekg_rgcn_linkprediction_b200 import _lib
    kg, (h, t, r, _) = _cfg1()
    m = _block_model(pkg, kg)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    lib = _lib.load()
    m.eval()
    with torch.no_grad():
        a = m.encoder(ei, et)
        n0 = lib.rgcn_launch_count()
        b = m.encoder(ei, et)
        assert lib.rgcn_launch_count() == n0 and b is a                 # served from the cache
        rank, ties = m.decoder.rank_tails(a, h[:256], r[:256], t[:256])
        assert rank.shape[0] == 256 and int(rank.min()) >= 1 and int(rank.max()) <= kg.num_nodes
        # the fused rank is the count over the dense scores, up to candidates within rounding of the true score
        s = (a[h[:256]] * m.decoder.relation_embeddings.weight[r[:256]]) @ a.t()
        true = s.gather(1, t[:256].view(-1, 1))
        tol = 1e-5 * float(s.abs().max())
        lo, hi = (s > true + tol).sum(1) + 1, (s > true - tol).sum(1) + 1
        assert bool(((rank.long() >= lo) & (rank.long() <= hi)).all())
        m.encoder.conv1.weight.mul_(1.5)                                 # a parameter change drops the cache
        c = m.encoder(ei, et)
        assert lib.rgcn_launch_count() > n0 and not torch.equal(c, a)


# ------------------------------------------------------------------------------------------------
# (4) captured training step
def test_graphed_step_with_fused_optimizer_tracks_torch(pkg):
    from primekg_rgcn_linkprediction_b200 import synth
    kg = synth.primekg_subgraph(20_000, seed=5)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    batches = [[t.to(DEV) for t in synth.link_batch(kg, 256, seed=10 + i)] for i in range(4)]
    ma, mb = _block_model(pkg, kg, seed=1), _block_model(pkg, kg, seed=1)
    ma.train(); mb.train()
    opt_a = pkg.FusedAdam(ma.parameters(), lr=1e-2, max_grad_norm=1.0)
    opt_b = torch.optim.Adam(mb.parameters(), lr=1e-2, foreach=False)
    step_a = pkg.GraphedTrainStep(ma, ei, et, batch_size=512, optimizer=opt_a)
    step_b = pkg.GraphedTrainStep(mb, ei, et, batch_size=512)
    params_b = list(mb.parameters())
    losses = []
    # 12 replays: the two runs differ in the last bits from the first update on, and Adam's division by sqrt(v) grows
    # that difference step by step once the loss of the four repeated batches nears zero
    for it in range(12):
        b = batches[it % 4]
        la = float(step_a(*b))
        lb = float(step_b(*b))
        torch.nn.utils.clip_grad_norm_(params_b, 1.0, foreach=False)
        opt_b.step()
        assert abs(la - lb) <= 1e-4 * abs(lb), (it, la, lb)
        losses.append(la)
    # whole tensors within 1e-3 (relative Frobenius); entries within 1 % of the tensor's scale, except the few (at most
    # 1e-5 of a tensor) whose gradient sits at rounding-noise level, where Adam's sqrt(v) step may go either way
    for (k, p), q in zip(ma.named_parameters(), params_b):
        p, q = p.detach(), q.detach()
        assert float((p - q).norm() / q.norm()) < 1e-3, k
        far = (p - q).abs() > 1e-2 * float(q.abs().max()) + 1e-3 * q.abs()
        assert int(far.sum()) <= max(1, int(1e-5 * q.numel())), (k, int(far.sum()))
    assert sum(losses[-4:]) < sum(losses[:4])


def test_graphed_step_arena_holds_every_block_gradient(pkg):
    """The dense weight gradient of a block layer is scratch: only the compact block gradient takes an arena slice, so
    the arena sized for the parameters holds every gradient and ``flat_grad`` is the one tensor to all-reduce."""
    from primekg_rgcn_linkprediction_b200 import synth
    kg = synth.primekg_subgraph(20_000, seed=5)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    b = [t.to(DEV) for t in synth.link_batch(kg, 256, seed=3)]
    ma, mb = _block_model(pkg, kg, seed=2), _block_model(pkg, kg, seed=2)
    ma.train(); mb.train()
    step = pkg.GraphedTrainStep(ma, ei, et, batch_size=512, flat_grads="arena")
    assert step.flat_grad is not None
    la = step(*b).clone()
    torch.cuda.synchronize()
    buf = step.arena.buf
    lo, hi = buf.data_ptr(), buf.data_ptr() + buf.numel() * 4
    for k, p in ma.named_parameters():
        assert p.grad is not None and lo <= p.grad.data_ptr() < hi, k
    ref = pkg.GraphedTrainStep(mb, ei, et, batch_size=512)
    lb = ref(*b).clone()
    assert torch.equal(la, lb)
    for (k, p), q in zip(ma.named_parameters(), mb.parameters()):
        _close_by_scale(p.grad, q.grad, k, rtol=1e-5, atol=1e-6)


def test_autograph_replay_equals_eager(pkg, monkeypatch):
    """The reference's loop: the same training call three times (eager), then replayed from the captured graphs."""
    monkeypatch.setenv("PRIMEKG_RGCN_AUTOGRAPH", "1")
    from primekg_rgcn_linkprediction_b200 import synth
    kg = synth.primekg_subgraph(20_000, seed=6)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    h, t, r, y = [x.to(DEV) for x in synth.link_batch(kg, 256, seed=4)]
    m = _block_model(pkg, kg, seed=4)
    m.train()
    losses, grads = [], []
    for _ in range(5):
        m.zero_grad()
        loss = F.binary_cross_entropy_with_logits(m(ei, et, h, t, r), y)
        loss.backward()
        losses.append(float(loss))
        grads.append(m.encoder.conv1.weight.grad.clone())
    assert any(e[1] is not None for e in m.__dict__.get("_autograph", {}).values())     # it was captured
    for l, g in zip(losses[1:], grads[1:]):
        assert abs(l - losses[0]) <= 1e-6 * abs(losses[0]), losses
        _close_by_scale(g, grads[0], "conv1.weight", rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------------------------------------
# (5) partitioned models at world size 1
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


def _run_partitioned(model, heads, tails, rels, labels):
    s = model(heads, tails, rels)
    loss = F.binary_cross_entropy_with_logits(s, labels)
    loss.backward()
    if hasattr(model, "allreduce_decoder_grads"):
        model.allreduce_decoder_grads()
    return s.detach().clone(), loss.detach().clone()


@pytest.mark.parametrize("kind", ["fused", "nccl"])
def test_partitioned_block_model_matches_single_gpu(pg, monkeypatch, kind):
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
    models = {}
    for name, nb in (("blocks", 4), ("dense", None)):
        models[name] = cls(plan, 0, R, d_e, H, dropout=0.0, seed=5, num_blocks=nb).to(DEV)
        models[name].encoder.build_graph(ei, et)
        models[name].train()
    mb, md = models["blocks"], models["dense"]
    assert mb.encoder.convs[0].weight.shape == (R, 4, 16, 32)
    with torch.no_grad():                                  # the dense shard holds the expanded matrices
        md.encoder.node_embeddings.copy_(mb.encoder.node_embeddings)
        for a, b in zip(mb.encoder.convs, md.encoder.convs):
            b.weight.copy_(expand_blocks(a.weight)); b.root.copy_(a.root); b.bias.copy_(a.bias)
        md.decoder.relation_embeddings.weight.copy_(mb.decoder.relation_embeddings.weight)
    heads = torch.randint(0, N, (B,), device=DEV)
    tails = torch.randint(0, N, (B,), device=DEV)
    rels = torch.randint(0, R, (B,), device=DEV)
    labels = (torch.rand(B, device=DEV) < 0.5).float()
    s, loss = _run_partitioned(mb, heads, tails, rels, labels)
    sd, lossd = _run_partitioned(md, heads, tails, rels, labels)
    assert torch.equal(s, sd) and torch.equal(loss, lossd)     # same kernels on the same operands
    for a, b in zip(mb.encoder.convs, md.encoder.convs):
        assert torch.equal(a.weight.grad, diag_blocks(b.weight.grad, 4))
        assert torch.equal(a.root.grad, b.root.grad) and torch.equal(a.bias.grad, b.bias.grad)
    # against the single-GPU block model, at the standard of the dense partitioned model's test
    ref = pkg.DrugDiseaseModel(N, R, d_e, H, dropout=0.0, decoder_dropout=0.0, num_blocks=4).to(DEV)
    with torch.no_grad():
        ref.encoder.node_embeddings.weight.copy_(mb.encoder.node_embeddings[:N])
        for mine, theirs in zip(mb.encoder.convs, ref.encoder._layers()):
            theirs.weight.copy_(mine.weight); theirs.root.copy_(mine.root); theirs.bias.copy_(mine.bias)
        ref.decoder.relation_embeddings.weight.copy_(mb.decoder.relation_embeddings.weight)
    ref.train()
    rs = ref(ei, et, heads, tails, rels)
    rloss = F.binary_cross_entropy_with_logits(rs, labels)
    rloss.backward()
    torch.testing.assert_close(s, rs.detach(), rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(loss, rloss.detach(), rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(mb.encoder.node_embeddings.grad[:N], ref.encoder.node_embeddings.weight.grad,
                               rtol=1e-3, atol=1e-6)
    for mine, theirs in zip(mb.encoder.convs, ref.encoder._layers()):
        for a, b in ((mine.weight, theirs.weight), (mine.root, theirs.root), (mine.bias, theirs.bias)):
            assert float((a.grad - b.grad).norm() / (b.grad.norm() + 1e-30)) < 1e-4


# ------------------------------------------------------------------------------------------------
# (6) training
def test_captured_training_tracks_the_oracle(pkg):
    """cfg1 with 4 blocks: the captured step (fused clip + Adam) lowers the loss over 30 steps, and its first steps
    track the oracle model trained the same way (dropout 0, same batches, torch's clip + Adam)."""
    from primekg_rgcn_linkprediction_b200 import synth
    kg, _ = _cfg1()
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    batches = [[t.to(DEV) for t in synth.link_batch(kg, 512, seed=100 + i)] for i in range(30)]
    model = _block_model(pkg, kg, seed=0)
    ref = ModelBlocksRef(kg.num_nodes, kg.num_relations, 64, 128, 0.0, 0.0, num_blocks=4)
    ref.load_state_dict(model.state_dict())
    ref.to(DEV)
    model.train(); ref.train()
    opt = pkg.FusedAdam(model.parameters(), lr=1e-2, max_grad_norm=1.0)
    opt_ref = torch.optim.Adam(ref.parameters(), lr=1e-2)
    step = pkg.GraphedTrainStep(model, ei, et, batch_size=1024, optimizer=opt)
    crit = torch.nn.BCEWithLogitsLoss()
    losses, ref_losses = [], []
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        for it, b in enumerate(batches):
            losses.append(float(step(*b)))
            if it < 6:
                loss = crit(ref(ei, et, b[0], b[1], b[2]), b[3])
                loss.backward()
                torch.nn.utils.clip_grad_norm_(ref.parameters(), 1.0)
                opt_ref.step(); opt_ref.zero_grad()
                ref_losses.append(float(loss))
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    assert sum(losses[-5:]) / 5 < losses[0] - 0.05, losses
    for a, b in zip(losses[:6], ref_losses):
        assert abs(a - b) < 2e-3 * max(1.0, abs(b)), (losses, ref_losses)

"""The peer-memory (fused exchange) partitioned path on ONE GPU: a world-size-1 process group, so every "peer"
buffer is the local one.  This exercises the real kernels — push, transform epilogue with peer stores, pull-reduce +
mask + plane split — and the layer wiring against the single-GPU model; the multi-GPU runs are
scripts/run_partitioned.py --exchange fused --check (profiles/)."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def pg(lib_built):
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


def test_peer_kernels(pg):
    from primekg_rgcn_linkprediction_b200 import ops
    from primekg_rgcn_linkprediction_b200.peer import PeerBuffer
    buf = PeerBuffer(4 * 3000 * 64, torch.device(DEV))
    assert buf.ptrs[0] == buf.local.data_ptr()
    torch.manual_seed(0)
    x = torch.randn(1000, 64, device=DEV)
    ops.p2p_push_rows(x, buf.peer_ptrs(0), 500, 64)
    buf.barrier()
    full = buf.view(3000, 64)
    assert torch.equal(full[500:1500], x)
    # pull-reduce with two "ranks" (the same buffer twice), extra term, mask and scale
    extra = torch.randn(1000, 64, device=DEV)
    mask = torch.randn(1000, 64, device=DEV)
    planes = ops.alloc_planes(1000, 64, "fp32", DEV)
    out, part = ops.p2p_reduce_split(buf.peer_ptrs(0) * 2, 500, 64, 1000, 64, torch.device(DEV), extra=extra,
                                     relu_mask=mask, mask_scale=2.0, want_fp32=True, planes=planes, colsum=True)
    want = ((extra + x) + x) * (mask > 0) * 2.0
    assert torch.equal(out, want)
    torch.testing.assert_close(planes[0].float() + planes[1].float(), want, rtol=2e-5, atol=1e-6)
    torch.testing.assert_close(part.sum(0), want.sum(0), rtol=1e-4, atol=1e-3)


@pytest.mark.parametrize("listed", [True, False])
@pytest.mark.parametrize("layers,dropout", [(2, 0.0), (3, 0.0), (2, 0.5)])
def test_fused_partition_matches_single_gpu(pg, monkeypatch, layers, dropout, listed):
    """``listed``: the last layer computes and exchanges only the rows the decoder reads (the default) / all rows."""
    import primekg_rgcn_linkprediction_b200 as pkg
    monkeypatch.setenv("PRIMEKG_RGCN_SPARSE_FWD", "1" if listed else "0")
    from primekg_rgcn_linkprediction_b200 import dist as D
    from primekg_rgcn_linkprediction_b200 import dist_fused as DF
    from primekg_rgcn_linkprediction_b200 import synth
    torch.manual_seed(0)
    N, R, d_e, H, B = 5000, 5, 64, 128, 512
    kg = synth.uniform_kg(N, 60_000, R, seed=3)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    plan = D.plan_partition(ei[1], N, 1)
    model = DF.FusedPartitionedModel(plan, 0, R, d_e, H, dropout=dropout, num_layers=layers, seed=5).to(DEV)
    model.encoder.build_graph(ei, et)
    model.train()
    heads = torch.randint(0, N, (B,), device=DEV)
    tails = torch.randint(0, N, (B,), device=DEV)
    rels = torch.randint(0, R, (B,), device=DEV)
    labels = (torch.rand(B, device=DEV) < 0.5).float()
    s = model(heads, tails, rels)
    F.binary_cross_entropy_with_logits(s, labels).backward()
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in model.parameters())
    ref = pkg.DrugDiseaseModel(N, R, d_e, H, dropout=dropout, decoder_dropout=0.0, num_layers=layers).to(DEV)
    with torch.no_grad():
        ref.encoder.node_embeddings.weight.copy_(model.encoder.node_embeddings[:N])
        for mine, theirs in zip(model.encoder.convs, ref.encoder._layers()):
            theirs.weight.copy_(mine.weight); theirs.root.copy_(mine.root); theirs.bias.copy_(mine.bias)
            if mine._drop_ctr is not None:
                # the same dropout stream, from the counter value before the forward above: the masks are keyed by
                # global node id, so the shard draws the single-GPU model's masks
                theirs._drop_seed, theirs._drop_ctr = mine._drop_seed, mine._drop_ctr - 1
        ref.decoder.relation_embeddings.weight.copy_(model.decoder.relation_embeddings.weight)
    ref.train()
    rs = ref(ei, et, heads, tails, rels)
    F.binary_cross_entropy_with_logits(rs, labels).backward()
    torch.testing.assert_close(s, rs, rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(model.encoder.node_embeddings.grad[:N], ref.encoder.node_embeddings.weight.grad,
                               rtol=1e-3, atol=1e-6)
    for mine, theirs in zip(model.encoder.convs, ref.encoder._layers()):
        for a, b in ((mine.weight, theirs.weight), (mine.root, theirs.root), (mine.bias, theirs.bias)):
            assert float((a.grad - b.grad).norm() / (b.grad.norm() + 1e-30)) < 1e-4


def test_only_one_forward_may_be_outstanding(pg):
    """The encoder's output lives in the peer buffer: a backward through an OLDER forward must refuse (a later forward
    rewrote the buffer through raw pointers, invisible to autograd's version counters); forward-only loops are fine and
    return the same values."""
    from primekg_rgcn_linkprediction_b200 import dist as D
    from primekg_rgcn_linkprediction_b200 import dist_fused as DF
    from primekg_rgcn_linkprediction_b200 import synth
    N, R = 2000, 3
    kg = synth.uniform_kg(N, 20_000, R, seed=4)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    plan = D.plan_partition(ei[1], N, 1)
    model = DF.FusedPartitionedModel(plan, 0, R, 64, 128, dropout=0.0, num_layers=2, seed=5).to(DEV)
    model.encoder.build_graph(ei, et)
    model.eval()
    with torch.no_grad():
        a = model.encoder().clone()
        b = model.encoder()
        assert torch.equal(a, b)
    model.train()
    heads = torch.randint(0, N, (64,), device=DEV)
    s1 = model(heads, heads.flip(0), torch.zeros(64, dtype=torch.long, device=DEV))
    s2 = model(heads, heads.flip(0), torch.zeros(64, dtype=torch.long, device=DEV))
    with pytest.raises(RuntimeError, match="only one forward"):
        s1.sum().backward()
    s2.sum().backward()
    assert model.encoder.node_embeddings.grad is not None


def test_peer_allreduce_world1_and_graph_capture(pg):
    """rgcn_p2p_allreduce with one rank: out = in * scale; flags / epochs advance on the device, so a captured graph
    replays it without host help; the data-parallel GraphedTrainStep(allreduce='peer') binds p.grad to the averaged buffer."""
    import primekg_rgcn_linkprediction_b200 as pkg
    from primekg_rgcn_linkprediction_b200 import synth
    from primekg_rgcn_linkprediction_b200.peer import PeerAllReduce
    ar = PeerAllReduce(1000, torch.device(DEV))
    torch.manual_seed(0)
    x = torch.randn(ar.n, device=DEV)
    ar.inp.copy_(x)
    out = ar(scale=0.5)
    torch.cuda.synchronize()
    assert torch.equal(out, x * 0.5)
    gr = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ar()
        with torch.cuda.graph(gr):
            ar(scale=2.0)
    torch.cuda.current_stream().wait_stream(side)
    for k in range(3):
        ar.inp.copy_(x + k)
        gr.replay()
        torch.cuda.synchronize()
        assert torch.equal(ar.out, (x + k) * 2.0)
    assert int(ar.epoch.item()) == 5
    ar.check()
    # the training step with the exchange captured inside
    kg = synth.primekg_subgraph(40_000, seed=3)
    heads, tails, rels, labels = (t.to(DEV) for t in synth.link_batch(kg, 256, seed=3))
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    torch.manual_seed(1)
    model = pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, 64, 128, dropout=0.0, decoder_dropout=0.0).to(DEV)
    model.train()
    plain = pkg.GraphedTrainStep(model, ei, et, batch_size=512, flat_grads="arena")
    plain.load_batch(heads, tails, rels, labels)
    plain()
    want = {k: p.grad.clone() for k, p in model.named_parameters()}
    for p in model.parameters():
        p.grad = None
    step = pkg.GraphedTrainStep(model, ei, et, batch_size=512, flat_grads="arena", allreduce="peer")
    step.load_batch(heads, tails, rels, labels)
    step()
    torch.cuda.synchronize()
    lo, hi = step.peer_ar.out.data_ptr(), step.peer_ar.out.data_ptr() + step.peer_ar.out.numel() * 4
    for k, p in model.named_parameters():
        assert lo <= p.grad.data_ptr() < hi, k
        assert torch.equal(p.grad, want[k]), k                    # one rank: the average is the gradient itself
    step.peer_ar.check()

"""Two-GPU tests of the peer-memory partitioned path (skipped on a one-GPU box): forward-only loops with skewed ranks,
the training forward's dropout masks against the single-GPU model's."""
import os
import socket

import pytest
import torch
import torch.distributed as dist

pytestmark = pytest.mark.gpu


def _two_rank_worker(rank, port, ret):
    import sys
    from conftest import ROOT
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=2, device_id=dev)
    try:
        import primekg_rgcn_linkprediction_b200 as pkg
        from primekg_rgcn_linkprediction_b200 import dist as D
        from primekg_rgcn_linkprediction_b200 import dist_fused as DF
        from primekg_rgcn_linkprediction_b200 import synth
        N, R = 20_000, 3
        kg = synth.uniform_kg(N, 400_000, R, seed=4)
        ei, et = kg.edge_index.to(dev), kg.edge_type.to(dev)
        plan = D.plan_partition(ei[1], N, 2)
        model = DF.FusedPartitionedModel(plan, rank, R, 64, 128, dropout=0.0, num_layers=2, seed=5).to(dev)
        model.encoder.build_graph(ei, et)
        model.eval()
        with torch.no_grad():
            out1 = model.encoder()
            if rank == 0:
                torch.cuda._sleep(200_000_000)          # ~0.1 s: rank 0's consumer of out1 lags behind rank 1
            kept = out1.clone()                          # the "decoder" reading the first output
            model.encoder.node_embeddings.mul_(2.0)      # the second forward pushes other values
            out2 = model.encoder()
            again = out2.clone()
            model.encoder.node_embeddings.mul_(0.5)
            out3 = model.encoder().clone()
        torch.cuda.synchronize()
        ok = bool(torch.equal(kept, out3)) and not bool(torch.equal(kept, again))
        ret[rank] = ok
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_forward_only_loop_with_skewed_ranks_two_gpus(lib_built):
    """ADVICE r1: a fast rank must not store the next forward's rows into a buffer a slow rank is still reading."""
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ret = mp.get_context("spawn").Manager().dict()
    mp.spawn(_two_rank_worker, args=(port, ret), nprocs=2, join=True)
    assert ret.get(0) is True and ret.get(1) is True


def _dropout_worker(rank, port, ret):
    import sys
    from conftest import ROOT
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=2, device_id=dev)
    try:
        import primekg_rgcn_linkprediction_b200 as pkg
        from primekg_rgcn_linkprediction_b200 import dist as D
        from primekg_rgcn_linkprediction_b200 import dist_fused as DF
        from primekg_rgcn_linkprediction_b200 import synth
        N, R = 20_000, 3
        kg = synth.uniform_kg(N, 400_000, R, seed=4)
        ei, et = kg.edge_index.to(dev), kg.edge_type.to(dev)
        plan = D.plan_partition(ei[1], N, 2)
        model = DF.FusedPartitionedModel(plan, rank, R, 64, 128, dropout=0.5, num_layers=3, seed=5).to(dev)
        model.encoder.build_graph(ei, et)
        model.train()
        torch.manual_seed(11)                             # the same dropout seeds on both ranks
        with torch.no_grad():
            out = model.encoder().clone()                 # all ranks' rows, padded id order
        shards = [torch.empty_like(model.encoder.node_embeddings) for _ in range(2)]
        dist.all_gather(shards, model.encoder.node_embeddings.detach().contiguous())
        ref = pkg.DrugDiseaseModel(N, R, 64, 128, dropout=0.5, decoder_dropout=0.0, num_layers=3).to(dev)
        with torch.no_grad():
            ref.encoder.node_embeddings.weight.copy_(torch.cat([shards[p][: plan.size(p)] for p in range(2)]))
            for mine, theirs in zip(model.encoder.convs, ref.encoder._layers()):
                theirs.weight.copy_(mine.weight); theirs.root.copy_(mine.root); theirs.bias.copy_(mine.bias)
                if mine._drop_ctr is not None:
                    theirs._drop_seed, theirs._drop_ctr = mine._drop_seed, mine._drop_ctr - 1
            ref.train()
            want = ref.encoder(ei, et)
        got = out[plan.to_padded(torch.arange(N, device=dev))]
        torch.testing.assert_close(got, want, rtol=1e-4, atol=1e-5)
        ret[rank] = True
    except Exception:
        import traceback
        ret[rank] = traceback.format_exc()
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_training_forward_dropout_equals_single_gpu_two_gpus(lib_built):
    """With dropout the fused mask is keyed by global node id: both shards draw the single-GPU model's masks."""
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ret = mp.get_context("spawn").Manager().dict()
    mp.spawn(_dropout_worker, args=(port, ret), nprocs=2, join=True)
    assert ret.get(0) is True and ret.get(1) is True, (ret.get(0), ret.get(1))


def _allreduce_worker(rank, port, ret):
    import sys
    from conftest import ROOT
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=2, device_id=dev)
    try:
        from primekg_rgcn_linkprediction_b200.peer import PeerAllReduce
        n = 2_300_000
        ar = PeerAllReduce(n, dev)
        ok = True
        for it in range(4):
            g = torch.Generator(device=dev).manual_seed(100 * it + rank)
            x = torch.randn(ar.n, generator=g, device=dev)
            ar.inp.copy_(x)
            if rank == it % 2:
                torch.cuda._sleep(50_000_000)                  # skew the ranks
            out = ar().clone()
            ref = x.clone()
            dist.all_reduce(ref)
            ref /= 2
            ok = ok and bool(torch.allclose(out, ref, rtol=0, atol=1e-6))
            both = [torch.empty_like(out) for _ in range(2)]
            dist.all_gather(both, out)
            ok = ok and bool(torch.equal(both[0], both[1]))   # rank-ordered sums: every rank holds the same bits
        ar.check()
        ret[rank] = ok
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_peer_allreduce_two_gpus(lib_built):
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ret = mp.get_context("spawn").Manager().dict()
    mp.spawn(_allreduce_worker, args=(port, ret), nprocs=2, join=True)
    assert ret.get(0) is True and ret.get(1) is True

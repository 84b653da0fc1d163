"""world_size-2 gloo tests (CPU) of the destination-range partitioned path: plan, padded relabelling, all-gather /
reduce-scatter / all-reduce with autograd, layer wiring.  The kernels are replaced by CPU stand-ins
(tests/cpu_ops_emulation.py); the 2-rank result must equal the single-process oracle on the unpartitioned graph."""
import os
import socket
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT


class _HashDropout(torch.nn.Module):
    """The fused dropout's keep masks (one per ReLU layer, in call order) applied as the reference's nn.Dropout."""

    def __init__(self, keeps, scale):
        super().__init__()
        self.keeps, self.scale = list(keeps), scale

    def forward(self, x):
        return torch.where(self.keeps.pop(0), x * self.scale, 0.0)


def _worker(rank, world, port, ret, dropout):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import cpu_ops_emulation as emu
        from oracle import rgcn_ref as O
        from primekg_rgcn_linkprediction_b200 import dist as D
        from primekg_rgcn_linkprediction_b200 import ops, synth
        emu.install(ops)
        torch.set_num_threads(1)
        N, R, d_e, H = 97, 3, 8, 12
        kg = synth.uniform_kg(N, 700, R, seed=5)
        # make it skewed: route a third of the edges into node 3 so the edge-balanced ranges are uneven
        ei = kg.edge_index.clone()
        ei[1, ::3] = 3
        et = kg.edge_type
        plan = D.plan_partition(ei[1], N, world)
        assert plan.bounds[0] == 0 and plan.bounds[-1] == N and sorted(plan.bounds) == plan.bounds
        assert plan.bounds[1] > 0
        enc = D.PartitionedRGCN(plan, rank, R, d_e, H, dropout=dropout, num_layers=3, seed=9)
        src, dst, rel = D.local_edges(ei, et, plan, rank)
        enc.set_graph(emu.CpuGraph(src, dst, rel, plan.max_n, world * plan.max_n, R))
        torch.manual_seed(7)                                   # the same dropout seeds on every rank, as in the models
        out = enc()                                            # [max_n, H], this rank's rows
        n_loc = plan.size(rank)
        g = torch.Generator().manual_seed(100)
        coef_full = torch.randn(N, H, generator=g)
        loss = (out[:n_loc] * coef_full[plan.bounds[rank]:plan.bounds[rank + 1]]).sum()
        loss.backward()
        # ---- single-process oracle on the unpartitioned graph with the same parameters ----
        shards = [torch.zeros(plan.max_n, d_e) for _ in range(world)]
        dist.all_gather(shards, enc.node_embeddings.detach())
        table = torch.cat([shards[p][: plan.size(p)] for p in range(world)], 0)
        ref = O.EncoderRef(N, R, d_e, H, 0.0, None, num_layers=3)
        if dropout > 0.0:
            # one mask per ReLU layer over ALL nodes, keyed by global node id: the shards must draw these very masks
            from test_gpu_gemm_conformance import drop_keep, drop_scale
            keeps = [drop_keep(N, 0, H, dropout, conv._drop_seed, int(conv._drop_ctr), device="cpu")
                     for conv in enc.convs[:-1]]
            ref.dropout = _HashDropout(keeps, drop_scale(dropout))
        with torch.no_grad():
            ref.node_embeddings.weight.copy_(table)
            for mine, theirs in zip(enc.convs, [ref.conv1, ref.conv2] + list(ref.extra)):
                theirs.weight.copy_(mine.weight); theirs.root.copy_(mine.root); theirs.bias.copy_(mine.bias)
        ref_out = ref(ei, et)
        (ref_out * coef_full).sum().backward()
        lo, hi = plan.bounds[rank], plan.bounds[rank + 1]
        torch.testing.assert_close(out[:n_loc].detach(), ref_out[lo:hi].detach(), rtol=1e-4, atol=1e-5)
        torch.testing.assert_close(enc.node_embeddings.grad[:n_loc], ref.node_embeddings.weight.grad[lo:hi],
                                   rtol=1e-4, atol=1e-5)
        assert float(enc.node_embeddings.grad[n_loc:].abs().sum()) == 0.0          # padding rows get no gradient
        for mine, theirs in zip(enc.convs, [ref.conv1, ref.conv2] + list(ref.extra)):
            torch.testing.assert_close(mine.weight.grad, theirs.weight.grad, rtol=1e-4, atol=1e-5)
            torch.testing.assert_close(mine.root.grad, theirs.root.grad, rtol=1e-4, atol=1e-5)
            torch.testing.assert_close(mine.bias.grad, theirs.bias.grad, rtol=1e-4, atol=1e-5)
        full = D.gather_embeddings(out.detach())
        pid = plan.to_padded(torch.arange(N))
        torch.testing.assert_close(full[pid], ref_out.detach(), rtol=1e-4, atol=1e-5)
        ret[rank] = "ok"
    except Exception as e:  # pragma: no cover
        import traceback
        ret[rank] = "FAIL: " + traceback.format_exc()
    finally:
        dist.destroy_process_group()


def test_partitioned_encoder_two_ranks_equals_single_process():
    _run_two_ranks(0.0)


def test_partitioned_encoder_two_ranks_dropout_masks_equal_single_process():
    """The fused dropout mask is keyed by global node id, so the 2-rank encoder draws the single-process masks."""
    _run_two_ranks(0.5)


def _run_two_ranks(dropout):
    world = 2
    mgr = mp.Manager()
    ret = mgr.dict()
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mp.spawn(_worker, args=(world, port, ret, dropout), nprocs=world, join=True)
    for r in range(world):
        assert ret.get(r) == "ok", ret.get(r)


def test_partition_plan_balances_in_edges():
    sys.path.insert(0, ROOT)
    from primekg_rgcn_linkprediction_b200 import dist as D
    from primekg_rgcn_linkprediction_b200 import synth
    kg = synth.primekg_subgraph(200_000, seed=2)
    for P in (2, 4, 8):
        plan = D.plan_partition(kg.edge_index[1], kg.num_nodes, P)
        deg = torch.bincount(kg.edge_index[1], minlength=kg.num_nodes)
        per = [int(deg[plan.bounds[p]:plan.bounds[p + 1]].sum()) for p in range(P)]
        assert sum(per) == kg.num_edges
        hub = int(deg.max())
        assert max(per) <= kg.num_edges / P + hub                # within one hub of perfectly balanced
        ids = torch.arange(kg.num_nodes)
        pid = plan.to_padded(ids)
        assert pid.unique().numel() == kg.num_nodes and int(pid.max()) < P * plan.max_n
        for p in range(P):                                        # owner-major, order preserving
            seg = pid[plan.bounds[p]:plan.bounds[p + 1]]
            assert torch.equal(seg, p * plan.max_n + torch.arange(seg.numel()))

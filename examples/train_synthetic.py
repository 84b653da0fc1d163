"""The reference's training epoch (src/train.py:247-347) on the fast path, on a synthetic PrimeKG-shaped graph.

Per step: positives in -> negatives drawn on the device -> full-graph 2-layer RGCN forward -> fused decoder + BCE loss +
accuracy -> backward, all replayed as ONE CUDA graph (``GraphedTrainStep`` with a ``NegativeSampler``), then the
reference's own clipping and Adam step (src/train.py:311-318).  ``--optimizer fused`` passes a ``FusedAdam(max_grad_norm=1.0)``
into the graphed step instead: clipping and Adam become the last kernels of the same graph, one replay per iteration.
``--negatives filtered`` redraws negatives that are edges of the graph; ``typed`` also keeps every replaced end to a node
type the relation takes on that side (the graph's three type blocks) and picks head or tail with the Bernoulli
probability of the relation; ``uniform`` (default) is the reference's sampler.
Loss and accuracy stay on the device and are read once per logging interval instead of twice per step (src/train.py:322,
:325).

    python examples/train_synthetic.py [--steps 300] [--hidden 128] [--batch 1024] [--optimizer torch|fused]
                                        [--negatives uniform|filtered|typed]
"""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import primekg_rgcn_linkprediction_b200 as pkg
from primekg_rgcn_linkprediction_b200 import synth


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--hidden", type=int, default=128)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--lr", type=float, default=0.01)
    ap.add_argument("--edges", type=int, default=849_456)
    ap.add_argument("--optimizer", choices=("torch", "fused"), default="torch")
    ap.add_argument("--negatives", choices=("uniform", "filtered", "typed"), default="uniform")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.manual_seed(42)
    kg = synth.primekg_subgraph(args.edges, seed=42)
    ei, et = kg.edge_index.to(dev), kg.edge_type.to(dev)
    model = pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, 64, args.hidden, dropout=0.5, decoder_dropout=0.1).to(dev)
    model.train()
    fused = args.optimizer == "fused"
    opt = (pkg.FusedAdam(model.parameters(), lr=args.lr, max_grad_norm=1.0) if fused
           else torch.optim.Adam(model.parameters(), lr=args.lr))
    kw = {}
    if args.negatives != "uniform":
        known = pkg.KnownTriples.from_graphs(kg.as_dict(), device=dev)
        kw["filter"] = known
        if args.negatives == "typed":
            node_type = torch.empty(kg.num_nodes, dtype=torch.int64)
            for i, (lo, hi) in enumerate(kg.blocks.values()):
                node_type[lo:hi] = i
            kw["constraints"] = pkg.RelationConstraints.from_node_types(known, node_type)
            kw["head_prob"] = known.bernoulli_head_prob()
    sampler = pkg.NegativeSampler(kg.num_nodes, 1, **kw)
    step = pkg.GraphedTrainStep(model, ei, et, batch_size=2 * args.batch, sampler=sampler,
                                optimizer=opt if fused else None)
    params = [p for p in model.parameters()]
    perm = torch.randperm(kg.num_edges, device=dev)
    loss_sum = torch.zeros((), device=dev)
    correct_sum = torch.zeros((), dtype=torch.int64, device=dev)
    first = last = None
    t0 = time.perf_counter()
    for it in range(args.steps):
        lo = (it * args.batch) % (kg.num_edges - args.batch)
        idx = perm[lo:lo + args.batch]
        loss = step.run_positives(ei[0, idx], ei[1, idx], et[idx])           # src/train.py:276-306 as one graph replay
        if not fused:                                                          # (fused: inside the replay)
            torch.nn.utils.clip_grad_norm_(params, 1.0)                        # src/train.py:311-315
            opt.step()                                                         # src/train.py:317
        loss_sum += loss
        correct_sum += step.correct
        if (it + 1) % 50 == 0:                                                 # one host read per logging interval
            avg, acc = float(loss_sum) / 50, int(correct_sum) / (50 * 2 * args.batch)
            first = avg if first is None else first
            last = avg
            print(f"step {it + 1:5d}  loss {avg:.4f}  accuracy {acc:.3f}  {(time.perf_counter() - t0) / (it + 1) * 1e3:.2f} ms/step")
            loss_sum.zero_(); correct_sum.zero_()
    if first is not None and last is not None and args.steps >= 100:
        assert last < first, "the loss did not go down"
        print(f"loss {first:.4f} -> {last:.4f}")
    if args.negatives != "uniform":
        print(f"negatives that kept a rejected draw: {int(sampler.exhausted)}")


if __name__ == "__main__":
    main()

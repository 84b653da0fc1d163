"""Filtered and type-constrained negative sampling on the B200: the sampler kernel's own time, the mean number of draws
per negative, and the captured cfg2 training iteration with each sampler; the card's name and power limit read in the
same run.

* kernel: ``NegativeSampler.batch`` for 1,024 edges of the cfg2 graph (``synth.primekg_subgraph()``) as positives and
  num_neg in {1, 4, 16}: plain (``rgcn_link_batch_ex`` with no tables, one thread per output entry), filtered (the whole
  graph as the filter) and filtered + typed (the graph's three node-type blocks), beside the one-block
  ``rgcn_link_batch``.  Each launch sits between two CUDA events; the launches are queued behind a device sleep so no
  host gap is timed; median over ``--launches`` launches after a warm-up.  The 10 MB lookup index stays in L2.
* tries: draws are a pure function of (seed, counter value, negative, attempt), so rerunning one batch with
  ``max_tries = j`` counts the negatives whose first j draws were all rejected; mean tries = 1 + sum_j of those counts
  over the number of negatives (``max_tries`` = 32).
* iteration: ``GraphedTrainStep(model, ..., sampler=..., optimizer=FusedAdam(...))`` at cfg2 (64 -> 256 -> 256, 1,024
  positives + 1,024 negatives, dropout 0.5 / 0.1), plain against filtered + typed sampler, alternated, each a host clock
  around ``--iters`` replays that end in a device synchronise; median over ``--repeats``.

Usage: python scripts/bench_sampler.py [--launches 400] [--iters 200] [--repeats 7] [--out FILE]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

DEV = torch.device("cuda:0")


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def kernel_us(fn, launches):
    for _ in range(20):
        fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(launches)]
    torch.cuda._sleep(200_000_000)              # the queue fills while the device sleeps: no host gap between events
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return statistics.median(a.elapsed_time(b) for a, b in ev) * 1e3


def mean_tries(s, pos, n_batches=20):
    n_neg = pos[0].numel() * s.num_neg_samples
    keep = s.max_tries
    total = 0.0
    for c in range(n_batches):
        rejected = []
        for j in range(1, keep):
            s.max_tries = j
            s._ctr.fill_(1000 + c)
            s.exhausted.zero_()
            s.batch(*pos)
            rejected.append(int(s.exhausted))
            if rejected[-1] == 0:
                break
        total += 1.0 + sum(rejected) / n_neg
    s.max_tries = keep
    return total / n_batches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=400)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_bench_sampler.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sampler.py needs a CUDA device")
    import primekg_rgcn_linkprediction_b200 as pkg
    from primekg_rgcn_linkprediction_b200 import ops, synth
    kg = synth.primekg_subgraph(849_456, seed=42)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    N = kg.num_nodes
    t0 = time.perf_counter()
    known = pkg.KnownTriples.from_graphs(kg.as_dict(), device=DEV)
    node_type = torch.empty(N, dtype=torch.int64)
    for i, (lo, hi) in enumerate(kg.blocks.values()):
        node_type[lo:hi] = i
    types = pkg.RelationConstraints.from_node_types(known, node_type)
    torch.cuda.synchronize()
    build_ms = (time.perf_counter() - t0) * 1e3
    g = torch.Generator().manual_seed(3)
    sel = torch.randint(0, kg.num_edges, (1024,), generator=g)
    pos = (kg.edge_index[0, sel].to(DEV), kg.edge_index[1, sel].to(DEV), kg.edge_type[sel].to(DEV))

    kernel, tries, same_bits = {}, {}, {}
    for k in (1, 4, 16):
        torch.manual_seed(k)
        samplers = {"plain": pkg.NegativeSampler(N, k),
                    "filtered": pkg.NegativeSampler(N, k, filter=known),
                    "filtered_typed": pkg.NegativeSampler(N, k, filter=known, constraints=types)}
        out = [tuple(torch.empty(1024 * (1 + k), dtype=dt, device=DEV) for dt in (torch.int64,) * 3 + (torch.float32,))
               for _ in range(2)]
        ctr = ops.rng_counter(DEV)
        plain = samplers["plain"]
        fns = {"link_batch_one_block": lambda: ops.link_batch(*pos, N, k, plain._seed, ctr, out=out[1])}
        for name, s in samplers.items():
            fns[name] = lambda s=s: s.batch(*pos, out=out[0])
        kernel[f"num_neg={k}"] = {name: round(kernel_us(fn, args.launches), 2) for name, fn in fns.items()}
        plain._ctr.fill_(77); ctr.fill_(77)
        plain.batch(*pos, out=out[0])
        ops.link_batch(*pos, N, k, plain._seed, ctr, out=out[1])
        same_bits[f"num_neg={k}"] = all(torch.equal(a, b) for a, b in zip(*out))
        tries[f"num_neg={k}"] = {name: round(mean_tries(s, pos), 5) for name, s in samplers.items() if name != "plain"}

    def model():
        torch.manual_seed(42)
        return pkg.DrugDiseaseModel(N, kg.num_relations, 64, 256, dropout=0.5, decoder_dropout=0.1).to(DEV).train()

    steps = {}
    for name, kw in (("plain", {}), ("filtered_typed", dict(filter=known, constraints=types))):
        m = model()
        torch.manual_seed(5)
        s = pkg.NegativeSampler(N, 1, **kw)
        steps[name] = pkg.GraphedTrainStep(m, ei, et, batch_size=2048, sampler=s,
                                           optimizer=pkg.FusedAdam(m.parameters(), lr=1e-3, max_grad_norm=1.0))
    for st in steps.values():
        for _ in range(20):
            st.run_positives(*pos)
    torch.cuda.synchronize()
    times = {k: [] for k in steps}
    for _ in range(args.repeats):
        for name, st in steps.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.iters):
                st.run_positives(*pos)
            torch.cuda.synchronize()
            times[name].append((time.perf_counter() - t0) / args.iters * 1e3)
    med = {k: statistics.median(v) for k, v in times.items()}

    res = {
        "script": "scripts/bench_sampler.py",
        "gpu": gpu_info(),
        "workload": "cfg2 graph: 30,926 nodes / 849,456 edges / 3 relations; 1,024 edge positives; filter = the whole "
                    f"graph ({len(known):,} distinct triples); types = the 3 node-type blocks",
        "index_build_ms": round(build_ms, 1),
        "kernel_us_median": kernel,
        "launches_per_median": args.launches,
        "plain_bitwise_equals_link_batch": same_bits,
        "mean_tries_per_negative": tries,
        "train_iter_ms_median": {k: round(v, 4) for k, v in med.items()},
        "train_iter_ms_min_max": {k: [round(min(v), 4), round(max(v), 4)] for k, v in times.items()},
        "train_iter_filtered_typed_over_plain": round(med["filtered_typed"] / med["plain"], 4),
        "train_iter": f"GraphedTrainStep(sampler, FusedAdam) 64->256->256, 1024 + 1024, {args.iters} iters x "
                      f"{args.repeats} repeats, alternated",
        "last_loss": {k: round(float(st.loss), 5) for k, st in steps.items()},
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

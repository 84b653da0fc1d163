"""Whole training iterations on cfg2 (the benchmark's workload), optimiser included: what the eager clip + Adam after
each graph replay costs, against the fused optimiser captured inside the step.

Arms, interleaved, each timed with a host clock around ``--iters`` iterations that end in a device synchronise:
  (a) GraphedTrainStep replay + torch clip_grad_norm_(1.0) + torch.optim.Adam (default: foreach)
  (b) the same with torch.optim.Adam(fused=True)
  (c) GraphedTrainStep(optimizer=FusedAdam(max_grad_norm=1.0)): one replay is the whole iteration
Also: device time of the optimiser's own kernels (50 steps captured in a CUDA graph, CUDA events around replays; warm
L2 back to back, and cold L2 with a 512 MiB write before every step, the write's own time subtracted), against the
algorithmic bytes (4 P for the norm pass, 28 P for the update) at the 7.7 TB/s data-sheet HBM rate.

    python scripts/bench_train_iter.py [--iters 200] [--repeats 5] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

HBM_TBPS = 7.7                      # HGX B200 data sheet, one GPU


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_train_iter.py needs a CUDA device")
    import primekg_rgcn_linkprediction_b200 as pkg
    from primekg_rgcn_linkprediction_b200 import synth
    dev = torch.device("cuda:0")
    kg = synth.primekg_subgraph(849_456, seed=42)
    ei, et = kg.edge_index.to(dev), kg.edge_type.to(dev)
    batch = [t.to(dev) for t in synth.link_batch(kg, 1024)]

    def model():
        torch.manual_seed(42)
        m = pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, 64, 256, dropout=0.5, decoder_dropout=0.1).to(dev)
        return m.train()

    arms = {}
    for name, kind in (("a_torch_adam", "foreach"), ("b_torch_adam_fused", "fused")):
        m = model()
        params = list(m.parameters())
        opt = torch.optim.Adam(params, lr=1e-3, fused=(kind == "fused"))
        step = pkg.GraphedTrainStep(m, ei, et, batch_size=batch[0].numel())
        step.load_batch(*batch)

        def it(step=step, params=params, opt=opt):
            step()
            torch.nn.utils.clip_grad_norm_(params, 1.0)
            opt.step()
        arms[name] = (it, step)
    mc = model()
    fopt = pkg.FusedAdam(mc.parameters(), lr=1e-3, max_grad_norm=1.0)
    step_c = pkg.GraphedTrainStep(mc, ei, et, batch_size=batch[0].numel(), optimizer=fopt)
    step_c.load_batch(*batch)
    arms["c_fused_adam_in_graph"] = (step_c, step_c)

    for it, _ in arms.values():                          # warm every arm (torch's optimiser state, allocator)
        for _ in range(10):
            it()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(args.repeats):
        for name, (it, _) in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.iters):
                it()
            torch.cuda.synchronize()
            times[name].append((time.perf_counter() - t0) / args.iters * 1e3)
    losses = {k: float(s.loss) for k, (_, s) in arms.items()}

    # the optimiser kernels alone: eager FusedAdam steps over cfg2's parameters, captured so no host gap is timed
    params = list(mc.parameters())
    P = sum(p.numel() for p in params)
    pairs = [(p, p.grad) for p in params]
    flush = torch.empty(512 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    n_in = 50
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graphs = {}
    with torch.cuda.stream(side):
        fopt._launch(pairs)
        flush.fill_(1.0)
        for kind in ("warm", "flush", "cold"):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                for _ in range(n_in):
                    if kind != "warm":
                        flush.fill_(1.0)
                    if kind != "flush":
                        fopt._launch(pairs)
            graphs[kind] = g
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()

    def graph_us(g, reps=10):
        g.replay()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            g.replay()
        b.record()
        b.synchronize()
        return a.elapsed_time(b) * 1e3 / (reps * n_in)

    kt = {k: [] for k in graphs}
    for _ in range(args.repeats):
        for k, g in graphs.items():
            kt[k].append(graph_us(g))
    warm_us = statistics.median(kt["warm"])
    cold_us = statistics.median(kt["cold"]) - statistics.median(kt["flush"])
    nbytes = 32 * P
    floor_us = nbytes / (HBM_TBPS * 1e12) * 1e6

    med = {k: statistics.median(v) for k, v in times.items()}
    out = {
        "script": "scripts/bench_train_iter.py",
        "gpu": gpu_info(),
        "workload": "cfg2: 30,926 nodes / 849,456 edges / 3 rel, 64->256->256, batch 1024+1024, dropout 0.5 / 0.1",
        "iters_per_repeat": args.iters, "repeats": args.repeats,
        "ms_per_iter_median": {k: round(v, 4) for k, v in med.items()},
        "ms_per_iter_min_max": {k: [round(min(v), 4), round(max(v), 4)] for k, v in times.items()},
        "c_vs_a": round(med["c_fused_adam_in_graph"] / med["a_torch_adam"], 4),
        "c_vs_b": round(med["c_fused_adam_in_graph"] / med["b_torch_adam_fused"], 4),
        "last_loss": {k: round(v, 5) for k, v in losses.items()},
        "optimizer_kernels": {
            "params": P, "algorithmic_bytes": nbytes, "hbm_floor_us_at_7.7TBps": round(floor_us, 2),
            "us_per_step_warm_l2": round(warm_us, 2), "us_per_step_cold_l2": round(cold_us, 2),
            "warm_l2_effective_TBps": round(nbytes / (warm_us * 1e-6) / 1e12, 2),
            "cold_l2_effective_TBps": round(nbytes / (cold_us * 1e-6) / 1e12, 2),
            "floor_over_cold": round(floor_us / cold_us, 3),
            "spread_us": {k: [round(min(v), 2), round(max(v), 2)] for k, v in kt.items()},
            "note": "warm: 50 back-to-back steps, the 74 MB working set stays in the 126 MB L2; cold: a 512 MiB write "
                    "before every step (its own time subtracted), the step reads from HBM",
        },
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

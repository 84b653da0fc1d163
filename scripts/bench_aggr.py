"""RGCNConv(aggr='mean' / 'sum' / 'max'): captured training steps and the walks' kernel times.

Workload: cfg2 (synth.primekg_subgraph(): 30,926 nodes, 849,456 edges, 3 relations) and cfg3 (synth.primekg_full():
129,375 nodes, ~8.1 M edges, 30 relations), 64 -> 256 -> 256, batch 1024 + 1024, dropout 0.5, the captured
``GraphedTrainStep`` replayed with the L2 overwritten before every step (CUDA events; two passes over the variants, the
second in reverse order).  The walks alone (forward: mean over the planes, max over the planes + fp32 maxima and tie
counts; backward: the transposed walks) are timed over back-to-back launches at the layer-2 shape (d = 256) with the
bytes each must move at least, against 7.7 TB/s.  "mean_unlisted" is the mean model with the listed last layer turned off
(PRIMEKG_RGCN_SPARSE_FWD=0): a max model's last layer walks all rows, and this isolates what that costs.  With
``--parent DIR`` (a checkout of the parent commit, built), ``bench.py --gpus 1 --quick`` runs alternately there and here,
``--ab`` times each, in the same call: the mean step before and after this change.  The card's name and power limit are
read in the same run.

Usage: python scripts/bench_aggr.py [--steps 10] [--out FILE] [--parent DIR --ab 3]"""
import argparse
import gc
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

DEV = torch.device("cuda:0")
HBM = 7.7e12
VARIANTS = [(cfg, aggr, mode) for cfg in ("cfg2", "cfg3") for mode in ("fp32", "bf16")
            for aggr in ("mean", "sum", "max", "mean_unlisted")]


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def time_steps(step, flush, steps):
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    ts = []
    for _ in range(steps):
        flush.fill_(0.0)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); step(); b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts)


def time_us(fn, flush, launches=20):
    fn(); torch.cuda.synchronize()
    ts = []
    for _ in range(launches):
        flush.fill_(0.0)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    return statistics.median(ts)


def walks(pkg, kg, d, flush):
    from primekg_rgcn_linkprediction_b200 import ops
    g = pkg.RelGraph.from_edges(kg.edge_index.to(DEV), kg.edge_type.to(DEV), kg.num_nodes, kg.num_relations)
    N, R, E = g.n_dst, g.R, g.E
    x = torch.randn(N, d, device=DEV)
    A = ops.alloc_planes(N, (R + 1) * d, "fp32", DEV)
    gA = torch.randn(N, (R + 1) * d, device=DEV)
    Hmax, Hcnt = ops.aggregate_max_fwd(g, x, A, x_root=x)
    # the least each walk must move: every input row once (the gathers repeat them, from L2 at best), the CSR, the output
    xb, blk, csr = N * d * 4, N * R * d * 4, (N * R + 1) * 4 + E * 4
    planes = N * (R + 1) * d * 4                                  # bf16 hi + lo = 4 bytes per element
    cases = {
        "mean_fwd": (lambda: ops.aggregate_fwd(g, x, planes=A, x_root=x), xb + csr + planes),
        "max_fwd": (lambda: ops.aggregate_max_fwd(g, x, A, x_root=x), xb + csr + planes + 2 * blk),
        "mean_bwd": (lambda: ops.aggregate_bwd(g, gA, d, init=gA[:, R * d:]), blk + xb + csr + E * 4 + xb),
        "max_bwd": (lambda: ops.aggregate_max_bwd(g, gA, Hmax, Hcnt, x, init=gA[:, R * d:]), 3 * blk + 2 * xb + csr + xb),
    }
    out = {}
    for k, (fn, nbytes) in cases.items():
        us = time_us(fn, flush)
        out[k] = {"us": round(us, 1), "min_bytes": nbytes, "TB_per_s": round(nbytes / us * 1e-6, 3),
                  "share_of_7.7TB_s": round(nbytes / us * 1e6 / HBM, 3)}
    return out


def parent_ab(parent, runs):
    """ms / step of ``bench.py --gpus 1 --steps 20 --warmup 3 --quick`` (the default mean workload), parent and this tree
    alternated ``runs`` times each in this process's call."""
    out = {"command": "bench.py --gpus 1 --steps 20 --warmup 3 --quick", "parent_ms": [], "this_ms": []}
    for _ in range(runs):
        for key, cwd in (("parent_ms", parent), ("this_ms", ROOT)):
            r = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", "20", "--warmup", "3", "--quick"],
                               cwd=cwd, capture_output=True, text=True)
            line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
            out[key].append(round(json.loads(line)["ms_per_step"], 4))
    for key in ("parent_ms", "this_ms"):
        v = out[key]
        out[key.replace("_ms", "_median_ms")] = statistics.median(v)
        out[key.replace("_ms", "_spread_ms")] = round(max(v) - min(v), 4)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_bench_aggr.json"))
    ap.add_argument("--parent", default=None, help="built checkout of the parent commit (mean step A/B)")
    ap.add_argument("--ab", type=int, default=3, help="bench.py runs per side, alternated")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_aggr.py measures on the GPU; there is none here")
    import primekg_rgcn_linkprediction_b200 as pkg
    from primekg_rgcn_linkprediction_b200 import synth
    kgs = {"cfg2": synth.primekg_subgraph(), "cfg3": synth.primekg_full()}
    data = {k: (kg, kg.edge_index.to(DEV), kg.edge_type.to(DEV), [t.to(DEV) for t in synth.link_batch(kg, 1024)])
            for k, kg in kgs.items()}
    flush = torch.empty(128 * 1024 * 1024, dtype=torch.float32, device=DEV)      # 512 MB > L2
    rec = {"card": gpu_info(), "steps_per_timing": args.steps,
           "workload": "cfg2: 30,926 nodes / 849,456 edges / 3 rel; cfg3: 129,375 nodes / ~8.1 M edges / 30 rel; "
                       "64->256->256, batch 1024+1024, dropout 0.5, GraphedTrainStep replay, L2 overwritten before "
                       "every step",
           "walks_d256": {k: walks(pkg, kgs[k], 256, flush) for k in ("cfg2", "cfg3")}}
    print(json.dumps(rec["walks_d256"]), flush=True)
    results = {}
    for order in (VARIANTS, VARIANTS[::-1]):
        for v in order:
            cfg, aggr, mode = v
            kg, ei, et, batch = data[cfg]
            gc.collect(); torch.cuda.empty_cache()
            torch.manual_seed(42)
            os.environ["PRIMEKG_RGCN_SPARSE_FWD"] = "0" if aggr == "mean_unlisted" else "1"
            model = pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, 64, 256, dropout=0.5, decoder_dropout=0.1,
                                         aggr=aggr.replace("_unlisted", "")).to(DEV)
            for c in model.encoder._layers():
                c.mode = mode
            model.train()
            step = pkg.GraphedTrainStep(model, ei, et, batch_size=2048)
            step.load_batch(*batch)
            ms = time_steps(step, flush, args.steps)
            r = results.setdefault(v, {"config": cfg, "aggr": aggr, "mode": mode, "ms_per_step_passes": []})
            r["ms_per_step_passes"].append(round(ms, 4))
            r["loss"] = float(step.loss)
            del model, step
            print(json.dumps(r), flush=True)
    os.environ.pop("PRIMEKG_RGCN_SPARSE_FWD", None)
    if args.parent:
        rec["mean_step_vs_parent"] = parent_ab(args.parent, args.ab)
        print(json.dumps(rec["mean_step_vs_parent"]), flush=True)
    rec["steps"] = []
    for v in VARIANTS:
        r = results[v]
        r["ms_per_step"] = round(statistics.mean(r["ms_per_step_passes"]), 4)
        rec["steps"].append(r)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec))


if __name__ == "__main__":
    main()

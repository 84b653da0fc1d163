"""Block-diagonal relation weights (RGCNConv(num_blocks=nb)) against the dense layer and the basis decomposition.

Workload: the cfg3 graph (synth.primekg_full(): 129,375 nodes, ~8.1 M edges, 30 relations), 64 -> 256 -> 256, batch
1024 + 1024, the captured ``GraphedTrainStep`` timed as ``bench_cfg.py`` does (L2 overwritten before every step, CUDA
events); plus a cfg2 point (30,926 nodes, 849,456 edges, R = 3).  Per variant: ms / step (two passes over the variants,
the second in reverse order), trainable parameter count, peak memory, and — in a separate ``torch.profiler`` run —
the device time per step of ``block_diag_expand`` and ``block_diag_gather`` (under programmatic dependent launch a
kernel starts early and waits for its predecessor, so this includes overlapped waiting), and each kernel timed alone
over back-to-back launches at the cfg3 / cfg2 layer shapes.  The card's name and power limit are read in the same run.

Usage: python scripts/bench_blocks.py [--steps 10] [--out FILE]"""
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

VARIANTS = [  # (config, label, mode, num_bases, num_blocks)
    ("cfg3", "dense", "fp32", None, None),
    ("cfg3", "bases8", "fp32", 8, None),
    ("cfg3", "blocks4", "fp32", None, 4),
    ("cfg3", "blocks16", "fp32", None, 16),
    ("cfg3", "blocks64", "fp32", None, 64),
    ("cfg3", "dense", "bf16", None, None),
    ("cfg3", "blocks16", "bf16", None, 16),
    ("cfg2", "dense", "fp32", None, None),
    ("cfg2", "blocks16", "fp32", None, 16),
]


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def build(pkg, kg, ei, et, batch, mode, bases, blocks):
    torch.manual_seed(42)
    model = pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, 64, 256, dropout=0.5, decoder_dropout=0.1,
                                 num_bases=bases, num_blocks=blocks).to(DEV)
    for c in model.encoder._layers():
        c.mode = mode
    model.train()
    step = pkg.GraphedTrainStep(model, ei, et, batch_size=2048)
    step.load_batch(*batch)
    return model, step


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


def kernel_us(step, steps=5):
    """Per-step device time of the two block kernels, from a profiled run of graph replays (includes PDL waits)."""
    from torch.profiler import ProfilerActivity, profile
    step(); torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            step()
        torch.cuda.synchronize()
    out = {"block_diag_expand": [0.0, 0], "block_diag_gather": [0.0, 0]}
    for ev in prof.events():
        for k in out:
            if k in ev.name and ev.device_type == torch.autograd.DeviceType.CUDA:
                out[k][0] += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
                out[k][1] += 1
    return {k: {"us_per_step": round(v[0] / steps, 3), "launches_per_step": v[1] / steps} for k, v in out.items()}


def standalone_us(R, nb, d_in, d_out, launches=200):
    """Each kernel alone, back to back over many launches (CUDA events): per-launch time and bytes moved."""
    from primekg_rgcn_linkprediction_b200 import _lib
    from primekg_rgcn_linkprediction_b200.graph import _ptr, _stream
    lib = _lib.load()
    bi, bo = d_in // nb, d_out // nb
    blocks = torch.randn(R, nb, bi, bo, device=DEV)
    W = torch.empty(R, d_in, d_out, device=DEV)
    calls = {"block_diag_expand": lambda: lib.rgcn_block_diag_expand(_ptr(blocks), R, nb, bi, bo, _ptr(W), _stream(DEV)),
             "block_diag_gather": lambda: lib.rgcn_block_diag_gather(_ptr(W), R, nb, bi, bo, _ptr(blocks), _stream(DEV))}
    nbytes = {"block_diag_expand": (W.numel() + blocks.numel()) * 4, "block_diag_gather": 2 * blocks.numel() * 4}
    out = {}
    for name, fn in calls.items():
        for _ in range(20):
            _lib.check(fn(), name)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(launches):
            fn()
        b.record()
        torch.cuda.synchronize()
        us = a.elapsed_time(b) * 1e3 / launches
        out[name] = {"us_per_launch": round(us, 3), "bytes": nbytes[name], "GB_per_s": round(nbytes[name] / us * 1e-3, 1)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_bench_blocks.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_blocks.py measures on the GPU; there is none here")
    import primekg_rgcn_linkprediction_b200 as pkg
    from primekg_rgcn_linkprediction_b200 import synth
    graphs = {}
    for name, kg in (("cfg3", synth.primekg_full()), ("cfg2", synth.primekg_subgraph())):
        batch = [t.to(DEV) for t in synth.link_batch(kg, 1024)]
        graphs[name] = (kg, kg.edge_index.to(DEV), kg.edge_type.to(DEV), batch)
    flush = torch.empty(128 * 1024 * 1024, dtype=torch.float32, device=DEV)      # 512 MB > L2
    rec = {"card": gpu_info(), "steps_per_timing": args.steps,
           "workload": "cfg3: 129,375 nodes / ~8.1 M edges / 30 rel; cfg2: 30,926 nodes / 849,456 edges / 3 rel; "
                       "64->256->256, batch 1024+1024, dropout 0.5 / 0.1, GraphedTrainStep replay, L2 overwritten "
                       "before every step",
           "variants": []}
    rec["kernels_alone"] = {f"R{R}_nb{nb}_{d_in}x{d_out}": standalone_us(R, nb, d_in, d_out)
                            for R, nb, d_in, d_out in ((30, 4, 64, 256), (30, 4, 256, 256), (30, 16, 256, 256),
                                                       (30, 64, 256, 256), (3, 16, 256, 256))}
    print(json.dumps(rec["kernels_alone"]), flush=True)
    results = {}
    for pass_no, order in enumerate((VARIANTS, VARIANTS[::-1])):
        for v in order:
            cfg, label, mode, bases, blocks = v
            kg, ei, et, batch = graphs[cfg]
            gc.collect(); torch.cuda.empty_cache()
            torch.cuda.reset_peak_memory_stats(DEV)
            model, step = build(pkg, kg, ei, et, batch, mode, bases, blocks)
            ms = time_steps(step, flush, args.steps)
            r = results.setdefault(v, {"config": cfg, "variant": label, "mode": mode, "num_bases": bases,
                                       "num_blocks": blocks, "ms_per_step_passes": []})
            r["ms_per_step_passes"].append(round(ms, 4))
            if pass_no == 0:
                r["params"] = sum(p.numel() for p in model.parameters())
                r["conv_weight_params"] = sum(c.weight.numel() + (0 if c.comp is None else c.comp.numel())
                                              for c in model.encoder._layers())
                r["loss"] = float(step.loss)
                r["peak_mem_GB"] = round(torch.cuda.max_memory_allocated(DEV) / 1e9, 3)
                if blocks is not None:
                    r["kernels"] = kernel_us(step)
            del model, step
            print(json.dumps(r), flush=True)
    for v in VARIANTS:
        r = results[v]
        r["ms_per_step"] = round(statistics.mean(r["ms_per_step_passes"]), 4)
        rec["variants"].append(r)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec))


if __name__ == "__main__":
    main()

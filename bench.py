#!/usr/bin/env python
"""Benchmark of the RGCN message-passing hot path (BASELINE.json metric: full-batch RGCN fwd+bwd
edges/sec; aggregation GB/s against the measured roofs of the box; transforms against the tensor peak).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--mode fp32|bf16] [--quick]
                    [--dump-outputs DIR]

One *step* = train-mode ``DrugDiseaseModel.forward`` on the full graph + BCEWithLogits + ``backward()``
(reference src/train.py:291-306; optimiser, clipping and sampling excluded, SURVEY.md §8d).
Headline workload at every N: cfg2 of BASELINE.json — the synthetic PrimeKG-shaped graph (30,926 nodes /
849,456 directed edges / 3 relations), 2-layer RGCN 64 -> 256 -> 256, batch 1,024 positives + 1,024
negatives, dropout 0.5 / decoder dropout 0.1, seed 42.  cfg1-4 fit one GPU, so N > 1 runs data-parallel
replicas for ``value`` (weak scaling: N * E edges per step); the node-range PARTITIONED path of north_star
config 5 is measured next to it at every N under ``partitioned`` (a cfg5-shaped graph sized per GPU:
1.25 M nodes / 50 M edges / 30 relations / 3 layers per rank => 10 M / 400 M at N = 8).

Prints ONE JSON line (rank 0).  Contract and every figure's definition: DESIGN.md §5.
"""
from __future__ import annotations

import argparse
import json
import os
import socket
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CFG = dict(num_nodes=30_926, num_edges=849_456, num_relations=3, embedding_dim=64, hidden_dim=256,
           batch_pos=1024, dropout=0.5, decoder_dropout=0.1, seed=42)
WORKLOAD = ("cfg2: synthetic PrimeKG-shaped KG 30,926 nodes / 849,456 edges / 3 relations, "
            "2-layer RGCN 64->256->256, batch 1024+1024, fwd+loss+bwd")
METRIC = "rgcn_fwd_bwd_edges_per_sec"
UNIT = "edges/s"
PARITY = ("operator restated, not PyG-pinned (torch_geometric is not installable here): RGCNConv checked against the "
          "restated loop path + a dense-adjacency re-derivation + fp64 gradcheck; everything around it pinned to the "
          "unmodified reference model file (tests/golden)")
# SURVEY.md §8d: algorithmic bytes of one cfg2 step in the reference's (dense) formulation
CFG2_STEP_BYTES = 2_406.3e6
PART = dict(nodes_per_gpu=1_250_000, edges_per_gpu=50_000_000, relations=30, layers=3, embedding=64, hidden=128, batch=2048)
DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1650.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


def cpu_model() -> str:
    try:
        for line in open("/proc/cpuinfo"):
            if line.lower().startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.path = gpu_index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "20"], stdout=open(self.path, "w"),
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return None
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                "window": "sampled every 20 ms from a 0.4 s pre-roll of the same graph replays through the timed region"}


# ---------------------------------------------------------------------------------------------
# workload + timing helpers
# ---------------------------------------------------------------------------------------------
def make_workload(rank: int):
    from primekg_rgcn_linkprediction_b200 import synth
    kg = synth.primekg_subgraph(CFG["num_edges"], seed=CFG["seed"])
    batch = synth.link_batch(kg, CFG["batch_pos"], seed=CFG["seed"] + 1000 * rank)   # a different mini-batch per rank
    return kg, batch


def rewind_dropout_counters(model):
    """Set the device-side step counters of the fused dropout (the layers' and the decoder's) back to 0.  A step's masks
    hash (seed, counter, element) and the untimed pre-roll runs as many steps as fit its time window, so without this
    the masks of the timed steps, and every output of them, would change from run to run."""
    for m in model.modules():
        ctr = getattr(m, "_drop_ctr", None)
        if ctr is not None:
            ctr.zero_()
        rng = getattr(m, "_drop_rng", None)
        if rng is not None:
            rng[1].zero_()


def dump_outputs(out_dir, gstep, model):
    """What the last step handed its caller, as float32 ``out_dir/<name>.npy``: the loss, the scores of the batch's
    pairs and every parameter gradient (``grad.<parameter name>``)."""
    arrays = {"loss": gstep.loss, "scores": gstep.scores}
    arrays.update((f"grad.{k}", p.grad) for k, p in model.named_parameters() if p.grad is not None)
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def algorithmic_bytes(E, N, R, d_in):
    """SURVEY.md §8d per-layer figures for the aggregation kernels (bytes per launch)."""
    fwd = E * (d_in * 4 + 4) + (N * R + 1) * 4
    bwd = E * (d_in * 4 + 8) + (N * R + 1) * 4
    return fwd, bwd


class Flusher:
    def __init__(self, dev):
        self.buf = torch.empty(512 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)

    def __call__(self):
        self.buf.fill_(1.0)            # 512 MiB write > 126 MB L2


def event_time(fn, iters, flush=None, warm=3):
    """Mean CUDA-event duration (ms) of ``fn`` on the launching stream; ``flush`` runs before every timed call."""
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(iters):
        if flush is not None:
            flush()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.mean(ts)


def time_aggregation(graph, d, iters, flush, comp=None):
    from primekg_rgcn_linkprediction_b200 import ops
    x = torch.randn(graph.n_src, d, device="cuda")
    gA = torch.randn(graph.n_dst, (graph.R + 1) * d, device="cuda")
    return {"aggregate_fwd": event_time(lambda: ops.aggregate_fwd(graph, x, comp=comp), iters, flush),
            "aggregate_bwd": event_time(lambda: ops.aggregate_bwd(graph, gA, d, init=gA[:, graph.R * d:]), iters, flush)}


def ncu_record(name):
    """Per-launch DRAM / L2 bytes of the dominant kernel from the committed ncu capture of this round (profiles/)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        return json.load(open(p)).get(name)
    return None


# ---------------------------------------------------------------------------------------------
# roofline block
# ---------------------------------------------------------------------------------------------
def roofline_block(pkg, kg, ei, et, flush, clocks, iters):
    """Three measured rates for the dominant kernel (layer-2 forward aggregation, gather width 256):
    gathered (algorithmic) GB/s, the L2 gather ceiling MEASURED on this box by rgcn_probe_gather over the same index
    array, and the DRAM rate from the committed ncu capture; ``frac`` = achieved / the roof that binds (the L2 for cfg2,
    whose 31.7 MB of features are L2 resident).  Plus a genuinely DRAM-bound gather, the tensor-pipe fraction of the
    layer-2 forward GEMM and the whole-step HBM fraction on the dense-backward line."""
    from primekg_rgcn_linkprediction_b200 import ops, synth
    peaks, peak_src = measured_peaks()
    hbm = float(peaks["hbm_gbs"])
    graph = pkg.get_graph(ei, et, kg.num_nodes, kg.num_relations)
    d2 = CFG["hidden_dim"]
    kt = time_aggregation(graph, d2, iters, flush)
    fwd_b, bwd_b = algorithmic_bytes(kg.num_edges, kg.num_nodes, kg.num_relations, d2)
    achieved = fwd_b / (kt["aggregate_fwd"] * 1e-3) / 1e9

    # ---- L2 gather ceiling, measured here: same table size, same source-index array, nothing but the loads ----
    table = torch.randn(kg.num_nodes, d2, device="cuda")
    col = graph.col
    gathered = col.numel() * d2 * 4
    probe = {}
    for bps in (2, 4, 8):
        ms = event_time(lambda: ops.probe_gather(table, col, blocks_per_sm=bps), iters, flush)
        probe[f"csr_order_{bps}_blocks_per_sm"] = round(gathered / (ms * 1e-3) / 1e9, 1)
    uni = torch.randint(0, kg.num_nodes, (col.numel(),), device="cuda", dtype=torch.int32)
    ms = event_time(lambda: ops.probe_gather(table, uni, blocks_per_sm=8), iters, flush)
    probe["uniform_random_rows_8_blocks_per_sm"] = round(gathered / (ms * 1e-3) / 1e9, 1)
    ms = event_time(lambda: ops.probe_gather(table, None, n_idx=col.numel(), blocks_per_sm=8), iters, flush)
    probe["streaming_read_8_blocks_per_sm"] = round(gathered / (ms * 1e-3) / 1e9, 1)
    l2_peak = max(probe.values())
    ncu = ncu_record("aggregate_rows_fwd_d256") or {}
    dram_bytes = ncu.get("dram_bytes")
    dram_gbs = None if not dram_bytes else dram_bytes / (kt["aggregate_fwd"] * 1e-3) / 1e9
    roof = {"bound": "hbm", "binding_roof": "l2 (the gather working set is L2 resident: 31.7 MB of features < 126 MB)",
            "kernel": "hub_partial_kernel + aggregate_rows_kernel (layer-2 forward gather, d=256)",
            "achieved": round(achieved, 1), "peak": round(l2_peak, 1), "unit": "GB/s", "frac": round(achieved / l2_peak, 4),
            "peak_source": "L2-resident row gather MEASURED in this run (rgcn_probe_gather: the aggregation's access pattern "
                           "alone; best of the variants in l2_probe)",
            "traffic": dram_bytes, "traffic_source": ncu.get("source"),
            "algorithmic_bytes_per_launch": fwd_b, "avg_launch_ms": round(kt["aggregate_fwd"], 5),
            "output_bytes_per_launch": kg.num_nodes * (kg.num_relations + 0) * d2 * 4,
            "frac_incl_output_write": round((fwd_b + kg.num_nodes * kg.num_relations * d2 * 4) / (kt["aggregate_fwd"] * 1e-3) / 1e9 / l2_peak, 4),
            "rates": {"gathered_algorithmic_gbs": round(achieved, 1), "l2_probe_peak_gbs": round(l2_peak, 1),
                      "lts_t_bytes_gbs_ncu": (None if not ncu.get("lts_t_bytes") else
                                              round(ncu["lts_t_bytes"] / (ncu["ncu_time_us"] * 1e-6) / 1e9, 1)),
                      "dram_gbs": None if dram_gbs is None else round(dram_gbs, 1),
                      "hbm_peak_gbs": hbm, "hbm_peak_source": peak_src,
                      "frac_of_hbm_peak_dram_level": None if dram_gbs is None else round(dram_gbs / hbm, 4),
                      "frac_of_hbm_peak_algorithmic": round(achieved / hbm, 4),
                      "note": "algorithmic / HBM peak exceeds 1 because every source row is gathered ~27x out of the L2; "
                              "the DRAM-level fraction is what the HBM sees"},
            "l2_probe": probe,
            "bwd": {"achieved": round(bwd_b / (kt["aggregate_bwd"] * 1e-3) / 1e9, 1),
                    "avg_launch_ms": round(kt["aggregate_bwd"], 5), "algorithmic_bytes_per_launch": bwd_b,
                    "frac": round(bwd_b / (kt["aggregate_bwd"] * 1e-3) / 1e9 / l2_peak, 4)}}
    del table, uni

    # ---- layer-1 gather (d = 64): the narrow-row walk against its own measured ceiling ----
    try:
        d1 = CFG["embedding_dim"]
        k1 = time_aggregation(graph, d1, iters, flush)
        f1, b1 = algorithmic_bytes(kg.num_edges, kg.num_nodes, kg.num_relations, d1)
        t1 = torch.randn(kg.num_nodes, d1, device="cuda")
        p1 = max(col.numel() * d1 * 4 / (event_time(lambda: ops.probe_gather(t1, col, blocks_per_sm=b), iters, flush) * 1e-3) / 1e9
                 for b in (4, 8))
        roof["d64"] = {"fwd_achieved": round(f1 / (k1["aggregate_fwd"] * 1e-3) / 1e9, 1),
                       "bwd_achieved": round(b1 / (k1["aggregate_bwd"] * 1e-3) / 1e9, 1),
                       "l2_probe_peak": round(p1, 1), "fwd_frac": round(f1 / (k1["aggregate_fwd"] * 1e-3) / 1e9 / p1, 4),
                       "bwd_frac": round(b1 / (k1["aggregate_bwd"] * 1e-3) / 1e9 / p1, 4),
                       "unit": "GB/s", "fwd_ms": round(k1["aggregate_fwd"], 5), "bwd_ms": round(k1["aggregate_bwd"], 5),
                       "fwd_algorithmic_bytes_per_launch": f1, "bwd_algorithmic_bytes_per_launch": b1,
                       "kernel": "hub_partial_kernel + aggregate_rows_kernel<16, 1, ...> (layer-1 gathers, 256-byte rows)",
                       "note": "since the last layer runs on the listed rows only, these two dense walks are the largest "
                               "kernels of the default step (timeline: forward 11 + 29 us, backward 10 + 50 us with the "
                               "weight gradient running beside it); the d = 256 walk above is the dominant kernel of the "
                               "all-rows formulation (dense_last_layer) and the reference point carried over from round 1"}
        del t1
    except Exception as ex:  # pragma: no cover
        roof["d64"] = {"error": repr(ex)[:200]}

    # ---- a genuinely DRAM-bound gather: cfg5-shard shape, uniform sources, 2 GB of features, d = 128 ----
    try:
        n_big, e_big, r_big, d_big = 4_000_000, 64_000_000, 30, 128
        big = synth.scaled_kg(n_big, e_big, r_big, seed=7, power=1.0, device="cuda")
        gb = pkg.RelGraph.from_edges(big.edge_index, big.edge_type, n_big, r_big)
        del big
        xb = torch.randn(n_big, d_big, device="cuda")
        ms_f = event_time(lambda: ops.aggregate_fwd(gb, xb, out_bf16=True), 3, None, warm=1)
        fb, _ = algorithmic_bytes(e_big, n_big, r_big, d_big)
        out_b = n_big * r_big * d_big * 2
        ms_p = event_time(lambda: ops.probe_gather(xb, gb.col, blocks_per_sm=8), 3, None, warm=1)
        a_f = fb / (ms_f * 1e-3) / 1e9
        ncu_b = ncu_record("aggregate_rows_fwd_hbm_case") or {}
        roof["hbm_bound_case"] = {
            "workload": "cfg5-shard-shaped gather: 4,000,000 nodes / 64,000,000 edges / 30 relations, uniform sources, "
                        "d = 128 (2.05 GB of fp32 features, 16x the L2), output as bf16 rows",
            "bound": "hbm", "achieved": round(a_f, 1), "peak": hbm, "unit": "GB/s", "frac": round(a_f / hbm, 4),
            "achieved_incl_output_write": round((fb + out_b) / (ms_f * 1e-3) / 1e9, 1),
            "frac_incl_output_write": round((fb + out_b) / (ms_f * 1e-3) / 1e9 / hbm, 4),
            "algorithmic_bytes_per_launch": fb, "output_bytes_per_launch": out_b, "avg_launch_ms": round(ms_f, 4),
            "probe_gather_same_indices_gbs": round(e_big * d_big * 4 / (ms_p * 1e-3) / 1e9, 1),
            "traffic": ncu_b.get("dram_bytes"), "traffic_source": ncu_b.get("source")}
        del gb, xb
        torch.cuda.empty_cache()
    except Exception as ex:  # pragma: no cover
        roof["hbm_bound_case"] = {"error": repr(ex)[:200]}

    # ---- tensor roofline: the layer-2 forward transform alone (M = N nodes, K = (R+1) d, N = d_out) ----
    try:
        K = (kg.num_relations + 1) * d2
        A = torch.randn(kg.num_nodes, K, device="cuda")
        W = torch.randn(K, d2, device="cuda") * 0.05
        bias = torch.zeros(d2, device="cuda")
        tens = {}
        for mode, prods in (("fp32", 3), ("bf16", 1)):
            planes = ops.alloc_planes(kg.num_nodes, K, mode, A.device)
            ops.split_planes(A, planes)
            wp = ops.prepare_weights(W, None, mode)
            o = torch.empty(kg.num_nodes, d2, device="cuda")
            ms = event_time(lambda: ops.transform_fwd_w(planes, K, wp, d2, bias, True, mode, out=o), iters, flush)
            alg = 2.0 * kg.num_nodes * K * d2
            tens[mode] = {"avg_launch_ms": round(ms, 5), "algorithmic_tflops": round(alg / (ms * 1e-3) / 1e12, 1),
                          "executed_bf16_tflops": round(prods * alg / (ms * 1e-3) / 1e12, 1), "mma_products": prods,
                          "note": "the tcgen05 kernel alone (weights already converted, rgcn_transform_fwd_w), L2 flushed"}
        mode = "fp32"
        roof["tensor"] = {"bound": "tensor", "kernel": "gemm_kmajor_kernel<SPLIT> (layer-2 forward transform, 30,926 x 1,024 x 256)",
                          "achieved": tens[mode]["executed_bf16_tflops"], "peak": float(peaks["bf16_tflops"]),
                          "peak_sustained": float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])),
                          "unit": "TFLOP/s", "frac": round(tens[mode]["executed_bf16_tflops"] / float(peaks["bf16_tflops"]), 4),
                          "peak_source": peak_src + " (burst figure: the kernel is timed alone)",
                          "tensor_pipe_active_pct_ncu": (ncu_record("gemm_fwd_layer2") or {}).get("tensor_pipe_active_pct"),
                          "modes": tens}
        del A, W, planes
    except Exception as ex:  # pragma: no cover
        roof["tensor"] = {"error": repr(ex)[:200]}
    return roof


# ---------------------------------------------------------------------------------------------
# the other configs of BASELINE.json as one-liners (N = 1 only)
# ---------------------------------------------------------------------------------------------
def graphed_step_ms(pkg, kg, hidden, bases, mode, dev, flush, steps=10, batch_pos=1024):
    from primekg_rgcn_linkprediction_b200 import synth
    heads, tails, rels, labels = synth.link_batch(kg, batch_pos)
    torch.manual_seed(CFG["seed"])
    model = pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, 64, hidden, dropout=0.5, decoder_dropout=0.1,
                                 num_bases=bases).to(dev)
    for c in (model.encoder.conv1, model.encoder.conv2):
        c.mode = mode
    model.train()
    ei, et = kg.edge_index.to(dev), kg.edge_type.to(dev)
    step = pkg.GraphedTrainStep(model, ei, et, batch_size=2 * batch_pos)
    step.load_batch(heads.to(dev), tails.to(dev), rels.to(dev), labels.to(dev))
    ms = event_time(step, steps, flush)
    loss = float(step.loss)
    del step, model
    return ms, loss


def other_configs(pkg, dev, flush, mode):
    from primekg_rgcn_linkprediction_b200 import synth
    out = {}
    try:
        kg = synth.primekg_subgraph(CFG["num_edges"], seed=CFG["seed"])
        ms, loss = graphed_step_ms(pkg, kg, 128, None, mode, dev, flush)
        out["cfg1"] = {"workload": "30,926 nodes / 849,456 edges / 3 rel, 64->128->128 (src/train.py defaults), batch 1024+1024",
                       "ms_per_step": round(ms, 4), "edges_per_s": kg.num_edges / (ms * 1e-3), "loss": loss}
    except Exception as ex:  # pragma: no cover
        out["cfg1"] = {"error": repr(ex)[:200]}
    try:
        kg = synth.primekg_full()
        ms, loss = graphed_step_ms(pkg, kg, 256, 8, mode, dev, flush, steps=5)
        out["cfg3"] = {"workload": "129,375 nodes / 8,100,498 edges / 30 rel, num_bases = 8, 64->256->256, batch 1024+1024",
                       "ms_per_step": round(ms, 4), "edges_per_s": kg.num_edges / (ms * 1e-3), "loss": loss,
                       "hbm_floor_ms_survey_8d": 3.35}
        del kg
        torch.cuda.empty_cache()
    except Exception as ex:  # pragma: no cover
        out["cfg3"] = {"error": repr(ex)[:200]}
    try:
        d = CFG["hidden_dim"]
        torch.manual_seed(3)
        emb = torch.randn(30926, d, device=dev)
        drugs = torch.arange(5593, 11875, device=dev)
        diseases = torch.arange(0, 5593, device=dev)
        rel = torch.randn(d, device=dev)
        table = torch.randn(3, d, device=dev)
        nq = 15372
        heads = torch.randint(0, 30926, (nq,), device=dev)
        tails = torch.randint(0, 30926, (nq,), device=dev)
        rels = torch.zeros(nq, dtype=torch.int64, device=dev)
        pairs = drugs.numel() * diseases.numel()
        c4 = {"workload": "all 6,282 x 5,593 drug-disease pairs, d = 256; ranking of 15,372 test edges against 30,926 entities"}
        ms = event_time(lambda: pkg.score_all_pairs(emb, drugs, diseases, rel_vec=rel), 5, flush)
        c4["distmult_all_pairs"] = {"ms": round(ms, 4), "pairs_per_s": pairs / (ms * 1e-3)}
        ms = event_time(lambda: pkg.score_all_pairs(emb, drugs, diseases, cosine=True), 5, flush)
        c4["cosine_all_pairs"] = {"ms": round(ms, 4), "pairs_per_s": pairs / (ms * 1e-3)}
        if hasattr(pkg, "topk_all_pairs"):
            ms = event_time(lambda: pkg.topk_all_pairs(emb, drugs, diseases, k=10, cosine=True), 5, flush)
            c4["cosine_top10_fused"] = {"ms": round(ms, 4), "pairs_per_s": pairs / (ms * 1e-3)}
        ms = event_time(lambda: pkg.rank_true_tails(emb, table, heads, rels, tails), 3, flush, warm=1)
        c4["rank_15372_vs_30926"] = {"ms": round(ms, 4), "pairs_per_s": nq * 30926 / (ms * 1e-3)}
        out["cfg4"] = c4
    except Exception as ex:  # pragma: no cover
        out["cfg4"] = {"error": repr(ex)[:200]}
    return out


def library_gpu_baseline(kg, batch, dev, steps=5):
    """The "library Blackwell path" (BASELINE.md §3, SURVEY.md §8d): the restated reference (oracle/rgcn_ref.py — what
    PyG's loop path does) on the SAME B200 through stock torch CUDA ops (ATen index_select / index_add_ + cuBLAS)."""
    from oracle import rgcn_ref
    heads, tails, rels, labels = [t.to(dev) for t in batch]
    torch.manual_seed(CFG["seed"])
    model = rgcn_ref.ModelRef(kg.num_nodes, kg.num_relations, CFG["embedding_dim"], CFG["hidden_dim"], CFG["dropout"],
                              CFG["decoder_dropout"]).to(dev)
    model.train()
    ei, et = kg.edge_index.to(dev), kg.edge_type.to(dev)

    def step():
        model.zero_grad(set_to_none=True)
        rgcn_ref.train_step_ref(model, ei, et, heads, tails, rels, labels)

    ms = event_time(step, steps, None, warm=3)
    return {"value": kg.num_edges / (ms * 1e-3), "unit": UNIT, "ms_per_step": round(ms, 4), "device": "same B200",
            "kind": "oracle port through stock torch CUDA ops (ATen gather / index_add_ atomics + cuBLAS fp32), eager, "
                    "torch.backends.cuda.matmul.allow_tf32 = %s" % torch.backends.cuda.matmul.allow_tf32}


# ---------------------------------------------------------------------------------------------
# node-range partitioned path (north_star config 5), measured at every N
# ---------------------------------------------------------------------------------------------
def partitioned_record(rank, world, dev, steps=5, warmup=4):
    """Destination-range partition of a cfg5-shaped graph sized per GPU (weak scaling).  Both exchange forms are timed:
    our kernels over peer-mapped memory (dist_fused.py, the product path) and NCCL all-gather / reduce-scatter (dist.py).
    Timing: CUDA events per step, barrier + synchronize on both sides, max over ranks."""
    import torch.distributed as dist
    import primekg_rgcn_linkprediction_b200 as pkg
    from primekg_rgcn_linkprediction_b200 import dist as D
    from primekg_rgcn_linkprediction_b200 import dist_fused as DF
    from primekg_rgcn_linkprediction_b200 import synth
    nodes, edges = PART["nodes_per_gpu"] * world, PART["edges_per_gpu"] * world
    R, L, d_e, d_h, B = PART["relations"], PART["layers"], PART["embedding"], PART["hidden"], PART["batch"]
    rec = {"workload": f"cfg5-shaped synthetic KG sized per GPU: {nodes:,} nodes / {edges:,} edges / {R} relations, "
                       f"{L}-layer RGCN {d_e}->{d_h} x {L}, batch {B}, fwd+loss+bwd, fp32 mode",
           "scaling": "weak", "n_gpus": world, "nodes": nodes, "edges": edges}

    def build(exchange, plan, graph):
        cls = DF.FusedPartitionedModel if exchange == "fused" else D.PartitionedModel
        m = cls(plan, rank, R, d_e, d_h, dropout=0.0, decoder_dropout=0.0, num_layers=L, seed=42).to(dev)
        m.encoder.set_graph(graph)
        m.train()
        return m

    def make_step(model, n_nodes):
        g = torch.Generator(device=dev).manual_seed(7)
        heads = torch.randint(0, n_nodes, (B,), generator=g, device=dev)
        tails = torch.randint(0, n_nodes, (B,), generator=g, device=dev)
        rels = torch.randint(0, R, (B,), generator=g, device=dev)
        labels = (torch.rand(B, generator=g, device=dev) < 0.5).float()
        sl = slice(rank * B // world, (rank + 1) * B // world)

        def step():
            for p in model.parameters():
                p.grad = None
            s = model(heads[sl], tails[sl], rels[sl])
            loss = F.binary_cross_entropy_with_logits(s, labels[sl], reduction="sum") / B
            loss.backward()
            model.allreduce_decoder_grads()
            return loss.detach(), s.detach()
        return step, (heads, tails, rels, labels, sl)

    def timed(step):
        for _ in range(warmup):
            step()
        torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
        evs = []
        for _ in range(steps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); step(); b.record()
            evs.append((a, b))
        torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
        t = torch.tensor([sum(a.elapsed_time(b) for a, b in evs) / steps], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    # ---- equals-single-GPU check at a small size (N > 1: the split must reproduce the one-GPU model) ----
    if world > 1:
        try:
            n_s, e_s = 200_000, 4_000_000
            kg = synth.scaled_kg(n_s, e_s, R, seed=42, device=dev)
            plan = D.plan_partition(kg.edge_index[1], n_s, world)
            src, dst, rel = D.local_edges(kg.edge_index, kg.edge_type, plan, rank)
            graph = pkg.RelGraph(src, dst, rel, plan.max_n, world * plan.max_n, R)
            model = build("fused", plan, graph)
            step, (heads, tails, rels, labels, sl) = make_step(model, n_s)
            loss, scores = step()
            total = loss.clone()
            dist.all_reduce(total)
            shards = [torch.zeros_like(model.encoder.node_embeddings.data) for _ in range(world)]
            dist.all_gather(shards, model.encoder.node_embeddings.data)
            gsh = [torch.zeros_like(model.encoder.node_embeddings.grad) for _ in range(world)]
            dist.all_gather(gsh, model.encoder.node_embeddings.grad)
            if rank == 0:
                ref = pkg.DrugDiseaseModel(n_s, R, d_e, d_h, dropout=0.0, decoder_dropout=0.0, num_layers=L).to(dev)
                with torch.no_grad():
                    ref.encoder.node_embeddings.weight.copy_(torch.cat([shards[p][: plan.size(p)] for p in range(world)]))
                    for mine, theirs in zip(model.encoder.convs, ref.encoder._layers()):
                        theirs.weight.copy_(mine.weight); theirs.root.copy_(mine.root); theirs.bias.copy_(mine.bias)
                    ref.decoder.relation_embeddings.weight.copy_(model.decoder.relation_embeddings.weight)
                ref.train()
                rs = ref(kg.edge_index, kg.edge_type, heads, tails, rels)
                rl = F.binary_cross_entropy_with_logits(rs, labels)
                rl.backward()
                gg = torch.cat([gsh[p][: plan.size(p)] for p in range(world)])
                want = ref.encoder.node_embeddings.weight.grad
                rec["equals_single_gpu"] = {
                    "graph": f"{n_s:,} nodes / {e_s:,} edges / {R} relations / {L} layers",
                    "loss_abs_err": abs(float(rl) - float(total)), "score_max_abs_err": float((rs[sl] - scores).abs().max()),
                    "emb_grad_rel_fro": float((gg - want).norm() / (want.norm() + 1e-30)),
                    "w_grad_rel_fro_max": max(float((m.weight.grad - t.weight.grad).norm() / (t.weight.grad.norm() + 1e-30))
                                              for m, t in zip(model.encoder.convs, ref.encoder._layers()))}
                e = rec["equals_single_gpu"]
                e["ok"] = bool(e["loss_abs_err"] < 1e-5 and e["score_max_abs_err"] < 1e-4 and e["emb_grad_rel_fro"] < 1e-3
                               and e["w_grad_rel_fro_max"] < 1e-3)
                del ref
            del model, graph, kg, step
            torch.cuda.empty_cache()
            dist.barrier()
        except Exception as ex:  # pragma: no cover
            rec["equals_single_gpu"] = {"error": repr(ex)[:300]}

    # ---- the timed graph: every rank generates the same edge list on its device, keeps its destination range ----
    kg = synth.scaled_kg(nodes, edges, R, seed=42, device=dev)
    plan = D.plan_partition(kg.edge_index[1], nodes, world)
    src, dst, rel = D.local_edges(kg.edge_index, kg.edge_type, plan, rank)
    del kg
    torch.cuda.empty_cache()
    graph = pkg.RelGraph(src, dst, rel, plan.max_n, world * plan.max_n, R)
    local_edges = int(rel.numel())
    del src, dst, rel
    rec["max_shard_rows"] = plan.max_n
    rec["local_edges_rank0"] = local_edges
    dims = [d_e] + [d_h] * L
    # forward: every rank receives the other ranks' rows of each layer's input and of the output; backward: the transpose
    # (peer-memory form: of the OUTPUT only the 2 * batch rows some decoder reads travel, and of the last layer's gradient
    # only those rows are pulled; the NCCL form exchanges full matrices)
    fwd_in = (world - 1) * plan.max_n * 4 * sum(dims[:-1]) + (world - 1) * 2 * B * 4 * dims[-1]
    rec["exchange_bytes_per_gpu_per_step"] = {"forward_received": fwd_in, "backward_pulled": fwd_in,
                                              "nccl_form_each_direction": (world - 1) * plan.max_n * 4 * sum(dims),
                                              "weight_grad_allreduce": 4 * sum((R + 1) * dims[i] * dims[i + 1] + dims[i + 1] for i in range(L))}
    for exchange in ("fused", "nccl"):
        try:
            model = build(exchange, plan, graph)
            step, _ = make_step(model, nodes)
            ms = timed(step)
            rec["ms_per_step" if exchange == "fused" else "nccl_exchange_ms_per_step"] = ms
            if exchange == "fused":
                rec["value"] = edges / (ms * 1e-3)
                rec["unit"] = UNIT
                rec["exchange"] = "our kernels over peer-mapped memory (all-gather = the transform's epilogue stores, " \
                                  "reduce-scatter = rank-ordered pull fused with mask + operand conversion); the last " \
                                  "layer runs on the rows the decoders read only (listed-rows forward + row-sparse backward)"
            del model, step
            torch.cuda.empty_cache()
        except Exception as ex:  # pragma: no cover
            rec[exchange + "_error"] = repr(ex)[:300]
    if "ms_per_step" in rec and "nccl_exchange_ms_per_step" in rec:
        rec["fused_vs_nccl_speedup"] = rec["nccl_exchange_ms_per_step"] / rec["ms_per_step"]
        rec["nccl_form_note"] = ("dist.py: NCCL all-gather / reduce-scatter of full matrices, last layer over all rows "
                                 "forward (row-sparse backward as well): the ratio covers the exchange form AND the "
                                 "listed-rows last layer of the peer-memory path")
    rec["max_mem_GB"] = torch.cuda.max_memory_allocated() / 1e9
    rec["ceiling_survey_8d_edges_per_s"] = 2.4e9 * world
    return rec


# ---------------------------------------------------------------------------------------------
# the headline step
# ---------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import primekg_rgcn_linkprediction_b200 as pkg
    from primekg_rgcn_linkprediction_b200 import _lib
    import torch.distributed as dist

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    kg, (heads, tails, rels, labels) = make_workload(rank)
    torch.manual_seed(CFG["seed"])
    model = pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, CFG["embedding_dim"], CFG["hidden_dim"],
                                 dropout=CFG["dropout"], decoder_dropout=CFG["decoder_dropout"]).to(dev)
    for c in (model.encoder.conv1, model.encoder.conv2):
        c.mode = args.mode
    model.train()
    ei, et = kg.edge_index.to(dev), kg.edge_type.to(dev)
    params = [p for p in model.parameters()]
    flush = Flusher(dev)
    d_batch = [t.to(dev) for t in (heads, tails, rels, labels)]
    dump_bytes = 4 * (1 + d_batch[0].numel() + sum(p.numel() for p in params))     # loss, scores, gradients
    if args.dump_outputs and dump_bytes > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {dump_bytes} bytes of outputs exceed the {DUMP_LIMIT_BYTES} byte limit")

    def eager_step(b):
        for p in params:
            p.grad = None
        scores = model(ei, et, b[0], b[1], b[2])
        loss = F.binary_cross_entropy_with_logits(scores, b[3])
        loss.backward()
        return loss

    def allreduce_grads():
        if world > 1:
            flat = torch.cat([p.grad.reshape(-1) for p in params])
            dist.all_reduce(flat)
            flat /= world

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        eager_step(d_batch)
        allreduce_grads()
    barrier()
    # our kernels per step, counted on ONE truly eager step (the captured forms replay without passing the library's host
    # entry points, and the step in which the module captures its graphs would count the capture's warm-up passes too)
    ag_env = os.environ.get("PRIMEKG_RGCN_AUTOGRAPH")
    os.environ["PRIMEKG_RGCN_AUTOGRAPH"] = "0"
    try:
        l0 = lib.rgcn_launch_count()
        eager_step(d_batch)
        torch.cuda.synchronize()
        launches_per_step = int(lib.rgcn_launch_count() - l0)
    finally:
        if ag_env is None:
            del os.environ["PRIMEKG_RGCN_AUTOGRAPH"]
        else:
            os.environ["PRIMEKG_RGCN_AUTOGRAPH"] = ag_env
    for _ in range(6):                                 # (the module re-captures its graphs after the eager detour: not timed)
        eager_step(d_batch)
    barrier()

    def timed(run_one, steps):
        """K steps, each bracketed by CUDA events on the launching stream, L2 flushed between steps."""
        evs = []
        for _ in range(steps):
            flush()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); run_one(); b.record()
            evs.append((a, b))
        barrier()
        ms = sum(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps

    # ---- eager module API (what an unmodified src/train.py drives): device-resident, then from pinned host ----
    barrier()
    eager_ms = timed(lambda: (eager_step(d_batch), allreduce_grads()), args.steps)
    pinned = [t.pin_memory() for t in (heads, tails, rels, labels)]
    loss_host = torch.empty(1, dtype=torch.float32).pin_memory()

    def e2e_eager():
        b = [t.to(dev, non_blocking=True) for t in pinned]
        loss_host.copy_(eager_step(b).detach().reshape(1), non_blocking=True)
        allreduce_grads()

    for _ in range(2):
        e2e_eager()
    barrier()
    e2e_eager_value = world * kg.num_edges / (timed(e2e_eager, args.steps) * 1e-3)
    for p in params:
        p.grad = None

    # ---- the same step captured once into a CUDA graph (GraphedTrainStep) ----
    # N > 1: the backward kernels write every parameter gradient into ONE flat buffer (ops.GradArena), so the replicas
    # exchange a single tensor
    # and they exchange it with OUR two-shot all-reduce over peer-mapped memory, captured as the last kernels of the step's
    # CUDA graph (peer.PeerAllReduce); RGCN_DP_ALLREDUCE=nccl keeps the round-1 form (one NCCL all-reduce after the replay)
    peer_ar = world > 1 and os.environ.get("RGCN_DP_ALLREDUCE", "peer") == "peer"
    dp_exchange = "none"
    if world > 1:
        ok = torch.ones(1, device=dev)
        if peer_ar:
            try:
                from primekg_rgcn_linkprediction_b200.peer import PeerBuffer
                PeerBuffer(4096, dev)
            except Exception:
                ok.zero_()
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            peer_ar = bool(ok.item() > 0)
        dp_exchange = ("two-shot all-reduce by our kernels over peer-mapped memory, inside the captured graph" if peer_ar else
                       "one NCCL all-reduce of the flat gradient buffer after the graph replay")

    def make_step(**kw):
        return pkg.GraphedTrainStep(model, ei, et, batch_size=d_batch[0].numel(), flat_grads="arena" if world > 1 else False,
                                    allreduce="peer" if peer_ar else None, **kw)

    gstep = make_step()
    gstep.load_batch(*d_batch)
    flat_holder = [gstep.flat_grad]

    def allreduce_graphed():
        if world > 1 and not peer_ar:
            if flat_holder[0] is not None:
                dist.all_reduce(flat_holder[0], op=dist.ReduceOp.AVG)   # NCCL averages in the reduction: no scaling pass
                return
            grads = [p.grad for p in params]
            with dist._coalescing_manager(device=dev):
                for g in grads:
                    dist.all_reduce(g, op=dist.ReduceOp.AVG)

    allreduce_grads = allreduce_graphed     # noqa: F811
    for _ in range(max(args.warmup, 3)):
        gstep(); allreduce_grads()
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    t_pre = time.perf_counter()
    while time.perf_counter() - t_pre < 0.4:            # pre-roll: the sampler sees the same kernel mix under load
        for _ in range(20):
            gstep(); allreduce_grads()
        torch.cuda.synchronize()
    rewind_dropout_counters(model)
    barrier()
    t_wall0 = time.perf_counter()
    ms_per_step = timed(lambda: (gstep(), allreduce_grads()), args.steps)
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, gstep, model)
    value = world * kg.num_edges / (ms_per_step * 1e-3)
    dp_exchange_ok = None
    if peer_ar:
        try:
            gstep.peer_ar.check()                       # a wait that gave up (a peer never arrived) would void the number
            dp_exchange_ok = True
        except Exception as ex:  # pragma: no cover
            dp_exchange_ok = repr(ex)[:200]

    # ---- end to end: batch in pinned host memory, H2D of the step's inputs and D2H of the loss inside ----
    packed = pkg.GraphedTrainStep.pack_batch(heads, tails, rels, labels)
    h2d_packed = packed.numel() * packed.element_size()
    for p in params:
        p.grad = None
    ghost = make_step(host_io=True)
    ghost.host_batch.copy_(packed)
    flat_value = flat_holder[0]
    flat_holder[0] = ghost.flat_grad

    def e2e_graphed():
        ghost.replay_host()
        allreduce_grads()

    for _ in range(2):
        e2e_graphed()
    barrier()
    e2e_value = world * kg.num_edges / (timed(e2e_graphed, args.steps) * 1e-3)
    e2e_loss = float(ghost.host_loss)                 # read after the timed region's synchronisation
    flat_holder[0] = flat_value
    del ghost

    # ---- the same graphed step with the row-sparse hand-over off: the last layer's backward over all N rows, i.e.
    #      the dense formulation SURVEY.md §8d's byte counts describe (same gradients, see tests) ----
    sparse_env = os.environ.get("PRIMEKG_RGCN_SPARSE_BWD")
    dense_ms = None
    if sparse_env != "0":
        os.environ["PRIMEKG_RGCN_SPARSE_BWD"] = "0"
        try:
            del gstep
            for p in params:
                p.grad = None
            gdense = make_step()
            gdense.load_batch(*d_batch)
            flat_holder[0] = gdense.flat_grad
            for _ in range(3):
                gdense(); allreduce_grads()
            barrier()
            dense_ms = timed(lambda: (gdense(), allreduce_grads()), args.steps)
            del gdense
        finally:
            if sparse_env is None:
                del os.environ["PRIMEKG_RGCN_SPARSE_BWD"]
            else:
                os.environ["PRIMEKG_RGCN_SPARSE_BWD"] = sparse_env
    flat_holder[0] = None
    for p in params:
        p.grad = None

    # ---- the partitioned path (north_star config 5), every N, every rank ----
    part = None
    if not args.no_partitioned:
        try:
            if world == 1 and not dist.is_initialized():
                s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
                os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
                os.environ["MASTER_PORT"] = str(port)
                dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev)
            torch.cuda.empty_cache()
            part = partitioned_record(rank, world, dev, steps=3 if args.quick else 5)
        except Exception as ex:  # pragma: no cover
            part = {"error": repr(ex)[:300]}
        torch.cuda.empty_cache()

    if rank != 0:
        return None
    peaks, peak_src = measured_peaks()
    hbm = float(peaks["hbm_gbs"])
    roofline = roofline_block(pkg, kg, ei, et, flush, clocks, max(5, min(args.steps, 20)))
    step_dense = dense_ms if dense_ms is not None else ms_per_step
    roofline["whole_step"] = {
        "algorithmic_bytes_survey_8d": CFG2_STEP_BYTES,
        "dense_last_layer_ms": dense_ms, "frac_of_hbm_peak_dense_last_layer": round(CFG2_STEP_BYTES / (step_dense * 1e-3) / 1e9 / hbm, 4),
        "listed_rows_last_layer_ms": ms_per_step,
        "note": "SURVEY §8d's bytes describe the dense last layer (all N rows forward and backward), so the fraction is "
                "quoted on that line; the timed default step computes the last layer only at the 2*batch head / tail rows "
                "the decoder reads (same scores bit for bit, same gradients up to the split-K summation order)"}
    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
           "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None,
           "dtype": ("bf16x3-split / f32-accumulate (operands as bf16 hi + lo planes, three tensor-core products, ~17 mantissa "
                     "bits; gathers, means, loss in f32)" if args.mode == "fp32" else "bf16-transform / f32-accumulate"),
           "data": "synthetic", "parity": PARITY,
           "config": {"workload": WORKLOAD, "mode": args.mode, "l2": "flushed between steps (512 MiB write)",
                      "parallelism": "single GPU" if world == 1 else f"dp{world} replicas, parameter gradients written into one flat buffer; exchange: {dp_exchange}",
                      "timing": "CUDA events per step on the launching stream, max over ranks",
                      "step": "one CUDA-graph replay of forward + BCE loss + backward (GraphedTrainStep)",
                      "last_layer": ("dense over all N rows, forward and backward (PRIMEKG_RGCN_SPARSE_BWD=0)" if sparse_env == "0" else
                                     "listed rows: forward and backward of the LAST RGCNConv run on the 2*batch rows of the "
                                     "encoder output that the decoder reads (reference src/models/rgcn.py:325-326 "
                                     "node_embeddings[head], [tail]); scores bit-identical to the dense layer "
                                     "(tests/test_gpu_listed_fwd.py), identical gradients "
                                     "(tests/test_gpu_parity.py::test_layer_bwd_rows_equals_dense); the all-rows "
                                     "formulation is timed beside it as dense_last_layer")},
           "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_packed, "d2h_bytes_per_step": 8,
                   "api": "GraphedTrainStep(model, edge_index, edge_type, host_io=True): host_batch <- pack_batch(heads, tails, rels, labels); replay_host(); host_loss",
                   "loss_read_back": e2e_loss,
                   "eager_module_api_value": e2e_eager_value,
                   "note": "batch (heads, tails, rels, labels; one int64 [4, B] block) copied from pinned host memory and the loss copied back to pinned host memory inside every step (memcpy nodes of the captured graph); "
                           "the graph and the model stay device-resident as in reference src/train.py:122-135; "
                           "eager_module_api_value = the unmodified reference call model(...); loss; backward()"},
           "eager_ms_per_step": eager_ms,
           "dense_last_layer": (None if dense_ms is None else
                                {"ms_per_step": dense_ms, "value": world * kg.num_edges / (dense_ms * 1e-3), "unit": UNIT,
                                 "note": "same graphed step with the last layer computed for all N rows, forward and "
                                         "backward, as PyG does (PRIMEKG_RGCN_SPARSE_BWD=0)"}),
           "gpu_launches": launches_per_step * args.steps, "gpu_launches_per_step": launches_per_step,
           "wall_s_timed_region": t_wall, "clocks": clocks, "roofline": roofline, "partitioned": part}
    out["dense_last_layer_bwd"] = out["dense_last_layer"]        # (round-1 name of the same record)
    if world > 1:
        out["dp_exchange"] = {"form": dp_exchange, "all_ranks_arrived": dp_exchange_ok}
    if world == 1 and not args.quick:
        out["configs"] = other_configs(pkg, dev, flush, args.mode)
        try:
            out["library_gpu_baseline"] = library_gpu_baseline(kg, (heads, tails, rels, labels), dev)
        except Exception as ex:  # pragma: no cover
            out["library_gpu_baseline"] = {"error": repr(ex)[:200]}
    return out


# ---------------------------------------------------------------------------------------------
# CPU reference arm / cpu_baseline
# ---------------------------------------------------------------------------------------------
def cpu_reference_steps(steps, warmup, budget_s, threads=None):
    """Times the oracle (the restated reference path, oracle/rgcn_ref.py) on the host cores.
    Returns (edges_per_s, cores, sample description, ms_per_step)."""
    from oracle import rgcn_ref
    from primekg_rgcn_linkprediction_b200 import synth
    cores = threads or os.cpu_count() or 1
    torch.set_num_threads(cores)
    kg = synth.primekg_subgraph(CFG["num_edges"], seed=CFG["seed"])
    heads, tails, rels, labels = synth.link_batch(kg, CFG["batch_pos"], seed=CFG["seed"])
    torch.manual_seed(CFG["seed"])
    model = rgcn_ref.ModelRef(kg.num_nodes, kg.num_relations, CFG["embedding_dim"], CFG["hidden_dim"],
                              CFG["dropout"], CFG["decoder_dropout"])
    model.train()
    ei, et = kg.edge_index, kg.edge_type

    def step(ei, et):
        model.zero_grad(set_to_none=True)
        rgcn_ref.train_step_ref(model, ei, et, heads, tails, rels, labels)

    t0 = time.perf_counter(); step(ei, et); t_first = time.perf_counter() - t0
    frac = min(1.0, budget_s / max(1e-9, (steps + warmup) * t_first))
    sample = f"full step: all {kg.num_edges:,} edges"
    if frac < 1.0:
        keep = max(2, int(kg.num_edges * frac) // 2 * 2)
        ei, et = ei[:, :keep].contiguous(), et[:keep].contiguous()      # whole (a->b),(b->a) pairs
        sample = f"first {keep:,} of {kg.num_edges:,} edges per step (bounded sample, {cores} threads)"
    for _ in range(max(0, warmup - 1)):
        step(ei, et)
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter(); step(ei, et); ts.append(time.perf_counter() - t0)
    ms = statistics.mean(ts) * 1e3
    return et.numel() / (ms * 1e-3), cores, sample, ms


def run_reference(args):
    value, cores, sample, ms = cpu_reference_steps(args.steps, args.warmup, budget_s=150.0)
    return {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "parity": PARITY,
            "config": {"workload": WORKLOAD, "mode": "fp32", "device": "host CPU: " + cpu_model()},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                             "cpu_model": cpu_model()},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "PyG is not installable here; this is the restated reference path (oracle/rgcn_ref.py) in "
                    "PyTorch on the host cores"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default=os.environ.get("PRIMEKG_RGCN_MODE", "fp32"), choices=["fp32", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-partitioned", action="store_true", help="skip the node-range partitioned record")
    ap.add_argument("--quick", action="store_true", help="headline + roofline only (no other configs, no library baseline)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss, scores and parameter gradients of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to the GPU path (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank == 0:
            print(json.dumps(run_reference(args)), flush=True)
        return 0

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (B200); there is no CPU fallback for the product path")
    import __graft_entry__ as entry
    if rank == 0:
        entry.build()
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    out = run_ours(args, rank, world, local_rank)
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            v, cores, sample, ms = cpu_reference_steps(3, 1, budget_s=25.0)
            out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                                   "ms_per_step": ms, "cpu_model": cpu_model()}
            if not args.quick:
                v1, _, sample1, ms1 = cpu_reference_steps(2, 1, budget_s=12.0, threads=1)
                out["cpu_baseline"]["one_thread"] = {"value": v1, "unit": UNIT, "cores": 1, "sample": sample1, "ms_per_step": ms1}
        print(json.dumps(out), flush=True)
    if dist.is_initialized():
        if world > 1:
            dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())

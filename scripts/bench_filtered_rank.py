"""Filtered ranking and novel-link top-k against their raw forms on the B200: CUDA-graph replay, device events, the card's
name and power limit read in the same run.

* evaluate size: ``rank_true_tails(method="tc")`` for 15,372 queries drawn as edges of the cfg2 graph
  (``synth.primekg_subgraph()``) against all 30,926 entities at d = 256, raw against ``filter=`` the whole graph
  (per-query known-tail lists: mean ~240, hub keys ~7,450 entries);
* the one-off ``KnownTriples`` build over the graph's 849,456 edges;
* BASELINE cfg4: per drug the 10 best of 5,593 diseases (6,282 drugs), DistMult and cosine, raw against ``exclude=``.
  The cfg2 graph has no drug-disease relation, so a seeded power-law set of drug-disease pairs is added as relation 3;
  DistMult excludes that relation, cosine every relation (``exclude_relation=None``).

Raw and filtered calls alternate, each timed as the minimum over ``--repeats`` graph replays.
Usage: python scripts/bench_filtered_rank.py [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import primekg_rgcn_linkprediction_b200 as pkg
from primekg_rgcn_linkprediction_b200 import synth

DEV = "cuda:0"


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def graphed(fn, rep):
    """``rep`` calls of fn captured in one CUDA graph (after a warm-up call outside it)."""
    fn()
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            for _ in range(rep):
                fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    return gr


def replay_ms(gr, rep):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    gr.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / rep


def ab(fns, rep, repeats):
    """{name: [ms per call, one per round]}, the graphs replayed alternately."""
    graphs = {k: graphed(f, rep) for k, f in fns.items()}
    out = {k: [] for k in fns}
    for _ in range(repeats):
        for k, g in graphs.items():
            out[k].append(replay_ms(g, rep))
    return out


def summary(ts):
    return {"ms_min": round(min(ts), 4), "ms_median": round(sorted(ts)[len(ts) // 2], 4), "ms_max": round(max(ts), 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_filtered_rank needs a CUDA device")
    res = {"gpu": gpu_info(), "torch": torch.__version__}

    # ---- evaluate size ----
    kg = synth.primekg_subgraph()
    g = torch.Generator().manual_seed(11)
    sel = torch.randperm(kg.num_edges, generator=g)[:15372].to(DEV)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    heads, tails, rels = ei[0, sel], ei[1, sel], et[sel]
    torch.manual_seed(12)
    emb = torch.randn(kg.num_nodes, 256, device=DEV)
    table = torch.randn(kg.num_relations, 256, device=DEV)

    build_ms = []
    for _ in range(4):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        known = pkg.KnownTriples(ei[0], et, ei[1], kg.num_nodes, kg.num_relations)
        torch.cuda.synchronize()
        build_ms.append((time.perf_counter() - t0) * 1e3)
    b, e, _ = known.lists(heads, rels)
    n = (e - b).double()
    res["known_triples_build"] = {"edges": kg.num_edges, "distinct_triples": len(known),
                                  "ms_first": round(build_ms[0], 2), "ms_min_warm": round(min(build_ms[1:]), 2),
                                  "note": "host clock around the build, ending in a device synchronise"}
    res["evaluate_lists"] = {"queries": heads.numel(), "mean": round(float(n.mean()), 1),
                             "median": float(n.median()), "max": int(n.max()), "total": int(n.sum())}

    raw = pkg.rank_true_tails(emb, table, heads, rels, tails, method="tc")
    flt = pkg.rank_true_tails(emb, table, heads, rels, tails, method="tc", filter=known)
    t = ab({"raw": lambda: pkg.rank_true_tails(emb, table, heads, rels, tails, method="tc"),
            "filtered": lambda: pkg.rank_true_tails(emb, table, heads, rels, tails, method="tc", filter=known)},
           rep=2, repeats=args.repeats)
    res["rank_15372_x_30926_d256"] = {
        "raw": summary(t["raw"]), "filtered": summary(t["filtered"]),
        "filtered_over_raw": round(min(t["filtered"]) / min(t["raw"]), 3),
        "mrr_raw": pkg.ranking_metrics(raw[0])["mrr"], "mrr_filtered": pkg.ranking_metrics(flt[0])["mrr"],
        "mean_rank_raw": float(raw[0].double().mean()), "mean_rank_filtered": float(flt[0].double().mean())}

    # ---- cfg4 top-k with known drug-disease links excluded ----
    gd = torch.Generator().manual_seed(21)
    npairs = 40000
    dr = synth._draw(*synth.CFG1_BLOCKS["drug"], npairs, gd, 2.5).to(DEV)
    di = synth._draw(*synth.CFG1_BLOCKS["disease"], npairs, gd, 2.5).to(DEV)
    known4 = pkg.KnownTriples(torch.cat([ei[0], dr]), torch.cat([et, torch.full_like(dr, 3)]), torch.cat([ei[1], di]),
                              kg.num_nodes, 4)
    torch.manual_seed(3)
    emb4 = torch.randn(kg.num_nodes, 256, device=DEV)
    drugs = torch.arange(*synth.CFG1_BLOCKS["drug"], device=DEV)
    diseases = torch.arange(*synth.CFG1_BLOCKS["disease"], device=DEV)
    rel = torch.randn(256, device=DEV)
    bx, ex, _ = known4.lists(drugs, 3, diseases)
    res["cfg4_lists"] = {"drug_disease_pairs_drawn": npairs, "mean": round(float((ex - bx).double().mean()), 2),
                         "max": int((ex - bx).max())}
    for name, kw, xr in (("distmult", dict(rel_vec=rel), 3), ("cosine", dict(cosine=True), None)):
        f_raw = lambda: pkg.topk_all_pairs(emb4, drugs, diseases, k=10, **kw)
        f_exc = lambda: pkg.topk_all_pairs(emb4, drugs, diseases, k=10, exclude=known4, exclude_relation=xr, **kw)
        t = ab({"raw": f_raw, "exclude": f_exc}, rep=5, repeats=args.repeats)
        v0, i0 = f_raw()
        v1, i1 = f_exc()
        res[f"cfg4_topk10_{name}_6282x5593_d256"] = {
            "raw": summary(t["raw"]), "exclude": summary(t["exclude"]),
            "exclude_over_raw": round(min(t["exclude"]) / min(t["raw"]), 3),
            "rows_whose_list_changed": int((i0 != i1).any(1).sum())}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

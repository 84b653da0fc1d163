"""Generates the golden fixtures in this directory.  Needs a checkout of the original
PrimeKG-RGCN-LinkPrediction project in ``$PRIMEKG_RGCN_REFERENCE``; the fixtures it writes are committed.

It imports the UNMODIFIED reference ``$PRIMEKG_RGCN_REFERENCE/src/models/rgcn.py``.  That file imports
``torch_geometric.nn.RGCNConv`` (third party, not installable here), so a stub module provides
``RGCNConv = oracle.rgcn_ref.RGCNConvRef`` — everything else (encoder wiring, ReLU/dropout placement,
DistMult decoder, composite forward, predict_all_tails) is executed by the reference's own code.

    python tests/golden/make_golden.py
"""
import importlib.util
import os
import sys
import types

import numpy as np
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = os.environ.get("PRIMEKG_RGCN_REFERENCE", "")
if not REF or not os.path.isfile(os.path.join(REF, "src", "models", "rgcn.py")):
    sys.exit("set PRIMEKG_RGCN_REFERENCE to a checkout of the original PrimeKG-RGCN-LinkPrediction project")

from oracle import rgcn_ref  # noqa: E402


def load_reference_models():
    tg = types.ModuleType("torch_geometric")
    tgnn = types.ModuleType("torch_geometric.nn")
    tgnn.RGCNConv = rgcn_ref.RGCNConvRef
    tg.nn = tgnn
    sys.modules["torch_geometric"] = tg
    sys.modules["torch_geometric.nn"] = tgnn
    spec = importlib.util.spec_from_file_location("reference_rgcn", os.path.join(REF, "src/models/rgcn.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def rand_graph(n, e, r, seed):
    g = torch.Generator().manual_seed(seed)
    und = e // 2
    a = torch.randint(0, n, (und,), generator=g)
    # heavy tail so a few rows become hubs (> 128 in-edges of one relation) even on a small graph
    b = torch.floor(n * torch.rand(und, generator=g).pow(3.0)).long().clamp_(max=n - 1)
    t = torch.randint(0, r, (und,), generator=g)
    ei = torch.stack([torch.stack([a, b], 1).reshape(-1), torch.stack([b, a], 1).reshape(-1)], 0)
    return ei.contiguous(), t.repeat_interleave(2).contiguous()


def make_case(ref, name, n, e, r, emb, hid, bases, scale, seed, batch=64):
    torch.manual_seed(seed)
    model = ref.DrugDiseaseModel(num_nodes=n, num_relations=r, embedding_dim=emb, hidden_dim=hid, dropout=0.0,
                                 decoder_dropout=0.0, num_bases=bases)
    with torch.no_grad():
        for k, p in model.named_parameters():
            if scale != 1.0 and ("weight" in k or "root" in k or "comp" in k):
                p.mul_(scale)
            if k.endswith("bias"):
                p.uniform_(-0.1, 0.1)          # PyG zero-inits the bias; make it observable
    ei, et = rand_graph(n, e, r, seed + 1)
    g = torch.Generator().manual_seed(seed + 2)
    sel = torch.randperm(ei.size(1), generator=g)[:batch]
    heads = torch.cat([ei[0, sel], torch.randint(0, n, (batch,), generator=g)])
    tails = torch.cat([ei[1, sel], torch.randint(0, n, (batch,), generator=g)])
    rels = torch.cat([et[sel], et[sel]])
    labels = torch.cat([torch.ones(batch), torch.zeros(batch)])
    state = {k: v.detach().clone() for k, v in model.state_dict().items()}

    model.train()                                     # dropout p = 0 => deterministic
    scores = model(ei, et, heads, tails, rels)        # reference src/models/rgcn.py:300-331
    loss = F.binary_cross_entropy_with_logits(scores, labels)   # reference src/train.py:300
    loss.backward()                                   # reference src/train.py:306
    grads = {k: p.grad.detach().clone() for k, p in model.named_parameters()}
    emb_out = model.get_embeddings(ei, et)            # reference :397-415
    all_tails = model.predict_all_tails(ei, et, heads[:8], rels[:8])   # reference :362-395
    # LinkPredictor on gathered rows (reference :189-213)
    dec = model.decoder(emb_out[heads], emb_out[tails], rels).detach()
    out = dict(name=name, num_nodes=n, num_relations=r, embedding_dim=emb, hidden_dim=hid, num_bases=bases,
               edge_index=ei, edge_type=et, heads=heads, tails=tails, rels=rels, labels=labels, state_dict=state,
               scores=scores.detach(), loss=loss.detach(), grads=grads, embeddings=emb_out,
               all_tail_scores=all_tails, decoder_scores=dec)
    torch.save(out, os.path.join(HERE, f"{name}.pt"))
    print(name, "loss", float(loss), "|scores|max", float(scores.abs().max()), "E", ei.size(1))


def make_micro():
    """Hand-computable graph: 5 nodes, 2 relations, a duplicate edge, an isolated node (4), a node with
    only relation-1 in-edges (3).  Integer features, identity-like weights => exact expected values."""
    ei = torch.tensor([[0, 1, 1, 2, 0, 2],
                       [1, 0, 0, 0, 3, 3]])            # 1->0 twice (multi-edge kept)
    et = torch.tensor([0, 0, 0, 0, 1, 1])
    x = torch.tensor([[1., 2., 3., 4.], [10., 20., 30., 40.], [100., 200., 300., 400.], [7., 7., 7., 7.], [5., 6., 7., 8.]])
    W = torch.stack([torch.eye(4), 2 * torch.eye(4)])
    root = 3 * torch.eye(4)
    bias = torch.tensor([1., 1., 1., 1.])
    # node 0: rel0 in-neighbours {1, 1, 2} -> mean (10+10+100)/3 = 40 ; rel1: none
    # node 1: rel0 {0} -> x0 ;  node 3: rel1 {0, 2} -> mean (1+100)/2 = 50.5, times 2
    expected = torch.stack([
        torch.tensor([40., 80., 120., 160.]) + 3 * x[0] + 1,
        x[0] + 3 * x[1] + 1,
        3 * x[2] + 1,
        2 * torch.tensor([50.5, 101., 151.5, 202.]) + 3 * x[3] + 1,
        3 * x[4] + 1])
    got = rgcn_ref.rgcn_conv_ref(x, ei, et, W, root, bias)
    assert torch.equal(got, expected), (got, expected)
    torch.save(dict(edge_index=ei, edge_type=et, x=x, weight=W, root=root, bias=bias, expected=expected),
               os.path.join(HERE, "micro.pt"))
    print("micro ok")


def make_real_fixture(ref):
    """The reference's shipped validation graph (data/processed/val_data.pt: 15,362 directed drug-gene
    edges, all relation 0, real power-law degrees, multi-edges): stored as compressed int32 plus the
    reference model's output on it at a few sampled rows."""
    d = torch.load(os.path.join(REF, "data/processed/val_data.pt"))
    ei, et, n, r = d["edge_index"], d["edge_type"], d["num_nodes"], d["num_relations"]
    keep = (ei[0] < n) & (ei[1] < n)                  # reference src/train.py:572-586
    ei, et = ei[:, keep], et[keep]
    torch.manual_seed(7)
    model = ref.DrugDiseaseModel(num_nodes=n, num_relations=r, embedding_dim=64, hidden_dim=128, dropout=0.5,
                                 decoder_dropout=0.1)
    with torch.no_grad():
        for k, p in model.named_parameters():
            if "conv" in k and not k.endswith("bias"):
                p.mul_(4.0)
    emb = model.get_embeddings(ei, et)
    touched = torch.unique(ei)
    g = torch.Generator().manual_seed(3)
    rows = torch.cat([touched[torch.randperm(touched.numel(), generator=g)[:96]],
                      torch.randint(0, n, (32,), generator=g)])
    np.savez_compressed(os.path.join(HERE, "val_graph.npz"), edge_index=ei.numpy().astype(np.int32),
                        edge_type=et.numpy().astype(np.int8), num_nodes=n, num_relations=r,
                        rows=rows.numpy().astype(np.int32), emb_rows=emb[rows].numpy(),
                        emb_colsum=emb.double().sum(0).numpy(), seed=7, conv_scale=4.0)
    print("val_graph", ei.shape, "rows", rows.numel())


if __name__ == "__main__":
    ref = load_reference_models()
    make_micro()
    make_case(ref, "small_full", n=150, e=2400, r=3, emb=16, hid=32, bases=None, scale=1.8, seed=11)
    make_case(ref, "small_basis", n=140, e=2000, r=6, emb=16, hid=24, bases=2, scale=1.6, seed=23)
    make_case(ref, "small_default_init", n=100, e=500, r=3, emb=64, hid=128, bases=None, scale=1.0, seed=5, batch=32)
    make_real_fixture(ref)

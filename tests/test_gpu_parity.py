"""GPU parity tests: the sm_100a kernels (through the C ABI) against the CPU oracle, the golden
fixtures produced by the unmodified reference model file, and size-independent properties at the
benchmark's full size.

Tolerances (BASELINE.json north_star): bit-exact for CSR / index construction; rtol 1e-4 for fp32
embeddings, losses and scores; 2e-2 in the bf16-transform mode.  Gradients of sums over ~10^3 terms
are compared at rtol 1e-3 / small atol (different but fixed summation orders).
"""
import os

import pytest
import torch
import torch.nn.functional as F

from conftest import load_golden, load_val_graph
from oracle import rgcn_ref as O

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture(scope="module")
def pkg(lib_built):
    return lib_built


def _graphs():
    from primekg_rgcn_linkprediction_b200 import synth
    v = load_val_graph()
    out = {
        "uniform_small": (synth.uniform_kg(100, 500, 3, seed=1), None),
        "uniform_r30": (synth.uniform_kg(5000, 60_000, 30, seed=2), None),
        "primekg_100k": (synth.primekg_subgraph(100_000, seed=3), None),
        "one_relation": (synth.uniform_kg(257, 4000, 1, seed=4), None),
    }
    g = {k: (kg.edge_index, kg.edge_type, kg.num_nodes, kg.num_relations) for k, (kg, _) in out.items()}
    g["val_fixture"] = (v["edge_index"], v["edge_type"], v["num_nodes"], v["num_relations"])
    g["empty"] = (torch.zeros(2, 0, dtype=torch.int64), torch.zeros(0, dtype=torch.int64), 17, 3)
    # ragged: isolated nodes, a node with only relation-1 in-edges, a multi-edge, a self loop
    g["ragged"] = (torch.tensor([[0, 1, 1, 2, 0, 2, 6, 6], [1, 0, 0, 0, 3, 3, 6, 0]]),
                   torch.tensor([0, 0, 0, 0, 1, 1, 2, 2]), 9, 3)
    return g


GRAPHS = None


def graphs():
    global GRAPHS
    if GRAPHS is None:
        GRAPHS = _graphs()
    return GRAPHS


GRAPH_NAMES = ["uniform_small", "uniform_r30", "primekg_100k", "one_relation", "val_fixture", "empty", "ragged"]


# ------------------------------------------------------------------------------------------------
# (1) graph preprocessing: bit-exact
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", GRAPH_NAMES)
def test_csr_bit_exact(pkg, name):
    ei, et, N, R = graphs()[name]
    g = pkg.RelGraph.from_edges(ei.to(DEV), et.to(DEV), N, R)
    rowptr, col, perm, rowptr_t, row_t, perm_t = O.csr_oracle(ei, et, N, R)
    for got, want, what in ((g.rowptr, rowptr, "rowptr"), (g.col, col, "col"), (g.perm, perm, "perm"),
                            (g.rowptr_t, rowptr_t, "rowptr_t"), (g.row_t, row_t, "row_t"), (g.perm_t, perm_t, "perm_t")):
        assert torch.equal(got.cpu().to(torch.int64), want), what
    cnt = (rowptr[1:] - rowptr[:-1]).clamp(min=1).to(torch.float32)
    assert torch.equal(g.inv_cnt.cpu(), 1.0 / cnt)
    if ei.size(1):
        w = (1.0 / cnt)[(ei[1] * R + et)[perm_t]]
        assert torch.equal(g.w_t.cpu(), w)
        assert g.max_seg == int((rowptr[1:] - rowptr[:-1]).max())
        assert g.max_seg_t == int((rowptr_t[1:] - rowptr_t[:-1]).max())


def test_csr_rejects_out_of_range(pkg):
    ei = torch.tensor([[0, 5], [1, 0]], device=DEV)
    with pytest.raises(IndexError):
        pkg.RelGraph.from_edges(ei, torch.tensor([0, 0], device=DEV), 5, 1)
    with pytest.raises(IndexError):
        pkg.RelGraph.from_edges(torch.tensor([[0], [1]], device=DEV), torch.tensor([3], device=DEV), 5, 3)
    with pytest.raises(IndexError):
        pkg.RelGraph.from_edges(torch.tensor([[0], [-1]], device=DEV), torch.tensor([0], device=DEV), 5, 3)


def test_graph_cache_identity_and_invalidation(pkg):
    ei, et, N, R = graphs()["uniform_small"]
    ei, et = ei.to(DEV), et.to(DEV)
    pkg.clear_graph_cache()
    g1 = pkg.get_graph(ei, et, N, R)
    assert pkg.get_graph(ei, et, N, R) is g1                 # same tensors every step => cache hit
    et[0] = (et[0] + 1) % R                                  # in-place edit bumps _version
    g2 = pkg.get_graph(ei, et, N, R)
    assert g2 is not g1
    rowptr = O.csr_oracle(ei.cpu(), et.cpu(), N, R)[0]
    assert torch.equal(g2.rowptr.cpu().to(torch.int64), rowptr)


# ------------------------------------------------------------------------------------------------
# (3) aggregation forward / backward
# ------------------------------------------------------------------------------------------------
def _means_ref(x, ei, et, N, R):
    out = []
    for r in range(R):
        m = et == r
        s = torch.zeros(N, x.size(1), dtype=x.dtype).index_add_(0, ei[1][m], x[ei[0][m]])
        c = torch.zeros(N, dtype=x.dtype).index_add_(0, ei[1][m], torch.ones(int(m.sum()), dtype=x.dtype)).clamp_(min=1)
        out.append(s / c[:, None])
    return torch.cat(out, 1)


@pytest.mark.parametrize("name", GRAPH_NAMES)
@pytest.mark.parametrize("d", [16, 64, 128, 256, 100])
def test_aggregate_fwd(pkg, name, d):
    from primekg_rgcn_linkprediction_b200 import ops
    ei, et, N, R = graphs()[name]
    if N * R * d > 60_000_000:
        pytest.skip("oracle too slow at this size")
    torch.manual_seed(0)
    x = torch.randn(N, d)
    g = pkg.RelGraph.from_edges(ei.to(DEV), et.to(DEV), N, R)
    H = ops.aggregate_fwd(g, x.to(DEV)).cpu()
    want = _means_ref(x, ei, et, N, R)
    torch.testing.assert_close(H, want, rtol=1e-5, atol=1e-5)
    # segments below the hub threshold are summed serially in original edge order => identical bits
    cnt = (g.rowptr[1:] - g.rowptr[:-1]).cpu().view(N, R)
    small = (cnt <= g.fwd.threshold)[:, :, None].expand(N, R, d).reshape(N, R * d)
    assert torch.equal(H[small], want[small])
    Hb = ops.aggregate_fwd(g, x.to(DEV), out_bf16=True).cpu()
    assert torch.equal(Hb, H.to(torch.bfloat16))


@pytest.mark.parametrize("name", ["uniform_small", "uniform_r30", "primekg_100k", "val_fixture", "ragged", "empty"])
@pytest.mark.parametrize("d", [64, 256])
def test_aggregate_bwd(pkg, name, d):
    from primekg_rgcn_linkprediction_b200 import ops
    ei, et, N, R = graphs()[name]
    if N * R * d > 60_000_000:
        pytest.skip("oracle too slow at this size")
    torch.manual_seed(1)
    x = torch.randn(N, d, dtype=torch.float64, requires_grad=True)
    gA = torch.randn(N, (R + 1) * d)
    H = _means_ref(x, ei, et, N, R)
    (H * gA[:, : R * d].double()).sum().backward()
    want = x.grad.float() + gA[:, R * d:]
    g = pkg.RelGraph.from_edges(ei.to(DEV), et.to(DEV), N, R)
    gAd = gA.to(DEV)
    got = ops.aggregate_bwd(g, gAd, d, init=gAd[:, R * d:]).cpu()
    torch.testing.assert_close(got, want, rtol=1e-4, atol=1e-4)
    got2 = ops.aggregate_bwd(g, gAd, d, init=gAd[:, R * d:]).cpu()
    assert torch.equal(got, got2)                            # deterministic: no atomics


def test_aggregate_appends_root_rows(pkg):
    """x_root appended as the last block by the row walk = the separate split_planes call, bit for bit."""
    from primekg_rgcn_linkprediction_b200 import ops
    ei, et, N, R = graphs()["primekg_100k"]
    g = pkg.RelGraph.from_edges(ei.to(DEV), et.to(DEV), N, R)
    torch.manual_seed(5)
    for d in (64, 256, 100):
        x = torch.randn(N, d, device=DEV)
        A = ops.alloc_planes(N, (R + 1) * d, "fp32", DEV)
        B = ops.alloc_planes(N, (R + 1) * d, "fp32", DEV)
        ops.aggregate_fwd(g, x, planes=A, x_root=x)
        ops.aggregate_fwd(g, x, planes=B)
        ops.split_planes(x, B, col0=R * d)
        assert torch.equal(A[0], B[0]) and torch.equal(A[1], B[1])


def test_aggregate_basis_mix(pkg):
    from primekg_rgcn_linkprediction_b200 import ops
    ei, et, N, R = graphs()["uniform_r30"]
    torch.manual_seed(2)
    d, B = 64, 8
    x = torch.randn(N, d)
    comp = torch.randn(R, B)
    g = pkg.RelGraph.from_edges(ei.to(DEV), et.to(DEV), N, R)
    Z = ops.aggregate_fwd(g, x.to(DEV), comp=comp.to(DEV)).cpu()
    H = _means_ref(x, ei, et, N, R).view(N, R, d)
    want = torch.einsum("nrd,rb->nbd", H, comp).reshape(N, B * d)
    torch.testing.assert_close(Z, want, rtol=1e-4, atol=1e-4)


# ------------------------------------------------------------------------------------------------
# the layer and the whole model against the goldens of the unmodified reference file
# ------------------------------------------------------------------------------------------------
def test_micro_graph_exact(pkg):
    g = load_golden("micro")
    conv = pkg.RGCNConv(4, 4, 2)
    with torch.no_grad():
        conv.weight.copy_(g["weight"]); conv.root.copy_(g["root"]); conv.bias.copy_(g["bias"])
    conv.to(DEV)
    out = conv(g["x"].to(DEV), g["edge_index"].to(DEV), g["edge_type"].to(DEV))
    torch.testing.assert_close(out.cpu(), g["expected"], rtol=1e-6, atol=1e-4)


def _product_model(pkg, g, mode="fp32"):
    m = pkg.DrugDiseaseModel(g["num_nodes"], g["num_relations"], g["embedding_dim"], g["hidden_dim"], dropout=0.0,
                             decoder_dropout=0.0, num_bases=g["num_bases"])
    m.load_state_dict(g["state_dict"], strict=True)          # reference-trained checkpoints load as they are
    for c in (m.encoder.conv1, m.encoder.conv2):
        c.mode = mode
    return m.to(DEV)


@pytest.mark.parametrize("name", ["small_full", "small_basis", "small_default_init"])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_model_matches_reference_goldens(pkg, name, mode):
    g = load_golden(name)
    m = _product_model(pkg, g, mode)
    rtol, atol = (1e-4, 1e-5) if mode == "fp32" else (2e-2, 2e-2)
    ei, et = g["edge_index"].to(DEV), g["edge_type"].to(DEV)
    m.train()
    scores = m(ei, et, g["heads"].to(DEV), g["tails"].to(DEV), g["rels"].to(DEV))
    loss = F.binary_cross_entropy_with_logits(scores, g["labels"].to(DEV))
    loss.backward()
    smax = float(g["scores"].abs().max())
    torch.testing.assert_close(scores.detach().cpu(), g["scores"], rtol=rtol, atol=atol * max(1.0, smax))
    torch.testing.assert_close(loss.detach().cpu(), g["loss"], rtol=rtol, atol=atol)
    for k, p in m.named_parameters():
        want = g["grads"][k]
        scale = float(want.abs().max()) + 1e-12
        if mode == "fp32":
            torch.testing.assert_close(p.grad.cpu(), want, rtol=1e-3, atol=2e-5 * scale,
                                       msg=lambda s: f"{name}/{mode}/{k}: {s}")
        else:
            # bf16 operands perturb the logits by ~1e-2, which the sigmoid amplifies element-wise; the
            # gradient is checked in norm
            rel = float((p.grad.cpu() - want).norm() / (want.norm() + 1e-30))
            assert rel < 0.15, f"{name}/{mode}/{k}: relative Frobenius error {rel:.3e}"
    emb = m.get_embeddings(ei, et)
    emax = float(g["embeddings"].abs().max())
    torch.testing.assert_close(emb.cpu(), g["embeddings"], rtol=rtol, atol=atol * max(1.0, emax))
    if mode == "fp32":
        all_t = m.predict_all_tails(ei, et, g["heads"][:8].to(DEV), g["rels"][:8].to(DEV))
        torch.testing.assert_close(all_t.cpu(), g["all_tail_scores"], rtol=1e-4, atol=1e-4 * max(1.0, smax))
        dec = m.decoder(emb[g["heads"].to(DEV)], emb[g["tails"].to(DEV)], g["rels"].to(DEV))
        torch.testing.assert_close(dec.cpu(), g["decoder_scores"], rtol=1e-4, atol=1e-5 * max(1.0, smax))
        pred = m.predict(ei, et, g["heads"].to(DEV), g["tails"].to(DEV), g["rels"].to(DEV))
        torch.testing.assert_close(pred.cpu(), g["scores"], rtol=1e-4, atol=1e-5 * max(1.0, smax))


def test_real_fixture_graph_rows(pkg):
    """The reference's own validation graph: seeded init must consume the RNG in the reference's order and
    the encoder must reproduce the reference's rows."""
    v = load_val_graph()
    torch.manual_seed(v["seed"])
    m = pkg.DrugDiseaseModel(v["num_nodes"], v["num_relations"], 64, 128, dropout=0.5, decoder_dropout=0.1)
    with torch.no_grad():
        for k, p in m.named_parameters():
            if "conv" in k and not k.endswith("bias"):
                p.mul_(v["conv_scale"])
    m.to(DEV)
    emb = m.get_embeddings(v["edge_index"].to(DEV), v["edge_type"].to(DEV)).cpu()
    torch.testing.assert_close(emb[v["rows"]], v["emb_rows"], rtol=1e-4, atol=1e-5)
    # a column sum over 30,926 rows: tolerance relative to the sum of magnitudes (summation-order noise)
    tol = 1e-5 * emb.double().abs().sum(0)
    assert torch.all((emb.double().sum(0) - v["emb_colsum"]).abs() <= tol + 1e-6)


def test_decoder_rows_backward(pkg):
    torch.manual_seed(4)
    B, d, R = 37, 128, 3
    dec = pkg.LinkPredictor(R, d).to(DEV)
    ref = O.DecoderRef(R, d)
    ref.load_state_dict(dec.state_dict())
    h = torch.randn(B, d, requires_grad=True)
    t = torch.randn(B, d, requires_grad=True)
    rel = torch.randint(0, R, (B,))
    hd, td = h.detach().to(DEV).requires_grad_(), t.detach().to(DEV).requires_grad_()
    s = dec(hd, td, rel.to(DEV))
    s.sum().backward()
    sr = ref(h, t, rel)
    sr.sum().backward()
    torch.testing.assert_close(s.detach().cpu(), sr.detach(), rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(hd.grad.cpu(), h.grad, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(td.grad.cpu(), t.grad, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(dec.relation_embeddings.weight.grad.cpu(), ref.relation_embeddings.weight.grad,
                               rtol=1e-4, atol=1e-4)


def test_decoder_dropout_path_trains(pkg):
    torch.manual_seed(5)
    g = load_golden("small_full")
    m = pkg.DrugDiseaseModel(g["num_nodes"], g["num_relations"], g["embedding_dim"], g["hidden_dim"], dropout=0.5,
                             decoder_dropout=0.1).to(DEV)
    m.train()
    s = m(g["edge_index"].to(DEV), g["edge_type"].to(DEV), g["heads"].to(DEV), g["tails"].to(DEV), g["rels"].to(DEV))
    F.binary_cross_entropy_with_logits(s, g["labels"].to(DEV)).backward()
    for k, p in m.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all(), k


def test_encoder_deterministic(pkg):
    g = load_golden("small_full")
    m = _product_model(pkg, g)
    ei, et = g["edge_index"].to(DEV), g["edge_type"].to(DEV)
    outs, grads = [], []
    for _ in range(2):
        m.zero_grad()
        e = m.encoder(ei, et)
        e.square().sum().backward()
        outs.append(e.detach().clone())
        grads.append(m.encoder.node_embeddings.weight.grad.clone())
    assert torch.equal(outs[0], outs[1]) and torch.equal(grads[0], grads[1])


# ------------------------------------------------------------------------------------------------
# reference self-tests (src/models/rgcn.py:422-570): shapes
# ------------------------------------------------------------------------------------------------
def test_reference_shape_selftests(pkg):
    torch.manual_seed(0)
    enc = pkg.DrugDiseaseRGCN(100, 3, 64, 128).to(DEV)
    ei = torch.randint(0, 100, (2, 500), device=DEV)
    et = torch.randint(0, 3, (500,), device=DEV)
    assert enc(ei, et).shape == (100, 128)
    dec = pkg.LinkPredictor(3, 128).to(DEV)
    h, t = torch.randn(32, 128, device=DEV), torch.randn(32, 128, device=DEV)
    rel = torch.randint(0, 3, (32,), device=DEV)
    assert dec(h, t, rel).shape == (32,)
    assert dec.score_all_tails(h, rel, torch.randn(100, 128, device=DEV)).shape == (32, 100)
    model = pkg.DrugDiseaseModel(100, 3, 64, 128).to(DEV)
    heads, tails = torch.randint(0, 100, (32,), device=DEV), torch.randint(0, 100, (32,), device=DEV)
    assert model(ei, et, heads, tails, rel).shape == (32,)
    assert model.predict(ei, et, heads, tails, rel).shape == (32,)
    assert model.predict_all_tails(ei, et, heads, rel).shape == (32, 100)
    assert model.get_embeddings(ei, et).shape == (100, 128)
    assert enc.get_node_embeddings(heads).shape == (32, 64)
    sub = enc(ei, et, node_indices=torch.arange(100, device=DEV))
    assert sub.shape == (100, 128)


def test_error_behaviour(pkg):
    conv = pkg.RGCNConv(8, 8, 2).to(DEV)
    x = torch.randn(5, 8, device=DEV)
    ei = torch.tensor([[0, 1], [1, 2]], device=DEV)
    with pytest.raises(ValueError):
        conv(x, ei, None)
    with pytest.raises(IndexError):
        conv(x, torch.tensor([[0, 7], [1, 2]], device=DEV), torch.tensor([0, 1], device=DEV))
    with pytest.raises(RuntimeError):
        pkg.RGCNConv(8, 8, 2)(x.cpu(), ei.cpu(), torch.tensor([0, 1]))


# ------------------------------------------------------------------------------------------------
# full benchmark size (cfg2: 30,926 nodes / 849,456 edges / 3 relations, 64 -> 256 -> 256)
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def cfg2():
    from primekg_rgcn_linkprediction_b200 import synth
    kg = synth.primekg_subgraph()
    return kg, synth.link_batch(kg, 1024)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_full_size_step_against_oracle_on_device(pkg, cfg2, mode):
    """cfg2 at full size: the oracle restatement runs on the same GPU through stock torch ops."""
    kg, (heads, tails, rels, labels) = cfg2
    torch.manual_seed(42)
    m = pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, 64, 256, dropout=0.0, decoder_dropout=0.0)
    with torch.no_grad():
        for k, p in m.named_parameters():
            if "conv" in k and not k.endswith("bias"):
                p.mul_(4.0)
    ref = O.ModelRef(kg.num_nodes, kg.num_relations, 64, 256, 0.0, 0.0)
    ref.load_state_dict(m.state_dict())
    for c in (m.encoder.conv1, m.encoder.conv2):
        c.mode = mode
    m.to(DEV).train(); ref.to(DEV).train()
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    b = [t.to(DEV) for t in (heads, tails, rels, labels)]
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        s = m(ei, et, b[0], b[1], b[2])
        loss = F.binary_cross_entropy_with_logits(s, b[3])
        loss.backward()
        rl, rs = O.train_step_ref(ref, ei, et, b[0], b[1], b[2], b[3])
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    rtol, atol = (1e-4, 1e-5) if mode == "fp32" else (2e-2, 2e-2)
    smax = float(rs.abs().max())
    torch.testing.assert_close(s.detach(), rs, rtol=rtol, atol=atol * max(1.0, smax))
    torch.testing.assert_close(loss.detach(), rl, rtol=rtol, atol=atol)
    for (k, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
        scale = float(q.grad.abs().max()) + 1e-12
        # 7.9 M ReLU inputs: a few sit within rounding distance of 0 and flip between two correct fp32
        # implementations, which changes single gradient entries by a finite amount => norm + loose elementwise
        rel = float((p.grad - q.grad).norm() / (q.grad.norm() + 1e-30))
        assert rel < (5e-3 if mode == "fp32" else 0.15), f"{mode}/{k}: relative Frobenius error {rel:.3e}"
        if mode == "fp32":
            torch.testing.assert_close(p.grad, q.grad, rtol=1e-2, atol=1e-2 * scale, msg=lambda t: f"{mode}/{k}: {t}")



def test_full_size_gradients_with_matched_relu_pattern(pkg, cfg2):
    """Why ``test_full_size_step_against_oracle_on_device`` holds the gradients only in norm: with 7.9 M hidden
    activations a few ReLU inputs sit within rounding distance of zero and their 0 / 1 derivative differs between two
    correct fp32 evaluation orders.  SHOWN here, not asserted: (1) the activation patterns of the two implementations
    differ ONLY at elements whose oracle pre-activation is below 2e-5 * max|z| (the forward's rounding band);
    (2) once the oracle differentiates through OUR pattern (h = z * [ours > 0]) every gradient agrees element-wise
    at rtol 1e-3 — the bar of the small golden fixtures — with an absolute floor of 1e-4 of the tensor's scale."""
    kg, (heads, tails, rels, labels) = cfg2
    torch.manual_seed(42)
    m = pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, 64, 256, dropout=0.0, decoder_dropout=0.0)
    with torch.no_grad():
        for k, p in m.named_parameters():
            if "conv" in k and not k.endswith("bias"):
                p.mul_(4.0)
    ref = O.ModelRef(kg.num_nodes, kg.num_relations, 64, 256, 0.0, 0.0)
    ref.load_state_dict(m.state_dict())
    for c in (m.encoder.conv1, m.encoder.conv2):
        c.mode = "fp32"
    m.to(DEV).train(); ref.to(DEV).train()
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    b = [t.to(DEV) for t in (heads, tails, rels, labels)]
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        s = m(ei, et, b[0], b[1], b[2])
        F.binary_cross_entropy_with_logits(s, b[3]).backward()
        with torch.no_grad():
            graph = pkg.get_graph(ei, et, kg.num_nodes, kg.num_relations)
            ours_on = m.encoder.conv1.forward_graph(m.encoder.node_embeddings.weight, graph, relu=True) > 0
        enc = ref.encoder
        z1 = enc.conv1(enc.node_embeddings.weight, ei, et)
        flips = ours_on != (z1 > 0)
        band = 2e-5 * float(z1.detach().abs().max())
        n_flip = int(flips.sum())
        assert n_flip < 1e-3 * z1.numel(), n_flip
        if n_flip:
            worst = float(z1.detach().abs()[flips].max())
            assert worst < band, f"{n_flip} ReLU flips, the largest at |z| = {worst:.3e} (band {band:.3e})"
        h = z1 * ours_on.to(z1.dtype)                      # relu(z1) up to the band; derivative = OUR pattern
        emb = enc.conv2(h, ei, et)
        rs = ref.decoder(emb[b[0]], emb[b[1]], b[2])
        F.binary_cross_entropy_with_logits(rs, b[3]).backward()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    torch.testing.assert_close(s.detach(), rs.detach(), rtol=1e-4, atol=1e-5 * max(1.0, float(rs.abs().max())))
    for (k, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
        scale = float(q.grad.abs().max()) + 1e-30
        torch.testing.assert_close(p.grad, q.grad, rtol=1e-3, atol=1e-4 * scale,
                                   msg=lambda t: f"{k} ({n_flip} pattern flips inside the band): {t}")


@pytest.mark.parametrize("decoder_dropout", [0.0, 0.1])
def test_step_is_bitwise_deterministic(pkg, cfg2, decoder_dropout):
    """SURVEY §7.2: determinism end to end.  Two runs of the same step (hub-heavy batch: repeated head / tail nodes; the
    decoder's backward sums them in position order, csrc/decoder.cu link_bwd_rows_kernel) give bit-identical gradients
    for EVERY parameter, the embedding table and the relation table included."""
    kg, (heads, tails, rels, labels) = cfg2
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    b = [t.to(DEV) for t in (heads, tails, rels, labels)]
    assert torch.unique(torch.cat([b[0], b[1]])).numel() < 2 * b[0].numel()          # the batch does repeat nodes
    runs = []
    for _ in range(2):
        torch.manual_seed(7)
        m = pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, 64, 256, dropout=0.0,
                                 decoder_dropout=decoder_dropout).to(DEV)
        m.train()
        s = m(ei, et, b[0], b[1], b[2])
        F.binary_cross_entropy_with_logits(s, b[3]).backward()
        loss2, _, _ = m.link_loss(ei, et, b[0], b[1], b[2], b[3])
        g2 = torch.autograd.grad(loss2, [m.encoder.node_embeddings.weight, m.decoder.relation_embeddings.weight])
        runs.append(({k: p.grad.clone() for k, p in m.named_parameters()}, [g.clone() for g in g2]))
    for k in runs[0][0]:
        assert torch.equal(runs[0][0][k], runs[1][0][k]), k
    for a, c in zip(runs[0][1], runs[1][1]):
        assert torch.equal(a, c)


def test_decoder_backward_rows_matches_reference_formula(pkg):
    """The deterministic decoder backward against autograd of the plain formula (repeated nodes, self pairs h == t,
    a relation nobody uses, d not a multiple of 128)."""
    torch.manual_seed(11)
    N, d, R, B = 50, 72, 4, 300
    emb = torch.randn(N, d, device=DEV, requires_grad=True)
    dec = pkg.LinkPredictor(R, d).to(DEV)
    heads = torch.randint(0, 12, (B,), device=DEV)                  # 12 nodes only: every node repeats many times
    tails = torch.randint(0, N, (B,), device=DEV)
    tails[:20] = heads[:20]                                          # self pairs
    rels = torch.randint(0, R - 1, (B,), device=DEV)                 # relation R-1 unused: its gradient row is exactly 0
    coef = torch.randn(B, device=DEV)
    s = dec.score_pairs(emb, heads, tails, rels)
    (s * coef).sum().backward()
    e2 = emb.detach().clone().requires_grad_()
    t2 = dec.relation_embeddings.weight.detach().clone().requires_grad_()
    s2 = (e2[heads] * t2[rels] * e2[tails]).sum(1)
    (s2 * coef).sum().backward()
    torch.testing.assert_close(s.detach(), s2.detach(), rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(emb.grad, e2.grad, rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(dec.relation_embeddings.weight.grad, t2.grad, rtol=1e-4, atol=1e-4)
    assert float(dec.relation_embeddings.weight.grad[R - 1].abs().sum()) == 0.0
    assert float(emb.grad[torch.tensor([i for i in range(N) if i not in set(heads.tolist()) | set(tails.tolist())],
                                       device=DEV, dtype=torch.long)].abs().sum()) == 0.0


def test_out_of_range_pair_is_skipped_and_flagged(pkg):
    """The reference's ``node_embeddings[idx]`` raises a device assert on a bad index; the fused decoder skips the pair
    (NaN score, no gradient, no out-of-bounds access) and ``ops.raise_on_bad_pairs`` reports it."""
    from primekg_rgcn_linkprediction_b200 import ops
    torch.manual_seed(12)
    N, d, R, B = 40, 64, 3, 16
    emb = torch.randn(N, d, device=DEV, requires_grad=True)
    dec = pkg.LinkPredictor(R, d).to(DEV)
    heads = torch.randint(0, N, (B,), device=DEV)
    tails = torch.randint(0, N, (B,), device=DEV)
    rels = torch.randint(0, R, (B,), device=DEV)
    ops.raise_on_bad_pairs(emb.device)                               # clean slate
    good = dec.score_pairs(emb, heads, tails, rels).detach()
    ops.raise_on_bad_pairs(emb.device)                               # nothing to report
    bad_h, bad_r = heads.clone(), rels.clone()
    bad_h[3] = N + 5
    bad_r[7] = -1
    s = dec.score_pairs(emb, bad_h, tails, bad_r)
    assert torch.isnan(s[3]) and torch.isnan(s[7])
    keep = torch.ones(B, dtype=torch.bool, device=DEV)
    keep[3] = keep[7] = False
    torch.testing.assert_close(s.detach()[keep], good[keep], rtol=0, atol=0)
    torch.nan_to_num(s, nan=0.0).sum().backward()
    assert torch.isfinite(emb.grad).all() and torch.isfinite(dec.relation_embeddings.weight.grad).all()
    e2 = emb.detach().clone().requires_grad_()
    (e2[heads[keep]] * dec.relation_embeddings.weight.detach()[rels[keep]] * e2[tails[keep]]).sum().backward()
    torch.testing.assert_close(emb.grad, e2.grad, rtol=1e-4, atol=1e-5)          # the two bad pairs left no trace
    with pytest.raises(IndexError):
        ops.raise_on_bad_pairs(emb.device)
    ops.raise_on_bad_pairs(emb.device)                               # the flag is cleared by the report


def test_fused_dropout_hash_statistics(pkg):
    """The fused dropout draws its mask from a counter-based hash (csrc/transform.cu), not from torch's Philox stream;
    what a dropout mask needs is tested here on 2.6 M elements per step: keep rate, independence of neighbouring elements
    along rows and columns (2 x 2 chi-square, 1 degree of freedom), no serial correlation at lags 1..4 in memory order,
    independence between consecutive steps, and 16-bit resolution of p."""
    from primekg_rgcn_linkprediction_b200 import ops
    n, K, d_out = 20_000, 8, 128
    A = torch.zeros(n, K, device=DEV)
    planes = ops.alloc_planes(n, K, "bf16", A.device)
    ops.split_planes(A, planes)
    W = torch.zeros(K, d_out, device=DEV)
    bias = torch.ones(d_out, device=DEV)
    ctr = ops.dropout_counter(A.device)

    def mask(p, seed):
        out = ops.transform_fwd(planes, K, 0, W, None, bias, True, "bf16", p, seed, ctr)       # = 1 / (1 - p) where kept
        return out > 0

    def chi2(a, c):                                       # 2 x 2 contingency of two boolean tensors
        a, c = a.reshape(-1).double(), c.reshape(-1).double()
        nn_ = a.numel()
        o = torch.stack([(a * c).sum(), (a * (1 - c)).sum(), ((1 - a) * c).sum(), ((1 - a) * (1 - c)).sum()])
        pa, pc = a.mean(), c.mean()
        e = nn_ * torch.stack([pa * pc, pa * (1 - pc), (1 - pa) * pc, (1 - pa) * (1 - pc)])
        return float(((o - e) ** 2 / e).sum())

    for p in (0.5, 0.1, 0.9):
        m0, m1 = mask(p, 1234), mask(p, 1234)              # consecutive steps of one stream
        tot = m0.numel()
        sd = (p * (1 - p) / tot) ** 0.5
        assert abs(float(m0.float().mean()) - (1 - p)) < 5 * sd + 2.0 ** -16
        assert chi2(m0[:, :-1], m0[:, 1:]) < 20.0          # chi-square(1): P(> 20) ~ 8e-6
        assert chi2(m0[:-1, :], m0[1:, :]) < 20.0
        assert chi2(m0, m1) < 20.0
        flat = m0.reshape(-1).double() - (1 - p)
        for lag in (1, 2, 3, 4):
            rho = float((flat[:-lag] * flat[lag:]).mean() / (p * (1 - p)))
            assert abs(rho) < 5.0 / tot ** 0.5, (p, lag, rho)
        assert (m0 != m1).any()
        assert (mask(p, 99) != mask(p, 1234)).any()        # another seed, another stream
    # per-row and per-column keep counts are binomial: the largest z-score over 20,000 rows stays below 6
    m = mask(0.5, 5)
    z_rows = (m.double().sum(1) - 0.5 * d_out) / (0.25 * d_out) ** 0.5
    z_cols = (m.double().sum(0) - 0.5 * n) / (0.25 * n) ** 0.5
    assert float(z_rows.abs().max()) < 6.0 and float(z_cols.abs().max()) < 6.0


def test_full_size_properties(pkg, cfg2):
    """Size-independent properties at 849,456 edges: linearity of the aggregation, the count-weighted
    checksum  sum_i cnt(i, r) * H_r[i] = sum_{e of type r} x[src[e]], and adjointness <agg(x), g> = <x, agg^T(g)>."""
    from primekg_rgcn_linkprediction_b200 import ops
    kg, _ = cfg2
    N, R, d = kg.num_nodes, kg.num_relations, 64
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    g = pkg.get_graph(ei, et, N, R)
    torch.manual_seed(9)
    x, y = torch.randn(N, d, device=DEV), torch.randn(N, d, device=DEV)
    Hx, Hy, Hxy = ops.aggregate_fwd(g, x), ops.aggregate_fwd(g, y), ops.aggregate_fwd(g, 2.0 * x + y)
    torch.testing.assert_close(Hxy, 2.0 * Hx + Hy, rtol=1e-4, atol=1e-4)
    cnt = (g.rowptr[1:] - g.rowptr[:-1]).view(N, R).double()
    for r in range(R):
        lhs = (Hx[:, r * d:(r + 1) * d].double() * cnt[:, r:r + 1]).sum(0)
        rhs = x[ei[0][et == r]].double().sum(0)
        torch.testing.assert_close(lhs, rhs, rtol=1e-6, atol=1e-3)
    gA = torch.randn(N, (R + 1) * d, device=DEV)
    gA[:, R * d:] = 0
    gx = ops.aggregate_bwd(g, gA, d, init=gA[:, R * d:])
    torch.testing.assert_close((Hx.double() * gA[:, : R * d].double()).sum(), (x.double() * gx.double()).sum(),
                               rtol=1e-6, atol=1e-2)


@pytest.mark.parametrize("flat", [False, True])
def test_graphed_step_matches_eager(pkg, flat):
    """GraphedTrainStep replays the same kernels: loss and every gradient equal the eager step bit for bit
    (dropout off so both draw nothing), and a second batch through the static buffers works."""
    g = load_golden("small_full")
    m = _product_model(pkg, g)
    m.train()
    ei, et = g["edge_index"].to(DEV), g["edge_type"].to(DEV)
    b = [g[k].to(DEV) for k in ("heads", "tails", "rels", "labels")]
    def eager():
        # in its own scope: a live autograd graph would keep the parameters' AccumulateGrad nodes bound to the
        # default stream, which a later capture on another stream may not depend on
        m.zero_grad()
        loss = F.binary_cross_entropy_with_logits(m(ei, et, b[0], b[1], b[2]), b[3])
        loss.backward()
        return loss.detach().clone(), {k: p.grad.clone() for k, p in m.named_parameters()}

    want_loss, want = eager()
    step = pkg.GraphedTrainStep(m, ei, et, batch_size=b[0].numel(), flat_grads=flat)
    assert (step.flat_grad is not None) == flat
    got_loss = step(*b).clone()
    torch.testing.assert_close(got_loss, want_loss, rtol=1e-6, atol=1e-7)
    for k, p in m.named_parameters():
        if "node_embeddings" in k or "relation" in k:      # decoder scatter uses fp32 atomics on repeated nodes
            torch.testing.assert_close(p.grad, want[k], rtol=1e-4, atol=1e-6)
        else:
            torch.testing.assert_close(p.grad, want[k], rtol=1e-5, atol=1e-7)
    perm = torch.randperm(b[0].numel(), device=DEV)
    l2 = step(b[0][perm], b[1][perm], b[2][perm], b[3][perm]).clone()
    torch.testing.assert_close(l2, got_loss, rtol=1e-5, atol=1e-6)      # same pairs, permuted => same mean loss


def test_graph_state_round_trip(pkg, tmp_path):
    """CSR + CSR^T stored next to edge_index (the reference's loaders ignore extra keys) and reloaded."""
    ei, et, N, R = graphs()["primekg_100k"]
    ei, et = ei.to(DEV), et.to(DEV)
    g = pkg.RelGraph.from_edges(ei, et, N, R)
    blob = {"edge_index": ei.cpu(), "edge_type": et.cpu(), "num_nodes": N, "num_relations": R, **pkg.graph_state(g)}
    f = tmp_path / "full_graph.pt"
    torch.save(blob, f)
    back = torch.load(f)                                   # weights_only default: plain tensors / ints only
    g2 = pkg.graph_from_state(back, DEV)
    for k in ("rowptr", "col", "perm", "rowptr_t", "row_t", "perm_t", "inv_cnt", "w_t"):
        assert torch.equal(getattr(g, k), getattr(g2, k)), k
    assert (g2.fwd.n_hubs, g2.fwd.n_chunks, g2.bwd.n_hubs) == (g.fwd.n_hubs, g.fwd.n_chunks, g.bwd.n_hubs)
    from primekg_rgcn_linkprediction_b200 import ops
    x = torch.randn(N, 64, device=DEV)
    assert torch.equal(ops.aggregate_fwd(g, x), ops.aggregate_fwd(g2, x))
    pkg.clear_graph_cache()
    pkg.register_graph(ei, et, g2)
    assert pkg.get_graph(ei, et, N, R) is g2


def test_trainer_loop_like_reference(pkg):
    """The calls src/train.py makes, in its order (NegativeSampler :59-97, forward :291-297, BCEWithLogits :300,
    backward :306, clip :311-315, Adam :317-318, eval forward :389-395), on our modules: parameters move, the loss
    falls, and the first steps track the oracle trained the same way (dropout 0, same negatives)."""
    from primekg_rgcn_linkprediction_b200 import synth
    kg = synth.primekg_subgraph(60_000, seed=11)
    torch.manual_seed(0)
    model = pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, 64, 128, dropout=0.0, decoder_dropout=0.0)
    ref = O.ModelRef(kg.num_nodes, kg.num_relations, 64, 128, 0.0, 0.0)
    ref.load_state_dict(model.state_dict())
    model.to(DEV); ref.to(DEV)
    opt = torch.optim.Adam(model.parameters(), lr=1e-2)
    opt_ref = torch.optim.Adam(ref.parameters(), lr=1e-2)
    crit = torch.nn.BCEWithLogitsLoss()
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    g = torch.Generator(device=DEV).manual_seed(1)
    losses, ref_losses = [], []
    for it in range(12):
        sel = torch.randint(0, kg.num_edges, (512,), generator=g, device=DEV)
        ph, pt, pr = ei[0, sel], ei[1, sel], et[sel]
        corrupt = torch.rand(512, generator=g, device=DEV) < 0.5
        rnd = torch.randint(0, kg.num_nodes, (512,), generator=g, device=DEV)
        heads = torch.cat([ph, torch.where(corrupt, rnd, ph)])
        tails = torch.cat([pt, torch.where(~corrupt, rnd, pt)])
        rels = torch.cat([pr, pr])
        labels = torch.cat([torch.ones(512, device=DEV), torch.zeros(512, device=DEV)])
        for m, o, acc in ((model, opt, losses), (ref, opt_ref, ref_losses)):
            m.train()
            loss = crit(m(ei, et, heads, tails, rels), labels)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(m.parameters(), 1.0)
            o.step(); o.zero_grad()
            acc.append(float(loss))
    assert losses[-1] < losses[0] - 0.05, losses
    for a, b in zip(losses[:6], ref_losses[:6]):
        assert abs(a - b) < 2e-3 * max(1.0, abs(b)), (losses, ref_losses)
    model.eval()
    with torch.no_grad():
        s = model(ei, et, heads, tails, rels)
    assert torch.isfinite(s).all()


def test_cfg3_full_size_basis_forward_backward(pkg):
    """BASELINE cfg3: full-PrimeKG-shaped synthetic KG (129,375 nodes / ~8.1 M edges / 30 relations), basis
    decomposition B = 8, one layer 64 -> 256 forward + backward against the oracle run on the same device."""
    from primekg_rgcn_linkprediction_b200 import synth
    kg = synth.primekg_full()
    assert kg.num_nodes == 129_375 and kg.num_relations == 30 and kg.num_edges == 8_100_498
    torch.manual_seed(3)
    conv = pkg.RGCNConv(64, 256, 30, num_bases=8).to(DEV)
    ref = O.RGCNConvRef(64, 256, 30, num_bases=8).to(DEV)
    ref.load_state_dict(conv.state_dict())
    x = (torch.randn(kg.num_nodes, 64, device=DEV) * 0.5).requires_grad_()
    xr = x.detach().clone().requires_grad_()
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    coef = torch.randn(kg.num_nodes, 256, device=DEV)
    out = conv(x, ei, et)
    (out * coef).sum().backward()
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        want = ref(xr, ei, et)
        (want * coef).sum().backward()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    torch.testing.assert_close(out.detach(), want.detach(), rtol=1e-4, atol=1e-4 * float(want.abs().max()))
    for got, exp, name in ((x.grad, xr.grad, "x"), (conv.weight.grad, ref.weight.grad, "weight"),
                           (conv.comp.grad, ref.comp.grad, "comp"), (conv.root.grad, ref.root.grad, "root"),
                           (conv.bias.grad, ref.bias.grad, "bias")):
        rel = float((got - exp).norm() / (exp.norm() + 1e-30))
        assert rel < 1e-4, (name, rel)


def _bce_logits(kind):
    if kind == "random":
        torch.manual_seed(8)
        return torch.randn(2048, device=DEV) * 6, (torch.rand(2048, device=DEV) < 0.5).float()
    if kind == "band":
        # sigmoid(x) rounds to 0.5 in fp32 for 0 < x < ~9e-8, where x > 0 and sigmoid(x) > 0.5 disagree; labels 1, 0, 0,
        # 1, 0, 0, ... so that the two labels do not cancel in the count; then +-0, +- the smallest subnormal and +-1e4
        sweep = torch.linspace(-2e-7, 2e-7, 40_001, device=DEV)
        special = torch.tensor([0.0, -0.0, 2.0 ** -149, -(2.0 ** -149), 1e4, -1e4], device=DEV).repeat(2)
        return (torch.cat([sweep, special]),
                torch.cat([(torch.arange(sweep.numel(), device=DEV) % 3 == 0).float(),
                           torch.tensor([1.0] * 6 + [0.0] * 6, device=DEV)]))
    g = torch.Generator(device=DEV).manual_seed(9)                  # long: the single block's per-thread loop
    return (torch.randn(1_000_000, device=DEV, generator=g) * 4,
            (torch.rand(1_000_000, device=DEV, generator=g) < 0.5).float())


def test_fused_bce_matches_torch(pkg):
    """Loss, gradient and accuracy count against torch, for each set of logits of ``_bce_logits``."""
    from primekg_rgcn_linkprediction_b200 import ops
    for kind in ("random", "band", "long"):
        x, y = _bce_logits(kind)
        x.requires_grad_()
        n = x.numel()
        xr = x.detach().clone().requires_grad_()
        loss, correct = ops.bce_with_logits(x, y, with_accuracy=True)
        (loss * 3.0).backward()
        ref = F.binary_cross_entropy_with_logits(xr, y)
        (ref * 3.0).backward()
        torch.testing.assert_close(loss, ref, rtol=1e-6, atol=1e-7, msg=lambda m: f"{kind} logits: {m}")
        torch.testing.assert_close(x.grad, xr.grad, rtol=1e-5, atol=1e-9, msg=lambda m: f"{kind} logits: {m}")
        want = int(((torch.sigmoid(xr) > 0.5).float() == y).sum())                 # reference src/train.py:321-322
        assert int(correct) == want, f"{kind} logits: accuracy count {int(correct)} != {want}"
        # against float64: each thread adds n / 1024 terms in order, then two 32-wide butterflies
        x64 = x.detach().double()
        l64 = x64.clamp_min(0) - x64 * y.double() + torch.log1p(torch.exp(-x64.abs()))
        assert abs(float(loss) - float(l64.mean())) <= (n / 1024 + 40) * 2.0 ** -24 * float(l64.abs().mean()), kind


# ------------------------------------------------------------------------------------------------
# fused ReLU + dropout epilogue (reference F.relu + nn.Dropout, src/models/rgcn.py:124-125)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("p", [0.5, 0.1])
def test_fused_dropout_layer(pkg, p):
    """Train-mode layer with the dropout in the GEMM epilogue: every element is either 0 or the no-dropout value
    / (1 - p); the kept fraction is 1 - p; the gradient is the no-dropout gradient of the same masked function; a
    second call draws a different mask."""
    from primekg_rgcn_linkprediction_b200 import synth
    from primekg_rgcn_linkprediction_b200.conv import RGCNConv
    from primekg_rgcn_linkprediction_b200.graph import get_graph
    torch.manual_seed(3)
    kg = synth.uniform_kg(3000, 40_000, 3, seed=11)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    conv = RGCNConv(64, 128, 3).to(DEV)
    x = torch.randn(3000, 64, device=DEV, requires_grad=True)
    graph = get_graph(ei, et, 3000, 3)
    base = conv.forward_graph(x, graph, relu=True).detach()
    out = conv.forward_graph(x, graph, relu=True, dropout_p=p)
    kept = out != 0
    pos = base > 0
    assert not (kept & ~pos).any()                                   # nothing appears where ReLU gave 0
    frac = float((kept & pos).sum()) / float(pos.sum())
    assert abs(frac - (1 - p)) < 0.01, frac
    torch.testing.assert_close(out[kept], base[kept] / (1 - p), rtol=1e-6, atol=0)
    # backward: same as differentiating relu(z) * mask / (1 - p) with the mask held fixed
    coef = torch.randn_like(out)
    (out * coef).sum().backward()
    gx, gw = x.grad.clone(), conv.weight.grad.clone()
    x.grad = None
    conv.zero_grad()
    base2 = conv.forward_graph(x, graph, relu=True)
    (base2 * coef * kept / (1 - p)).sum().backward()
    torch.testing.assert_close(gx, x.grad, rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(gw, conv.weight.grad, rtol=1e-4, atol=1e-4)
    out2 = conv.forward_graph(x, graph, relu=True, dropout_p=p).detach()
    assert ((out2 != 0) != kept).float().mean() > 0.05              # fresh mask per call
    # columns are not correlated with rows: every column keeps about 1 - p of its positives
    col_frac = (kept & pos).float().sum(0) / pos.float().sum(0).clamp(min=1)
    assert float((col_frac - (1 - p)).abs().max()) < 0.08


def test_fused_dropout_changes_under_graph_replay(pkg):
    """The device-side dropout counter advances inside the captured graph: two replays give different masks."""
    from primekg_rgcn_linkprediction_b200 import synth
    from primekg_rgcn_linkprediction_b200.graphed import GraphedTrainStep
    torch.manual_seed(1)
    kg = synth.primekg_subgraph(20_000, seed=5)
    model = pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, 64, 128, dropout=0.5, decoder_dropout=0.0).to(DEV)
    model.train()
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    B = 256
    step = GraphedTrainStep(model, ei, et, B)
    heads = torch.randint(0, kg.num_nodes, (B,), device=DEV)
    tails = torch.randint(0, kg.num_nodes, (B,), device=DEV)
    rels = torch.randint(0, kg.num_relations, (B,), device=DEV)
    labels = (torch.rand(B, device=DEV) > 0.5).float()
    l1 = float(step(heads, tails, rels, labels))
    s1 = step.scores.clone()
    l2 = float(step(heads, tails, rels, labels))
    s2 = step.scores.clone()
    assert l1 == l1 and l2 == l2
    assert not torch.equal(s1, s2)
    model.eval()                                                      # eval: no dropout, deterministic
    with torch.no_grad():
        a = model(ei, et, heads, tails, rels)
        b = model(ei, et, heads, tails, rels)
    assert torch.equal(a, b)


@pytest.mark.parametrize("overlap", ["0", "1"])
def test_hub_rows_mixed_modes(pkg, overlap, monkeypatch):
    monkeypatch.setenv("RGCN_OVERLAP_HUBS", overlap)     # "1": hub chunks on a side stream + finish kernel (opt-in)
    _hub_rows_mixed_modes(pkg)


def _hub_rows_mixed_modes(pkg):
    """Graph where several relations of the same rows are hubs (> 128 edges) next to short segments: the row pass
    skips what needs chunk partials and the hub-row pass fills it in, for all three mixing modes."""
    from primekg_rgcn_linkprediction_b200 import ops
    from primekg_rgcn_linkprediction_b200.graph import RelGraph
    g = torch.Generator().manual_seed(7)
    N, R, E = 600, 4, 30_000
    src = torch.randint(0, N, (E,), generator=g)
    dst = torch.randint(0, N, (E,), generator=g)
    rel = torch.randint(0, R, (E,), generator=g)
    dst[: E // 2] = torch.randint(0, 5, (E // 2,), generator=g)       # rows 0..4: every relation a hub (~750 edges)
    src[E // 2: E // 2 + 4000] = 7                                     # node 7: hub in the transposed CSR
    dst[-300:] = 9
    rel[-300:] = 2                                                    # row 9: one hub relation, three short ones
    graph = RelGraph(src.to(DEV), dst.to(DEV), rel.to(DEV), N, N, R)
    assert graph.fwd.n_hubs >= 21 and graph.bwd.n_hubs >= 1
    for d in (8, 64, 256):
        x = torch.randn(N, d, generator=g)
        H = ops.aggregate_fwd(graph, x.to(DEV)).cpu()
        Href = _means_ref(x, torch.stack([src, dst]), rel, N, R)
        torch.testing.assert_close(H, Href, rtol=1e-5, atol=1e-5)
        comp = torch.randn(R, 3, generator=g)
        Z = ops.aggregate_fwd(graph, x.to(DEV), comp=comp.to(DEV)).cpu()
        Zref = torch.einsum("rb,nrd->nbd", comp, Href.reshape(N, R, d)).reshape(N, 3 * d)
        torch.testing.assert_close(Z, Zref, rtol=1e-4, atol=1e-4)
        gH = torch.randn(N, R * d, generator=g)
        init = torch.randn(N, d, generator=g)
        gx = ops.aggregate_bwd(graph, gH.to(DEV), d, init=init.to(DEV)).cpu()
        cnt = torch.bincount(dst * R + rel, minlength=N * R).clamp(min=1).float()
        contrib = gH.reshape(N, R, d)[dst, rel] / cnt[dst * R + rel][:, None]
        gref = init.clone().index_add_(0, src, contrib)
        torch.testing.assert_close(gx, gref, rtol=1e-4, atol=1e-4)
        assert torch.equal(ops.aggregate_fwd(graph, x.to(DEV)).cpu(), H)                            # same bits again


# ------------------------------------------------------------------------------------------------
# basis decomposition in the B-accumulator (Z) form
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dims", [(64, 64), (128, 64), (64, 256), (256, 256)])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_basis_z_form_layer(pkg, dims, mode, monkeypatch):
    """The Z form (relations mixed in the aggregation, K = (B+1) d_in, mirrored backward with the coefficient
    gradient as a side output) against the oracle's materialised-W_r loop, on a hub-heavy graph, with ReLU."""
    from primekg_rgcn_linkprediction_b200 import synth
    from primekg_rgcn_linkprediction_b200.conv import _RGCNBasisLayerFn  # noqa: F401  (the form under test)
    monkeypatch.setenv("PRIMEKG_RGCN_BASIS_FORM", "z")
    d_in, d_out = dims
    kg = synth.primekg_subgraph(20_000, seed=9)
    R, B = kg.num_relations, 2
    torch.manual_seed(4)
    conv = pkg.RGCNConv(d_in, d_out, R, num_bases=B, mode=mode).to(DEV)
    ref = O.RGCNConvRef(d_in, d_out, R, num_bases=B).to(DEV)
    ref.load_state_dict(conv.state_dict())
    with torch.no_grad():
        conv.bias.normal_(); ref.bias.copy_(conv.bias)
    x = (torch.randn(kg.num_nodes, d_in, device=DEV) * 0.5).requires_grad_()
    xr = x.detach().clone().requires_grad_()
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    from primekg_rgcn_linkprediction_b200.graph import get_graph
    graph = get_graph(ei, et, kg.num_nodes, R)
    assert conv._use_z_form(graph) and graph.bwd.n_hubs > 0 and graph.fwd.n_hubs > 0
    coef = torch.randn(kg.num_nodes, d_out, device=DEV)
    out = conv.forward_graph(x, graph, relu=True)
    (out * coef).sum().backward()
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        pre = ref(xr, ei, et)
        # the ReLU mask is taken from the product's output: an element within rounding distance of zero may fall on
        # either side, and one flipped element out of 10^6 already shows up at 1e-3 in the gradient norm
        want = pre * (out.detach() > 0)
        (want * coef).sum().backward()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    tol = 1e-4 if mode == "fp32" else 2e-2
    torch.testing.assert_close(out.detach(), torch.relu(pre.detach()), rtol=tol, atol=tol * float(want.abs().max()))
    for got, exp, name in ((x.grad, xr.grad, "x"), (conv.weight.grad, ref.weight.grad, "weight"),
                           (conv.comp.grad, ref.comp.grad, "comp"), (conv.root.grad, ref.root.grad, "root"),
                           (conv.bias.grad, ref.bias.grad, "bias")):
        rel = float((got - exp).norm() / (exp.norm() + 1e-30))
        assert rel < (2e-4 if mode == "fp32" else 3e-2), (name, rel)
    # deterministic
    x.grad = None
    conv.zero_grad()
    out2 = conv.forward_graph(x, graph, relu=True)
    (out2 * coef).sum().backward()
    assert torch.equal(out, out2)


def test_basis_forms_agree_r30(pkg, monkeypatch):
    """30 relations / 8 bases: the Z form and the materialised-W_r form of the same layer give the same numbers."""
    from primekg_rgcn_linkprediction_b200 import synth
    kg = synth.uniform_kg(5000, 60_000, 30, seed=2)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    torch.manual_seed(6)
    conv = pkg.RGCNConv(128, 128, 30, num_bases=8).to(DEV)
    x0 = torch.randn(5000, 128, device=DEV)
    coef = torch.randn(5000, 128, device=DEV)
    res = {}
    for form in ("w", "z"):
        monkeypatch.setenv("PRIMEKG_RGCN_BASIS_FORM", form)
        x = x0.clone().requires_grad_()
        conv.zero_grad()
        out = conv(x, ei, et)
        (out * coef).sum().backward()
        res[form] = (out.detach(), x.grad, conv.weight.grad.clone(), conv.comp.grad.clone(), conv.root.grad.clone())
    for a, b in zip(res["w"], res["z"]):
        assert float((a - b).norm() / (a.norm() + 1e-30)) < 1e-4


def test_eval_encoder_output_is_cached(pkg):
    """evaluate.py re-encodes the full graph once per batch of test edges (reference src/evaluate.py:251-254); in eval
    mode under no_grad the second call launches nothing, and any parameter change or a train-mode call recomputes."""
    from primekg_rgcn_linkprediction_b200 import _lib
    g = load_golden("small_full")
    m = _product_model(pkg, g)
    ei, et = g["edge_index"].to(DEV), g["edge_type"].to(DEV)
    lib = _lib.load()
    m.eval()
    with torch.no_grad():
        a = m.encoder(ei, et)
        n0 = lib.rgcn_launch_count()
        b = m.encoder(ei, et)
        assert lib.rgcn_launch_count() == n0 and b is a            # served from the cache
        c = m.get_embeddings(ei, et)
        assert lib.rgcn_launch_count() == n0 and torch.equal(c, a)
        m.encoder.conv1.root.mul_(1.5)                             # in-place parameter change (an optimizer step)
        d = m.encoder(ei, et)
        assert lib.rgcn_launch_count() > n0 and not torch.equal(d, a)
        n1 = lib.rgcn_launch_count()
        d.add_(1.0)                                                # a caller scribbles on the returned tensor
        e = m.encoder(ei, et)
        assert lib.rgcn_launch_count() > n1 and not torch.equal(e, d)
    n2 = lib.rgcn_launch_count()
    f = m.encoder(ei, et)                                          # autograd on: never cached
    assert lib.rgcn_launch_count() > n2 and f.requires_grad
    m.train()
    with torch.no_grad():
        n3 = lib.rgcn_launch_count()
        m.encoder(ei, et)
        assert lib.rgcn_launch_count() > n3
    # writes that bypass the version counter (p.data, raw pointers, replayed graphs) are covered by the cache's lifetime:
    # every train() / eval() switch, .to(), load_state_dict and invalidate_eval_cache() drops it
    m.eval()
    with torch.no_grad():
        a = m.encoder(ei, et)
        assert m.encoder._eval_cache is not None and m.encoder._eval_cache[1] is not None     # holds the graph itself
        m.encoder.conv2.root.data.mul_(1.25)                       # no version bump
        m.train(); m.eval()                                        # what a training epoch between two validations does
        assert m.encoder._eval_cache is None
        b = m.encoder(ei, et)
        assert not torch.equal(a, b)
        sd = {k: v.clone() for k, v in m.state_dict().items()}
        m.encoder(ei, et)
        m.load_state_dict(sd)
        assert m.encoder._eval_cache is None
        m.encoder(ei, et)
        m.encoder.invalidate_eval_cache()
        assert m.encoder._eval_cache is None
        m.encoder(ei, et)
        m.to(DEV)
        assert m.encoder._eval_cache is None


# ------------------------------------------------------------------------------------------------
# row-sparse output gradient of the last layer (csrc/rowsparse.cu)
@pytest.mark.parametrize("name", ["uniform_small", "uniform_r30", "primekg_100k", "val_fixture", "ragged"])
@pytest.mark.parametrize("d", [16, 64, 128, 256])
def test_aggregate_bwd_rows_equals_dense_bitwise(pkg, name, d):
    """gH zero outside a row list (with duplicates): the walk that skips the absent edges returns the dense walk's bits,
    hub segments included."""
    from primekg_rgcn_linkprediction_b200 import ops
    ei, et, N, R = graphs()[name]
    g = pkg.RelGraph.from_edges(ei.to(DEV), et.to(DEV), N, R)
    gen = torch.Generator().manual_seed(5)
    n_list = max(2, N // 8)
    rows = torch.randint(0, N, (n_list,), generator=gen)
    rows[1] = rows[0]                                                   # a duplicate
    if ei.numel():
        rows[2 % n_list] = int(torch.bincount(ei[1], minlength=N).argmax())   # the biggest hub is listed
    uniq = torch.unique(rows)
    m_c = (n_list + 127) // 128 * 128
    K = (R + 1) * d
    dense = torch.zeros(N, K)
    dense[uniq] = torch.randn(uniq.numel(), K, generator=gen)
    slot = torch.full((N,), m_c, dtype=torch.int32)
    compact = torch.zeros(m_c + 1, K)
    for c in range(n_list - 1, -1, -1):                                 # first position wins
        slot[rows[c]] = c
    for i in uniq.tolist():
        compact[slot[i]] = dense[i]
    dd, cd = dense.to(DEV), compact.to(DEV)
    want = ops.aggregate_bwd(g, dd, d, init=dd[:, R * d:])
    got = ops.aggregate_bwd(g, cd, d, init=cd[:, R * d:], slot=slot.to(DEV), zero_row=m_c)
    assert torch.equal(got, want)


def _step_grads(pkg, g, sparse, monkeypatch, extra_consumer=False, mode="fp32"):
    from primekg_rgcn_linkprediction_b200 import rowsparse
    monkeypatch.setenv("PRIMEKG_RGCN_SPARSE_BWD", "1" if sparse else "0")
    monkeypatch.setattr(rowsparse, "MAX_FRACTION", 1e9)      # the fixture graphs are small: list longer than N / 2
    rowsparse.clear()
    rowsparse.stats.update(claimed=0, declined=0)
    m = _product_model(pkg, g, mode)
    m.train()
    ei, et = g["edge_index"].to(DEV), g["edge_type"].to(DEV)
    if extra_consumer:
        emb = m.encoder(ei, et)
        scores = m.decoder.score_pairs(emb, g["heads"].to(DEV), g["tails"].to(DEV), g["rels"].to(DEV))
        loss = F.binary_cross_entropy_with_logits(scores, g["labels"].to(DEV)) + 1e-3 * emb.square().mean()
    else:
        scores = m(ei, et, g["heads"].to(DEV), g["tails"].to(DEV), g["rels"].to(DEV))
        loss = F.binary_cross_entropy_with_logits(scores, g["labels"].to(DEV))
    loss.backward()
    return {k: p.grad.clone() for k, p in m.named_parameters()}, dict(rowsparse.stats)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("name,d_in,d_out", [("uniform_r30", 64, 128), ("primekg_100k", 256, 256), ("val_fixture", 64, 64)])
def test_layer_bwd_rows_equals_dense(pkg, name, d_in, d_out, mode):
    """One layer's backward on a row-sparse output gradient, compact form against dense form on the SAME gO: the input
    gradient bit for bit (dgrad rows and the walk do not depend on the other rows), the weight gradients up to the
    summation order of the split-K reduction."""
    from primekg_rgcn_linkprediction_b200 import ops
    ei, et, N, R = graphs()[name]
    g = pkg.RelGraph.from_edges(ei.to(DEV), et.to(DEV), N, R)
    gen = torch.Generator().manual_seed(11)
    x = torch.randn(N, d_in, generator=gen).to(DEV)
    W = (torch.randn(R * d_in, d_out, generator=gen) / d_in ** 0.5).to(DEV)
    root = (torch.randn(d_in, d_out, generator=gen) / d_in ** 0.5).to(DEV)
    bias = torch.zeros(d_out, device=DEV)
    _, A, _wp = ops.layer_fwd(g, x, x, W, root, bias, False, mode)
    n_list = min(4096, N // 4)
    rows = torch.randint(0, N, (n_list,), generator=gen)
    rows[1::7] = rows[0]                                               # duplicates
    rows[3] = int(torch.bincount(ei[1], minlength=N).argmax())          # a hub
    gO = torch.zeros(N, d_out)
    uniq = torch.unique(rows)
    gO[uniq] = torch.randn(uniq.numel(), d_out, generator=gen)
    gO = gO.to(DEV)
    dense = ops.layer_bwd(g, gO, None, 1.0, A, W, root, d_in, mode, True, True, True, True)
    comp = ops.layer_bwd(g, gO, None, 1.0, A, W, root, d_in, mode, True, True, True, True, rows=rows.to(DEV))
    assert torch.equal(comp[0], dense[0])                               # g_x
    assert comp[1] is None
    for a, b, what in zip(comp[2:], dense[2:], ("g_weight", "g_root", "g_bias")):
        scale = float(b.abs().max()) + 1e-30
        torch.testing.assert_close(a, b, rtol=1e-4, atol=2e-5 * scale, msg=lambda s: f"{what}: {s}")
    only_x = ops.layer_bwd(g, gO, None, 1.0, A, W, root, d_in, mode, True, True, False, False, rows=rows.to(DEV))
    assert torch.equal(only_x[0], dense[0]) and only_x[2] is None


def _close_by_scale(a, b, what, rtol=1e-4, atol=2e-5):
    scale = float(b.abs().max()) + 1e-30
    torch.testing.assert_close(a, b, rtol=rtol, atol=atol * scale, msg=lambda s: f"{what}: {s}")


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_sparse_last_layer_backward_equals_dense(pkg, monkeypatch, mode):
    """The loss reads 2 * batch rows of the encoder output (reference src/models/rgcn.py:325-326): the compact backward of
    the last layer must give the dense backward's gradients."""
    g = load_golden("small_full")
    dense, st0 = _step_grads(pkg, g, False, monkeypatch, mode=mode)
    sparse, st1 = _step_grads(pkg, g, True, monkeypatch, mode=mode)
    assert st0 == {"claimed": 0, "declined": 0} and st1 == {"claimed": 1, "declined": 0}
    for k in dense:
        _close_by_scale(sparse[k], dense[k], k)
    if mode == "fp32":
        for k, want in g["grads"].items():                               # and the reference's goldens
            _close_by_scale(sparse[k].cpu(), want, k, rtol=1e-3)


def test_sparse_backward_declines_when_gradient_is_not_row_sparse(pkg, monkeypatch):
    """A second consumer of the embeddings makes autograd add a dense contribution: the announcement must not be
    honoured, and the gradients must equal those of the run with the hand-over switched off."""
    g = load_golden("small_full")
    dense, _ = _step_grads(pkg, g, False, monkeypatch, extra_consumer=True)
    guarded, st = _step_grads(pkg, g, True, monkeypatch, extra_consumer=True)
    assert st["claimed"] == 0
    for k in dense:
        _close_by_scale(guarded[k], dense[k], k)


def test_sparse_backward_full_size_cfg2(pkg, cfg2, monkeypatch):
    """cfg2 at full size (849,456 edges, hubs of 10^4 edges, 4,096 listed rows with duplicates)."""
    from primekg_rgcn_linkprediction_b200 import rowsparse
    kg, (heads, tails, rels, labels) = cfg2
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    b = [t.to(DEV) for t in (heads, tails, rels, labels)]
    res = {}
    for sparse in (False, True):
        monkeypatch.setenv("PRIMEKG_RGCN_SPARSE_BWD", "1" if sparse else "0")
        rowsparse.stats.update(claimed=0, declined=0)
        torch.manual_seed(42)
        m = pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, 64, 256, dropout=0.0, decoder_dropout=0.0).to(DEV).train()
        F.binary_cross_entropy_with_logits(m(ei, et, b[0], b[1], b[2]), b[3]).backward()
        assert rowsparse.stats["claimed"] == int(sparse)
        res[sparse] = {k: p.grad.clone() for k, p in m.named_parameters()}
    for k in res[False]:
        rel = float((res[True][k] - res[False][k]).norm() / (res[False][k].norm() + 1e-30))
        assert rel < 1e-5, f"{k}: relative Frobenius difference {rel:.3e}"


# ------------------------------------------------------------------------------------------------
# fused tail of the training step (SURVEY §8f row 2): sampler, decoder + loss + accuracy in one kernel pair
def test_link_loss_matches_unfused_step(pkg):
    """model.link_loss == model(...) -> BCEWithLogitsLoss -> sigmoid > 0.5 accuracy (reference src/train.py:291-300,
    :321-322) and the oracle's goldens; gradients equal those of the unfused step."""
    g = load_golden("small_full")
    ei, et = g["edge_index"].to(DEV), g["edge_type"].to(DEV)
    b = [g[k].to(DEV) for k in ("heads", "tails", "rels", "labels")]
    m = _product_model(pkg, g)
    m.train()
    s0 = m(ei, et, b[0], b[1], b[2])
    l0 = F.binary_cross_entropy_with_logits(s0, b[3])
    l0.backward()
    want = {k: p.grad.clone() for k, p in m.named_parameters()}
    m.zero_grad()
    loss, scores, correct = m.link_loss(ei, et, *b)
    loss.backward()
    torch.testing.assert_close(scores, s0.detach(), rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(loss.detach(), l0.detach(), rtol=1e-6, atol=1e-7)
    torch.testing.assert_close(loss.detach().cpu(), g["loss"], rtol=1e-4, atol=1e-5)
    assert int(correct) == int(((torch.sigmoid(s0) > 0.5).float() == b[3]).sum())
    for k, p in m.named_parameters():
        _close_by_scale(p.grad, want[k], k, rtol=1e-4, atol=1e-5)
    # deterministic loss: the block partials are reduced in a fixed order
    l2, _, _ = m.link_loss(ei, et, *b)
    assert torch.equal(l2.detach(), loss.detach())


def test_link_loss_dropout_mask_is_shared_by_forward_and_backward(pkg):
    """Relation dropout of reference src/models/rgcn.py:207-208 by counter-based mask.  With all-ones embeddings and
    relation table, score[p] = (kept elements of pair p) / (1 - p): the keep rate is read off the scores, and
    sum_k dL/dtable[r, k] = sum_{p: rel = r} g_p * score_p holds only if the backward regenerates the same mask."""
    from primekg_rgcn_linkprediction_b200 import ops
    n, d, R, N, p = 4096, 256, 3, 500, 0.25
    gen = torch.Generator().manual_seed(3)
    emb = torch.ones(N, d, device=DEV, requires_grad=True)
    table = torch.ones(R, d, device=DEV, requires_grad=True)
    h = torch.randint(0, N, (n,), generator=gen).to(DEV)
    t = torch.randint(0, N, (n,), generator=gen).to(DEV)
    r = torch.randint(0, R, (n,), generator=gen).to(DEV)
    y = (torch.rand(n, generator=gen) < 0.5).float().to(DEV)
    ctr = ops.rng_counter(DEV)
    loss, s, _ = ops.link_loss(emb, table, h, t, r, y, p, 1234, ctr)
    assert int(ctr) == 1
    kept = s * (1 - p) / d
    assert abs(float(kept.mean()) - (1 - p)) < 0.01 and float(kept.std()) > 0.0
    assert float((s * (1 - p) - (s * (1 - p)).round()).abs().max()) < 1e-2    # each element is 0 or 1 / (1 - p)
    loss.backward()
    g = (torch.sigmoid(s) - y) / n
    want = torch.zeros(R, device=DEV).index_add_(0, r, g * s)
    torch.testing.assert_close(table.grad.sum(1), want, rtol=1e-4, atol=1e-6)
    # next call: counter advanced => another mask
    _, s2, _ = ops.link_loss(emb, table, h, t, r, y, p, 1234, ctr)
    assert int(ctr) == 2 and not torch.equal(s2, s)
    # no dropout: plain DistMult
    _, s3, _ = ops.link_loss(emb, table, h, t, r, y, 0.0, 0, None)
    assert torch.equal(s3, torch.full_like(s3, float(d)))


def test_negative_sampler_properties(pkg):
    """Device-side NegativeSampler (reference src/train.py:59-97, :281-288): layout, labels, exactly-one-end corruption,
    range, rates; fresh draws per call and per CUDA-graph replay."""
    N, n, k = 30926, 1024, 3
    gen = torch.Generator().manual_seed(9)
    ph = torch.randint(0, N, (n,), generator=gen).to(DEV)
    pt = torch.randint(0, N, (n,), generator=gen).to(DEV)
    pr = torch.randint(0, 3, (n,), generator=gen).to(DEV)
    torch.manual_seed(0)
    smp = pkg.NegativeSampler(N, k)
    H, T, Rr, Y = smp.batch(ph, pt, pr)
    assert H.numel() == n * (1 + k) and torch.equal(H[:n], ph) and torch.equal(T[:n], pt) and torch.equal(Rr[:n], pr)
    assert torch.equal(Y, torch.cat([torch.ones(n), torch.zeros(n * k)]).to(DEV))
    rh, rt = ph.repeat_interleave(k), pt.repeat_interleave(k)
    assert torch.equal(Rr[n:], pr.repeat_interleave(k))
    keep_h, keep_t = H[n:] == rh, T[n:] == rt
    assert bool((keep_h | keep_t).all())                               # never both ends replaced
    assert int(H.min()) >= 0 and int(H.max()) < N and int(T.min()) >= 0 and int(T.max()) < N
    frac_head = float((~keep_h).float().mean())
    assert 0.45 < frac_head < 0.55
    ent = torch.where(~keep_h, H[n:], T[n:]).double()
    assert abs(float(ent.mean()) / N - 0.5) < 0.03 and float(ent.std()) / N > 0.25
    nh, nt, nr = smp.sample(ph, pt, pr)                                # reference interface, next counter value
    assert nh.numel() == n * k and not torch.equal(nh, H[n:])
    # graph replay draws fresh negatives
    out = tuple(torch.empty_like(x) for x in (H, T, Rr, Y))
    smp.batch(ph, pt, pr, out=out)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            smp.batch(ph, pt, pr, out=out)
    torch.cuda.current_stream().wait_stream(side)
    gr.replay(); a = out[0].clone()
    gr.replay(); b2 = out[0].clone()
    assert not torch.equal(a, b2)


def test_graphed_step_uses_fused_loss_and_reports_accuracy(pkg):
    g = load_golden("small_full")
    m = _product_model(pkg, g)
    m.train()
    ei, et = g["edge_index"].to(DEV), g["edge_type"].to(DEV)
    b = [g[k].to(DEV) for k in ("heads", "tails", "rels", "labels")]
    step = pkg.GraphedTrainStep(m, ei, et, batch_size=b[0].numel())
    assert step.fused_loss
    loss = step(*b)
    torch.testing.assert_close(loss.cpu(), g["loss"], rtol=1e-4, atol=1e-5)
    assert int(step.correct) == int(((g["scores"] > 0).float() == g["labels"]).sum())


# ------------------------------------------------------------------------------------------------
# cross-layer hand-over: the backward walk writes the upstream layer's masked G planes itself
@pytest.mark.parametrize("name,d", [("primekg_100k", 256), ("uniform_r30", 64), ("val_fixture", 128), ("ragged", 16)])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("slot_form", [False, True])
def test_walk_writes_masked_planes(pkg, name, d, mode, slot_form):
    """Second output of rgcn_aggregate_bwd[_rows] == rgcn_split_planes(gX, relu_mask, scale) on the walk's own result:
    planes bit for bit, column sums up to the order of the partial rows."""
    from primekg_rgcn_linkprediction_b200 import ops
    ei, et, N, R = graphs()[name]
    g = pkg.RelGraph.from_edges(ei.to(DEV), et.to(DEV), N, R)
    gen = torch.Generator().manual_seed(21)
    K = (R + 1) * d
    mask = (torch.randn(N, d, generator=gen).clamp_min(0.0)).to(DEV)            # ~half zeros, like a ReLU output
    scale = 1.0 / (1.0 - 0.3)
    kw = {}
    if slot_form:
        n_list = max(2, N // 6)
        rows = torch.randint(0, N, (n_list,), generator=gen)
        m_c = (n_list + 127) // 128 * 128
        slot = torch.full((N,), m_c, dtype=torch.int32)
        for c in range(n_list - 1, -1, -1):
            slot[rows[c]] = c
        gA = torch.zeros(m_c + 1, K)
        uniq = torch.unique(rows)
        gA[slot[uniq].long()] = torch.randn(uniq.numel(), K, generator=gen)
        kw = dict(slot=slot.to(DEV), zero_row=m_c)
    else:
        gA = torch.randn(N, K, generator=gen)
    gA = gA.to(DEV)
    planes = ops.alloc_planes(N, d, mode, DEV)
    ncs = torch.empty(int(pkg._lib.load().rgcn_aggregate_row_blocks(g.bwd.ref, d)) or 1, d, device=DEV)
    gx = ops.aggregate_bwd(g, gA, d, init=gA[:, R * d:], masked=(mask, scale, planes, ncs), **kw)
    want_gx = ops.aggregate_bwd(g, gA, d, init=gA[:, R * d:], **kw)
    assert torch.equal(gx, want_gx)
    ref = ops.alloc_planes(N, d, mode, DEV)
    cs = ops.split_planes(gx, ref, relu_mask=mask, colsum=True, mask_scale=scale)
    assert torch.equal(planes[0], ref[0])
    if mode == "fp32":
        assert torch.equal(planes[1], ref[1])
    a, b = ncs.sum(0), cs.sum(0)
    torch.testing.assert_close(a, b, rtol=1e-4, atol=1e-4 * float(b.abs().max() + 1e-30))


@pytest.mark.parametrize("p_drop", [0.0, 0.5])
def test_cross_layer_planes_handover_equals_separate_pass(pkg, monkeypatch, p_drop):
    """Two-layer model, training step: with the hand-overs on, layer 1's backward takes the planes layer 2's walk wrote
    (claimed == 1) and every gradient equals the run with the hand-overs off."""
    from primekg_rgcn_linkprediction_b200 import rowsparse
    g = load_golden("small_full")
    ei, et = g["edge_index"].to(DEV), g["edge_type"].to(DEV)
    b = [g[k].to(DEV) for k in ("heads", "tails", "rels", "labels")]
    res = {}
    for on in (False, True):
        monkeypatch.setenv("PRIMEKG_RGCN_SPARSE_BWD", "1" if on else "0")
        monkeypatch.setenv("PRIMEKG_RGCN_PLANES_HANDOVER", "1")          # opt-in (measured slower on cfg2)
        monkeypatch.setattr(rowsparse, "MAX_FRACTION", 1e9)
        rowsparse.clear()
        rowsparse.plane_stats.update(claimed=0, declined=0)
        torch.manual_seed(77)                                            # same dropout seed in both runs
        m = pkg.DrugDiseaseModel(g["num_nodes"], g["num_relations"], g["embedding_dim"], g["hidden_dim"], dropout=p_drop,
                                 decoder_dropout=0.0, num_bases=g["num_bases"])
        m.load_state_dict(g["state_dict"], strict=True)
        m.to(DEV).train()
        F.binary_cross_entropy_with_logits(m(ei, et, b[0], b[1], b[2]), b[3]).backward()
        assert rowsparse.plane_stats["claimed"] == int(on)
        res[on] = {k: p.grad.clone() for k, p in m.named_parameters()}
    for k in res[False]:
        _close_by_scale(res[True][k], res[False][k], k)


# ------------------------------------------------------------------------------------------------
# edge cases of the row-sparse backward and the fused step tail
@pytest.mark.parametrize("case", ["single_row", "all_duplicates", "every_node", "n_129", "isolated_rows"])
def test_layer_bwd_rows_edge_cases(pkg, case):
    """Row lists of awkward shapes: one entry, one node repeated, every node listed (nothing to skip), a length just past
    a multiple of 128, rows without any edge."""
    from primekg_rgcn_linkprediction_b200 import ops
    ei, et, N, R = graphs()["uniform_r30" if case != "isolated_rows" else "ragged"]
    d_in, d_out = 64, 128
    g = pkg.RelGraph.from_edges(ei.to(DEV), et.to(DEV), N, R)
    gen = torch.Generator().manual_seed(31)
    x = torch.randn(N, d_in, generator=gen).to(DEV)
    W = (torch.randn(R * d_in, d_out, generator=gen) / 8).to(DEV)
    root = (torch.randn(d_in, d_out, generator=gen) / 8).to(DEV)
    _, A, _wp = ops.layer_fwd(g, x, x, W, root, torch.zeros(d_out, device=DEV), False, "fp32")
    rows = {"single_row": torch.tensor([N // 2]), "all_duplicates": torch.full((300,), 7),
            "every_node": torch.randperm(N, generator=gen), "n_129": torch.randint(0, N, (129,), generator=gen),
            "isolated_rows": torch.tensor([4, 5, 7, 8, 4])}[case]
    gO = torch.zeros(N, d_out)
    uniq = torch.unique(rows)
    gO[uniq] = torch.randn(uniq.numel(), d_out, generator=gen)
    gO = gO.to(DEV)
    dense = ops.layer_bwd(g, gO, None, 1.0, A, W, root, d_in, "fp32", True, True, True, True)
    comp = ops.layer_bwd(g, gO, None, 1.0, A, W, root, d_in, "fp32", True, True, True, True, rows=rows.to(DEV))
    assert torch.equal(comp[0], dense[0])
    for a, b, what in zip(comp[2:], dense[2:], ("g_weight", "g_root", "g_bias")):
        _close_by_scale(a, b, what)


def test_sparse_backward_three_layers_and_long_lists(pkg, monkeypatch):
    """num_layers = 3 (the extension pattern of the reference's guide): only the last layer takes the compact backward;
    a row list longer than MAX_FRACTION * N falls back to the dense one.  Gradients equal the hand-over-off run."""
    from primekg_rgcn_linkprediction_b200 import rowsparse, synth
    kg = synth.uniform_kg(4000, 60_000, 5, seed=8)
    heads, tails, rels, labels = synth.link_batch(kg, 256, seed=8)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    b = [t.to(DEV) for t in (heads, tails, rels, labels)]
    res = {}
    for tag, env, frac in (("off", "0", 0.5), ("on", "1", 0.5), ("too_long", "1", 0.01)):
        monkeypatch.setenv("PRIMEKG_RGCN_SPARSE_BWD", env)
        monkeypatch.setattr(rowsparse, "MAX_FRACTION", frac)
        rowsparse.clear()
        rowsparse.stats.update(claimed=0, declined=0)
        torch.manual_seed(3)
        m = pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, 32, 64, dropout=0.0, decoder_dropout=0.0,
                                 num_layers=3).to(DEV).train()
        F.binary_cross_entropy_with_logits(m(ei, et, b[0], b[1], b[2]), b[3]).backward()
        assert rowsparse.stats == {"off": dict(claimed=0, declined=0), "on": dict(claimed=1, declined=0),
                                   "too_long": dict(claimed=0, declined=1)}[tag]
        res[tag] = {k: p.grad.clone() for k, p in m.named_parameters()}
    for tag in ("on", "too_long"):
        for k in res["off"]:
            _close_by_scale(res[tag][k], res["off"][k], f"{tag}/{k}")


def test_negative_sampler_edge_cases(pkg):
    """num_neg_samples = 0 (positives only), a single positive, and the reference's default of one negative each."""
    ph = torch.tensor([3, 1, 4], device=DEV); pt = torch.tensor([1, 5, 9], device=DEV); pr = torch.tensor([0, 1, 2], device=DEV)
    h, t, r, y = pkg.NegativeSampler(10, 0).batch(ph, pt, pr)
    assert torch.equal(h, ph) and torch.equal(t, pt) and torch.equal(r, pr) and torch.equal(y, torch.ones(3, device=DEV))
    h, t, r, y = pkg.NegativeSampler(10, 1).batch(ph[:1], pt[:1], pr[:1])
    assert h.numel() == 2 and y.tolist() == [1.0, 0.0] and int(r[1]) == 0
    assert (int(h[1]) == 3) != (int(t[1]) == 1) or (int(h[1]) == 3 and int(t[1]) == 1)   # at most one end replaced
    with pytest.raises(RuntimeError):
        pkg.NegativeSampler(10, 1).batch(ph.cpu(), pt.cpu(), pr.cpu())                    # no CPU path


def test_link_loss_rejects_bad_input(pkg):
    from primekg_rgcn_linkprediction_b200 import ops
    emb = torch.randn(10, 8, device=DEV); table = torch.randn(2, 8, device=DEV)
    idx = torch.zeros(4, dtype=torch.int64, device=DEV); y = torch.zeros(4, device=DEV)
    with pytest.raises(ValueError):
        ops.link_loss(emb, table, idx, idx[:3], idx, y)                                  # ragged batch
    with pytest.raises(ValueError):
        ops.link_loss(emb, table, idx, idx, idx, y, p_drop=0.5)                          # dropout without a counter
    with pytest.raises(RuntimeError):
        ops.link_loss(emb.cpu(), table.cpu(), idx.cpu(), idx.cpu(), idx.cpu(), y.cpu())  # no CPU path


def test_graphed_step_with_device_sampler(pkg):
    """The whole of src/train.py:276-306 as one CUDA graph: positives in, negatives drawn on the device per replay."""
    g = load_golden("small_full")
    m = _product_model(pkg, g)
    m.train()
    ei, et = g["edge_index"].to(DEV), g["edge_type"].to(DEV)
    n_pos = 16
    ph, pt, pr = ei[0, :n_pos].clone(), ei[1, :n_pos].clone(), et[:n_pos].clone()
    torch.manual_seed(1)
    smp = pkg.NegativeSampler(g["num_nodes"], 1)
    step = pkg.GraphedTrainStep(m, ei, et, batch_size=2 * n_pos, sampler=smp)
    l1 = float(step.run_positives(ph, pt, pr)); neg1 = (step.heads[n_pos:].clone(), step.tails[n_pos:].clone())
    l2 = float(step.run_positives(ph, pt, pr)); neg2 = (step.heads[n_pos:].clone(), step.tails[n_pos:].clone())
    assert torch.equal(step.heads[:n_pos], ph) and torch.equal(step.labels, torch.cat([torch.ones(n_pos), torch.zeros(n_pos)]).to(DEV))
    assert not (torch.equal(neg1[0], neg2[0]) and torch.equal(neg1[1], neg2[1]))            # fresh negatives per replay
    assert l1 == l1 and l2 == l2 and all(p.grad is not None and torch.isfinite(p.grad).all() for p in m.parameters())
    # the replayed step equals the eager step on the batch it drew
    want = F.binary_cross_entropy_with_logits(m(ei, et, step.heads, step.tails, step.rels), step.labels)
    torch.testing.assert_close(torch.tensor(l2), want.detach().cpu(), rtol=1e-5, atol=1e-6)
    with pytest.raises(RuntimeError):
        step(ph, pt, pr, step.labels)


def test_graphed_step_grad_arena(pkg):
    """flat_grads="arena": every parameter gradient is a slice of one flat buffer (what a data-parallel caller
    all-reduces in one call) and equals the plain graphed step's gradient."""
    g = load_golden("small_full")
    ei, et = g["edge_index"].to(DEV), g["edge_type"].to(DEV)
    b = [g[k].to(DEV) for k in ("heads", "tails", "rels", "labels")]
    m = _product_model(pkg, g)
    m.train()
    plain = pkg.GraphedTrainStep(m, ei, et, batch_size=b[0].numel())
    plain(*b)
    want = {k: p.grad.clone() for k, p in m.named_parameters()}
    step = pkg.GraphedTrainStep(m, ei, et, batch_size=b[0].numel(), flat_grads="arena")
    assert step.flat_grad is not None
    loss = step(*b)
    torch.testing.assert_close(loss.cpu(), g["loss"], rtol=1e-4, atol=1e-5)
    lo, hi = step.flat_grad.data_ptr(), step.flat_grad.data_ptr() + step.flat_grad.numel() * 4
    for k, p in m.named_parameters():
        assert lo <= p.grad.data_ptr() < hi, k
        _close_by_scale(p.grad, want[k], k, rtol=1e-4, atol=1e-5)
    # an in-place all-reduce stand-in on the flat tensor is seen by every p.grad
    before = m.encoder.conv1.root.grad.clone()
    step.flat_grad.mul_(2.0)
    assert torch.equal(m.encoder.conv1.root.grad, before * 2.0)
    # basis layers: autograd assembles weight / comp gradients itself -> no flat tensor, ordinary gradients
    gb = load_golden("small_basis")
    mb = _product_model(pkg, gb)
    mb.train()
    sb = pkg.GraphedTrainStep(mb, gb["edge_index"].to(DEV), gb["edge_type"].to(DEV), batch_size=gb["heads"].numel(),
                              flat_grads="arena")
    sb(*[gb[k].to(DEV) for k in ("heads", "tails", "rels", "labels")])
    assert sb.flat_grad is None and all(p.grad is not None for p in mb.parameters())


@pytest.mark.parametrize("R,B,din,dout", [(30, 8, 64, 256), (3, 2, 16, 8), (7, 16, 12, 20), (64, 1, 4, 4)])
def test_basis_combine_matches_matmul(pkg, R, B, din, dout):
    """W_r = sum_b comp[r, b] V_b (PyG: (comp @ weight.view(B, -1)).view(R, in, out)) and its backward on our kernels
    against the fp64 matmul and autograd; deterministic."""
    from primekg_rgcn_linkprediction_b200 import ops
    gen = torch.Generator().manual_seed(17)
    comp = torch.randn(R, B, generator=gen).to(DEV).requires_grad_()
    V = torch.randn(B, din, dout, generator=gen).to(DEV).requires_grad_()
    coef = torch.randn(R, din, dout, generator=gen).to(DEV)
    W = ops.basis_combine(comp, V)
    (W * coef).sum().backward()
    c64, v64 = comp.detach().double().requires_grad_(), V.detach().double().requires_grad_()
    W64 = (c64 @ v64.view(B, -1)).view(R, din, dout)
    (W64 * coef.double()).sum().backward()
    torch.testing.assert_close(W.detach(), W64.detach().float(), rtol=1e-5, atol=1e-5)
    _close_by_scale(comp.grad, c64.grad.float(), "g_comp", rtol=1e-4, atol=1e-5)
    _close_by_scale(V.grad, v64.grad.float(), "g_V", rtol=1e-5, atol=1e-5)
    g1 = comp.grad.clone()
    comp.grad = None; V.grad = None
    (ops.basis_combine(comp, V) * coef).sum().backward()
    assert torch.equal(comp.grad, g1)


def test_graphed_step_packed_batch(pkg):
    """One pinned [4, B] block per step (heads, tails, rels, labels bits) == the four separate copies."""
    g = load_golden("small_full")
    m = _product_model(pkg, g)
    m.train()
    ei, et = g["edge_index"].to(DEV), g["edge_type"].to(DEV)
    b = [g[k] for k in ("heads", "tails", "rels", "labels")]
    step = pkg.GraphedTrainStep(m, ei, et, batch_size=b[0].numel())
    l_sep = step(*[t.to(DEV) for t in b]).clone()
    grads = {k: p.grad.clone() for k, p in m.named_parameters()}
    packed = pkg.GraphedTrainStep.pack_batch(*b)
    assert packed.is_pinned() and packed.shape == (4, b[0].numel())
    step.heads.zero_(); step.labels.zero_()
    l_packed = step.run_packed(packed).clone()
    assert torch.equal(step.heads.cpu(), b[0]) and torch.equal(step.labels.cpu(), b[3])
    torch.testing.assert_close(l_packed, l_sep, rtol=1e-6, atol=1e-7)
    for k, p in m.named_parameters():
        _close_by_scale(p.grad, grads[k], k, rtol=1e-4, atol=1e-5)
    with pytest.raises(ValueError):
        step.load_packed(packed[:3])


def test_graphed_step_host_io(pkg):
    """host_io=True: the batch's H2D copy and the loss's D2H copy are nodes of the captured graph."""
    g = load_golden("small_full")
    m = _product_model(pkg, g)
    m.train()
    ei, et = g["edge_index"].to(DEV), g["edge_type"].to(DEV)
    b = [g[k] for k in ("heads", "tails", "rels", "labels")]
    step = pkg.GraphedTrainStep(m, ei, et, batch_size=b[0].numel(), host_io=True)
    step.host_batch.copy_(pkg.GraphedTrainStep.pack_batch(*b, pin=False))
    out = step.replay_host()
    torch.cuda.synchronize()
    assert out is step.host_loss and out.is_pinned()
    torch.testing.assert_close(step.host_loss[0], g["loss"], rtol=1e-4, atol=1e-5)
    assert int(step.host_correct) == int(((g["scores"] > 0).float() == g["labels"]).sum())
    for k, want in g["grads"].items():
        _close_by_scale(dict(m.named_parameters())[k].grad.cpu(), want, k, rtol=1e-3)
    # another batch through the same staging block
    perm = torch.randperm(b[0].numel())
    step.host_batch.copy_(pkg.GraphedTrainStep.pack_batch(*[t[perm] for t in b], pin=False))
    step.replay_host(); torch.cuda.synchronize()
    torch.testing.assert_close(step.host_loss[0], g["loss"], rtol=1e-4, atol=1e-5)
    with pytest.raises(RuntimeError):
        pkg.GraphedTrainStep(m, ei, et, batch_size=b[0].numel()).replay_host()


# ------------------------------------------------------------------------------------------------
# pipelined layer forward: the walk of row chunk c + 1 under the transform of chunk c (csrc/layer.cu)
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("d_in,d_out,relu", [(64, 256, True), (256, 256, False), (128, 96, True)])
def test_pipelined_layer_forward_equals_sequential(pkg, mode, d_in, d_out, relu):
    """Same kernels, same per-row arithmetic, two streams: bit-identical outputs and operand planes, on the
    PrimeKG-shaped graph (hub rows, chunk-wise row order) and on a large uniform graph without a row order."""
    from primekg_rgcn_linkprediction_b200 import ops, synth
    for kg in (synth.primekg_subgraph(200_000, seed=3), synth.uniform_kg(70_000, 300_000, 5, seed=8)):
        ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
        g = pkg.RelGraph.from_edges(ei, et, kg.num_nodes, kg.num_relations)
        assert (g.fwd.row_order is None) or g.fwd.order_chunk_rows > 0
        torch.manual_seed(5)
        R = kg.num_relations
        x = torch.randn(kg.num_nodes, d_in, device=DEV)
        W = torch.randn(R * d_in, d_out, device=DEV) * 0.1
        root = torch.randn(d_in, d_out, device=DEV) * 0.1
        bias = torch.randn(d_out, device=DEV)
        outs = []
        for pipeline in (1, 2):
            ctr = ops.dropout_counter(x.device)
            drop = (0.5, 123, ctr) if relu else (0.0, 0, None)
            out, A, wp = ops.layer_fwd(g, x, x, W, root, bias, relu, mode, *drop, pipeline=pipeline)
            torch.cuda.synchronize()
            outs.append((out, A[0], A[1], wp))
        assert torch.equal(outs[0][0], outs[1][0])
        assert torch.equal(outs[0][1], outs[1][1])
        if mode == "fp32":
            assert torch.equal(outs[0][2], outs[1][2])
        if relu:
            assert 0.2 < float((outs[0][0] > 0).float().mean()) < 0.3          # ~half survive ReLU, half of those dropout


def test_chunkwise_row_order_is_a_blockwise_permutation(pkg):
    from primekg_rgcn_linkprediction_b200 import synth
    from primekg_rgcn_linkprediction_b200.graph import ORDER_CHUNK_ROWS
    kg = synth.primekg_subgraph(100_000, seed=2)
    g = pkg.RelGraph.from_edges(kg.edge_index.to(DEV), kg.edge_type.to(DEV), kg.num_nodes, kg.num_relations)
    for ori in (g.fwd, g.bwd):
        assert ori.order_chunk_rows == ORDER_CHUNK_ROWS
        order = ori.row_order.long()
        assert torch.equal(torch.sort(order).values, torch.arange(kg.num_nodes, device=DEV))
        pos = torch.arange(kg.num_nodes, device=DEV)
        assert torch.equal(order // ORDER_CHUNK_ROWS, pos // ORDER_CHUNK_ROWS)      # every block keeps its own rows
        deg = (ori.rowptr[kg.num_relations::kg.num_relations] - ori.rowptr[:-1:kg.num_relations]).long()
        d = deg[order]
        same_block = (pos[1:] // ORDER_CHUNK_ROWS) == (pos[:-1] // ORDER_CHUNK_ROWS)
        assert torch.all(d[1:][same_block] <= d[:-1][same_block])                   # decreasing edge count inside a block


# ------------------------------------------------------------------------------------------------
# bf16-transform mode: the walk gathers a bf16 copy of the features (csrc/aggregate.cu, *_bf16_kernel)
@pytest.mark.parametrize("d", [64, 128, 256, 72])
def test_bf16_feature_walk_equals_fp32_walk_over_the_same_values(pkg, d):
    """Same bf16 values, fp32 sums in the same edge order, true division, one rounding to bf16 at the end: without hub
    segments the operand plane is bit-identical to the fp32-feature walk over the up-converted copy; with hubs (other
    chunk grouping at some widths) it agrees to one bf16 ulp.  The self-loop block is the copy itself."""
    from primekg_rgcn_linkprediction_b200 import ops, synth
    for kg, exact in ((synth.uniform_kg(20_000, 150_000, 4, seed=3), True), (synth.primekg_subgraph(120_000, seed=5), False)):
        ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
        g = pkg.RelGraph.from_edges(ei, et, kg.num_nodes, kg.num_relations)
        R = kg.num_relations
        torch.manual_seed(d)
        x16 = ops.to_bf16(torch.randn(kg.num_nodes, d, device=DEV))
        x = x16.float().contiguous()
        W = torch.randn(R * d, 64, device=DEV) * 0.1
        root = torch.randn(d, 64, device=DEV) * 0.1
        bias = torch.zeros(64, device=DEV)
        _, A_ref, _ = ops.layer_fwd(g, x, x, W, root, bias, False, "bf16")
        out, A, _, out16 = ops.layer_fwd(g, x, x, W, root, bias, True, "bf16", x_bf16=x16, want_out_bf16=True)
        K = (R + 1) * d
        if exact:
            assert torch.equal(A[0][:, :K], A_ref[0][:, :K])
        else:
            torch.testing.assert_close(A[0][:, :K].float(), A_ref[0][:, :K].float(), rtol=2.0 ** -7, atol=1e-6)
            same_rows = (A[0][:, :K] == A_ref[0][:, :K]).all(1).float().mean()
            assert float(same_rows) > 0.97                                   # only rows with a hub segment may differ
        assert torch.equal(A[0][:, R * d:K], x16[:, :d])
        assert torch.equal(out16, out.to(torch.bfloat16))                    # the epilogue's bf16 copy of the output


def test_bf16_mode_hands_the_bf16_copy_from_layer_to_layer(pkg, monkeypatch):
    """Encoder in bf16 mode: layer 1 gathers a bf16 copy of the table, its epilogue leaves the bf16 copy of its output and
    layer 2 claims it; results stay within the bf16 budget of the fp32-gather form (PRIMEKG_RGCN_BF16_GATHER=0)."""
    from primekg_rgcn_linkprediction_b200 import rowsparse
    g = load_golden("small_full")
    m = _product_model(pkg, g)
    for c in (m.encoder.conv1, m.encoder.conv2):
        c.mode = "bf16"
    ei, et = g["edge_index"].to(DEV), g["edge_type"].to(DEV)
    m.train()
    claimed = []
    orig = rowsparse.claim_bf16
    monkeypatch.setattr(rowsparse, "claim_bf16", lambda x: claimed.append(orig(x)) or claimed[-1])
    a = m.encoder(ei, et)
    assert len(claimed) == 2 and claimed[0] is None and claimed[1] is not None and claimed[1].dtype == torch.bfloat16
    a.sum().backward()
    ga = m.encoder.node_embeddings.weight.grad.clone()
    monkeypatch.setenv("PRIMEKG_RGCN_BF16_GATHER", "0")
    m.zero_grad()
    b = m.encoder(ei, et)
    b.sum().backward()
    scale = float(b.abs().max())
    torch.testing.assert_close(a, b, rtol=2e-2, atol=2e-2 * scale)
    gb = m.encoder.node_embeddings.weight.grad
    assert float((ga - gb).norm() / gb.norm()) < 2e-2


# ------------------------------------------------------------------------------------------------
# the unmodified training call as two captured CUDA graphs (autograph.py)
def test_training_call_graph_capture_equals_eager(pkg, monkeypatch):
    """model(...) -> BCEWithLogitsLoss -> backward() of reference src/train.py:291-306, driven eagerly: after three
    identical calls the model replays captured graphs.  Same kernels => the same scores and gradients as a twin model
    that stays eager (dropout off so the two draw nothing), on batches that change every step."""
    from primekg_rgcn_linkprediction_b200 import autograph, synth
    kg = synth.primekg_subgraph(120_000, seed=5)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    torch.manual_seed(3)
    twins = []
    for _ in range(2):
        torch.manual_seed(3)
        twins.append(pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, embedding_dim=64, hidden_dim=128, dropout=0.0,
                                          decoder_dropout=0.0).to(DEV).train())
    graphed, eager = twins
    alive = {}                       # the previous step's scores and loss stay referenced while the next call runs, as
    for step in range(8):            # the variables of the reference's for-loop do (src/train.py:291-306)
        h, t, r, y = [x.to(DEV) for x in synth.link_batch(kg, 256, seed=100 + step)]
        outs = []
        for m, on in ((graphed, "1"), (eager, "0")):
            monkeypatch.setenv("PRIMEKG_RGCN_AUTOGRAPH", on)
            for p in m.parameters():
                p.grad = None
            s = m(ei, et, h, t, r)
            loss = torch.nn.functional.binary_cross_entropy_with_logits(s, y)
            loss.backward()
            alive[on] = (s, loss)
            outs.append((s.detach().clone(), [p.grad.clone() for p in m.parameters()]))
        (s1, g1), (s0, g0) = outs
        assert torch.equal(s1, s0), step
        for a, b in zip(g1, g0):
            torch.testing.assert_close(a, b, rtol=1e-6, atol=1e-7 * float(b.abs().max()) + 1e-12)
    state = graphed.__dict__["_autograph"]
    assert any(e[1] is not None for e in state.values())              # the capture happened
    assert "_autograph" not in eager.__dict__ or all(e[1] is None for e in eager.__dict__["_autograph"].values())
    # eval-mode and no-grad calls stay eager and see the current parameters
    graphed.eval()
    with torch.no_grad():
        torch.testing.assert_close(graphed(ei, et, h, t, r), eager.eval()(ei, et, h, t, r))
    graphed.invalidate_graphs()
    assert "_autograph" not in graphed.__dict__

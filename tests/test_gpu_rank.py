"""GPU tests of the all-pairs scoring / ranking kernels against the oracle (reference src/models/rgcn.py:234-241,
src/evaluate.py:260-276, src/compare_methods.py:384-397)."""
import pytest
import torch

from oracle import rgcn_ref as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def pkg(lib_built):
    return lib_built


@pytest.mark.parametrize("N,d,B", [(1000, 128, 77), (30926, 128, 1024), (513, 24, 5)])
def test_score_all_tails_matches_oracle(pkg, N, d, B):
    torch.manual_seed(0)
    R = 3
    dec = pkg.LinkPredictor(R, d).to(DEV)
    ref = O.DecoderRef(R, d)
    ref.load_state_dict(dec.state_dict())
    emb = torch.randn(N, d)
    heads = torch.randint(0, N, (B,))
    rels = torch.randint(0, R, (B,))
    with torch.no_grad():
        got = dec.score_all_tails(emb.to(DEV)[heads.to(DEV)], rels.to(DEV), emb.to(DEV)).cpu()
        want = ref.score_all_tails(emb[heads], rels, emb)
    assert got.shape == (B, N)
    torch.testing.assert_close(got, want, rtol=1e-4, atol=1e-4 * float(want.abs().max()))


def test_score_all_tails_backward(pkg):
    torch.manual_seed(1)
    N, d, B, R = 200, 32, 9, 3
    dec = pkg.LinkPredictor(R, d).to(DEV)
    ref = O.DecoderRef(R, d)
    ref.load_state_dict(dec.state_dict())
    h, T = torch.randn(B, d, requires_grad=True), torch.randn(N, d, requires_grad=True)
    rels = torch.randint(0, R, (B,))
    hd, Td = h.detach().to(DEV).requires_grad_(), T.detach().to(DEV).requires_grad_()
    coef = torch.randn(B, N)
    (dec.score_all_tails(hd, rels.to(DEV), Td) * coef.to(DEV)).sum().backward()
    (ref.score_all_tails(h, rels, T) * coef).sum().backward()
    torch.testing.assert_close(hd.grad.cpu(), h.grad, rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(Td.grad.cpu(), T.grad, rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(dec.relation_embeddings.weight.grad.cpu(), ref.relation_embeddings.weight.grad,
                               rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("method", ["tc", "tc_block", "simt"])
@pytest.mark.parametrize("N,d,B", [(30926, 128, 1024), (777, 64, 130), (30926, 256, 2500)])
def test_rank_true_tails_brackets_reference_rank(pkg, N, d, B, method):
    """rank = 1 + #greater must lie inside the oracle's [optimistic, pessimistic] bracket evaluated with an epsilon
    band (two fp32 summation orders), and equal the exact count computed from our own score matrix."""
    torch.manual_seed(2)
    R = 3
    emb = torch.randn(N, d, device=DEV)
    table = torch.randn(R, d, device=DEV)
    heads = torch.randint(0, N, (B,), device=DEV)
    tails = torch.randint(0, N, (B,), device=DEV)
    rels = torch.randint(0, R, (B,), device=DEV)
    emb[5] = emb[9]                                   # an exact duplicate entity => exact score ties
    tails[0] = 5
    rank, ties = pkg.rank_true_tails(emb, table, heads, rels, tails, method=method)
    scores = O.distmult_allpairs_ref(emb.double(), heads, torch.arange(N, device=DEV), table[rels].double())
    s_true = scores.gather(1, tails.view(-1, 1))
    eps = 1e-4 * scores.abs().max()
    lo = (scores > s_true + eps).sum(1) + 1
    hi = (scores >= s_true - eps).sum(1)
    assert torch.all((rank >= lo) & (rank <= hi))
    assert torch.all(rank + ties <= hi)                  # rank .. rank + ties is the reference's (unstable argsort) range
    assert int(ties[0]) >= 1                          # the duplicate of the true tail is an exact tie
    # exactness against our own fp32 scores
    from primekg_rgcn_linkprediction_b200.rank import _prep, scores_from_rows
    S = scores_from_rows(_prep(emb, heads, table, rels, False), emb, method="simt" if method == "simt" else "tc")
    st = S.gather(1, tails.view(-1, 1))
    others = torch.ones_like(S, dtype=torch.bool)
    others.scatter_(1, tails.view(-1, 1), False)
    assert torch.equal(rank, ((S > st) & others).sum(1) + 1)
    assert torch.equal(ties, ((S == st) & others).sum(1))
    m = pkg.ranking_metrics(rank)
    assert 0 < m["mrr"] <= 1 and m["hits@100"] >= m["hits@10"]


@pytest.mark.parametrize("method", ["tc", "simt"])
def test_all_pairs_drug_disease_sweep(pkg, method):
    """BASELINE cfg4: all 6,282 x 5,593 drug-disease pairs, DistMult and cosine; on the tensor cores (three bf16 products,
    fp32 accumulation) and through the fp32 FMA tiles."""
    torch.manual_seed(3)
    emb = torch.randn(30926, 128, device=DEV)
    drugs = torch.arange(5593, 11875, device=DEV)
    diseases = torch.arange(0, 5593, device=DEV)
    rel = torch.randn(128, device=DEV)
    got = pkg.score_all_pairs(emb, drugs, diseases, rel_vec=rel, method=method)
    want = O.distmult_allpairs_ref(emb, drugs, diseases, rel)
    assert got.shape == (6282, 5593)
    torch.testing.assert_close(got, want, rtol=1e-4, atol=1e-4 * float(want.abs().max()))
    gotc = pkg.score_all_pairs(emb, drugs, diseases, cosine=True, method=method)
    wantc = O.cosine_allpairs_ref(emb, drugs, diseases)
    torch.testing.assert_close(gotc, wantc, rtol=1e-5, atol=1e-5 if method == "simt" else 2e-5)


# (queries, candidates): BASELINE cfg4 (5,593 diseases x 6,282 drugs), then few queries against many candidates, where a
# row receives a partial list from every CTA run over its row tile (up to 2 (#SMs + 1) lists), and fewer candidates than k
TOPK_SHAPES = [(5593, 6282), (1, 1025), (100, 5593), (128, 30926), (1000, 30926), (2048, 30926), (7, 5)]


@pytest.mark.parametrize("nq,ncand", TOPK_SHAPES)
@pytest.mark.parametrize("cosine", [False, True])
@pytest.mark.parametrize("k", [1, 10, 16])
def test_fused_topk_matches_sorted_score_matrix(pkg, cosine, k, nq, ncand):
    """``topk_all_pairs`` (score block consumed in the GEMM epilogue) against a sort of the materialised tensor-core score
    matrix: same values bit for bit, same candidates, ties broken by the lower position; missing entries (fewer
    candidates than k) are -inf / -1."""
    torch.manual_seed(4)
    emb = torch.randn(30926, 128, device=DEV)
    c0 = 5593 if ncand == 6282 else 0
    queries = torch.arange(nq, device=DEV) + (0 if c0 else 30926 - nq)
    cands = torch.arange(c0, c0 + ncand, device=DEV)
    if ncand >= 3:
        emb[cands[2 * ncand // 3]] = emb[cands[ncand // 3]]          # duplicate candidates => exact ties
    rel = torch.randn(128, device=DEV)
    kw = dict(cosine=True) if cosine else dict(rel_vec=rel)
    val, ids = pkg.topk_all_pairs(emb, queries, cands, k=k, **kw)
    S = pkg.score_all_pairs(emb, queries, cands, **kw)
    assert val.shape == (nq, k) and ids.shape == (nq, k)
    # reference order: value descending, position ascending; entries beyond the candidate count are -inf / -1
    kk = min(k, ncand)
    order = torch.argsort(S, dim=1, descending=True, stable=True)[:, :kk]
    want_val = torch.full((nq, k), float("-inf"), device=DEV)
    want_ids = torch.full((nq, k), -1, dtype=torch.int64, device=DEV)
    want_val[:, :kk] = S.gather(1, order)
    want_ids[:, :kk] = cands[order]
    assert torch.equal(ids[:, kk:], want_ids[:, kk:]) and torch.equal(val[:, kk:], want_val[:, kk:])
    if kk > 1:
        assert torch.all(val[:, :kk - 1] >= val[:, 1:kk])
    if not cosine:
        # DistMult: the sweep and the matrix are the same products in the same order => the same bits, and exact ties
        # (the duplicated candidate) are broken like the stable sort: lower position first
        assert torch.equal(val, want_val)
        assert torch.equal(ids, want_ids)
    else:
        # cosine: the matrix folds (s + 1) / 2 into the contraction, the fused form applies it to the accumulator
        torch.testing.assert_close(val[:, :kk], want_val[:, :kk], rtol=0, atol=2e-6)
        pos = ids[:, :kk] - c0
        assert bool(((pos >= 0) & (pos < ncand)).all())
        torch.testing.assert_close(S.gather(1, pos), val[:, :kk], rtol=0, atol=2e-6)   # the candidates carry these scores
        assert bool((pos.sort(1).values[:, 1:] != pos.sort(1).values[:, :-1]).all()) if kk > 1 else True


def test_fused_rank_matches_block_rank_at_evaluate_size(pkg):
    """The ranking evaluation of src/evaluate.py:219-291 at its real size (15,372 test edges x 30,926 entities, d = 256):
    counts taken in the epilogue == counts from materialised 2,048-query score blocks."""
    torch.manual_seed(6)
    N, d, nq = 30926, 256, 15372
    emb = torch.randn(N, d, device=DEV)
    table = torch.randn(3, d, device=DEV)
    heads = torch.randint(0, N, (nq,), device=DEV)
    tails = torch.randint(0, N, (nq,), device=DEV)
    rels = torch.randint(0, 3, (nq,), device=DEV)
    r1, t1 = pkg.rank_true_tails(emb, table, heads, rels, tails, method="tc")
    r2, t2 = pkg.rank_true_tails(emb, table, heads, rels, tails, method="tc_block")
    assert torch.equal(r1, r2) and torch.equal(t1, t2)
    cand = torch.arange(5593, 11875, device=DEV)
    tpos = torch.randint(0, cand.numel(), (500,), device=DEV)
    r3, t3 = pkg.rank_true_tails(emb, table, heads[:500], rels[:500], tpos, candidates=cand, method="tc")
    r4, t4 = pkg.rank_true_tails(emb, table, heads[:500], rels[:500], tpos, candidates=cand, method="tc_block")
    assert torch.equal(r3, r4) and torch.equal(t3, t4)

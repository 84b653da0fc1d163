"""GPU tests of filtered ranking and known-link exclusion (``rank_true_tails(filter=)``, ``topk_all_pairs(exclude=)``).

Every method's filtered counts must equal the count taken from that method's OWN materialised score matrix with the known
set masked out (the tc matrix for ``tc`` / ``tc_block``, the fp32 FMA matrix for ``simt``): the filter takes excluded
columns out of the very bits the sweep computes.  The masks here are built independently of ``KnownTriples``: a dense
[queries, nodes] bit matrix scattered from the raw triples."""
import pytest
import torch

from oracle import rgcn_ref as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
METHODS = ["tc", "tc_block", "simt"]


@pytest.fixture(scope="module")
def pkg(lib_built):
    return lib_built


def known_mask(h, r, t, qh, qr, num_nodes, R, cand=None):
    """[nq, num_nodes] (or [nq, len(cand)]) bool: True where (qh[i], qr[i], column) is one of the triples (h, r, t)."""
    qk = qh * R + qr
    uq, inv = torch.unique(qk, return_inverse=True)
    tk = h * R + r
    idx = torch.searchsorted(uq, tk).clamp(max=uq.numel() - 1)
    hit = uq[idx] == tk
    M = torch.zeros(uq.numel(), num_nodes, dtype=torch.bool, device=DEV)
    M[idx[hit], t[hit]] = True
    m = M[inv]
    return m if cand is None else m[:, cand]


def own_scores(emb, table, heads, rels, method, cand=None):
    from primekg_rgcn_linkprediction_b200.rank import _prep, scores_from_rows
    return scores_from_rows(_prep(emb, heads, table, rels, False), emb, b_idx=cand,
                            method="simt" if method == "simt" else "tc")


def masked_counts(S, tails, mask):
    """(rank, ties) over the columns that are neither the true tail nor masked."""
    st = S.gather(1, tails.view(-1, 1))
    keep = ~mask
    keep.scatter_(1, tails.view(-1, 1), False)
    return ((S > st) & keep).sum(1) + 1, ((S == st) & keep).sum(1)


def check_method(pkg, emb, table, heads, rels, tails, known, triples, method, cand=None):
    """Filtered (rank, ties) == the masked count of the method's own matrix; returns (rank, ties, S, mask)."""
    h, r, t = triples
    rank, ties = pkg.rank_true_tails(emb, table, heads, rels, tails, candidates=cand, method=method, filter=known)
    S = own_scores(emb, table, heads, rels, method, cand)
    mask = known_mask(h, r, t, heads, rels, emb.size(0), table.size(0), cand)
    want_r, want_t = masked_counts(S, tails, mask)
    assert torch.equal(rank, want_r), f"{method}: {int((rank != want_r).sum())} ranks differ"
    assert torch.equal(ties, want_t), f"{method}: {int((ties != want_t).sum())} tie counts differ"
    return rank, ties, S, mask


@pytest.fixture(scope="module")
def evaluate_case(pkg):
    """The ranking evaluation at its real size: 15,372 queries drawn as edges of the cfg2 graph, all 30,926 entities,
    d = 256, the whole graph as the filter (hub (head, relation) keys hold thousands of known tails)."""
    from primekg_rgcn_linkprediction_b200 import synth
    kg = synth.primekg_subgraph()
    g = torch.Generator().manual_seed(11)
    sel = torch.randperm(kg.num_edges, generator=g)[:15372]
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    heads, tails, rels = ei[0, sel.to(DEV)], ei[1, sel.to(DEV)], et[sel.to(DEV)]
    torch.manual_seed(12)
    emb = torch.randn(kg.num_nodes, 256, device=DEV)
    table = torch.randn(kg.num_relations, 256, device=DEV)
    known = pkg.KnownTriples.from_graphs(kg.as_dict(), device=DEV)
    return dict(emb=emb, table=table, heads=heads, rels=rels, tails=tails, known=known, triples=(ei[0], et, ei[1]))


@pytest.mark.parametrize("method", METHODS)
def test_filtered_rank_at_evaluate_size(pkg, evaluate_case, method):
    c = evaluate_case
    args = (c["emb"], c["table"], c["heads"], c["rels"], c["tails"])
    rank, ties, S, mask = check_method(pkg, *args, c["known"], c["triples"], method)
    raw_r, raw_t = pkg.rank_true_tails(*args, method=method)
    assert torch.all(rank <= raw_r)
    # raw - filtered = the known other tails scoring strictly above the threshold
    st = S.gather(1, c["tails"].view(-1, 1))
    others = mask.clone()
    others.scatter_(1, c["tails"].view(-1, 1), False)
    assert torch.equal(raw_r - rank, ((S > st) & others).sum(1))
    assert torch.equal(raw_t - ties, ((S == st) & others).sum(1))
    assert int((raw_r - rank).max()) > 1000                 # hub keys: the raw protocol's bias is large on this graph
    r2, t2 = pkg.rank_true_tails(*args, method=method, filter=c["known"])
    assert torch.equal(rank, r2) and torch.equal(ties, t2)   # deterministic


def test_filtered_rank_lies_in_the_oracle_bracket(pkg, evaluate_case):
    """fp64 oracle with the known set masked, the epsilon band of test_rank_true_tails_brackets_reference_rank."""
    c = evaluate_case
    emb, heads, rels, tails = c["emb"], c["heads"], c["rels"], c["tails"]
    rank, ties = pkg.rank_true_tails(emb, c["table"], heads, rels, tails, filter=c["known"])
    N = emb.size(0)
    for q0 in range(0, heads.numel(), 4096):
        q = slice(q0, q0 + 4096)
        scores = O.distmult_allpairs_ref(emb.double(), heads[q], torch.arange(N, device=DEV), c["table"][rels[q]].double())
        mask = known_mask(*c["triples"], heads[q], rels[q], N, c["table"].size(0))
        keep = ~mask
        keep.scatter_(1, tails[q].view(-1, 1), True)          # the true tail itself is in the bracket's count
        s_true = scores.gather(1, tails[q].view(-1, 1))
        eps = 1e-4 * scores.abs().max()
        lo = ((scores > s_true + eps) & keep).sum(1) + 1
        hi = ((scores >= s_true - eps) & keep).sum(1)
        assert torch.all((rank[q] >= lo) & (rank[q] <= hi))
        assert torch.all(rank[q] + ties[q] <= hi)


def _random_case(N, d, B, R=3, n_known=4000, seed=0, n_other=200):
    torch.manual_seed(seed)
    emb = torch.randn(N, d, device=DEV)
    table = torch.randn(R, d, device=DEV)
    heads = torch.randint(0, N, (B,), device=DEV)
    rels = torch.randint(0, R, (B,), device=DEV)
    tails = torch.randint(0, N, (B,), device=DEV)
    # known triples: around the queries' own keys (heavy lists), plus unrelated ones; half the queries keep empty lists
    qi = torch.randint(0, B // 2 + 1, (n_known,), device=DEV)
    h = torch.cat([heads[qi], torch.randint(0, N, (n_other,), device=DEV)])
    r = torch.cat([rels[qi], torch.randint(0, R, (n_other,), device=DEV)])
    t = torch.randint(0, N, (h.numel(),), device=DEV)
    return emb, table, heads, rels, tails, (h, r, t)


@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("N,d,B", [(777, 64, 130), (1025, 32, 1), (5593, 128, 100), (30926, 128, 300)])
def test_filtered_rank_matches_masked_own_matrix(pkg, method, N, d, B):
    """Small and few-query shapes: 1 x 1,025 and 100 x 5,593 put many CTA runs on one row tile, so runs start mid-row
    and the cursor starts at a lower bound inside the list."""
    emb, table, heads, rels, tails, tri = _random_case(N, d, B, n_known=min(N * (B // 2 + 1) // 3, 60000), seed=N + B)
    known = pkg.KnownTriples(*tri, N, 3)
    rank, ties, S, mask = check_method(pkg, emb, table, heads, rels, tails, known, tri, method)
    raw_r, raw_t = pkg.rank_true_tails(emb, table, heads, rels, tails, method=method)
    empty = ~mask.any(1)
    assert torch.equal(rank[empty], raw_r[empty]) and torch.equal(ties[empty], raw_t[empty])
    if B > 1:
        assert bool(empty.any()) and bool((~empty).any())


@pytest.mark.parametrize("method", METHODS)
def test_filter_none_and_empty_filter_are_the_raw_call(pkg, method):
    emb, table, heads, rels, tails, _ = _random_case(30926, 128, 1024, seed=5)
    emb[5] = emb[9]
    tails[0] = 5                                     # an exact tie
    raw = pkg.rank_true_tails(emb, table, heads, rels, tails, method=method)
    none = pkg.rank_true_tails(emb, table, heads, rels, tails, method=method, filter=None)
    z = torch.zeros(0, dtype=torch.int64, device=DEV)
    empty = pkg.KnownTriples(z, z, z, 30926, 3)
    assert len(empty) == 0
    filt = pkg.rank_true_tails(emb, table, heads, rels, tails, method=method, filter=empty)
    for a, b in ((raw, none), (raw, filt)):
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert int(raw[1][0]) >= 1


@pytest.mark.parametrize("method", METHODS)
def test_candidates_subset_with_filter_outside_it(pkg, method):
    """Candidates = the drug block; the filter names nodes inside and outside it (those outside are ignored)."""
    emb, table, heads, rels, _, (h, r, t) = _random_case(30926, 128, 700, n_known=40000, seed=7)
    cand = torch.arange(5593, 11875, device=DEV)
    tpos = torch.randint(0, cand.numel(), (700,), device=DEV)
    known = pkg.KnownTriples(h, r, t, 30926, 3)
    assert bool(((t < 5593) | (t >= 11875)).any()) and bool(((t >= 5593) & (t < 11875)).any())
    check_method(pkg, emb, table, heads, rels, tpos, known, (h, r, t), method, cand=cand)
    # a second call with the same candidates tensor reuses the cached mapping
    r2 = pkg.rank_true_tails(emb, table, heads, rels, tpos, candidates=cand, method=method, filter=known)
    r1 = pkg.rank_true_tails(emb, table, heads, rels, tpos, candidates=cand.clone(), method=method, filter=known)
    assert torch.equal(r1[0], r2[0]) and torch.equal(r1[1], r2[1])
    with pytest.raises(ValueError, match="distinct"):
        pkg.rank_true_tails(emb, table, heads, rels, tpos, candidates=torch.cat([cand, cand[:1]]), method=method,
                            filter=known)


@pytest.mark.parametrize("method", METHODS)
def test_list_covering_every_other_candidate(pkg, method):
    """Every candidate but the true tail is known: rank 1, ties 0 (n = 300, not a multiple of 128)."""
    N = 300
    torch.manual_seed(8)
    emb = torch.randn(N, 64, device=DEV)
    table = torch.randn(2, 64, device=DEV)
    heads = torch.tensor([3, 3, 7], device=DEV)
    rels = torch.tensor([1, 1, 0], device=DEV)
    tails = torch.tensor([0, 299, 150], device=DEV)
    all_t = torch.arange(N, device=DEV)
    h = torch.cat([torch.full((N,), 3, device=DEV), torch.full((N,), 7, device=DEV)])
    r = torch.cat([torch.full((N,), 1, device=DEV), torch.zeros(N, dtype=torch.int64, device=DEV)])
    known = pkg.KnownTriples(h, r, torch.cat([all_t, all_t]), N, 2)      # the true tails are listed too
    rank, ties = pkg.rank_true_tails(emb, table, heads, rels, tails, method=method, filter=known)
    assert rank.tolist() == [1, 1, 1] and ties.tolist() == [0, 0, 0]


@pytest.mark.parametrize("method", METHODS)
def test_hub_list_of_more_than_7000_entries(pkg, method):
    N = 30926
    emb, table, heads, rels, tails, _ = _random_case(N, 128, 257, seed=9)
    heads[:] = 17
    rels[:] = 2
    hub = torch.randperm(N, device=DEV)[:7450]
    tri = (torch.full((7450,), 17, device=DEV), torch.full((7450,), 2, device=DEV), hub)
    known = pkg.KnownTriples(*tri, N, 3)
    assert len(known) == 7450
    check_method(pkg, emb, table, heads, rels, tails, known, tri, method)


@pytest.mark.parametrize("method", METHODS)
def test_known_columns_at_tile_and_chunk_edges(pkg, method):
    """Known positions at columns 0, 127, 128 and the last (n = 1,000, not a multiple of 128), all scoring above or
    exactly at the threshold; one of them an exact duplicate of the true tail, whose tie must not count once it is
    filtered."""
    N, T = 1000, 500
    torch.manual_seed(10)
    emb = torch.randn(N, 64, device=DEV)
    table = torch.randn(1, 64, device=DEV)
    heads = torch.randint(0, N, (200,), device=DEV)
    rels = torch.zeros(200, dtype=torch.int64, device=DEV)
    tails = torch.full((200,), T, device=DEV)
    edge = torch.tensor([0, 127, 128, N - 1], device=DEV)
    emb[edge[:3]] = 4 * emb[T]                       # above the threshold wherever the true score is positive
    emb[N - 1] = emb[T]                              # an exact duplicate of the true tail: an exact tie
    S = own_scores(emb, table, heads, rels, method)
    heads = heads[S[:, T] > 0]
    rels, tails = rels[:heads.numel()], tails[:heads.numel()]
    tri = (heads.repeat_interleave(4), torch.zeros(4 * heads.numel(), dtype=torch.int64, device=DEV),
           edge.repeat(heads.numel()))
    known = pkg.KnownTriples(*tri, N, 1)
    rank, ties, _, _ = check_method(pkg, emb, table, heads, rels, tails, known, tri, method)
    raw_r, raw_t = pkg.rank_true_tails(emb, table, heads, rels, tails, method=method)
    assert torch.equal(raw_r - rank, torch.full_like(rank, 3))
    assert torch.equal(raw_t - ties, torch.ones_like(ties))


@pytest.mark.parametrize("method", METHODS)
def test_duplicate_triples_are_deduplicated(pkg, method):
    emb, table, heads, rels, tails, (h, r, t) = _random_case(777, 64, 130, seed=13)
    once = pkg.KnownTriples(h, r, t, 777, 3)
    thrice = pkg.KnownTriples(h.repeat(3), r.repeat(3), t.repeat(3), 777, 3)
    assert len(once) == len(thrice) == torch.unique(torch.stack([h, r, t]), dim=1).size(1)
    a = pkg.rank_true_tails(emb, table, heads, rels, tails, method=method, filter=once)
    b = check_method(pkg, emb, table, heads, rels, tails, thrice, (h, r, t), method)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.parametrize("method", METHODS)
def test_head_side_through_the_reversed_view(pkg, method):
    """Filtered head ranks: rank_true_tails(tails as queries, heads as targets, filter=known.reversed()) equals the masked
    count of the transposed problem."""
    emb, table, heads, rels, tails, (h, r, t) = _random_case(2000, 64, 400, seed=14)
    known = pkg.KnownTriples(h, r, t, 2000, 3)
    rev = known.reversed()
    assert rev.reversed() is known and len(rev) == len(known)
    check_method(pkg, emb, table, tails, rels, heads, rev, (t, r, h), method)


def test_link_predictor_rank_tails_passes_the_filter(pkg):
    emb, table, heads, rels, tails, tri = _random_case(777, 64, 130, seed=15)
    dec = pkg.LinkPredictor(3, 64).to(DEV)
    known = pkg.KnownTriples(*tri, 777, 3)
    got = dec.rank_tails(emb, heads, rels, tails, filter=known)
    want = pkg.rank_true_tails(emb, dec.relation_embeddings.weight, heads, rels, tails, filter=known)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])


def test_known_triples_rejects_out_of_range_ids_on_the_device(pkg):
    h = torch.tensor([0, 1], device=DEV)
    with pytest.raises(ValueError, match="out of range"):
        pkg.KnownTriples(h, torch.tensor([0, 3], device=DEV), h, 10, 3)
    with pytest.raises(ValueError, match="out of range"):
        pkg.KnownTriples(h, h, torch.tensor([0, 10], device=DEV), 10, 3)


# ---- top-k of novel links ------------------------------------------------------------------------------------------
TOPK_SHAPES = [(5593, 6282), (1, 1025), (100, 5593), (128, 30926), (1000, 30926), (2048, 30926), (7, 5)]


@pytest.mark.parametrize("nq,ncand", TOPK_SHAPES)
@pytest.mark.parametrize("cosine", [False, True])
@pytest.mark.parametrize("k", [1, 10, 16])
def test_topk_excludes_known_links(pkg, cosine, k, nq, ncand):
    """Against a stable sort of the materialised matrix with the excluded entries at -inf.  Relation 1 holds each row's
    raw best candidates (every other row) and, for row 0, all but two candidates; relation 2 holds more of the raw
    best.  ``exclude_relation=1`` leaves relation 2's links in, ``exclude_relation=None`` takes both out."""
    torch.manual_seed(4)
    N = 30926
    emb = torch.randn(N, 128, device=DEV)
    c0 = 5593 if ncand == 6282 else 0
    queries = torch.arange(nq, device=DEV) + (0 if c0 else N - nq)
    cands = torch.arange(c0, c0 + ncand, device=DEV)
    if ncand >= 3:
        emb[cands[2 * ncand // 3]] = emb[cands[ncand // 3]]
    rel = torch.randn(128, device=DEV)
    kw = dict(cosine=True) if cosine else dict(rel_vec=rel)
    S = pkg.score_all_pairs(emb, queries, cands, **kw)
    order = torch.argsort(S, dim=1, descending=True, stable=True)
    rows = torch.arange(nq, device=DEV)
    # relation 1: the 3 raw best of every other row but row 0; relation 2: raw places 4..6 of every third row
    sel1 = rows[2::2].repeat_interleave(min(3, ncand))
    p1 = order[rows[2::2], :min(3, ncand)].reshape(-1)
    sel2 = rows[::3].repeat_interleave(min(3, max(ncand - 3, 0)))
    p2 = order[rows[::3], 3:6].reshape(-1)
    keep2 = order[0, :2] if ncand > 2 else order[0, :0]
    p0 = torch.tensor([j for j in range(ncand) if j not in set(keep2.tolist())], device=DEV, dtype=torch.int64)
    h = torch.cat([queries[sel1], queries[sel2], queries[0].repeat(p0.numel())])
    r = torch.cat([torch.ones_like(sel1), torch.full_like(sel2, 2), torch.ones_like(p0)])
    t = torch.cat([cands[p1], cands[p2], cands[p0]])
    known = pkg.KnownTriples(h, r, t, N, 3)
    for exclude_relation in (1, None):
        if exclude_relation is None:           # any relation: compare with every triple's relation set to 0
            excl = known_mask(h, torch.zeros_like(r), t, queries, torch.zeros_like(queries), N, 3, cands)
        else:
            excl = known_mask(h, r, t, queries, torch.full_like(queries, exclude_relation), N, 3, cands)
        val, ids = pkg.topk_all_pairs(emb, queries, cands, k=k, exclude=known, exclude_relation=exclude_relation, **kw)
        Sm = S.masked_fill(excl, float("-inf"))
        kk = min(k, ncand)
        o = torch.argsort(Sm, dim=1, descending=True, stable=True)[:, :kk]
        n_adm = (~excl).sum(1, keepdim=True)
        real = torch.arange(kk, device=DEV).view(1, -1) < n_adm
        want_val = torch.full((nq, k), float("-inf"), device=DEV)
        want_ids = torch.full((nq, k), -1, dtype=torch.int64, device=DEV)
        want_val[:, :kk] = torch.where(real, Sm.gather(1, o), float("-inf"))
        want_ids[:, :kk] = torch.where(real, cands[o], -1)
        assert val.shape == (nq, k) and ids.shape == (nq, k)
        if ncand > 2 and k > 2:
            assert ids[0, 2:].eq(-1).all() and val[0, 2:].eq(float("-inf")).all()   # fewer than k admissible
        pad = ~torch.cat([real, torch.zeros(nq, k - kk, dtype=torch.bool, device=DEV)], 1)
        assert torch.equal(ids[pad], want_ids[pad]) and torch.equal(val[pad], want_val[pad])
        if not cosine:
            assert torch.equal(val, want_val)
            assert torch.equal(ids, want_ids)
        else:
            torch.testing.assert_close(val[~pad], want_val[~pad], rtol=0, atol=2e-6)
            pos = (ids - c0).clamp(min=0)
            assert not bool(excl.gather(1, pos)[~pad].any())                    # nothing returned is excluded
            torch.testing.assert_close(S.gather(1, pos)[~pad], val[~pad], rtol=0, atol=2e-6)


def test_topk_with_an_empty_exclusion_is_the_raw_call(pkg):
    torch.manual_seed(16)
    emb = torch.randn(30926, 128, device=DEV)
    drugs, diseases = torch.arange(5593, 11875, device=DEV), torch.arange(0, 5593, device=DEV)
    z = torch.zeros(0, dtype=torch.int64, device=DEV)
    empty = pkg.KnownTriples(z, z, z, 30926, 3)
    for kw in (dict(rel_vec=torch.randn(128, device=DEV)), dict(cosine=True)):
        a = pkg.topk_all_pairs(emb, diseases, drugs, k=10, **kw)
        b = pkg.topk_all_pairs(emb, diseases, drugs, k=10, exclude=empty, **kw)
        c = pkg.topk_all_pairs(emb, diseases, drugs, k=10, exclude=empty, exclude_relation=2, **kw)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
        assert torch.equal(a[0], c[0]) and torch.equal(a[1], c[1])
    with pytest.raises(ValueError, match="exclude_relation"):
        pkg.topk_all_pairs(emb, diseases, drugs, k=10, exclude=empty, exclude_relation=3)

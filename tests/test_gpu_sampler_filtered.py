"""Filtered, type-constrained and Bernoulli negatives of the device sampler (``rgcn_link_batch_ex`` behind
``NegativeSampler(filter=, constraints=, head_prob=)``): bit-identity with the plain sampler, no known negative, admissible
types only, uniformity under rejection, exhaustion, the side frequencies, reproducibility and CUDA-graph capture."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
M32 = np.uint64(0xFFFFFFFF)


@pytest.fixture(scope="module")
def pkg(lib_built):
    return lib_built


@pytest.fixture(scope="module")
def cfg1():
    from primekg_rgcn_linkprediction_b200 import synth
    return synth.primekg_subgraph()


@pytest.fixture(scope="module")
def cfg1_known(pkg, cfg1):
    return pkg.KnownTriples.from_graphs(cfg1.as_dict(), device=DEV)


def _node_types(kg):
    nt = torch.empty(kg.num_nodes, dtype=torch.int64)
    for i, (lo, hi) in enumerate(kg.blocks.values()):
        nt[lo:hi] = i
    return nt


def _positives(kg, n, seed):
    g = torch.Generator().manual_seed(seed)
    sel = torch.randint(0, kg.num_edges, (n,), generator=g)
    return kg.edge_index[0, sel].to(DEV), kg.edge_index[1, sel].to(DEV), kg.edge_type[sel].to(DEV)


def _codes(h, r, t, R, N):
    return (np.asarray(h, dtype=np.int64) * R + np.asarray(r, dtype=np.int64)) * N + np.asarray(t, dtype=np.int64)


# ---- numpy port of the kernel's counter-based draws (csrc/decoder.cu: pcg32, draw2, redraw) -------------------------
def _pcg32(x):
    x = np.asarray(x, dtype=np.uint64) & M32
    state = (x * np.uint64(747796405) + np.uint64(2891336453)) & M32
    word = (((state >> ((state >> np.uint64(28)) + np.uint64(4))) ^ state) * np.uint64(277803737)) & M32
    return ((word >> np.uint64(22)) ^ word) & M32


def _draw2(seed, ctr, i):
    i = np.asarray(i, dtype=np.uint64)
    k = (_pcg32(np.uint64(seed) ^ (np.uint64(ctr) & M32)) + (np.uint64(ctr >> 32) * np.uint64(0x9E3779B9))) & M32
    a = _pcg32(i ^ k)
    return a, _pcg32((a + np.uint64(0x85EBCA6B) + i) & M32)


def _redraw(x, i, j):
    return _pcg32((_pcg32(x ^ ((np.uint64(j) * np.uint64(0x9E3779B9)) & M32)) + np.asarray(i, dtype=np.uint64)) & M32)


def _head_side(x, p):
    """The kernel's side choice for head probability p (float32): x >= (1 - p) 2^32."""
    thr = np.floor((1.0 - np.asarray(p, dtype=np.float32).astype(np.float64)) * 4294967296.0).astype(np.uint64)
    return x >= thr


# ---- 1. bit-identity with rgcn_link_batch ------------------------------------------------------------------------------
@pytest.mark.parametrize("multi_block", [False, True])
@pytest.mark.parametrize("num_neg", [1, 3, 16])
@pytest.mark.parametrize("n_pos", [1, 1000, 1025, 4096])
def test_no_options_is_bitwise_link_batch(pkg, n_pos, num_neg, multi_block):
    from primekg_rgcn_linkprediction_b200 import ops
    N, R = 30926, 3
    g = torch.Generator().manual_seed(n_pos * 31 + num_neg)
    ph, pt, pr = (torch.randint(0, hi, (n_pos,), generator=g).to(DEV) for hi in (N, N, R))
    c0 = 7 + (5 << 32)                                  # the counter's high word enters the draws too
    ctr_a, ctr_b = ops.rng_counter(DEV), ops.rng_counter(DEV)
    ctr_a.fill_(c0); ctr_b.fill_(c0)
    want = ops.link_batch(ph, pt, pr, N, num_neg, 0x5EED, ctr_a)
    ticket = torch.zeros(1, dtype=torch.int32, device=DEV) if multi_block else None
    got = ops.link_batch_ex(ph, pt, pr, N, num_neg, 0x5EED, ctr_b, ticket=ticket, max_tries=32)
    for a, b in zip(want, got):
        assert torch.equal(a, b)
    assert int(ctr_a) == int(ctr_b) == c0 + 1
    if multi_block:
        assert int(ticket) == 0
        # an explicit p = 1/2 per relation and the sampler's own path give the same bits
        ctr_b.fill_(c0)
        got = ops.link_batch_ex(ph, pt, pr, N, num_neg, 0x5EED, ctr_b, ticket=ticket, num_rel=R,
                                head_prob=torch.full((R,), 0.5, device=DEV))
        for a, b in zip(want, got):
            assert torch.equal(a, b)
        torch.manual_seed(3)
        s = pkg.NegativeSampler(N, num_neg)
        s.batch(ph, pt, pr)
        s._ctr.fill_(c0)
        got = s.batch(ph, pt, pr)
        ctr_a.fill_(c0)
        want = ops.link_batch(ph, pt, pr, N, num_neg, s._seed, ctr_a)
        for a, b in zip(want, got):
            assert torch.equal(a, b)
        assert int(s._ctr) == c0 + 1 and int(s.exhausted) == 0


# ---- 2. filtered negatives on cfg1 --------------------------------------------------------------------------------------
def test_filtered_negatives_are_never_known(pkg, cfg1, cfg1_known):
    N, R, n, k = cfg1.num_nodes, cfg1.num_relations, 1024, 4
    ph, pt, pr = _positives(cfg1, n, seed=2)
    torch.manual_seed(2)
    s = pkg.NegativeSampler(N, k, filter=cfg1_known)
    H, T, Rr, Y = s.batch(ph, pt, pr)
    assert H.numel() == n * (1 + k)
    assert torch.equal(H[:n], ph) and torch.equal(T[:n], pt) and torch.equal(Rr[:n], pr)
    assert torch.equal(Y, torch.cat([torch.ones(n), torch.zeros(n * k)]).to(DEV))
    assert torch.equal(Rr[n:], pr.repeat_interleave(k))
    ch, ct = H[n:] != ph.repeat_interleave(k), T[n:] != pt.repeat_interleave(k)
    assert bool((ch ^ ct).all())                        # exactly one end changes (the positive itself is known)
    assert int(s.exhausted) == 0
    known = np.unique(_codes(cfg1.edge_index[0], cfg1.edge_type, cfg1.edge_index[1], R, N))
    neg = _codes(H[n:].cpu(), Rr[n:].cpu(), T[n:].cpu(), R, N)
    assert not np.isin(neg, known).any()
    # the plain sampler does draw known triples here (the reason for the filter)
    s0 = pkg.NegativeSampler(N, k)
    H0, T0, R0, _ = s0.batch(ph, pt, pr)
    assert np.isin(_codes(H0[n:].cpu(), R0[n:].cpu(), T0[n:].cpu(), R, N), known).any()


# ---- 3. type constraints on the full graph ------------------------------------------------------------------------------
def test_typed_negatives_have_admissible_types(pkg):
    from primekg_rgcn_linkprediction_b200 import synth
    kg = synth.primekg_full()
    N, R, n, k = kg.num_nodes, kg.num_relations, 4096, 4
    nt = _node_types(kg)
    known = pkg.KnownTriples.from_graphs(kg.as_dict(), device=DEV)
    cons = pkg.RelationConstraints.from_node_types(known, nt)
    T_ = int(nt.max()) + 1
    ok_head = np.zeros((R, T_), dtype=bool)
    ok_tail = np.zeros((R, T_), dtype=bool)
    ntn = nt.numpy()
    ok_head[kg.edge_type.numpy(), ntn[kg.edge_index[0].numpy()]] = True
    ok_tail[kg.edge_type.numpy(), ntn[kg.edge_index[1].numpy()]] = True
    assert ok_head.sum() < R * T_                       # the constraints constrain
    ph, pt, pr = _positives(kg, n, seed=3)
    for filt in (None, known):
        torch.manual_seed(3)
        s = pkg.NegativeSampler(N, k, filter=filt, constraints=cons)
        H, T, Rr, _ = s.batch(ph, pt, pr)
        h, t, r = H[n:].cpu().numpy(), T[n:].cpu().numpy(), Rr[n:].cpu().numpy()
        hp, tp = ph.repeat_interleave(k).cpu().numpy(), pt.repeat_interleave(k).cpu().numpy()
        head_side = h != hp
        assert (~head_side | (t == tp)).all()          # at most one end changes
        assert ok_head[r[head_side], ntn[h[head_side]]].all()
        assert ok_tail[r[~head_side], ntn[t[~head_side]]].all()
        assert 0.4 < head_side.mean() < 0.6
        if filt is not None:
            assert ((h != hp) ^ (t != tp)).all() and int(s.exhausted) == 0
            kn = np.unique(_codes(kg.edge_index[0], kg.edge_type, kg.edge_index[1], R, N))
            assert not np.isin(_codes(h, r, t, R, N), kn).any()


# ---- 4. uniformity under rejection --------------------------------------------------------------------------------------
@pytest.mark.parametrize("typed", [False, True])
def test_accepted_draws_are_uniform_over_unknown_admissible(pkg, typed):
    from scipy.stats import chisquare
    g = torch.Generator().manual_seed(4)
    if typed:                                           # 40 admissible tails among 100 nodes, 30 of them known
        N, adm = 100, torch.arange(50, 90)
    else:                                               # all 40 nodes admissible, 30 known
        N, adm = 40, torch.arange(40)
    known_t = adm[torch.randperm(40, generator=g)[:30]]
    extra = torch.tensor([0, 1, 2]) if typed else torch.zeros(0, dtype=torch.int64)   # known, but not admissible
    tails = torch.cat([known_t, extra])
    known = pkg.KnownTriples(torch.zeros_like(tails).to(DEV), torch.zeros_like(tails).to(DEV), tails.to(DEV), N, 1)
    cons = pkg.RelationConstraints.from_lists([None], [adm], N, device=DEV) if typed else None
    free = sorted(set(adm.tolist()) - set(known_t.tolist()))
    n, k = 1000, 16
    ph = torch.zeros(n, dtype=torch.int64, device=DEV)
    pt = torch.full((n,), int(known_t[0]), dtype=torch.int64, device=DEV)
    pr = torch.zeros(n, dtype=torch.int64, device=DEV)
    torch.manual_seed(4)
    s = pkg.NegativeSampler(N, k, filter=known, constraints=cons, head_prob=0.0, max_tries=128)
    H, T, _, _ = s.batch(ph, pt, pr)
    assert int(s.exhausted) == 0 and bool((H[n:] == 0).all())
    t = T[n:].cpu()
    assert set(t.tolist()) <= set(free)
    counts = torch.bincount(t, minlength=N)[free].numpy()
    assert counts.sum() == n * k
    assert chisquare(counts).pvalue > 1e-3, counts


# ---- 5. exhaustion -----------------------------------------------------------------------------------------------------
def test_exhausted_queries_keep_their_last_draw(pkg):
    N, k, tries = 16, 4, 5
    tails = torch.arange(N)                                          # (0, 0, every node) is known
    known = pkg.KnownTriples(torch.zeros(N, dtype=torch.int64, device=DEV), torch.zeros(N, dtype=torch.int64, device=DEV),
                             tails.to(DEV), N, 1)
    ph = torch.tensor([0, 0, 0, 1, 1], device=DEV)                   # (1, 0, .) has no known tail
    pt = torch.tensor([3, 7, 3, 5, 2], device=DEV)
    pr = torch.zeros(5, dtype=torch.int64, device=DEV)
    torch.manual_seed(5)
    s = pkg.NegativeSampler(N, k, filter=known, head_prob=0.0, max_tries=tries)
    H, T, _, Y = s.batch(ph, pt, pr)
    torch.cuda.synchronize()
    assert int(s.exhausted) == 3 * k and bool((Y[5:] == 0).all())
    i = np.arange(5 * k, dtype=np.uint64)
    x, y0 = _draw2(s._seed, 0, i)
    last = _redraw(x, i, tries - 1)
    want = np.where(np.arange(5 * k) < 3 * k, (last * np.uint64(N)) >> np.uint64(32), (y0 * np.uint64(N)) >> np.uint64(32))
    assert T[5:].cpu().numpy().tolist() == want.astype(np.int64).tolist()
    assert bool((H[5:] == ph.repeat_interleave(k)).all())
    H2, T2, _, _ = s.batch(ph, pt, pr)
    torch.cuda.synchronize()
    assert int(s.exhausted) == 6 * k                                 # a running count


# ---- 6. Bernoulli head probability --------------------------------------------------------------------------------------
def test_bernoulli_head_prob_and_side_frequencies(pkg):
    N, n_per = 5000, 4000
    rng = np.random.default_rng(6)
    # r0: 20 heads x many tails (tph large), r1: the reverse, r2: both sides wide
    spec = [(20, N), (N, 20), (N, N)]
    h = np.concatenate([rng.integers(0, a, n_per) for a, _ in spec])
    t = np.concatenate([rng.integers(0, b, n_per) for _, b in spec])
    r = np.repeat(np.arange(3), n_per)
    known = pkg.KnownTriples(*(torch.from_numpy(v).to(DEV) for v in (h, r, t)), N, 3)
    want = []
    for rel in range(3):
        trip = np.unique(np.stack([h[r == rel], t[r == rel]], 1), axis=0)
        tph = len(trip) / len(np.unique(trip[:, 0]))
        hpt = len(trip) / len(np.unique(trip[:, 1]))
        want.append(tph / (tph + hpt))
    p = known.bernoulli_head_prob()
    np.testing.assert_allclose(p.cpu().numpy(), np.array(want, dtype=np.float32), rtol=1e-6)
    assert p[0] > 0.9 and p[1] < 0.1
    n, k = 6000, 8
    sel = rng.integers(0, len(h), n)
    ph, pt, pr = (torch.from_numpy(v[sel]).to(DEV) for v in (h, t, r))
    torch.manual_seed(6)
    s = pkg.NegativeSampler(N, k, filter=known, head_prob=p)
    H, T, Rr, _ = s.batch(ph, pt, pr)
    assert int(s.exhausted) == 0
    head_side = (H[n:] != ph.repeat_interleave(k)).cpu().numpy()
    assert ((T[n:] != pt.repeat_interleave(k)).cpu().numpy() ^ head_side).all()
    rr = Rr[n:].cpu().numpy()
    # exactly the kernel's coin (numpy port), and within binomial tolerance of p
    x, _ = _draw2(s._seed, 0, np.arange(n * k, dtype=np.uint64))
    assert (head_side == _head_side(x, p.cpu().numpy()[rr])).all()
    for rel in range(3):
        m = rr == rel
        cnt, pr_ = head_side[m].sum(), float(p[rel])
        assert abs(cnt - pr_ * m.sum()) <= 5 * np.sqrt(m.sum() * pr_ * (1 - pr_)) + 1, (rel, cnt, m.sum(), pr_)
    for prob in (0.0, 1.0):
        s = pkg.NegativeSampler(N, k, filter=known, head_prob=prob)
        H, T, _, _ = s.batch(ph, pt, pr)
        kept_head = bool((H[n:] == ph.repeat_interleave(k)).all())
        kept_tail = bool((T[n:] == pt.repeat_interleave(k)).all())
        assert (kept_head, kept_tail) == ((False, True) if prob == 1.0 else (True, False))


# ---- 7. reproducibility, replay, the captured training step, bad relation ids -------------------------------------------
def test_counter_reset_reproduces_and_graph_replays_differ(pkg, cfg1, cfg1_known):
    N, n, k = cfg1.num_nodes, 1024, 16
    cons = pkg.RelationConstraints.from_node_types(cfg1_known, _node_types(cfg1))
    ph, pt, pr = _positives(cfg1, n, seed=7)
    torch.manual_seed(7)
    s = pkg.NegativeSampler(N, k, filter=cfg1_known, constraints=cons, head_prob=cfg1_known.bernoulli_head_prob())
    a = [x.clone() for x in s.batch(ph, pt, pr)]
    b = [x.clone() for x in s.batch(ph, pt, pr)]
    assert int(s._ctr) == 2 and not (torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]))
    s._ctr.zero_()
    c = s.batch(ph, pt, pr)
    assert all(torch.equal(x, y) for x, y in zip(a, c))
    out = tuple(torch.empty_like(x) for x in a)
    s.batch(ph, pt, pr, out=out)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            s.batch(ph, pt, pr, out=out)
    torch.cuda.current_stream().wait_stream(side)
    c0 = int(s._ctr)
    gr.replay()
    r1 = [x.clone() for x in out]
    gr.replay()
    torch.cuda.synchronize()
    assert int(s._ctr) == c0 + 2
    assert not (torch.equal(r1[0], out[0]) and torch.equal(r1[1], out[1]))
    s._ctr.fill_(c0 + 1)
    again = s.batch(ph, pt, pr)
    assert all(torch.equal(x, y) for x, y in zip(again, out))


def test_graphed_train_step_with_filtered_typed_sampler(pkg):
    from primekg_rgcn_linkprediction_b200 import synth
    kg = synth.primekg_subgraph(num_directed_edges=40_000, seed=1)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    known = pkg.KnownTriples.from_graphs(kg.as_dict(), device=DEV)
    cons = pkg.RelationConstraints.from_node_types(known, _node_types(kg))
    torch.manual_seed(8)
    m = pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, 64, 128, dropout=0.1, decoder_dropout=0.1).to(DEV).train()
    smp = pkg.NegativeSampler(kg.num_nodes, 4, filter=known, constraints=cons, head_prob=known.bernoulli_head_prob())
    opt = pkg.FusedAdam(m.parameters(), lr=1e-3, max_grad_norm=1.0)
    n_pos = 256
    step = pkg.GraphedTrainStep(m, ei, et, batch_size=5 * n_pos, sampler=smp, optimizer=opt)
    ph, pt, pr = _positives(kg, n_pos, seed=8)
    losses, negs = [], []
    for _ in range(3):
        losses.append(float(step.run_positives(ph, pt, pr)))
        negs.append(step.tails[n_pos:].clone())
    assert all(np.isfinite(losses)) and not torch.equal(negs[1], negs[2])
    kn = np.unique(_codes(kg.edge_index[0], kg.edge_type, kg.edge_index[1], kg.num_relations, kg.num_nodes))
    got = _codes(step.heads[n_pos:].cpu(), step.rels[n_pos:].cpu(), step.tails[n_pos:].cpu(), kg.num_relations, kg.num_nodes)
    assert not np.isin(got, kn).any() and int(smp.exhausted) == 0


def test_out_of_range_relation_is_drawn_unconstrained_and_flagged(pkg, cfg1, cfg1_known):
    from primekg_rgcn_linkprediction_b200 import ops
    N, R, n, k = cfg1.num_nodes, cfg1.num_relations, 64, 4
    cons = pkg.RelationConstraints.from_node_types(cfg1_known, _node_types(cfg1))
    ph, pt, pr = _positives(cfg1, n, seed=9)
    pr[5], pr[9] = R, -1 - (1 << 40)
    torch.manual_seed(9)
    s = pkg.NegativeSampler(N, k, filter=cfg1_known, constraints=cons, head_prob=torch.zeros(R))
    H, T, Rr, Y = s.batch(ph, pt, pr)
    torch.cuda.synchronize()
    assert int(H.min()) >= 0 and int(H.max()) < N and int(T.min()) >= 0 and int(T.max()) < N
    assert int(Rr[n + 5 * k]) == R and int(Rr[n + 9 * k]) == -1 - (1 << 40)
    # the bad pairs draw with the default coin (head_prob = 0 is never read for them): the numpy port's side
    x, _ = _draw2(s._seed, 0, np.arange(n * k, dtype=np.uint64))
    for q in (5, 9):
        head_side = x[q * k:(q + 1) * k] >= np.uint64(1 << 31)
        hq, tq = H[n + q * k:n + (q + 1) * k].cpu().numpy(), T[n + q * k:n + (q + 1) * k].cpu().numpy()
        assert (tq[head_side] == int(pt[q])).all() and (hq[~head_side] == int(ph[q])).all()
    good = torch.ones(n, dtype=torch.bool, device=DEV)
    good[5] = good[9] = False
    assert bool((H[n:][good.repeat_interleave(k)] == ph.repeat_interleave(k)[good.repeat_interleave(k)]).all())
    ops.raise_on_bad_pairs(torch.device(DEV))                        # clean slate
    emb = torch.randn(N, 16, device=DEV)
    table = torch.randn(R, 16, device=DEV)
    loss, scores, _ = ops.link_loss(emb, table, H, T, Rr, Y)
    torch.cuda.synchronize()
    with pytest.raises(IndexError):
        ops.raise_on_bad_pairs(torch.device(DEV))

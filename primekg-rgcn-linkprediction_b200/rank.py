"""All-pairs scoring and ranking on device (SURVEY.md §8a `score_all_tails`, §8f rows 1 and 3, BASELINE cfg4).

* ``score_all_pairs``  — DistMult ``(h * r) @ T^T`` (reference src/models/rgcn.py:234-241) or cosine ``(cos + 1) / 2``
  (src/compare_methods.py:384-397; src/medical_validation.py:222-239) over index lists, gathers fused.
* ``rank_true_tails``  — 1-indexed rank of the true tail among all candidates, the quantity the Python loop at
  src/evaluate.py:266-276 extracts with one ``argsort`` per row.

Both are a dense contraction ``A' @ B^T`` over the feature width and run on the tensor cores by default (``method="tc"``):
the prepared query rows become bf16 hi / lo operand planes and the candidate rows the K-major "weight" operand of the
tcgen05 kernel behind ``rgcn_transform_dgrad`` (three bf16 products with fp32 accumulation, 3-7e-6 relative error — the
fp32 mode of the encoder).  ``alpha`` / ``beta`` ride along as one extra K column, so the cosine rescale costs nothing.
The ranking counts come from the score block itself (``rgcn_rank_count``), a block of queries at a time.
``method="simt"`` keeps the fp32 FMA tile kernels of ``csrc/rank.cu`` (every output accumulated in ascending k order with
``fmaf``; they never materialise the [queries, candidates] block when ranking).

Filtered ranking (Bordes et al. 2013) and top-k of novel links take a ``KnownTriples`` index: per query a sorted list
of candidate positions to leave out.  The tensor-core epilogues skip them as they sweep (``rgcn_scores_rank_excl_w``,
``rgcn_scores_topk_excl_w``); ``tc_block`` and ``simt`` count unfiltered and then take the excluded positions back out
with the counting pass's own score bits (``rgcn_rank_excl_correct``).
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import _lib
from .graph import _ptr, _stream

_RANK_BLOCK = 2048       # queries ranked per score block of the tensor-core path (2048 x 30,926 fp32 = 253 MB)

ExclLists = Tuple[torch.Tensor, torch.Tensor, torch.Tensor]     # (begin [n] int64, end [n] int64, positions int32)


def _lex_order(major: torch.Tensor, minor: torch.Tensor) -> torch.Tensor:
    """Permutation sorting by (major, minor): two stable sorts, no packed key that could overflow."""
    o = torch.argsort(minor, stable=True)
    return o[torch.argsort(major[o], stable=True)]


def _check_candidates(cand: torch.Tensor, num_nodes: int) -> None:
    """A candidate list that positions are mapped into must name distinct nodes of the graph."""
    if cand.numel() and (int(cand.min()) < 0 or int(cand.max()) >= num_nodes):
        raise ValueError("candidates hold node ids outside the filter's graph")
    if torch.unique(cand).numel() != cand.numel():
        raise ValueError("candidates must be distinct when a filter / exclusion is given")


class KnownTriples:
    """Known (head, relation, tail) triples on the device, indexed by (head, relation) with the tails of each key sorted
    and distinct (multi-edges are deduplicated).  The filter of ``rank_true_tails(filter=...)`` (filtered MRR / Hits@K:
    the other known true tails of a query's (head, relation) leave the candidate set) and the exclusion of
    ``topk_all_pairs(exclude=...)`` (only links that are not known yet).

    Head-side filtered ranking needs no second function: DistMult is symmetric, so
    ``rank_true_tails(emb, table, tails, rels, heads, filter=known.reversed())`` ranks every true head among all heads.
    """

    def __init__(self, heads: torch.Tensor, rels: torch.Tensor, tails: torch.Tensor, num_nodes: int, num_relations: int):
        for name, t in (("heads", heads), ("rels", rels), ("tails", tails)):
            if not isinstance(t, torch.Tensor) or t.dim() != 1 or t.numel() != heads.numel():
                raise ValueError("KnownTriples: heads, rels and tails must be 1-D tensors of one length")
            if t.dtype.is_floating_point or t.dtype == torch.bool:
                raise ValueError(f"KnownTriples: {name} must hold integer ids")
        if not (0 < num_nodes < 2 ** 31 and num_relations > 0):
            raise ValueError("KnownTriples: need 0 < num_nodes < 2^31 and num_relations > 0")
        heads, rels, tails = heads.to(torch.int64), rels.to(torch.int64), tails.to(torch.int64)
        if heads.numel():
            lo = torch.stack([heads.min(), rels.min(), tails.min()])
            hi = torch.stack([heads.max() - num_nodes, rels.max() - num_relations, tails.max() - num_nodes])
            if bool((lo < 0).any()) or bool((hi >= 0).any()):
                raise ValueError(f"KnownTriples: ids out of range (num_nodes={num_nodes}, num_relations={num_relations})")
        if not (heads.is_cuda and rels.is_cuda and tails.is_cuda):
            raise ValueError("KnownTriples: heads, rels and tails must be CUDA tensors (the index lives on the device)")
        self.num_nodes, self.num_relations = int(num_nodes), int(num_relations)
        self.device = heads.device
        key = heads * num_relations + rels
        o = _lex_order(key, tails)
        key, tails = key[o], tails[o]
        keep = torch.ones_like(key, dtype=torch.bool)
        keep[1:] = (key[1:] != key[:-1]) | (tails[1:] != tails[:-1])
        self.keys = key[keep].contiguous()                      # head * num_relations + rel, ascending
        self.tails = tails[keep].to(torch.int32).contiguous()   # ascending within each key
        self._reversed: Optional["KnownTriples"] = None
        self._any: Optional["KnownTriples"] = None
        self._cand = None                                       # (candidates tensor, its version, keys, positions)

    @classmethod
    def from_graphs(cls, *graphs, device=None) -> "KnownTriples":
        """Every edge of the given graphs (the reference's dicts ``{'edge_index', 'edge_type', 'num_nodes',
        'num_relations'}``, e.g. train + val + test) as known triples; ``device`` moves CPU-held graphs over."""
        if not graphs:
            raise ValueError("KnownTriples.from_graphs needs at least one graph")
        ei = torch.cat([g["edge_index"].to(device) if device is not None else g["edge_index"] for g in graphs], 1)
        et = torch.cat([g["edge_type"].to(device) if device is not None else g["edge_type"] for g in graphs])
        return cls(ei[0], et, ei[1], max(int(g["num_nodes"]) for g in graphs),
                   max(int(g["num_relations"]) for g in graphs))

    def __len__(self) -> int:
        return int(self.keys.numel())

    def reversed(self) -> "KnownTriples":
        """The (tail, relation) -> head view, for filtered head ranking."""
        if self._reversed is None:
            R = self.num_relations
            self._reversed = KnownTriples(self.tails.to(torch.int64), self.keys % R, self.keys // R, self.num_nodes, R)
            self._reversed._reversed = self
        return self._reversed

    def any_relation(self) -> "KnownTriples":
        """The relation-agnostic view: head -> every tail it links to under any relation (query it with relation 0)."""
        if self._any is None:
            R = self.num_relations
            self._any = KnownTriples(self.keys // R, torch.zeros_like(self.keys), self.tails.to(torch.int64),
                                     self.num_nodes, 1)
        return self._any

    def bernoulli_head_prob(self) -> torch.Tensor:
        """float32 [num_relations]: tph / (tph + hpt) per relation, the head-replacement probability of Wang et al.
        2014 (``NegativeSampler(head_prob=...)``).  tph = mean number of tails per (head, relation), hpt = mean number of
        heads per (tail, relation); 1/2 for a relation without triples."""
        R = self.num_relations
        rel = self.keys % R
        n = torch.bincount(rel, minlength=R).to(torch.float64)
        n_heads = torch.bincount(torch.unique_consecutive(self.keys) % R, minlength=R).to(torch.float64)
        n_tails = torch.bincount(torch.unique(self.tails.to(torch.int64) * R + rel) % R, minlength=R).to(torch.float64)
        tph, hpt = n / n_heads.clamp(min=1), n / n_tails.clamp(min=1)
        p = torch.where(n > 0, tph / (tph + hpt).clamp(min=1e-300), torch.full_like(n, 0.5))
        return p.to(torch.float32)

    def _on_candidates(self, candidates: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """(keys, positions) with the tails mapped to positions in ``candidates`` (non-candidates dropped, positions
        ascending per key); cached for the last candidates tensor."""
        c = self._cand
        if c is not None and c[0] is candidates and c[1] == candidates._version:
            return c[2], c[3]
        cand = candidates.to(self.device, torch.int64).reshape(-1)
        n = cand.numel()
        _check_candidates(cand, self.num_nodes)
        inv = torch.full((self.num_nodes,), -1, dtype=torch.int64, device=self.device)
        inv[cand] = torch.arange(n, dtype=torch.int64, device=self.device)
        pos = inv[self.tails.to(torch.int64)]
        keep = pos >= 0
        keys, pos = self.keys[keep], pos[keep]
        o = _lex_order(keys, pos)
        keys, pos = keys[o].contiguous(), pos[o].to(torch.int32).contiguous()
        self._cand = (candidates, candidates._version, keys, pos)
        return keys, pos

    def lists(self, heads: torch.Tensor, rels, candidates: Optional[torch.Tensor] = None) -> ExclLists:
        """Per query (heads[i], rels[i]) its known tails as the kernels' exclusion lists: (begin, end, positions), the
        positions being node ids (``candidates=None``: ranges straight into the index) or positions in ``candidates``.
        ``rels`` may be one int for all queries."""
        heads = heads.to(self.device, torch.int64).reshape(-1)
        if isinstance(rels, int):
            rels = torch.full_like(heads, rels)
        rels = rels.to(self.device, torch.int64).reshape(-1)
        keys, pos = (self.keys, self.tails) if candidates is None else self._on_candidates(candidates)
        q = heads * self.num_relations + rels
        begin = torch.searchsorted(keys, q)
        end = torch.searchsorted(keys, q, right=True)
        # an id outside the index must not alias another key: empty list
        bad = (heads < 0) | (heads >= self.num_nodes) | (rels < 0) | (rels >= self.num_relations)
        end = torch.where(bad, begin, end)
        if pos.numel() == 0:                # every range is empty, but the kernels take a non-null list pointer
            pos = torch.zeros(1, dtype=torch.int32, device=self.device)
        return begin.contiguous(), end.contiguous(), pos


def _prep(emb: torch.Tensor, idx: Optional[torch.Tensor], rel_table: Optional[torch.Tensor],
          rel: Optional[torch.Tensor], normalize: bool) -> torch.Tensor:
    lib = _lib.load()
    if not emb.is_cuda:
        raise RuntimeError("all-pairs scoring needs CUDA tensors: there is no CPU implementation of this path")
    emb = emb.detach().to(torch.float32)
    if emb.stride(1) != 1:
        emb = emb.contiguous()
    n = emb.size(0) if idx is None else idx.numel()
    d = emb.size(1)
    idx = None if idx is None else idx.to(torch.int64).contiguous()
    if rel is not None:
        rel = rel.to(torch.int64).contiguous()
        rel_table = rel_table.detach().to(torch.float32).contiguous()
    out = torch.empty(n, d, dtype=torch.float32, device=emb.device)
    _lib.check(lib.rgcn_rows_prepare(_ptr(emb), emb.stride(0), _ptr(idx), n, d, _ptr(rel_table) if rel is not None else None,
                                     _ptr(rel), int(normalize), _ptr(out), out.stride(0), _stream(emb.device)),
               "rgcn_rows_prepare")
    return out


def _tc_block(A: torch.Tensor, Bext: torch.Tensor, alpha: float, beta: float) -> torch.Tensor:
    """[rows(A), rows(Bext)] = alpha * A @ Bext[:, :d]^T + beta on the tensor cores.  ``Bext`` is the candidate operand
    from ``_tc_candidates`` ([nb_pad, d + 8] when alpha / beta ride along, else [nb_pad, d])."""
    from . import ops
    d = A.size(1)
    dk = Bext.size(1)
    if dk != d:
        Ae = torch.zeros(A.size(0), dk, dtype=torch.float32, device=A.device)
        torch.mul(A, alpha, out=Ae[:, :d])
        Ae[:, d] = 1.0
        A = Ae
    planes = ops.alloc_planes(A.size(0), dk, "fp32", A.device)
    ops.split_planes(A, planes)
    return ops.transform_dgrad(planes, dk, Bext, None, "fp32")


def _tc_candidates(B: torch.Tensor, b_idx: Optional[torch.Tensor], alpha: float, beta: float) -> torch.Tensor:
    """Candidate rows as the K-major operand: gathered, padded to a multiple of 8 rows with zeros and — when the scores
    are to be rescaled — widened by 8 columns of which the first holds ``beta`` (it meets the constant 1 of the queries)."""
    nb = B.size(0) if b_idx is None else b_idx.numel()
    d = B.size(1)
    ext = alpha != 1.0 or beta != 0.0
    Be = torch.zeros((nb + 7) // 8 * 8, d + (8 if ext else 0), dtype=torch.float32, device=B.device)
    if b_idx is None:
        Be[:nb, :d] = B
    else:
        lib = _lib.load()
        view = Be[:nb, :d]
        _lib.check(lib.rgcn_rows_prepare(_ptr(B), B.stride(0), _ptr(b_idx), nb, d, None, None, 0, _ptr(view), Be.stride(0),
                                         _stream(B.device)), "rgcn_rows_prepare")
    if ext:
        Be[:nb, d] = beta
    return Be


def scores_from_rows(A: torch.Tensor, B: torch.Tensor, b_idx: Optional[torch.Tensor] = None, alpha: float = 1.0,
                     beta: float = 0.0, method: str = "tc") -> torch.Tensor:
    """out[i, j] = alpha * <A[i], B[b_idx[j]]> + beta  (fp32, fused gather of the candidate rows)."""
    lib = _lib.load()
    A = A.detach().to(torch.float32).contiguous()
    B = B.detach().to(torch.float32)
    if B.stride(1) != 1 or B.stride(0) % 4 or B.data_ptr() % 16:
        B = B.contiguous()
    b_idx = None if b_idx is None else b_idx.to(torch.int64).contiguous()
    nb = B.size(0) if b_idx is None else b_idx.numel()
    if method == "tc" and A.size(0) > 0 and nb > 0 and A.size(1) % 4 == 0:
        out = _tc_block(A, _tc_candidates(B, b_idx, alpha, beta), alpha, beta)
        return out[:, :nb]
    if method not in ("tc", "simt"):
        raise ValueError("method must be 'tc' (tensor cores) or 'simt' (fp32 FMA tiles)")
    out = torch.empty(A.size(0), nb, dtype=torch.float32, device=A.device)
    _lib.check(lib.rgcn_allpairs_scores(_ptr(A), A.stride(0), A.size(0), _ptr(B), B.stride(0), _ptr(b_idx), nb,
                                        A.size(1), alpha, beta, _ptr(out), out.stride(0), _stream(A.device)),
               "rgcn_allpairs_scores")
    return out


def score_all_pairs(emb: torch.Tensor, a_idx: torch.Tensor, b_idx: torch.Tensor,
                    rel_vec: Optional[torch.Tensor] = None, cosine: bool = False, method: str = "tc") -> torch.Tensor:
    """[len(a_idx), len(b_idx)] scores.  DistMult: (emb[a] * rel_vec) . emb[b];  cosine: (cos(emb[a], emb[b]) + 1) / 2."""
    if cosine:
        A = _prep(emb, a_idx, None, None, True)
        Bn = _prep(emb, b_idx, None, None, True)
        return scores_from_rows(A, Bn, None, 0.5, 0.5, method=method)
    if rel_vec is not None:
        table = rel_vec.reshape(1, -1)
        A = _prep(emb, a_idx, table, torch.zeros(a_idx.numel(), dtype=torch.int64, device=emb.device), False)
    else:
        A = _prep(emb, a_idx, None, None, False)
    return scores_from_rows(A, emb, b_idx, method=method)


def _query_planes(A: torch.Tensor):
    from . import ops
    planes = ops.alloc_planes(A.size(0), A.size(1), "fp32", A.device)
    ops.split_planes(A, planes)
    return planes


def _candidate_rows(B: torch.Tensor, idx: Optional[torch.Tensor]) -> torch.Tensor:
    """fp32 candidate rows [n, d], gathered through ``idx`` when given (contiguous)."""
    if idx is None:
        return B.contiguous()
    lib = _lib.load()
    out = torch.empty(idx.numel(), B.size(1), dtype=torch.float32, device=B.device)
    _lib.check(lib.rgcn_rows_prepare(_ptr(B), B.stride(0), _ptr(idx), idx.numel(), B.size(1), None, None, 0, _ptr(out),
                                     out.stride(0), _stream(B.device)), "rgcn_rows_prepare")
    return out


def _rank_fused(A: torch.Tensor, B: torch.Tensor, cand: Optional[torch.Tensor], tails: torch.Tensor,
                excl: Optional[ExclLists] = None):
    """Tensor-core sweep whose epilogue counts instead of storing (``rgcn_scores_rank_excl_w``); the threshold comes
    from the diagonal tiles of queries x (their own true tails) with the same K order, so it carries the sweep's own
    bits.  ``excl``: per-query positions the epilogue leaves out."""
    from . import ops
    lib = _lib.load()
    nq, d = A.shape
    C = _candidate_rows(B, cand)
    nb = C.size(0)
    Q = _query_planes(A)
    cand_planes = ops.prepare_weights(C, None, "fp32")
    true_rows = torch.empty(nq, d, dtype=torch.float32, device=A.device)
    _lib.check(lib.rgcn_rows_prepare(_ptr(C), C.stride(0), _ptr(tails), nq, d, None, None, 0, _ptr(true_rows), d,
                                     _stream(A.device)), "rgcn_rows_prepare")
    tail_planes = ops.prepare_weights(true_rows, None, "fp32")
    thr = torch.empty(nq, dtype=torch.float32, device=A.device)
    greater = torch.zeros(nq, dtype=torch.int32, device=A.device)
    equal = torch.zeros(nq, dtype=torch.int32, device=A.device)
    st = _stream(A.device)
    _lib.check(lib.rgcn_scores_diag_w(_ptr(Q[0]), _ptr(Q[1]), Q[0].stride(0), d, _ptr(tail_planes), nq, _ptr(thr), st),
               "rgcn_scores_diag_w")
    xb, xe, xp = excl if excl is not None else (None, None, None)
    _lib.check(lib.rgcn_scores_rank_excl_w(_ptr(Q[0]), _ptr(Q[1]), Q[0].stride(0), d, _ptr(cand_planes), nb, nq,
                                           _ptr(thr), _ptr(tails), _ptr(greater), _ptr(equal), _ptr(xb), _ptr(xe),
                                           _ptr(xp), st), "rgcn_scores_rank_excl_w")
    return greater, equal


def topk_from_rows(A: torch.Tensor, B: torch.Tensor, k: int, b_idx: Optional[torch.Tensor] = None, alpha: float = 1.0,
                   beta: float = 0.0, excl: Optional[ExclLists] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """(values [n_a, k], positions [n_a, k]): per row of ``A`` the k best rows of ``B[b_idx]`` by alpha * <a, b> + beta,
    sorted by value (ties: lower position first); positions index ``b_idx`` (or B).  Tensor cores, the score block is
    consumed in the epilogue (``rgcn_scores_topk_excl_w``), k <= 16.  ``excl`` (``KnownTriples.lists``): per row of A
    the positions that are never returned; a row left with fewer than k candidates ends in -inf / -1."""
    from . import ops
    lib = _lib.load()
    if not (1 <= k <= 16):
        raise ValueError("fused top-k serves 1 <= k <= 16")
    A = A.detach().to(torch.float32).contiguous()
    B = B.detach().to(torch.float32)
    if B.stride(1) != 1:
        B = B.contiguous()
    C = _candidate_rows(B, None if b_idx is None else b_idx.to(torch.int64).contiguous())
    na, d = A.shape
    nb = C.size(0)
    if na == 0 or nb == 0 or d % 4:
        raise ValueError("topk_from_rows needs non-empty operands with a feature width that is a multiple of 4")
    Q = _query_planes(A)
    cand_planes = ops.prepare_weights(C, None, "fp32")
    slots = int(lib.rgcn_scores_topk_slots(na, nb))
    dev = A.device
    cv = torch.empty(na, slots, 16, dtype=torch.float32, device=dev)
    ci = torch.empty(na, slots, 16, dtype=torch.int32, device=dev)
    ctr = torch.empty(na, dtype=torch.int32, device=dev)
    ov = torch.empty(na, k, dtype=torch.float32, device=dev)
    oi = torch.empty(na, k, dtype=torch.int64, device=dev)
    xb, xe, xp = excl if excl is not None else (None, None, None)
    _lib.check(lib.rgcn_scores_topk_excl_w(_ptr(Q[0]), _ptr(Q[1]), Q[0].stride(0), d, _ptr(cand_planes), nb, na, int(k),
                                           float(alpha), float(beta), _ptr(cv), _ptr(ci), _ptr(ctr), slots, _ptr(ov),
                                           _ptr(oi), _ptr(xb), _ptr(xe), _ptr(xp), _stream(dev)),
               "rgcn_scores_topk_excl_w")
    return ov, oi


def topk_all_pairs(emb: torch.Tensor, a_idx: torch.Tensor, b_idx: torch.Tensor, k: int = 10,
                   rel_vec: Optional[torch.Tensor] = None, cosine: bool = False,
                   exclude: Optional[KnownTriples] = None, exclude_relation: Optional[int] = None
                   ) -> Tuple[torch.Tensor, torch.Tensor]:
    """Per row of ``a_idx`` the k best of ``b_idx`` — DistMult ``(emb[a] * rel_vec) . emb[b]`` or cosine ``(cos + 1) / 2`` —
    without the [len(a), len(b)] matrix: (scores [len(a), k], node ids [len(a), k]).  The device form of the per-disease /
    per-drug sweeps + top-k filters of src/compare_methods.py:384-397, src/medical_validation.py:222-239 and
    src/case_studies.py:260-274 (fused L2 normalisation, fused rescale).

    ``exclude``: return novel links only — ``b`` is left out for row ``a`` when (a, exclude_relation, b) is a known
    triple, or, with ``exclude_relation=None``, when (a, r, b) is known for any relation r.  ``b_idx`` must then be
    distinct; a row with fewer than k admissible candidates ends in -inf / -1."""
    excl = None
    if exclude is not None:
        if exclude_relation is None:
            view, rel = exclude.any_relation(), 0
        else:
            if not 0 <= int(exclude_relation) < exclude.num_relations:
                raise ValueError(f"exclude_relation={exclude_relation} outside [0, {exclude.num_relations})")
            view, rel = exclude, int(exclude_relation)
        excl = view.lists(a_idx, rel, b_idx)
    elif exclude_relation is not None:
        raise ValueError("exclude_relation needs exclude=")
    b_idx = b_idx.to(torch.int64)
    if cosine:
        A = _prep(emb, a_idx, None, None, True)
        Bn = _prep(emb, b_idx, None, None, True)
        val, pos = topk_from_rows(A, Bn, k, None, 0.5, 0.5, excl=excl)
    else:
        if rel_vec is not None:
            A = _prep(emb, a_idx, rel_vec.reshape(1, -1), torch.zeros(a_idx.numel(), dtype=torch.int64, device=emb.device), False)
        else:
            A = _prep(emb, a_idx, None, None, False)
        val, pos = topk_from_rows(A, emb, k, b_idx, excl=excl)
    ids = torch.where(pos >= 0, b_idx[pos.clamp(min=0)], pos)
    return val, ids


def rank_true_tails(emb: torch.Tensor, rel_table: torch.Tensor, heads: torch.Tensor, rels: torch.Tensor,
                    tails: torch.Tensor, candidates: Optional[torch.Tensor] = None, method: str = "tc",
                    filter: Optional[KnownTriples] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """(rank, ties): rank[i] = 1 + #{candidates scoring strictly above the true tail} (int64, 1-indexed like
    src/evaluate.py:274); ties[i] = #{other candidates with exactly the true tail's score}.  ``candidates`` = index list
    of admissible tails (default: all entities); ``tails`` then holds POSITIONS in that list.
    ``method``: "tc" = tensor cores, counts taken in the GEMM epilogue (no score block); "tc_block" = tensor cores through
    materialised 2,048-query score blocks (round 1); "simt" = fp32 FMA tiles.
    ``filter``: the filtered protocol (Bordes et al. 2013) — every known tail of (heads[i], rels[i]) other than the true
    one leaves row i's candidate set, so it counts in neither rank nor ties (``candidates`` must then be distinct).
    Filtered head ranks: ``rank_true_tails(emb, rel_table, tails, rels, heads, filter=known.reversed())`` (DistMult
    is symmetric)."""
    lib = _lib.load()
    excl = None if filter is None else filter.lists(heads, rels, candidates)
    A = _prep(emb, heads, rel_table, rels, False)
    B = emb.detach().to(torch.float32)
    if B.stride(1) != 1 or B.stride(0) % 4 or B.data_ptr() % 16:
        B = B.contiguous()
    cand = None if candidates is None else candidates.to(torch.int64).contiguous()
    nb = B.size(0) if cand is None else cand.numel()
    nq = A.size(0)
    tails = tails.to(torch.int64).contiguous()
    greater = torch.empty(nq, dtype=torch.int32, device=A.device)
    equal = torch.empty(nq, dtype=torch.int32, device=A.device)
    if method == "tc" and nq > 0 and nb > 0 and A.size(1) % 4 == 0:
        greater, equal = _rank_fused(A, B, cand, tails, excl)
        return greater.to(torch.int64) + 1, equal.to(torch.int64)
    st = _stream(A.device)

    def correct(q0, q1, thr, S=None):
        # filtered counts: the excluded positions' own scores (block bits, or recomputed as the FMA tiles compute them)
        # leave the unfiltered counts of rows q0 .. q1
        if excl is None:
            return
        xb, xe, xp = excl
        if S is not None:
            ops = (_ptr(S), S.stride(0), None, 0, None, 0, None, A.size(1))
        else:
            ops = (None, 0, _ptr(A), A.stride(0), _ptr(B), B.stride(0), _ptr(cand), A.size(1))
        _lib.check(lib.rgcn_rank_excl_correct(*ops, q1 - q0, nb, _ptr(tails[q0:q1]), _ptr(thr), _ptr(xb[q0:q1]),
                                              _ptr(xe[q0:q1]), _ptr(xp), _ptr(greater[q0:q1]), _ptr(equal[q0:q1]), st),
                   "rgcn_rank_excl_correct")

    if method in ("tc", "tc_block") and nq > 0 and nb > 0 and A.size(1) % 4 == 0:
        Bext = _tc_candidates(B, cand, 1.0, 0.0)
        # queries per score block: at most _RANK_BLOCK, and at most ~1 GiB of scores for very large candidate sets
        qb = max(128, min(_RANK_BLOCK, (1 << 28) // max(Bext.size(0), 1) // 128 * 128))
        thr = None if excl is None else torch.empty(nq, dtype=torch.float32, device=A.device)
        for q0 in range(0, nq, qb):
            q1 = min(q0 + qb, nq)
            S = _tc_block(A[q0:q1], Bext, 1.0, 0.0)
            _lib.check(lib.rgcn_rank_count(_ptr(S), S.stride(0), q1 - q0, nb, _ptr(tails[q0:q1]),
                                           None if thr is None else _ptr(thr[q0:q1]), _ptr(greater[q0:q1]),
                                           _ptr(equal[q0:q1]), st), "rgcn_rank_count")
            correct(q0, q1, None if thr is None else thr[q0:q1], S)
        return greater.to(torch.int64) + 1, equal.to(torch.int64)
    if method not in ("tc", "tc_block", "simt"):
        raise ValueError("method must be 'tc' (tensor cores, fused count), 'tc_block' or 'simt' (fp32 FMA tiles)")
    thr = torch.empty(nq, dtype=torch.float32, device=A.device)
    _lib.check(lib.rgcn_allpairs_rank(_ptr(A), A.stride(0), nq, _ptr(B), B.stride(0), _ptr(cand), nb, A.size(1),
                                      _ptr(tails), _ptr(thr), _ptr(greater), _ptr(equal), st),
               "rgcn_allpairs_rank")
    correct(0, nq, thr)
    return greater.to(torch.int64) + 1, equal.to(torch.int64)


def ranking_metrics(ranks: torch.Tensor, k_values=(1, 3, 10, 50, 100), ties: Optional[torch.Tensor] = None,
                    tie_policy: str = "optimistic") -> dict:
    """MRR / mean / median rank / Hits@K as assembled at src/evaluate.py:278-291.

    ``median_rank`` is numpy's median (the MEAN of the two middle order statistics for an even count, as
    ``np.median(ranks)`` at src/evaluate.py:283; ``torch.median`` would return the lower one).
    Ties: ``rank_true_tails`` returns the OPTIMISTIC rank 1 + #{strictly greater}; the reference's position in an
    unstable ``argsort`` is arbitrary inside [rank, rank + ties].  ``tie_policy="mean"`` (needs ``ties``) reports the
    expected rank rank + ties / 2 instead, ``"pessimistic"`` rank + ties."""
    r = ranks.to(torch.float64)
    if tie_policy != "optimistic":
        if ties is None:
            raise ValueError("tie_policy needs the tie counts returned by rank_true_tails")
        if tie_policy == "mean":
            r = r + ties.to(torch.float64) / 2
        elif tie_policy == "pessimistic":
            r = r + ties.to(torch.float64)
        else:
            raise ValueError("tie_policy must be optimistic, mean or pessimistic")
    out = {"mrr": float((1.0 / r).mean()), "mean_rank": float(r.mean()),
           "median_rank": float(torch.quantile(r, 0.5)) if r.numel() else float("nan"), "tie_policy": tie_policy}
    for k in k_values:
        out[f"hits@{k}"] = float((r <= k).double().mean())
    return out

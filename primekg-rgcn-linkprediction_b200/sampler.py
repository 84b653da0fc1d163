"""Device-side negative sampler with the interface of the reference's ``NegativeSampler`` (src/train.py:43-97).

``sample(pos_head, pos_tail, pos_rel)`` returns the corrupted triples like the reference; ``batch(...)`` returns the whole
mini-batch the training loop assembles from them (src/train.py:281-288: positives, then negatives, labels 1 / 0) from one
kernel.  Random numbers come from a counter-based generator (seed drawn from torch's generator at construction, device
counter advanced by every call), so a captured CUDA graph draws fresh negatives on every replay.  By default, the same
distribution as the reference (head or tail with probability 1/2, replacement uniform over all nodes,
``repeat_interleave`` order), not the same stream of numbers as ``torch.rand`` / ``torch.randint``.

Options, all applied inside the same kernel (``rgcn_link_batch_ex``) and so inside a captured training step:

* ``filter`` (a ``KnownTriples``): filtered negatives — a corruption that is a known triple is redrawn;
* ``constraints`` (a ``RelationConstraints``): type-constrained negatives (Krompaß et al. 2015) — an end of relation r
  is replaced only by a node that r admits on that side;
* ``head_prob``: the probability of replacing the head, one float or one per relation — e.g.
  ``KnownTriples.bernoulli_head_prob()``, the Bernoulli choice of Wang et al. 2014.

A negative is redrawn at most ``max_tries - 1`` times; one that is still rejected keeps its last draw (label 0 all the
same) and adds one to the device counter ``exhausted``.
"""
from __future__ import annotations

import math
from typing import Optional, Sequence, Union

import torch

from . import ops
from .rank import KnownTriples, _lex_order


def _int_tensor(t, what: str) -> torch.Tensor:
    t = torch.as_tensor(t)
    if t.numel() and (t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool):
        raise ValueError(f"{what} must hold integer ids")
    return t.reshape(-1).to(torch.int64)


class RelationConstraints:
    """Admissible heads and tails per relation: a type-constrained negative of relation r replaces its head (tail)
    only by a node of r's admissible-head (-tail) list; an empty list admits every node.  Stored CSR style, as the
    sampler kernel reads it: ``head_offsets`` int64 [R + 1] into ``head_nodes`` int32 (distinct within a relation),
    ``tail_offsets`` / ``tail_nodes`` likewise.  Every table must live on the device the sampler runs on."""

    def __init__(self, head_offsets: torch.Tensor, head_nodes: torch.Tensor, tail_offsets: torch.Tensor,
                 tail_nodes: torch.Tensor, num_nodes: int, num_relations: int):
        if not (0 < num_nodes < 2 ** 31 and num_relations > 0):
            raise ValueError("RelationConstraints: need 0 < num_nodes < 2^31 and num_relations > 0")
        self.num_nodes, self.num_relations = int(num_nodes), int(num_relations)
        self.device = head_offsets.device
        tables = []
        for side, off, nodes in (("head", head_offsets, head_nodes), ("tail", tail_offsets, tail_nodes)):
            if off.device != self.device or nodes.device != self.device:
                raise ValueError("RelationConstraints: all tables must be on one device")
            off, nodes = _int_tensor(off, f"{side}_offsets"), _int_tensor(nodes, f"{side}_nodes")
            if off.numel() != num_relations + 1:
                raise ValueError(f"RelationConstraints: {side}_offsets must have num_relations + 1 = "
                                 f"{num_relations + 1} entries")
            if int(off[0]) != 0 or int(off[-1]) != nodes.numel() or bool((off[1:] < off[:-1]).any()):
                raise ValueError(f"RelationConstraints: {side}_offsets must rise from 0 to len({side}_nodes)")
            if nodes.numel() and (int(nodes.min()) < 0 or int(nodes.max()) >= num_nodes):
                raise ValueError(f"RelationConstraints: {side}_nodes holds ids outside [0, {num_nodes})")
            rel = torch.repeat_interleave(torch.arange(num_relations, device=self.device), off[1:] - off[:-1])
            o = _lex_order(rel, nodes)
            r_s, n_s = rel[o], nodes[o]
            if bool(((r_s[1:] == r_s[:-1]) & (n_s[1:] == n_s[:-1])).any()):
                raise ValueError(f"RelationConstraints: a relation lists a {side} twice (it would be drawn more often)")
            if nodes.numel() == 0:              # every list empty, but the kernel takes a non-null pointer
                nodes = torch.zeros(1, dtype=torch.int64, device=self.device)
            tables += [off.contiguous(), nodes.to(torch.int32).contiguous()]
        self.head_offsets, self.head_nodes, self.tail_offsets, self.tail_nodes = tables

    def tables(self):
        """(head_offsets, head_nodes, tail_offsets, tail_nodes), the ``constraints`` of ``ops.link_batch_ex``."""
        return self.head_offsets, self.head_nodes, self.tail_offsets, self.tail_nodes

    def admissible(self, relation: int, side: str) -> torch.Tensor:
        """The admissible ``side`` ("head" / "tail") list of ``relation``, int64 (empty: every node)."""
        off, nodes = (self.head_offsets, self.head_nodes) if side == "head" else (self.tail_offsets, self.tail_nodes)
        return nodes[int(off[relation]):int(off[relation + 1])].to(torch.int64)

    @classmethod
    def from_lists(cls, heads: Sequence, tails: Sequence, num_nodes: int, device=None) -> "RelationConstraints":
        """Explicit lists: ``heads[r]`` / ``tails[r]`` are the admissible heads / tails of relation r (integer sequences
        or tensors; ``None`` or empty = every node).  Duplicates are dropped."""
        if len(heads) != len(tails) or len(heads) == 0:
            raise ValueError("RelationConstraints.from_lists: heads and tails need one list per relation")
        tables = []
        for side, lists in (("head", heads), ("tail", tails)):
            parts = [torch.zeros(0, dtype=torch.int64)]
            for r, x in enumerate(lists):
                t = torch.zeros(0, dtype=torch.int64) if x is None else _int_tensor(x, f"{side}s[{r}]").cpu()
                if t.numel() and (int(t.min()) < 0 or int(t.max()) >= num_nodes):
                    raise ValueError(f"RelationConstraints: {side}s[{r}] holds ids outside [0, {num_nodes})")
                parts.append(torch.unique(t))
            off = torch.zeros(len(lists) + 1, dtype=torch.int64)
            off[1:] = torch.cumsum(torch.tensor([p.numel() for p in parts[1:]], dtype=torch.int64), 0)
            tables += [off.to(device), torch.cat(parts).to(device)]
        return cls(*tables, num_nodes, len(heads))

    @classmethod
    def from_node_types(cls, known: KnownTriples, node_type: torch.Tensor) -> "RelationConstraints":
        """Constraints from node types: the admissible heads (tails) of relation r are all nodes whose type occurs as
        a head (tail) of r in ``known``.  ``node_type``: integer tensor [num_nodes] of types >= 0.  A relation that
        admits every type on a side, or that has no triples, gets an empty list there (every node: the same draws
        without a table read)."""
        N, R = known.num_nodes, known.num_relations
        if not isinstance(node_type, torch.Tensor) or node_type.dim() != 1 or node_type.numel() != N:
            raise ValueError(f"node_type must be a 1-D tensor of num_nodes = {N} entries")
        dev = known.device
        nt = _int_tensor(node_type, "node_type").to(dev)
        if int(nt.min()) < 0:
            raise ValueError("node_type must hold types >= 0")
        T = int(nt.max()) + 1
        count = torch.bincount(nt, minlength=T)
        start = torch.cumsum(count, 0) - count
        order = torch.argsort(nt, stable=True)              # nodes grouped by type, ascending within a type
        rels = known.keys % R
        tables = []
        for ends in (known.keys // R, known.tails.to(torch.int64)):
            present = torch.zeros(R, T, dtype=torch.bool, device=dev)
            present[rels, nt[ends]] = True
            present[present.sum(1) == int((count > 0).sum())] = False      # every type: empty list
            pr, pt = present.nonzero(as_tuple=True)                        # relation-major
            cnt = count[pt]
            seg = torch.repeat_interleave(torch.arange(pr.numel(), device=dev), cnt)
            within = torch.arange(int(cnt.sum()), device=dev) - (torch.cumsum(cnt, 0) - cnt)[seg]
            nodes, rel_of = order[start[pt][seg] + within], pr[seg]
            nodes = nodes[_lex_order(rel_of, nodes)]
            off = torch.zeros(R + 1, dtype=torch.int64, device=dev)
            off[1:] = torch.cumsum(torch.bincount(rel_of, minlength=R), 0)
            tables += [off, nodes]
        return cls(*tables, N, R)


class NegativeSampler:
    """``NegativeSampler(num_nodes, num_neg_samples)`` draws the reference's negatives; ``filter``, ``constraints`` and
    ``head_prob`` (a float, or a float tensor [num_relations]) select filtered, type-constrained and Bernoulli
    negatives (module docstring).  ``exhausted`` is the device counter (int64 [1]) of negatives that kept a rejected
    draw, created with the step counter by the first call.  After its first call, ``batch`` neither allocates (given
    ``out``) nor synchronises, so ``GraphedTrainStep(sampler=...)`` captures it."""

    def __init__(self, num_nodes: int, num_neg_samples: int = 1, *, filter: Optional[KnownTriples] = None,
                 constraints: Optional[RelationConstraints] = None, head_prob: Union[float, torch.Tensor] = 0.5,
                 max_tries: int = 32):
        self.num_nodes = int(num_nodes)
        self.num_neg_samples = int(num_neg_samples)
        self._seed = int(torch.randint(0, 2 ** 31 - 1, (1,)).item())
        self._ctr = None
        self.exhausted: Optional[torch.Tensor] = None
        self._ticket = None
        if isinstance(max_tries, bool) or int(max_tries) != max_tries or max_tries < 1:
            raise ValueError("max_tries must be an integer >= 1")
        self.max_tries = int(max_tries)
        if filter is not None and not isinstance(filter, KnownTriples):
            raise TypeError("filter must be a KnownTriples")
        if constraints is not None and not isinstance(constraints, RelationConstraints):
            raise TypeError("constraints must be a RelationConstraints")
        tabled = [t for t in (filter, constraints) if t is not None]
        for t in tabled:
            if t.num_nodes != self.num_nodes:
                raise ValueError(f"{type(t).__name__} has num_nodes={t.num_nodes}, the sampler {self.num_nodes}")
        rel_counts = {t.num_relations for t in tabled}
        if isinstance(head_prob, torch.Tensor):
            rel_counts.add(head_prob.numel())
        if len(rel_counts) > 1:
            raise ValueError(f"filter, constraints and head_prob disagree on the number of relations: {sorted(rel_counts)}")
        self.num_relations = rel_counts.pop() if rel_counts else 0
        if len({t.device for t in tabled}) > 1:
            raise ValueError("filter and constraints must be on one device")
        self._device = tabled[0].device if tabled else None
        self._filter = None if filter is None else (filter.keys, filter.tails)
        self._types = None if constraints is None else constraints.tables()
        self._head_prob = self._check_head_prob(head_prob)

    def _check_head_prob(self, head_prob) -> Optional[torch.Tensor]:
        R = self.num_relations
        if isinstance(head_prob, torch.Tensor):
            if head_prob.dim() != 1 or not head_prob.dtype.is_floating_point:
                raise ValueError(f"head_prob must be a float or a 1-D float tensor of num_relations = {R} entries")
            hp = head_prob.detach().to(torch.float32)
            if not bool(((hp >= 0) & (hp <= 1)).all()):
                raise ValueError("head_prob must lie in [0, 1]")
            return hp.to(self._device).contiguous() if self._device is not None else hp.contiguous()
        p = float(head_prob)
        if not (math.isfinite(p) and 0.0 <= p <= 1.0):
            raise ValueError("head_prob must lie in [0, 1]")
        if p == 0.5:
            return None                         # the kernel's default: exactly the reference's coin
        if R == 0:
            raise ValueError("head_prob other than 1/2 needs the number of relations: pass filter=, constraints= or a "
                             "[num_relations] tensor")
        return torch.full((R,), p, dtype=torch.float32, device=self._device)

    def _counter(self, device):
        if self._ctr is None or self._ctr.device != device:
            if self._device is not None and self._device != device:
                raise ValueError(f"the sampler's tables are on {self._device}, the positives on {device}")
            self._ctr = ops.rng_counter(device)
            self.exhausted = torch.zeros(1, dtype=torch.int64, device=device)
            self._ticket = torch.zeros(1, dtype=torch.int32, device=device)
            if self._head_prob is not None:
                self._head_prob = self._head_prob.to(device)
        return self._ctr

    def batch(self, pos_head: torch.Tensor, pos_tail: torch.Tensor, pos_rel: torch.Tensor, out=None):
        """(all_heads, all_tails, all_rels, labels) of src/train.py:281-288."""
        if not pos_head.is_cuda:
            raise RuntimeError("the device-side sampler needs CUDA tensors")
        ctr = self._counter(pos_head.device)
        return ops.link_batch_ex(pos_head, pos_tail, pos_rel, self.num_nodes, self.num_neg_samples, self._seed, ctr,
                                 out=out, num_rel=self.num_relations, head_prob=self._head_prob, filter=self._filter,
                                 constraints=self._types, max_tries=self.max_tries, exhausted=self.exhausted,
                                 ticket=self._ticket)

    def sample(self, pos_head: torch.Tensor, pos_tail: torch.Tensor, pos_rel: torch.Tensor):
        n = pos_head.numel()
        h, t, r, _ = self.batch(pos_head, pos_tail, pos_rel)
        return h[n:], t[n:], r[n:]

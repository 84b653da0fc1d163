"""CPU tests of the filtered / type-constrained negative sampler's host side: the entry point is exported, its argument
struct matches the header, it rejects bad arguments before any CUDA call, and NegativeSampler / RelationConstraints
validate their inputs at construction."""
import ctypes
import os
import shutil
import subprocess

import pytest
import torch

from conftest import ROOT


def test_sampler_entry_point_is_exported(lib_built):
    from primekg_rgcn_linkprediction_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    assert hasattr(lib, "rgcn_link_batch_ex") and "rgcn_link_batch_ex" in _lib.PROTOTYPES
    assert _lib.load().rgcn_abi_version() == _lib.ABI_VERSION == 8


def test_link_batch_args_match_header_layout(tmp_path):
    from primekg_rgcn_linkprediction_b200 import _lib
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    A = _lib.LinkBatchArgs
    names = [f for f, _ in A._fields_]
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "rgcn_b200.h"\n'
                   'int main(void){printf("%zu", sizeof(rgcn_link_batch_args));' +
                   "".join(f'printf(" %zu", offsetof(rgcn_link_batch_args, {n}));' for n in names) +
                   'printf("\\n");return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(t) for t in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [ctypes.sizeof(A)] + [getattr(A, n).offset for n in names]


def _fake(addr=4096):
    return ctypes.c_void_p(addr)          # never dereferenced: validation fails first


def _args(**kw):
    from primekg_rgcn_linkprediction_b200 import _lib
    a = _lib.LinkBatchArgs(pos_head=_fake(), pos_tail=_fake(), pos_rel=_fake(), n_pos=16, num_neg=4, num_rel=3,
                           num_nodes=100, seed=1, max_tries=8, counter=_fake(), heads=_fake(), tails=_fake(),
                           rels=_fake(), labels=_fake(), ticket=_fake())
    for k, v in kw.items():
        setattr(a, k, v)
    return a


@pytest.mark.parametrize("case,msg", [
    (dict(n_pos=-1), "bad sizes"), (dict(num_neg=-1), "bad sizes"), (dict(num_nodes=0), "bad sizes"),
    (dict(num_nodes=1 << 32), "bad sizes"), (dict(num_rel=-1), "bad sizes"), (dict(n_filter=-1), "bad sizes"),
    (dict(n_pos=1 << 31, num_neg=2), "2^32"),
    (dict(max_tries=0), "max_tries"), (dict(max_tries=-3), "max_tries"),
    (dict(filter_keys=_fake()), "filter_keys and filter_tails"),
    (dict(filter_tails=_fake(), n_filter=10), "filter_keys and filter_tails"),
    (dict(n_filter=10), "filter_keys and filter_tails"),
    (dict(head_offsets=_fake()), "four type-constraint tables"),
    (dict(head_offsets=_fake(), head_nodes=_fake(), tail_offsets=_fake()), "four type-constraint tables"),
    (dict(tail_nodes=_fake()), "four type-constraint tables"),
    (dict(num_rel=0, head_prob=_fake()), "num_rel > 0"),
    (dict(num_rel=0, filter_keys=_fake(), filter_tails=_fake(), n_filter=5), "num_rel > 0"),
    (dict(num_nodes=1 << 31, filter_keys=_fake(), filter_tails=_fake(), n_filter=5), "< 2^31"),
    (dict(counter=None), "null argument"), (dict(labels=None), "null argument"),
])
def test_link_batch_ex_rejects_bad_arguments_without_gpu(lib_built, case, msg):
    """Argument validation happens before any CUDA call, so it is testable here."""
    from primekg_rgcn_linkprediction_b200 import _lib
    lib = _lib.load()
    rc = lib.rgcn_link_batch_ex(ctypes.byref(_args(**case)), None)
    assert rc == 1, case
    assert "link_batch" in _lib.last_error() and msg in _lib.last_error(), _lib.last_error()
    assert lib.rgcn_link_batch_ex(None, None) == 1 and "null args" in _lib.last_error()
    # nothing to draw: no CUDA call, success
    assert lib.rgcn_link_batch_ex(ctypes.byref(_args(n_pos=0)), None) == 0


@pytest.fixture
def cpu_known(monkeypatch):
    """KnownTriples on the CPU (it insists on CUDA tensors; nothing here launches a kernel)."""
    from primekg_rgcn_linkprediction_b200 import KnownTriples
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))
    # node types [0, 0, 1, 1, 2, 2, 3, 3]; relation 2 has no triples
    h = [0, 1, 2, 4, 0, 0, 2, 4, 6, 4]
    r = [0, 0, 1, 1, 1, 3, 3, 3, 3, 1]
    t = [2, 3, 4, 6, 5, 6, 7, 6, 7, 6]          # the last triple repeats (4, 1, 6)
    return KnownTriples(torch.tensor(h), torch.tensor(r), torch.tensor(t), 8, 4)


NODE_TYPE = torch.tensor([0, 0, 1, 1, 2, 2, 3, 3])


def test_constraints_from_node_types_hand_worked(lib_built, cpu_known):
    from primekg_rgcn_linkprediction_b200 import RelationConstraints
    c = RelationConstraints.from_node_types(cpu_known, NODE_TYPE)
    # r0: heads of type 0 -> {0, 1}, tails of type 1 -> {2, 3}
    # r1: heads of types 1, 2, 0 -> {0 .. 5}, tails of types 2, 3 -> {4 .. 7}
    # r2: no triples -> every node (empty list)
    # r3: heads of every type -> every node (empty list), tails of type 3 -> {6, 7}
    heads = [[0, 1], [0, 1, 2, 3, 4, 5], [], []]
    tails = [[2, 3], [4, 5, 6, 7], [], [6, 7]]
    for r in range(4):
        assert c.admissible(r, "head").tolist() == heads[r], r
        assert c.admissible(r, "tail").tolist() == tails[r], r
    assert c.head_offsets.tolist() == [0, 2, 8, 8, 8] and c.tail_offsets.tolist() == [0, 2, 6, 6, 8]
    assert c.head_nodes.dtype == c.tail_nodes.dtype == torch.int32
    e = RelationConstraints.from_lists(heads, [[3, 2, 2], [4, 5, 6, 7], None, [7, 6]], 8)
    for r in range(4):
        assert e.admissible(r, "head").tolist() == heads[r] and e.admissible(r, "tail").tolist() == tails[r]


def test_bernoulli_head_prob_hand_worked(lib_built, cpu_known):
    # r3: 4 triples, 4 distinct heads (tph 1), 2 distinct tails (hpt 2) -> 1 / 3; r2 has no triples -> 1/2
    p = cpu_known.bernoulli_head_prob()
    assert p.dtype == torch.float32
    torch.testing.assert_close(p, torch.tensor([0.5, 0.5, 0.5, 1 / 3]))


def test_constraints_reject_bad_input(lib_built, cpu_known):
    from primekg_rgcn_linkprediction_b200 import RelationConstraints
    with pytest.raises(ValueError, match="outside"):
        RelationConstraints.from_lists([[0, 8]], [[1]], 8)
    with pytest.raises(ValueError, match="outside"):
        RelationConstraints.from_lists([[0]], [[-1]], 8)
    with pytest.raises(ValueError, match="one list per relation"):
        RelationConstraints.from_lists([[0], [1]], [[1]], 8)
    with pytest.raises(ValueError, match="integer"):
        RelationConstraints.from_lists([[0.5]], [[1]], 8)
    off, nodes = torch.tensor([0, 2]), torch.tensor([1, 2])
    with pytest.raises(ValueError, match="num_relations \\+ 1"):
        RelationConstraints(off, nodes, off, nodes, 8, 2)
    with pytest.raises(ValueError, match="rise from 0"):
        RelationConstraints(torch.tensor([0, 3]), nodes, off, nodes, 8, 1)
    with pytest.raises(ValueError, match="twice"):
        RelationConstraints(off, torch.tensor([1, 1]), off, nodes, 8, 1)
    with pytest.raises(ValueError, match="outside"):
        RelationConstraints(off, nodes, off, torch.tensor([1, 8]), 8, 1)
    with pytest.raises(ValueError, match="num_nodes"):
        RelationConstraints.from_node_types(cpu_known, NODE_TYPE[:7])
    with pytest.raises(ValueError, match=">= 0"):
        RelationConstraints.from_node_types(cpu_known, NODE_TYPE - 1)


def test_negative_sampler_validates_at_construction(lib_built, cpu_known):
    from primekg_rgcn_linkprediction_b200 import NegativeSampler, RelationConstraints
    types = RelationConstraints.from_node_types(cpu_known, NODE_TYPE)
    NegativeSampler(8, 4, filter=cpu_known, constraints=types, head_prob=cpu_known.bernoulli_head_prob(), max_tries=1)
    with pytest.raises(ValueError, match="num_nodes"):
        NegativeSampler(9, 4, filter=cpu_known)
    with pytest.raises(ValueError, match="num_nodes"):
        NegativeSampler(9, 4, constraints=types)
    three = RelationConstraints.from_lists([[0], [1], [2]], [[0], [1], [2]], 8)
    with pytest.raises(ValueError, match="number of relations"):
        NegativeSampler(8, 4, filter=cpu_known, constraints=three)
    with pytest.raises(ValueError, match="number of relations"):
        NegativeSampler(8, 4, filter=cpu_known, head_prob=torch.full((3,), 0.5))
    for p in (-0.1, 1.5, float("nan"), float("inf")):
        with pytest.raises(ValueError, match="\\[0, 1\\]"):
            NegativeSampler(8, 4, filter=cpu_known, head_prob=p)
    with pytest.raises(ValueError, match="\\[0, 1\\]"):
        NegativeSampler(8, 4, filter=cpu_known, head_prob=torch.tensor([0.5, 0.5, float("nan"), 0.5]))
    with pytest.raises(ValueError, match="\\[0, 1\\]"):
        NegativeSampler(8, 4, filter=cpu_known, head_prob=torch.tensor([0.5, 0.5, 1.01, 0.5]))
    with pytest.raises(ValueError, match="1-D float"):
        NegativeSampler(8, 4, filter=cpu_known, head_prob=torch.full((2, 2), 0.5))
    with pytest.raises(ValueError, match="1-D float"):
        NegativeSampler(8, 4, filter=cpu_known, head_prob=torch.zeros(4, dtype=torch.int64))
    with pytest.raises(ValueError, match="number of relations"):
        NegativeSampler(8, 4, head_prob=0.3)                  # nothing says how many relations there are
    for bad in (0, -1, 2.5, True):
        with pytest.raises(ValueError, match="max_tries"):
            NegativeSampler(8, 4, filter=cpu_known, max_tries=bad)
    with pytest.raises(TypeError, match="KnownTriples"):
        NegativeSampler(8, 4, filter=(cpu_known.keys, cpu_known.tails))
    # the plain sampler keeps its constructor
    s = NegativeSampler(8, 2)
    assert s.num_relations == 0 and s.exhausted is None
    s = NegativeSampler(8, 2, head_prob=torch.tensor([0.0, 1.0]))
    assert s.num_relations == 2

"""CPU tests of the filtered ranking / novel-link top-k host side: the excluding entry points are exported and validate
their arguments before any CUDA call; KnownTriples and the candidate mapping reject bad input."""
import ctypes

import pytest
import torch

NEW_SYMBOLS = ("rgcn_scores_rank_excl_w", "rgcn_scores_topk_excl_w", "rgcn_rank_excl_correct")


def test_excluding_entry_points_are_exported(lib_built):
    from primekg_rgcn_linkprediction_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for n in NEW_SYMBOLS:
        assert hasattr(lib, n) and n in _lib.PROTOTYPES
    assert _lib.load().rgcn_abi_version() == _lib.ABI_VERSION == 8


def _fake(addr=4096):
    return ctypes.c_void_p(addr)          # never dereferenced: validation fails first


@pytest.mark.parametrize("nulls", [(1, 0, 0), (0, 1, 0), (0, 0, 1), (1, 1, 0), (0, 1, 1)])
def test_partially_null_exclusion_lists_are_rejected(lib_built, nulls):
    from primekg_rgcn_linkprediction_b200 import _lib
    lib = _lib.load()
    xb, xe, xp = (None if n else _fake() for n in nulls)
    rc = lib.rgcn_scores_rank_excl_w(_fake(), _fake(), 64, 64, _fake(256), 100, 10, _fake(), _fake(), _fake(), _fake(),
                                     xb, xe, xp, None)
    assert rc == 1 and "all null or none" in _lib.last_error()
    rc = lib.rgcn_scores_topk_excl_w(_fake(), _fake(), 64, 64, _fake(256), 100, 10, 5, 1.0, 0.0, _fake(), _fake(),
                                     _fake(), 1000, _fake(), _fake(), xb, xe, xp, None)
    assert rc == 1 and "all null or none" in _lib.last_error()


def test_excluding_entry_points_reject_bad_sizes(lib_built):
    from primekg_rgcn_linkprediction_b200 import _lib
    lib = _lib.load()
    rc = lib.rgcn_scores_rank_excl_w(_fake(), _fake(), 64, 64, _fake(256), 100, -1, _fake(), _fake(), _fake(), _fake(),
                                     _fake(), _fake(), _fake(), None)
    assert rc == 1 and "bad sizes" in _lib.last_error()
    rc = lib.rgcn_scores_topk_excl_w(_fake(), _fake(), 64, 64, _fake(256), 100, 10, 17, 1.0, 0.0, _fake(), _fake(),
                                     _fake(), 1000, _fake(), _fake(), _fake(), _fake(), _fake(), None)
    assert rc == 1 and "1 <= k" in _lib.last_error()
    for nq, ncand in ((-1, 10), (10, -1)):
        rc = lib.rgcn_rank_excl_correct(_fake(), 16, None, 0, None, 0, None, 16, nq, ncand, _fake(), _fake(), _fake(),
                                        _fake(), _fake(), _fake(), _fake(), None)
        assert rc == 1 and "negative size" in _lib.last_error()
    rc = lib.rgcn_rank_excl_correct(_fake(), 16, None, 0, None, 0, None, 16, 10, 10, _fake(), _fake(), None, _fake(),
                                    _fake(), _fake(), _fake(), None)
    assert rc == 1 and "null argument" in _lib.last_error()
    rc = lib.rgcn_rank_excl_correct(_fake(), 8, None, 0, None, 0, None, 16, 10, 10, _fake(), _fake(), _fake(), _fake(),
                                    _fake(), _fake(), _fake(), None)
    assert rc == 1 and "ld < n_cand" in _lib.last_error()
    rc = lib.rgcn_rank_excl_correct(None, 0, None, 0, None, 0, None, 16, 10, 10, _fake(), _fake(), _fake(), _fake(),
                                    _fake(), _fake(), _fake(), None)
    assert rc == 1 and "operands" in _lib.last_error()
    # nothing to do: no CUDA call, success
    assert lib.rgcn_rank_excl_correct(None, 0, None, 0, None, 0, None, 16, 0, 10, None, None, None, None, None, None,
                                      None, None) == 0


def test_known_triples_rejects_bad_input(lib_built):
    from primekg_rgcn_linkprediction_b200 import KnownTriples
    h = torch.tensor([0, 1, 2])
    r = torch.tensor([0, 1, 0])
    t = torch.tensor([3, 4, 5])
    with pytest.raises(ValueError, match="out of range"):
        KnownTriples(h, r, torch.tensor([3, 4, 6]), 6, 2)          # tail id 6 with 6 nodes
    with pytest.raises(ValueError, match="out of range"):
        KnownTriples(h, torch.tensor([0, 2, 0]), t, 6, 2)          # relation 2 with 2 relations
    with pytest.raises(ValueError, match="out of range"):
        KnownTriples(torch.tensor([-1, 1, 2]), r, t, 6, 2)
    with pytest.raises(ValueError, match="CUDA"):
        KnownTriples(h, r, t, 6, 2)                                # valid ids, but on the CPU
    with pytest.raises(ValueError, match="one length"):
        KnownTriples(h, r[:2], t, 6, 2)
    with pytest.raises(ValueError, match="integer"):
        KnownTriples(h.float(), r, t, 6, 2)
    with pytest.raises(ValueError, match="from_graphs needs"):
        KnownTriples.from_graphs()


def test_candidates_must_be_distinct_graph_nodes(lib_built):
    from primekg_rgcn_linkprediction_b200.rank import _check_candidates
    _check_candidates(torch.tensor([4, 0, 2]), 5)
    with pytest.raises(ValueError, match="distinct"):
        _check_candidates(torch.tensor([4, 0, 4]), 5)
    with pytest.raises(ValueError, match="outside"):
        _check_candidates(torch.tensor([4, 5]), 5)


def test_exclude_relation_needs_exclude(lib_built):
    import primekg_rgcn_linkprediction_b200 as pkg
    e = torch.zeros(4, 8)
    with pytest.raises(ValueError, match="exclude_relation needs exclude"):
        pkg.topk_all_pairs(e, torch.tensor([0]), torch.tensor([1, 2]), k=1, exclude_relation=0)

"""RGCNConv(aggr=, root_weight=, bias=, is_sorted=) on the host: the oracle's statement of PyG's loop path (mean equals
the pinned oracle, gradchecks, torch's tie rule for max by hand) and the constructor (aliases, rejected aggregations,
PyG-shaped state dicts for every combination, strict loads)."""
import itertools

import pytest
import torch

from aggr_oracle import RGCNConvAggrRef, aggregate_ref, rgcn_conv_aggr_ref
from oracle import rgcn_ref as O


def _graph(seed=0, N=12, E=60, R=3):
    g = torch.Generator().manual_seed(seed)
    ei = torch.randint(0, N, (2, E), generator=g)
    et = torch.randint(0, R, (E,), generator=g)
    return ei, et, N, R


def test_mean_oracle_equals_the_pinned_oracle_in_fp64():
    ei, et, N, R = _graph()
    g = torch.Generator().manual_seed(1)
    x = torch.randn(N, 8, dtype=torch.float64, generator=g)
    W = torch.randn(R, 8, 5, dtype=torch.float64, generator=g)
    root = torch.randn(8, 5, dtype=torch.float64, generator=g)
    b = torch.randn(5, dtype=torch.float64, generator=g)
    torch.testing.assert_close(rgcn_conv_aggr_ref(x, ei, et, W, root, b, "mean"), O.rgcn_conv_ref(x, ei, et, W, root, b),
                               rtol=0, atol=1e-12)


@pytest.mark.parametrize("aggr", ["sum", "add", "max"])
@pytest.mark.parametrize("root_bias", [(True, True), (False, True), (True, False), (False, False)])
def test_oracle_gradcheck_tie_free(aggr, root_bias):
    ei, et, N, R = _graph(2, N=7, E=25, R=2)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(N, 3, dtype=torch.float64, generator=g).requires_grad_()     # continuous draws: no ties
    W = torch.randn(R, 3, 2, dtype=torch.float64, generator=g).requires_grad_()
    root = torch.randn(3, 2, dtype=torch.float64, generator=g).requires_grad_() if root_bias[0] else None
    b = torch.randn(2, dtype=torch.float64, generator=g).requires_grad_() if root_bias[1] else None
    args = [t for t in (x, W, root, b) if t is not None]

    def f(*a):
        it = iter(a)
        xx, WW = next(it), next(it)
        rr = next(it) if root is not None else None
        bb = next(it) if b is not None else None
        return rgcn_conv_aggr_ref(xx, ei, et, WW, rr, bb, aggr)
    assert torch.autograd.gradcheck(f, args)


def _max_grad(vals):
    """Gradient of h = max of ``vals`` (all into one destination) for each source, by torch's autograd."""
    x = torch.tensor(vals, dtype=torch.float64).unsqueeze(1).requires_grad_()
    src = torch.arange(len(vals))
    h = aggregate_ref(x, src, torch.zeros(len(vals), dtype=torch.int64), 1, "max")
    h.sum().backward()
    return h.item(), x.grad.squeeze(1).tolist()


def test_max_ties_by_hand():
    # the zero initial value counts as a tie when the maximum is exactly 0
    assert _max_grad([0.0, 0.0]) == (0.0, [1 / 3, 1 / 3])
    assert _max_grad([1.0, 1.0, -2.0]) == (1.0, [0.5, 0.5, 0.0])
    assert _max_grad([-1.0, -3.0]) == (-1.0, [1.0, 0.0])          # an all-negative segment gives its max, not 0
    assert _max_grad([0.0, -1.0]) == (0.0, [0.5, 0.0])
    assert _max_grad([2.0]) == (2.0, [1.0])


def test_max_empty_segment_and_nan():
    x = torch.tensor([[1.0, float("nan")], [3.0, 2.0]])
    h = aggregate_ref(x, torch.tensor([0, 1]), torch.tensor([0, 0]), 3, "max")
    assert h[0, 0] == 3.0 and torch.isnan(h[0, 1])
    assert torch.equal(h[1:], torch.zeros(2, 2))


# ---- the constructor -------------------------------------------------------------------------------------------------
def _pkg():
    import primekg_rgcn_linkprediction_b200 as pkg
    return pkg


@pytest.mark.parametrize("aggr,canon", [("mean", "mean"), ("add", "sum"), ("sum", "sum"), ("max", "max")])
def test_aggr_aliases(aggr, canon):
    conv = _pkg().RGCNConv(8, 8, 3, aggr=aggr)
    assert conv._aggr == canon and conv.aggr == aggr
    assert ("aggr=" in repr(conv)) == (canon != "mean")


@pytest.mark.parametrize("aggr", ["min", "mul", "Max", ["mean", "max"], None, 1])
def test_unsupported_aggregations_raise(aggr):
    with pytest.raises(ValueError, match="mean, sum and max"):
        _pkg().RGCNConv(8, 8, 3, aggr=aggr)


def test_aggregation_module_raises():
    with pytest.raises(ValueError):
        _pkg().RGCNConv(8, 8, 3, aggr=torch.nn.Identity())


COMBOS = list(itertools.product([None, 2], [None, 4], ["mean", "add", "max"], [True, False], [True, False]))


@pytest.mark.parametrize("num_bases,num_blocks,aggr,root_weight,bias",
                         [c for c in COMBOS if not (c[0] is not None and c[1] is not None)])
def test_state_dict_is_pyg_shaped(num_bases, num_blocks, aggr, root_weight, bias):
    kw = dict(num_bases=num_bases, num_blocks=num_blocks, aggr=aggr, root_weight=root_weight, bias=bias)
    torch.manual_seed(0)
    ref = RGCNConvAggrRef(8, 16, 3, is_sorted=True, **kw)
    conv = _pkg().RGCNConv(8, 16, 3, is_sorted=True, **kw)
    sd, rsd = conv.state_dict(), ref.state_dict()
    assert list(sd) == list(rsd)
    assert all(sd[k].shape == rsd[k].shape for k in sd)
    assert (conv.root is None) != root_weight and (conv.bias is None) != bias
    conv.load_state_dict(rsd, strict=True)
    ref.load_state_dict(conv.state_dict(), strict=True)
    for k in sd:
        assert torch.equal(conv.state_dict()[k], rsd[k])
    # same draws in PyG's order: a seeded construction gives the reference's values
    torch.manual_seed(0)
    again = _pkg().RGCNConv(8, 16, 3, **kw)
    for k in sd:
        assert torch.equal(again.state_dict()[k], rsd[k]), k
    r = repr(conv)
    assert ("root_weight=False" in r) != root_weight and ("bias=False" in r) != bias


def test_models_take_aggr_and_keep_their_layout():
    pkg = _pkg()
    for aggr in ("mean", "sum", "max"):
        m = pkg.DrugDiseaseModel(100, 5, aggr=aggr)
        assert all(c._aggr == aggr for c in m.encoder._layers())
    ref = pkg.DrugDiseaseModel(1000, 30)
    big = pkg.DrugDiseaseModel(1000, 30, aggr="add")
    assert [(k, v.shape) for k, v in big.state_dict().items()] == [(k, v.shape) for k, v in ref.state_dict().items()]


def test_partitioned_encoder_rejects_max():
    from primekg_rgcn_linkprediction_b200 import dist as D
    plan = D.plan_partition(torch.tensor([0, 1, 2, 3]), 4, 1)
    with pytest.raises(ValueError, match="mean' and 'sum'"):
        D.PartitionedRGCN(plan, 0, 2, 8, 8, aggr="max")
    enc = D.PartitionedRGCN(plan, 0, 2, 8, 8, aggr="add")
    assert all(c._aggr == "sum" for c in enc.convs)

"""Block-diagonal relation weights, RGCNConv(num_blocks=nb), on the host: PyG's constructor rules, parameter layout
and init stream, the oracle against its independent dense formulation, and the argument checks of the two C entry
points (they return before any CUDA call)."""
import ctypes

import pytest
import torch

from blocks_oracle import (ModelBlocksRef, RGCNConvBlocksRef, diag_blocks, expand_blocks, rgcn_conv_blocks_ref)
from oracle import rgcn_ref as O


def _pkg():
    import primekg_rgcn_linkprediction_b200 as pkg
    return pkg


@pytest.mark.parametrize("kw,match", [(dict(num_bases=4, num_blocks=4), "both"),
                                      (dict(num_blocks=3), "divide"),
                                      (dict(num_blocks=128), "divide"),
                                      (dict(num_blocks=0), "divide")])
def test_constructor_rejects_pyg_invalid_arguments(kw, match):
    with pytest.raises(ValueError, match=match):
        _pkg().RGCNConv(64, 256, 30, **kw)


def test_constructor_keeps_the_multiple_of_four_rule():
    with pytest.raises(ValueError, match="multiples of 4"):
        _pkg().RGCNConv(6, 6, 3, num_blocks=3)              # divisible, but not a multiple of 4
    with pytest.raises(ValueError, match="divide"):
        _pkg().RGCNConv(64, 20, 3, num_blocks=8)            # 20 % 8


def test_block_layer_parameters_and_repr():
    conv = _pkg().RGCNConv(64, 256, 30, num_blocks=16)
    assert conv.weight.shape == (30, 16, 4, 16) and conv.comp is None
    assert conv.root.shape == (64, 256) and conv.bias.shape == (256,)
    assert [k for k, _ in conv.named_parameters()] == ["weight", "root", "bias"]
    assert "num_blocks=16" in repr(conv)
    assert "num_blocks" not in repr(_pkg().RGCNConv(64, 256, 30))
    with pytest.raises(RuntimeError, match="CUDA"):
        conv.relation_weights()                              # no CPU path


def test_model_state_dict_has_pyg_block_shapes():
    m = _pkg().DrugDiseaseModel(500, 30, 64, 256, num_blocks=4)
    sd = m.state_dict()
    assert not any(k.endswith(".comp") for k in sd)
    assert sd["encoder.conv1.weight"].shape == (30, 4, 16, 64)
    assert sd["encoder.conv2.weight"].shape == (30, 4, 64, 64)
    assert sd["encoder.conv1.root"].shape == (64, 256) and sd["encoder.conv2.bias"].shape == (256,)
    m3 = _pkg().DrugDiseaseModel(500, 30, 64, 256, num_blocks=4, num_layers=3)
    assert m3.state_dict()["encoder.extra_convs.0.weight"].shape == (30, 4, 64, 64)
    enc = _pkg().DrugDiseaseRGCN(500, 30, 64, 128, num_blocks=8)
    assert enc.conv2.weight.shape == (30, 8, 16, 16)


def test_seeded_init_draws_the_oracle_stream():
    torch.manual_seed(7)
    conv = _pkg().RGCNConv(64, 256, 30, num_blocks=4)
    torch.manual_seed(7)
    ref = RGCNConvBlocksRef(64, 256, 30, 4)
    for k, v in ref.state_dict().items():
        assert torch.equal(conv.state_dict()[k], v), k
    a = (6.0 / (16 + 64)) ** 0.5                             # glorot over the last two dims
    wmax = float(conv.weight.detach().abs().max())
    assert 0.9 * a < wmax <= a
    torch.manual_seed(11)
    m = _pkg().DrugDiseaseModel(300, 5, 64, 128, num_blocks=4)
    torch.manual_seed(11)
    r = ModelBlocksRef(300, 5, 64, 128, num_blocks=4)
    sd = m.state_dict()
    assert set(sd) == set(r.state_dict())
    for k, v in r.state_dict().items():
        assert torch.equal(sd[k], v), k
    m.load_state_dict(r.state_dict(), strict=True)           # checkpoints move both ways


def _tiny_graph(N=11, E=40, R=3, seed=0):
    g = torch.Generator().manual_seed(seed)
    ei = torch.randint(0, N, (2, E), generator=g)
    et = torch.randint(0, R, (E,), generator=g)
    return ei, et, g


@pytest.mark.parametrize("d_in,d_out,nb", [(8, 8, 1), (8, 12, 4), (6, 4, 2), (16, 32, 8)])
def test_oracle_block_layer_equals_dense_formulation(d_in, d_out, nb):
    ei, et, g = _tiny_graph()
    R = 3
    x = torch.randn(11, d_in, generator=g, dtype=torch.float64)
    w = torch.randn(R, nb, d_in // nb, d_out // nb, generator=g, dtype=torch.float64)
    root = torch.randn(d_in, d_out, generator=g, dtype=torch.float64)
    bias = torch.randn(d_out, generator=g, dtype=torch.float64)
    W = expand_blocks(w)
    assert W.shape == (R, d_in, d_out) and torch.equal(diag_blocks(W, nb), w)
    assert int((W != 0).sum()) == int((w != 0).sum())        # nothing off the blocks
    got = rgcn_conv_blocks_ref(x, ei, et, w, root, bias)
    torch.testing.assert_close(got, O.rgcn_conv_dense_ref(x, ei, et, W, root, bias), rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(got, O.rgcn_conv_ref(x, ei, et, W, root, bias), rtol=1e-12, atol=1e-12)


def test_oracle_block_layer_gradcheck():
    ei, et, g = _tiny_graph(N=7, E=20)
    x = torch.randn(7, 8, generator=g, dtype=torch.float64, requires_grad=True)
    w = torch.randn(3, 4, 2, 3, generator=g, dtype=torch.float64, requires_grad=True)
    root = torch.randn(8, 12, generator=g, dtype=torch.float64, requires_grad=True)
    bias = torch.randn(12, generator=g, dtype=torch.float64, requires_grad=True)
    assert torch.autograd.gradcheck(lambda *a: rgcn_conv_blocks_ref(a[0], ei, et, *a[1:]), (x, w, root, bias))


def test_block_entry_points_argument_errors_without_gpu(lib_built):
    from primekg_rgcn_linkprediction_b200 import _lib
    lib = _lib.load()
    for fn, name in ((lib.rgcn_block_diag_expand, "block_diag_expand"), (lib.rgcn_block_diag_gather, "block_diag_gather")):
        assert fn(None, 2, 4, 4, 4, None, None) == 1 and name in _lib.last_error()          # null matrices
        assert fn(256, 0, 4, 4, 4, 512, None) == 1 and "R, nb, bi, bo" in _lib.last_error()
        assert fn(256, 2, 4, 0, 4, 512, None) == 1
        assert fn(256, 2, 4, 4, -1, 512, None) == 1
        assert fn(256, 2, 1 << 12, 1 << 10, 4, 512, None) == 1 and "2^20" in _lib.last_error()
        assert fn(260, 2, 4, 4, 4, 512, None) == 1 and "16-byte" in _lib.last_error()
        assert fn(256, 1 << 10, 1, 1 << 11, 1 << 11, 512, None) == 1 and "2^31" in _lib.last_error()
        with pytest.raises(_lib.RGCNLibraryError):
            _lib.check(fn(None, 1, 1, 1, 1, None, None), name)
    assert ctypes.c_int32 in _lib.PROTOTYPES["rgcn_block_diag_expand"][1]

"""CPU tests of the optimiser step's host side: the C structs match their ctypes mirrors, rgcn_adam_step rejects bad
arguments before any CUDA call, and FusedAdam refuses what it does not implement."""
import ctypes
import os
import shutil
import subprocess

import pytest
import torch

from conftest import ROOT


def test_adam_structs_match_header_layout(tmp_path):
    from primekg_rgcn_linkprediction_b200 import _lib
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "rgcn_b200.h"\n'
                   'int main(void){printf("%zu %zu %zu %zu %zu %zu %d\\n", sizeof(rgcn_adam_segment),'
                   'offsetof(rgcn_adam_segment, numel), offsetof(rgcn_adam_segment, group), sizeof(rgcn_adam_hparams),'
                   'offsetof(rgcn_adam_hparams, weight_decay), offsetof(rgcn_adam_hparams, decoupled_weight_decay),'
                   'RGCN_ADAM_MAX_SEGMENTS);return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(t) for t in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    S, H = _lib.AdamSegment, _lib.AdamHparams
    want = [ctypes.sizeof(S), S.numel.offset, S.group.offset, ctypes.sizeof(H), H.weight_decay.offset,
            H.decoupled_weight_decay.offset, _lib.ADAM_MAX_SEGMENTS]
    assert got == want


def _segments(n, numel=8, group=0, null=None):
    from primekg_rgcn_linkprediction_b200 import _lib
    fake = 0x10000
    segs = (_lib.AdamSegment * max(n, 1))()
    for s in range(n):
        segs[s] = _lib.AdamSegment(fake, fake, fake, fake, fake, numel, group)
        if null:
            setattr(segs[s], null, None)
    return segs


@pytest.mark.parametrize("case", ["negative_segments", "too_many", "null_table", "null_hparams", "negative_numel",
                                  "bad_group", "null_grad", "null_step", "nan_max_norm", "small_workspace"])
def test_adam_step_argument_errors_without_gpu(lib_built, case):
    """Argument validation happens before any CUDA call, so it is testable here."""
    from primekg_rgcn_linkprediction_b200 import _lib
    lib = _lib.load()
    hp, ws = ctypes.c_void_p(0x20000), ctypes.c_void_p(0x30000)
    nbytes = lib.rgcn_adam_workspace_bytes(8, 1)
    args = dict(segs=_segments(1), n=1, hp=hp, groups=1, clip=1.0, ws=ws, nbytes=nbytes)
    if case == "negative_segments":
        args["n"] = -1
    elif case == "too_many":
        args.update(segs=_segments(_lib.ADAM_MAX_SEGMENTS + 1), n=_lib.ADAM_MAX_SEGMENTS + 1)
    elif case == "null_table":
        args["segs"] = None
    elif case == "null_hparams":
        args["hp"] = None
    elif case == "negative_numel":
        args["segs"] = _segments(1, numel=-4)
    elif case == "bad_group":
        args["segs"] = _segments(1, group=1)
    elif case == "null_grad":
        args["segs"] = _segments(1, null="grad")
    elif case == "null_step":
        args["segs"] = _segments(1, null="step")
    elif case == "nan_max_norm":
        args["clip"] = float("nan")
    elif case == "small_workspace":
        args["nbytes"] = 8
    rc = lib.rgcn_adam_step(args["segs"], args["n"], args["hp"], args["groups"], args["clip"], None, args["ws"],
                            args["nbytes"], None)
    assert rc == 1, case
    assert "adam_step" in _lib.last_error()
    with pytest.raises(_lib.RGCNLibraryError):
        _lib.check(rc, "rgcn_adam_step")


def test_adam_workspace_bytes_covers_every_block(lib_built):
    from primekg_rgcn_linkprediction_b200 import _lib
    lib = _lib.load()
    assert lib.rgcn_adam_workspace_bytes(-1, 1) == 0
    # 64 header bytes + one fp64 partial per 4096-float block (every segment may add a partial block)
    assert lib.rgcn_adam_workspace_bytes(2_300_000, 9) >= 64 + 8 * (2_300_000 // 4096 + 9)


def _p(*shape, **kw):
    return torch.nn.Parameter(torch.zeros(*shape, **kw))


@pytest.mark.parametrize("kw", [dict(amsgrad=True), dict(maximize=True), dict(differentiable=True),
                                dict(foreach=True), dict(fused=True), dict(max_grad_norm=-1.0)])
def test_fused_adam_rejects_unsupported_options(lib_built, kw):
    with pytest.raises(ValueError):
        lib_built.FusedAdam([_p(4)], **kw)


def test_fused_adam_rejects_cpu_parameters(lib_built):
    with pytest.raises(RuntimeError, match="CUDA"):
        lib_built.FusedAdam([_p(4)])
    with pytest.raises(RuntimeError, match="CUDA"):
        lib_built.FusedAdamW([_p(4)])


def test_fused_adam_rejects_bad_parameter_layouts(lib_built, monkeypatch):
    """dtype, layout and device checks (parameters pretend to be CUDA tensors: nothing is launched at construction)."""
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))
    with pytest.raises(ValueError, match="float32"):
        lib_built.FusedAdam([_p(4, dtype=torch.float64)])
    with pytest.raises(ValueError, match="contiguous"):
        lib_built.FusedAdam([torch.nn.Parameter(torch.zeros(4, 4).t())])
    with pytest.raises(ValueError, match="contiguous"):
        lib_built.FusedAdam([torch.nn.Parameter(torch.zeros(4).to_sparse())])
    with pytest.raises(ValueError, match="at most"):
        lib_built.FusedAdam([_p(4) for _ in range(65)])


def test_fused_adam_state_dict_groups_have_torch_adam_keys(lib_built, monkeypatch):
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))
    ps = [_p(4)]
    ours = lib_built.FusedAdam(ps, lr=1e-2, max_grad_norm=1.0).state_dict()["param_groups"][0]
    ref = torch.optim.Adam(ps, lr=1e-2).state_dict()["param_groups"][0]
    assert list(ours) == list(ref)
    w = lib_built.FusedAdamW(ps).state_dict()["param_groups"][0]
    assert list(w) == list(torch.optim.AdamW(ps).state_dict()["param_groups"][0])
    assert w["decoupled_weight_decay"] is True and w["weight_decay"] == 1e-2

"""CPU tests of the host side: the C-ABI library builds, loads and exports every symbol the header
declares (no compute without a GPU); module surface, state-dict layout, seeded init order; the synthetic
workload generator; loud failure on CPU tensors."""
import ctypes
import os
import re

import pytest
import torch

from conftest import ROOT, load_golden
from oracle import rgcn_ref as O


def _header_symbols():
    src = open(os.path.join(ROOT, "include", "rgcn_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"^\s*(?:int|size_t|int64_t|int32_t)\s+(rgcn_\w+)\s*\(", src, flags=re.M)))


def test_library_exports_every_header_symbol(lib_built):
    from primekg_rgcn_linkprediction_b200 import _lib
    names = _header_symbols()
    assert len(names) >= 12
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/rgcn_b200.h but not exported"
    assert set(names) == set(_lib.PROTOTYPES), "ctypes prototypes and header disagree"
    assert _lib.load().rgcn_abi_version() == _lib.ABI_VERSION == 8


def test_library_argument_errors_without_gpu(lib_built):
    """Argument validation happens before any CUDA call, so it is testable here."""
    from primekg_rgcn_linkprediction_b200 import _lib
    lib = _lib.load()
    rc = lib.rgcn_csr_build(None, None, None, -1, 1, 1, 1, None, None, None, None, None, None, None, None, None,
                            None, 0, None)
    assert rc == 1 and "negative" in _lib.last_error()
    g = _lib.CsrStruct()
    rc = lib.rgcn_aggregate_fwd(ctypes.byref(g), None, 0, 6, None, 0, None, None, 0, 0, None, 0, None, None, 0, None, 0, None)
    assert rc == 1
    with pytest.raises(_lib.RGCNLibraryError):
        _lib.check(rc, "rgcn_aggregate_fwd")


def test_csr_struct_matches_header_layout():
    from primekg_rgcn_linkprediction_b200 import _lib
    # 3 pointers, 2 int64, 4 int32, 4 pointers, 1 int64
    assert ctypes.sizeof(_lib.CsrStruct) == 3 * 8 + 2 * 8 + 4 * 4 + 4 * 8 + 8
    assert _lib.CsrStruct.hub_keys.offset == 56


def test_arg_structs_match_header_layout(tmp_path):
    """The header is plain C: compile it with gcc and compare sizeof / offsetof with the ctypes mirrors."""
    import shutil
    import subprocess
    from primekg_rgcn_linkprediction_b200 import _lib
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "rgcn_b200.h"\n'
                   'int main(void){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(rgcn_csr_t), sizeof(rgcn_layer_fwd_args),'
                   'sizeof(rgcn_layer_bwd_args), offsetof(rgcn_layer_bwd_args, rows), offsetof(rgcn_layer_bwd_args, ldac),'
                   'offsetof(rgcn_layer_fwd_args, gemm_workspace_bytes), offsetof(rgcn_layer_fwd_args, pipeline),'
                   'offsetof(rgcn_layer_bwd_args, w_planes), offsetof(rgcn_csr_t, order_chunk_rows),'
                   'offsetof(rgcn_layer_fwd_args, dropout_row0));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(t) for t in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    want = [ctypes.sizeof(_lib.CsrStruct), ctypes.sizeof(_lib.LayerFwdArgs), ctypes.sizeof(_lib.LayerBwdArgs),
            _lib.LayerBwdArgs.rows.offset, _lib.LayerBwdArgs.ldac.offset, _lib.LayerFwdArgs.gemm_workspace_bytes.offset,
            _lib.LayerFwdArgs.pipeline.offset, _lib.LayerBwdArgs.w_planes.offset, _lib.CsrStruct.order_chunk_rows.offset,
            _lib.LayerFwdArgs.dropout_row0.offset]
    assert got == want


def test_module_surface_and_state_dict(lib_built):
    pkg = lib_built
    m = pkg.DrugDiseaseModel(30926, 3)
    assert sum(p.numel() for p in m.parameters()) == 2_078_208         # reference results/results.json:29
    ref = O.ModelRef(30926, 3)
    assert list(m.state_dict().keys()) == list(ref.state_dict().keys())
    for k, v in ref.state_dict().items():
        assert m.state_dict()[k].shape == v.shape, k
    for attr in ("node_embeddings", "conv1", "conv2", "dropout", "num_nodes", "num_relations", "embedding_dim",
                 "hidden_dim"):
        assert hasattr(m.encoder, attr)
    assert hasattr(m.decoder, "relation_embeddings") and hasattr(m.decoder, "score_all_tails")
    for meth in ("forward", "predict", "predict_all_tails", "get_embeddings"):
        assert callable(getattr(m, meth))
    mb = pkg.DrugDiseaseModel(50, 6, 16, 24, num_bases=2)
    assert mb.encoder.conv1.weight.shape == (2, 16, 24) and mb.encoder.conv1.comp.shape == (6, 2)
    g = load_golden("small_basis")
    mb2 = pkg.DrugDiseaseModel(g["num_nodes"], g["num_relations"], g["embedding_dim"], g["hidden_dim"],
                               num_bases=g["num_bases"])
    mb2.load_state_dict(g["state_dict"], strict=True)


@pytest.mark.parametrize("bases", [None, 4])
def test_seeded_init_draws_the_reference_stream(lib_built, bases):
    """Same seed => same parameters as the restated reference constructor (PyG glorot for the conv
    layers, xavier_uniform_ for both embedding tables, in the reference's construction order)."""
    torch.manual_seed(123)
    a = lib_built.DrugDiseaseModel(300, 5, 32, 48, num_bases=bases)
    torch.manual_seed(123)
    b = O.ModelRef(300, 5, 32, 48, num_bases=bases)
    for (k, p), (k2, q) in zip(a.state_dict().items(), b.state_dict().items()):
        assert k == k2 and torch.equal(p, q), k


def test_cpu_tensors_fail_loudly(lib_built):
    pkg = lib_built
    m = pkg.DrugDiseaseModel(10, 2, 8, 8)
    ei = torch.tensor([[0, 1], [1, 2]])
    et = torch.tensor([0, 1])
    idx = torch.tensor([0])
    with pytest.raises(RuntimeError, match="no CPU"):
        m(ei, et, idx, idx, idx)
    with pytest.raises(RuntimeError, match="no CPU"):
        m.decoder(torch.randn(1, 8), torch.randn(1, 8), idx)
    with pytest.raises(RuntimeError):
        pkg.RGCNConv(8, 8, 2)(torch.randn(3, 8), ei, et)


def test_dropin_module_file_exports_the_reference_names(lib_built):
    import importlib
    mod = importlib.import_module("src.models.rgcn")
    for n in ("DrugDiseaseRGCN", "LinkPredictor", "DrugDiseaseModel"):
        assert getattr(mod, n) is getattr(lib_built, n)


def test_synthetic_primekg_subgraph_shape():
    from primekg_rgcn_linkprediction_b200 import synth
    kg = synth.primekg_subgraph()
    assert kg.num_nodes == 30_926 and kg.num_relations == 3 and kg.num_edges == 849_456
    ei, et = kg.edge_index, kg.edge_type
    assert ei.dtype == torch.int64 and et.dtype == torch.int64
    # consecutive (a->b),(b->a) columns of the same type: reference src/preprocess.py:228-234
    assert torch.equal(ei[0, 0::2], ei[1, 1::2]) and torch.equal(ei[1, 0::2], ei[0, 1::2])
    assert torch.equal(et[0::2], et[1::2])
    blocks = synth.CFG1_BLOCKS
    for r, (a, b, _) in enumerate(synth.CFG1_RELS):
        s, d = ei[0, 0::2][et[0::2] == r], ei[1, 0::2][et[0::2] == r]
        assert int(s.min()) >= blocks[a][0] and int(s.max()) < blocks[a][1]
        assert int(d.min()) >= blocks[b][0] and int(d.max()) < blocks[b][1]
    again = synth.primekg_subgraph()
    assert torch.equal(again.edge_index, ei)                         # seeded => reproducible
    deg = torch.bincount(ei[1], minlength=kg.num_nodes)
    assert int(deg.max()) > 2000 and float(deg.float().median()) < 30    # hubs + a long tail
    h, t, rl, y = synth.link_batch(kg, 1024)
    assert h.shape == t.shape == rl.shape == y.shape == (2048,) and int(y.sum()) == 1024


def test_synthetic_full_kg_shape():
    from primekg_rgcn_linkprediction_b200 import synth
    kg = synth.primekg_full(num_directed_edges=200_000)
    assert kg.num_nodes == 129_375 and kg.num_relations == 30 and kg.num_edges == 200_000
    assert int(kg.edge_type.max()) == 29 and int(kg.edge_index.max()) < 129_375


def test_rowsparse_handover_guards(lib_built, monkeypatch):
    """Host logic of the row-sparse hand-over (rowsparse.py), on CPU tensors: the announcement is honoured only for the very
    buffer that was announced, untouched, and is consumed by the first claim."""
    from primekg_rgcn_linkprediction_b200 import rowsparse
    monkeypatch.delenv("PRIMEKG_RGCN_SPARSE_BWD", raising=False)
    rowsparse.clear()
    rowsparse.stats.update(claimed=0, declined=0)
    dense = torch.zeros(100, 8)
    rows = torch.tensor([3, 7, 3])
    rowsparse.announce(dense, rows)
    got = rowsparse.claim(dense)
    assert got[0] is rows and got[1] is None and rowsparse.claim(dense) is None         # consumed
    rowsparse.announce(dense, rows)
    assert rowsparse.claim(dense.clone()) is None                                      # another buffer (engine summed a copy)
    rowsparse.announce(dense, rows)
    dense.add_(1.0)                                                                    # in-place accumulation bumps the version
    assert rowsparse.claim(dense) is None
    rowsparse.announce(dense, rows)
    assert rowsparse.claim(dense[:50]) is None                                         # same storage, other shape
    rowsparse.announce(dense, torch.arange(60))                                        # longer than MAX_FRACTION * N
    assert rowsparse.claim(dense) is None
    assert rowsparse.stats["claimed"] == 1 and rowsparse.stats["declined"] == 4
    monkeypatch.setenv("PRIMEKG_RGCN_SPARSE_BWD", "0")
    rowsparse.announce(dense, rows)
    assert rowsparse.claim(dense) is None                                              # switched off: nothing announced
    # second hand-over (masked planes): off by default, keyed on the mask tensor, scale and mode
    monkeypatch.setenv("PRIMEKG_RGCN_SPARSE_BWD", "1")
    mask = torch.ones(100, 8)
    rowsparse.announce_planes(dense, mask, 2.0, "fp32", "payload")
    assert rowsparse.claim_planes(dense, mask, 2.0, "fp32") is None                    # opt-in only
    monkeypatch.setenv("PRIMEKG_RGCN_PLANES_HANDOVER", "1")
    rowsparse.announce_planes(dense, mask, 2.0, "fp32", "payload")
    assert rowsparse.claim_planes(dense, mask, 2.0, "fp32") == "payload"
    rowsparse.announce_planes(dense, mask, 2.0, "fp32", "payload")
    assert rowsparse.claim_planes(dense, mask.clone(), 2.0, "fp32") is None            # another mask tensor
    rowsparse.announce_planes(dense, mask, 2.0, "fp32", "payload")
    assert rowsparse.claim_planes(dense, mask, 1.0, "fp32") is None                    # another dropout scale
    rowsparse.clear()


def test_listed_rows_switches_and_output_mark(lib_built, monkeypatch):
    """Host logic of the listed-rows last layer: the environment switches, and the mark that lets the decoder's backward
    leave the unlisted gradient rows undefined — honoured only for the very tensor that was marked, untouched, consumed by
    the first look, dropped by any layer forward that computes all rows."""
    from primekg_rgcn_linkprediction_b200 import dist_fused, modules, ops, rowsparse
    for k in ("PRIMEKG_RGCN_SPARSE_FWD", "PRIMEKG_RGCN_SPARSE_BWD", "RGCN_MARK_SOURCES", "RGCN_PEER_PUSH"):
        monkeypatch.delenv(k, raising=False)
    assert modules.sparse_forward_enabled() and dist_fused.listed_last_layer() and ops.mark_sources()
    assert not dist_fused.push_after_transform()
    monkeypatch.setenv("PRIMEKG_RGCN_SPARSE_FWD", "0")
    assert not modules.sparse_forward_enabled() and not dist_fused.listed_last_layer()
    monkeypatch.setenv("PRIMEKG_RGCN_SPARSE_FWD", "1")
    monkeypatch.setenv("PRIMEKG_RGCN_SPARSE_BWD", "0")                 # the listed forward needs the row-sparse backward
    assert not modules.sparse_forward_enabled() and not dist_fused.listed_last_layer()
    monkeypatch.setenv("RGCN_MARK_SOURCES", "0")
    assert not ops.mark_sources() and ops.MARK_SOURCES_RATIO >= 8
    rowsparse.clear()
    out = torch.zeros(50, 8)
    assert not rowsparse.is_listed_output(out)
    rowsparse.mark_listed_output(out)
    assert rowsparse.is_listed_output(out) and not rowsparse.is_listed_output(out)          # consumed by the first look
    rowsparse.mark_listed_output(out)
    assert not rowsparse.is_listed_output(out.clone())                                      # another tensor
    rowsparse.mark_listed_output(out)
    out.add_(1.0)
    assert not rowsparse.is_listed_output(out)                                              # written since
    rowsparse.mark_listed_output(out)
    rowsparse.unmark_listed_output()                                                        # a dense layer forward ran
    assert not rowsparse.is_listed_output(out)
    rowsparse.clear()


def test_model_forward_on_cpu_indices_keeps_the_dense_encoder(lib_built, monkeypatch):
    """``DrugDiseaseModel._encode_for`` only takes the listed form for CUDA index tensors with autograd on; anything else
    goes through ``encoder(...)`` (here: stubbed, so the routing alone is checked on the CPU box)."""
    import primekg_rgcn_linkprediction_b200 as pkg
    m = pkg.DrugDiseaseModel(20, 2, 8, 8)
    calls = []
    monkeypatch.setattr(m.encoder, "_encode", lambda *a, **k: calls.append(("listed", a[3] if len(a) > 3 else k.get("read_rows"))) or "L")
    monkeypatch.setattr(type(m.encoder), "forward", lambda self, ei, et, node_indices=None: calls.append(("dense", None)) or "D")
    h = torch.tensor([1, 2]); t = torch.tensor([3, 4])
    assert m._encode_for(None, None, h, t) == "D"                                           # CPU indices
    with torch.no_grad():
        assert m._encode_for(None, None, h, t) == "D"
    assert [c[0] for c in calls] == ["dense", "dense"]


def test_grad_arena_slices(lib_built):
    """ops.GradArena: call-order slices of one flat buffer, 256-byte aligned, reset per step, overflow falls back."""
    from primekg_rgcn_linkprediction_b200 import ops
    arena = ops.GradArena(64 * 4, "cpu")
    a = arena.take(3, 5)
    b = arena.take(64)
    assert a.shape == (3, 5) and a.data_ptr() == arena.buf.data_ptr() and b.data_ptr() == arena.buf.data_ptr() + 64 * 4
    assert arena.used.numel() == 128
    assert arena.take(200) is None and arena.used.numel() == 128                        # too large: the caller allocates
    arena.reset()
    a2 = arena.take(3, 5)
    assert a2.data_ptr() == a.data_ptr()                                               # same slices every step
    ops.set_grad_arena(arena)
    try:
        arena.reset()
        g = ops.param_grad(4, 4, device=torch.device("cpu"))
        assert g.data_ptr() == arena.buf.data_ptr()
        big = ops.param_grad(1000, device=torch.device("cpu"))
        assert not (arena.buf.data_ptr() <= big.data_ptr() < arena.buf.data_ptr() + arena.buf.numel() * 4)
    finally:
        ops.set_grad_arena(None)
    assert ops.param_grad(4, device=torch.device("cpu")).data_ptr() != arena.buf.data_ptr()


def test_integration_doc_lists_every_abi_symbol():
    """INTEGRATION.md is the maintainer-facing map of the C ABI: every entry point of the header must appear in it."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, "include", "rgcn_b200.h")).read()
    doc = open(os.path.join(root, "INTEGRATION.md")).read()
    syms = sorted(set(re.findall(r"\b(rgcn_[a-z0-9_]+)\s*\(", hdr)))
    assert len(syms) >= 40
    missing = [s for s in syms if s not in doc]
    assert not missing, f"not documented in INTEGRATION.md: {missing}"


def test_ranking_metrics_median_is_numpys(lib_built):
    """src/evaluate.py:283 uses np.median: the MEAN of the two middle values for an even count."""
    import numpy as np
    from primekg_rgcn_linkprediction_b200 import ranking_metrics
    ranks = torch.tensor([1, 2, 10, 400, 7, 3])
    m = ranking_metrics(ranks, k_values=(1, 3, 10))
    assert m["median_rank"] == float(np.median(ranks.numpy())) == 5.0
    assert abs(m["mrr"] - float(np.mean(1.0 / ranks.numpy()))) < 1e-12 and m["hits@3"] == 0.5
    ties = torch.tensor([0, 2, 0, 0, 0, 1])
    mean = ranking_metrics(ranks, k_values=(3,), ties=ties, tie_policy="mean")
    assert mean["mean_rank"] == float((ranks.double() + ties.double() / 2).mean()) and mean["hits@3"] == 1 / 3
    with pytest.raises(ValueError):
        ranking_metrics(ranks, tie_policy="mean")

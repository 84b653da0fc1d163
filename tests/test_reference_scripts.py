"""The north_star boundary claim, exercised: the reference's OWN ``src/train.py`` and ``src/evaluate.py`` — imported
from the checkout of the original project named by ``$PRIMEKG_RGCN_REFERENCE``, where they lie, unmodified — run on
top of this repo's drop-in ``src/models/rgcn.py``.

No GPU here, so the kernels under the module trio are the CPU stand-ins of tests/cpu_ops_emulation.py (same role as in
tests/test_dist.py); everything above them — constructors, ``.to(device)``, the graph cache, autograd wiring of both
layers, the fused decoder hand-over, eval-mode caching, state-dict keys, checkpoint save / load — is the product code.
The sequence of model-API calls the scripts make is recorded and must equal the committed
tests/golden/ref_call_sequence.json, which tests/test_gpu_reference_calls.py replays against the real kernels."""
import json
import os

import numpy as np
import pytest
import torch

import ref_harness as H
from conftest import GOLDEN

pytestmark = pytest.mark.skipif(not H.reference_present(),
                                reason="needs a checkout of the original project: set PRIMEKG_RGCN_REFERENCE")


@pytest.fixture(scope="module")
def ref_run(tmp_path_factory, lib_built):
    import cpu_ops_emulation as emu
    mp = pytest.MonkeyPatch()
    try:
        emu.install_full(mp, lib_built)
        rec = H.CallRecorder({})
        out = H.run_reference_scripts(str(tmp_path_factory.mktemp("ref_run")), rec)
        out["calls"] = rec.calls
        yield out
    finally:
        mp.undo()


def test_train_py_runs_unchanged(ref_run):
    ck = ref_run["checkpoint"]
    assert ck["epoch"] == 2 and len(ck["train_losses"]) == 2 and len(ck["val_losses"]) == 2
    assert all(np.isfinite(v) for v in ck["train_losses"] + ck["val_losses"])
    assert ck["train_losses"][1] < ck["train_losses"][0]            # Adam on BCE: the loss goes down
    # checkpoint keys = the reference's (src/train.py:430-441); state-dict keys = PyG's parameter names
    assert set(ck) >= {"epoch", "model_state_dict", "optimizer_state_dict", "best_val_loss", "best_val_acc", "args"}
    assert list(ck["model_state_dict"]) == [
        "encoder.node_embeddings.weight", "encoder.conv1.weight", "encoder.conv1.root", "encoder.conv1.bias",
        "encoder.conv2.weight", "encoder.conv2.root", "encoder.conv2.bias", "decoder.relation_embeddings.weight"]
    assert os.path.exists(ref_run["best_path"]) and os.path.exists(ref_run["final_path"])


def test_evaluate_py_loads_and_ranks(ref_run):
    info, ranking = ref_run["info"], ref_run["ranking"]
    assert info["num_nodes"] == H.DATA["num_nodes"] and info["num_relations"] == 3 and info["hidden_dim"] == 128
    assert info["num_parameters"] == 600 * 64 + (3 * 64 * 128 + 64 * 128 + 128) + (3 * 128 * 128 + 128 * 128 + 128) + 3 * 128
    assert 0 < ranking["mrr"] <= 1 and 1 <= ranking["median_rank"] <= 600 and ranking["hits@50"] >= ranking["hits@10"]
    n_test = int(ref_run["test"]["edge_index"].size(1))
    assert ref_run["scores"].shape == (2 * n_test,) and ref_run["labels"].sum() == n_test
    # the reference's rank loop (argsort per row) against this repo's ranking on the same embeddings
    from oracle import rgcn_ref as O
    m = ref_run["model"]
    with torch.no_grad():
        emb = m.encoder(ref_run["full"]["edge_index"], ref_run["full"]["edge_type"])
        ei, et = ref_run["test"]["edge_index"], ref_run["test"]["edge_type"]
        s = m.decoder.score_all_tails(emb[ei[0]], et, emb)
    opt, pes = O.rank_of_true_tail_ref(s, ei[1])
    mrr_lo, mrr_hi = float((1.0 / pes.double()).mean()), float((1.0 / opt.double()).mean())
    assert mrr_lo - 1e-9 <= ranking["mrr"] <= mrr_hi + 1e-9


def test_call_sequence_matches_committed_fixture(ref_run):
    """What the scripts call, in order — the contract the GPU replay test is built from."""
    calls = ref_run["calls"]
    ops = [c["op"] for c in calls]
    assert ops.count("optimizer.step") == 2 * 5 and ops.count("backward") == 10      # 4,800 train columns / 1,024, 2 epochs
    assert "load_state_dict" in ops and "decoder.score_all_tails" in ops and "encoder.forward" in ops
    first = calls[0]
    assert first == dict(op="model.forward", graph="train", pairs=2048, training=True, grad=True)
    path = os.path.join(GOLDEN, "ref_call_sequence.json")
    assert os.path.exists(path), "run tests/golden/make_ref_calls.py"
    want = json.load(open(path))
    assert want["calls"] == calls, "the recorded call sequence changed: regenerate tests/golden/ref_call_sequence.json"

"""Self-contained CPU check of what the original project's scripts rely on.  tests/test_reference_scripts.py runs that
project's own src/train.py and src/evaluate.py, which are not part of this repository, so it skips without a checkout
of it.  The sequence of model-API calls those scripts make was recorded from them into
tests/golden/ref_call_sequence.json; here it is driven through this repo's drop-in ``src.models.rgcn`` (kernels = the CPU stand-ins of
tests/cpu_ops_emulation.py) on the same synthetic splits, under the recorder of tests/ref_harness.py.  Checked: the
drop-in makes no top-level model-API call of its own (the recorder sees the stored sequence again), the parameter count
and state-dict keys, a checkpoint written in train.py's layout and reloaded into a fresh model (same outputs, and the
same outputs as the oracle model loaded from that checkpoint), the training loss going down over the two epochs, and
``score_all_tails`` with evaluate.py's per-row argsort ranking against the oracle."""
import json
import os

import pytest
import torch
import torch.nn.functional as F

import ref_harness as H
from conftest import GOLDEN
from oracle import rgcn_ref as O

STATE_DICT_KEYS = ["encoder.node_embeddings.weight", "encoder.conv1.weight", "encoder.conv1.root",
                   "encoder.conv1.bias", "encoder.conv2.weight", "encoder.conv2.root", "encoder.conv2.bias",
                   "decoder.relation_embeddings.weight"]


def test_recorded_script_calls_replay_on_the_dropin(lib_built, tmp_path):
    import cpu_ops_emulation as emu
    from src.models.rgcn import DrugDiseaseModel
    doc = json.load(open(os.path.join(GOLDEN, "ref_call_sequence.json")))
    assert doc["data"] == json.loads(json.dumps(H.DATA))
    train, val, test, full, _ = H.build_splits(doc["data"])
    graphs = {"train": (train["edge_index"], train["edge_type"]), "full": (full["edge_index"], full["edge_type"])}
    m = doc["model"]
    N, R = m["num_nodes"], m["num_relations"]
    epochs = int(doc["train_argv"][doc["train_argv"].index("--epochs") + 1])

    def make_model():
        return DrugDiseaseModel(N, R, m["embedding_dim"], m["hidden_dim"])

    def oracle_from(state_dict):
        ref = O.ModelRef(N, R, m["embedding_dim"], m["hidden_dim"])
        ref.load_state_dict(state_dict)
        return ref.eval()

    g = torch.Generator().manual_seed(7)
    ckpt_path = tmp_path / "best_model.pt"
    test_ei, test_et = test["edge_index"], test["edge_type"]
    mp = pytest.MonkeyPatch()
    try:
        emu.install_full(mp, lib_built)
        torch.manual_seed(42)
        model = make_model()
        assert sum(p.numel() for p in model.parameters()) == m["num_parameters"]
        assert list(model.state_dict()) == STATE_DICT_KEYS
        rec = H.CallRecorder({int(ei.size(1)): name for name, (ei, _) in graphs.items()})
        opt = saved = ref = emb = last = None
        train_losses, n_ranked, n_checked = [], 0, 0
        with H.recording(rec):
            for c in doc["calls"]:
                op = c["op"]
                if op == "model.forward":
                    ei, et = graphs[c["graph"]]
                    pick = torch.randint(0, ei.size(1), (c["pairs"] // 2,), generator=g)
                    h, t, r, y = O.negative_batch_ref(ei[0][pick], ei[1][pick], et[pick], N, 1, generator=g)
                    model.train(c["training"])
                    with torch.set_grad_enabled(c["grad"]):
                        s = model(ei, et, h, t, r)
                    assert s.shape == (c["pairs"],) and s.requires_grad == c["grad"]
                    if ref is not None:                 # after evaluate.py's load_model: oracle on the same checkpoint
                        with torch.no_grad():
                            torch.testing.assert_close(s, ref(ei, et, h, t, r), rtol=1e-4, atol=1e-5)
                        n_checked += 1
                    last = (s, y)
                elif op == "backward":
                    loss = F.binary_cross_entropy_with_logits(*last)
                    loss.backward()
                    train_losses.append(float(loss.detach()))
                elif op == "clip_grad_norm_":
                    torch.nn.utils.clip_grad_norm_(model.parameters(), c["max_norm"])
                elif op == "optimizer.step":
                    if opt is None:
                        opt = getattr(torch.optim, c["optimizer"])(model.parameters(), lr=c["lr"],
                                                                   weight_decay=c["weight_decay"])
                    opt.step()
                    opt.zero_grad()
                elif op == "state_dict":
                    saved = model
                    torch.save({"epoch": len(train_losses), "model_state_dict": model.state_dict(),
                                "optimizer_state_dict": opt.state_dict(), "best_val_loss": 0.0, "best_val_acc": 0.0,
                                "args": {"argv": doc["train_argv"]}}, ckpt_path)
                elif op == "load_state_dict":
                    ck = torch.load(ckpt_path, map_location="cpu", weights_only=False)
                    assert list(ck["model_state_dict"]) == STATE_DICT_KEYS
                    model = make_model()
                    model.load_state_dict(ck["model_state_dict"])
                    model.eval()
                    ref = oracle_from(ck["model_state_dict"])
                elif op == "encoder.forward":
                    ei, et = graphs[c["graph"]]
                    model.train(c["training"])
                    with torch.set_grad_enabled(c["grad"]):
                        emb = model.encoder(ei, et)
                    with torch.no_grad():
                        torch.testing.assert_close(emb, ref.encoder(ei, et), rtol=1e-4, atol=1e-5)
                    n_checked += 1
                elif op == "decoder.score_all_tails":
                    sl = slice(n_ranked, n_ranked + c["heads"])           # evaluate.py walks the test edges in order
                    h, r, t = test_ei[0][sl], test_et[sl], test_ei[1][sl]
                    n_ranked += c["heads"]
                    with torch.no_grad():
                        s = model.decoder.score_all_tails(emb[h], r, emb)
                        assert s.shape == (c["heads"], c["tails"])
                        torch.testing.assert_close(s, ref.decoder.score_all_tails(emb[h], r, emb), rtol=1e-4, atol=1e-5)
                    best, worst = O.rank_of_true_tail_ref(s, t)
                    for i in range(c["heads"]):                   # the per-row argsort loop of evaluate.py
                        pos = int((torch.argsort(s[i], descending=True) == t[i]).nonzero()[0, 0]) + 1
                        assert int(best[i]) <= pos <= int(worst[i])
                    n_checked += 1
                elif op != "decoder.forward":
                    raise AssertionError(f"unknown recorded op {op}")
        assert rec.calls == doc["calls"], "the drop-in made model-API calls of its own"
        assert n_ranked == test_ei.size(1) and n_checked >= 6
        # the checkpoint round trip: the model evaluate.py loaded computes what the saved one did
        ei, et = graphs["full"]
        saved.eval()
        with torch.no_grad():
            assert torch.equal(model.encoder(ei, et), saved.encoder(ei, et))
    finally:
        mp.undo()
    per_epoch = len(train_losses) // epochs
    assert len(train_losses) == epochs * per_epoch
    means = [sum(train_losses[k * per_epoch:(k + 1) * per_epoch]) / per_epoch for k in range(epochs)]
    assert means[-1] < means[0], means                    # Adam on BCE: the loss goes down, as in train.py's log

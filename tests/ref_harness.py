"""TEST INFRASTRUCTURE: drives the reference's OWN scripts (``src/train.py``, ``src/evaluate.py`` of the checkout of the
original PrimeKG-RGCN-LinkPrediction project named by ``$PRIMEKG_RGCN_REFERENCE``, loaded from where they lie, never
copied) on top of this repo's drop-in ``src/models/rgcn.py``, and records the sequence of model-API calls they make.
Used by ``tests/test_reference_scripts.py`` (CPU: kernels replaced by ``tests/cpu_ops_emulation.py``) and by
``tests/golden/make_ref_calls.py`` (writes ``tests/golden/ref_call_sequence.json``, which
``tests/test_reference_call_replay.py`` drives through the drop-in on the CPU and ``tests/test_gpu_reference_calls.py``
replays against the real kernels on the B200)."""
import contextlib
import importlib.util
import os
import sys
import types

import torch

# the original project is not part of this repository: the tests that run its scripts skip without it
REF = os.environ.get("PRIMEKG_RGCN_REFERENCE", "")


def reference_present() -> bool:
    return bool(REF) and os.path.isfile(os.path.join(REF, "src", "train.py"))


# ---------------------------------------------------------------------------------------------------
# synthetic data/processed/ in the dict formats of reference src/preprocess.py:256-261 and :373-388
# ---------------------------------------------------------------------------------------------------
DATA = dict(num_nodes=600, num_relations=3, undirected=(2400, 300, 300), seed=123, invalid_val_pairs=3)


def build_splits(cfg=DATA):
    """(train, val, test, full, mappings): every undirected edge as two consecutive columns (a->b), (b->a) of one type
    (src/preprocess.py:228-241); ``full`` holds all of them; val carries a few rows with an index >= num_nodes, as the
    shipped val_data.pt does (train.py:572-586 filters them)."""
    g = torch.Generator().manual_seed(cfg["seed"])
    N, R = cfg["num_nodes"], cfg["num_relations"]
    out = []
    for k, und in enumerate(cfg["undirected"]):
        u = torch.rand(und, generator=g, dtype=torch.float64)
        a = torch.floor(N * u.pow(2.0)).clamp_(max=N - 1).to(torch.int64)         # skewed: hubs exist
        b = torch.randint(0, N, (und,), generator=g)
        r = torch.randint(0, R, (und,), generator=g)
        ei = torch.stack([torch.stack([a, b], 1).reshape(-1), torch.stack([b, a], 1).reshape(-1)], 0)
        et = r.repeat_interleave(2)
        out.append((ei, et))
    full_ei = torch.cat([e for e, _ in out], 1)
    full_et = torch.cat([t for _, t in out])

    def pack(ei, et):
        return {"edge_index": ei.contiguous(), "edge_type": et.contiguous(), "num_nodes": N, "num_relations": R}

    train, val, test = (pack(*o) for o in out)
    k = cfg["invalid_val_pairs"]
    if k:
        bad = torch.tensor([[N + 1, 5] * k, [5, N + 1] * k])
        val = pack(torch.cat([val["edge_index"], bad], 1), torch.cat([val["edge_type"], torch.zeros(2 * k, dtype=torch.int64)]))
    mappings = {"node2idx": {f"n{i}": i for i in range(N)}, "idx2node": {i: f"n{i}" for i in range(N)},
                "relation2idx": {f"r{i}": i for i in range(R)}, "idx2relation": {i: f"r{i}" for i in range(R)}}
    return train, val, test, pack(full_ei, full_et), mappings


def write_processed(dirpath, cfg=DATA):
    os.makedirs(dirpath, exist_ok=True)
    train, val, test, full, mappings = build_splits(cfg)
    for name, obj in (("train_data", train), ("val_data", val), ("test_data", test), ("full_graph", full),
                      ("mappings", mappings)):
        torch.save(obj, os.path.join(dirpath, name + ".pt"))
    return train, val, test, full


# ---------------------------------------------------------------------------------------------------
# loading the reference's scripts unchanged, with `src.models.rgcn` resolved to this repo's drop-in
# ---------------------------------------------------------------------------------------------------
def _stub_plotting_modules():
    """matplotlib / seaborn are not installed in this image; evaluate.py imports them at module level for its figure
    helpers (never called here).  Test-only stubs."""
    made = []
    for name in ("matplotlib", "matplotlib.pyplot", "seaborn"):
        if name not in sys.modules:
            m = types.ModuleType(name)
            def _getattr(attr):
                if attr.startswith("__"):
                    raise AttributeError(attr)
                return lambda *a, **k: None
            m.__dict__["__getattr__"] = _getattr
            sys.modules[name] = m
            made.append(name)
    if "matplotlib" in made:
        sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    return made


def load_reference_script(name: str):
    """Import the reference's src/<name>.py as a module.  Its ``from src.models.rgcn import DrugDiseaseModel`` finds this
    repo's ``src`` package, which is imported (and therefore in ``sys.modules``) first."""
    import src.models.rgcn as shim                       # this repo's drop-in
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    assert os.path.abspath(shim.__file__).startswith(root), shim.__file__
    _stub_plotting_modules()
    path = os.path.join(REF, "src", name + ".py")
    spec = importlib.util.spec_from_file_location("reference_" + name, path)
    mod = importlib.util.module_from_spec(spec)
    before = list(sys.path)
    try:
        spec.loader.exec_module(mod)
    finally:
        sys.path[:] = before                             # the script prepends the reference root to sys.path
    assert mod.DrugDiseaseModel is shim.DrugDiseaseModel
    return mod


# ---------------------------------------------------------------------------------------------------
# recorder of the model-API calls the scripts make
# ---------------------------------------------------------------------------------------------------
class CallRecorder:
    def __init__(self, graph_tags):
        self.calls, self.depth, self.tags = [], 0, graph_tags      # tags: number of edge columns -> "train" / "full" / ...

    def _tag(self, edge_index):
        return self.tags.get(int(edge_index.size(1)), f"E{int(edge_index.size(1))}")

    def add(self, **kw):
        if self.depth == 0:
            self.calls.append(kw)


@contextlib.contextmanager
def recording(rec: CallRecorder):
    import primekg_rgcn_linkprediction_b200 as pkg
    M, E, D = pkg.DrugDiseaseModel, pkg.DrugDiseaseRGCN, pkg.LinkPredictor
    saved = [(M, "forward", M.forward), (E, "forward", E.forward), (D, "score_all_tails", D.score_all_tails),
             (D, "forward", D.forward), (M, "state_dict", M.state_dict), (M, "load_state_dict", M.load_state_dict),
             (torch.Tensor, "backward", torch.Tensor.backward),
             (torch.nn.utils, "clip_grad_norm_", torch.nn.utils.clip_grad_norm_)]

    def nested(fn, make):
        def wrapper(*a, **k):
            rec.add(**make(*a, **k))
            rec.depth += 1
            try:
                return fn(*a, **k)
            finally:
                rec.depth -= 1
        return wrapper

    M.forward = nested(M.forward, lambda self, ei, et, h, t, r: dict(
        op="model.forward", graph=rec._tag(ei), pairs=int(h.numel()), training=self.training, grad=torch.is_grad_enabled()))
    E.forward = nested(E.forward, lambda self, ei, et, node_indices=None: dict(
        op="encoder.forward", graph=rec._tag(ei), training=self.training, grad=torch.is_grad_enabled()))
    D.score_all_tails = nested(D.score_all_tails, lambda self, h, r, allt: dict(
        op="decoder.score_all_tails", heads=int(h.size(0)), tails=int(allt.size(0))))
    D.forward = nested(D.forward, lambda self, h, t, r: dict(op="decoder.forward", pairs=int(r.numel())))
    M.state_dict = nested(M.state_dict, lambda self, *a, **k: dict(op="state_dict"))
    M.load_state_dict = nested(M.load_state_dict, lambda self, *a, **k: dict(op="load_state_dict"))
    torch.Tensor.backward = nested(torch.Tensor.backward, lambda self, *a, **k: dict(op="backward"))
    torch.nn.utils.clip_grad_norm_ = nested(torch.nn.utils.clip_grad_norm_, lambda params, max_norm, *a, **k: dict(
        op="clip_grad_norm_", max_norm=float(max_norm)))
    from torch.optim.optimizer import register_optimizer_step_post_hook
    handle = register_optimizer_step_post_hook(
        lambda opt, a, k: rec.add(op="optimizer.step", optimizer=type(opt).__name__,
                                  lr=float(opt.param_groups[0]["lr"]),
                                  weight_decay=float(opt.param_groups[0].get("weight_decay", 0.0))))
    try:
        yield rec
    finally:
        handle.remove()
        for obj, name, fn in saved:
            setattr(obj, name, fn)


# ---------------------------------------------------------------------------------------------------
# the run: train.py main() for two epochs, then evaluate.py's loader + ranking / scoring loops
# ---------------------------------------------------------------------------------------------------
TRAIN_ARGV = ["--epochs", "2", "--batch_size", "1024", "--device", "cpu", "--save_every", "1", "--hidden_dim", "128",
              "--embedding_dim", "64", "--lr", "0.001", "--seed", "42"]


def run_reference_scripts(workdir, rec=None):
    """Runs the reference's train.py ``main()`` and evaluate.py's ``load_model`` / ``ModelEvaluator`` in ``workdir``
    (CPU; the caller has installed the CPU kernel stand-ins).  Returns a dict of what the scripts produced."""
    data_dir = os.path.join(workdir, "data", "processed")
    out_dir = os.path.join(workdir, "output")
    train, val, test, full = write_processed(data_dir)
    if rec is not None:
        rec.tags.update({int(train["edge_index"].size(1)): "train", int(full["edge_index"].size(1)): "full"})
    cwd, argv = os.getcwd(), list(sys.argv)
    os.chdir(workdir)                                    # train.py opens ./training.log at import time
    try:
        ref_train = load_reference_script("train")
        sys.argv = ["train.py", "--data_dir", data_dir, "--output_dir", out_dir] + TRAIN_ARGV
        ctx = recording(rec) if rec is not None else contextlib.nullcontext()
        with ctx:
            ref_train.main()
            best = os.path.join(out_dir, "models", "best_model.pt")
            final = os.path.join(out_dir, "models", "final_model.pt")
            ref_eval = load_reference_script("evaluate")
            model, info = ref_eval.load_model(best, torch.device("cpu"))
            test_data, full_graph = ref_eval.load_test_data(data_dir)
            ev = ref_eval.ModelEvaluator(model, test_data, full_graph, torch.device("cpu"), batch_size=256)
            scores, labels = ev.compute_scores_and_labels(num_neg_samples=1)
            ranking = ev.compute_ranking_metrics(k_values=[10, 50])
        ckpt = torch.load(final, map_location="cpu", weights_only=False)
        return dict(info=info, ranking=ranking, scores=scores, labels=labels, checkpoint=ckpt, model=model,
                    best_path=best, final_path=final, test=test_data, full=full_graph)
    finally:
        sys.argv = argv
        os.chdir(cwd)

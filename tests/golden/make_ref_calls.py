"""Generates tests/golden/ref_call_sequence.json: the sequence of model-API calls the reference's UNMODIFIED
src/train.py (main(), two epochs) and src/evaluate.py (load_model, ModelEvaluator scoring + ranking loops) make on the
drop-in module trio, recorded on the CPU (kernels = tests/cpu_ops_emulation.py).  Needs a checkout of the original
project in ``$PRIMEKG_RGCN_REFERENCE``.

    python tests/golden/make_ref_calls.py
"""
import json
import os
import sys
import tempfile

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import cpu_ops_emulation as emu  # noqa: E402
import ref_harness as H  # noqa: E402


def main():
    import __graft_entry__ as entry
    entry.build()
    import primekg_rgcn_linkprediction_b200 as pkg
    mp = pytest.MonkeyPatch()
    try:
        emu.install_full(mp, pkg)
        rec = H.CallRecorder({})
        with tempfile.TemporaryDirectory() as d:
            out = H.run_reference_scripts(d, rec)
        doc = {"generator": "tests/golden/make_ref_calls.py", "data": H.DATA, "train_argv": H.TRAIN_ARGV,
               "eval_batch_size": 256, "model": {k: out["info"][k] for k in ("num_nodes", "num_relations", "embedding_dim",
                                                                               "hidden_dim", "num_parameters")},
               "calls": rec.calls}
        with open(os.path.join(HERE, "ref_call_sequence.json"), "w") as f:
            json.dump(doc, f, indent=0)
        print(f"{len(rec.calls)} calls recorded")
    finally:
        mp.undo()


if __name__ == "__main__":
    main()

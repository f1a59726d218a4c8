"""fuxictr_b200.patch.enable() on the REAL reference (oracle/_ref) without a GPU: class identity,
state_dict and CPU behaviour are untouched, and CUDA tensors would be routed to the kernels.  The
same boundary on a real device: tests/test_reference_boundary.py (-m gpu)."""
import os
import sys
import types

import pytest
import torch

from conftest import Golden, rel_err

from baseline import refenv  # noqa: E402

pytestmark = pytest.mark.skipif(not refenv.available(), reason=refenv.why_unavailable())


@pytest.fixture(scope="module")
def ref():
    R = refenv.import_reference()
    return types.SimpleNamespace(L=R.layers, FeatureMap=R.FeatureMap, DeepFM=refenv.load_model_class("DeepFM"))


def build_ref_deepfm(ref, g):
    from collections import OrderedDict
    fm = ref.FeatureMap("synthetic", "/tmp")
    fm.features = OrderedDict((k, dict(v)) for k, v in g.meta["specs"])
    fm.labels = g.meta["labels"]
    fm.default_emb_dim = g.meta["kwargs"]["embedding_dim"]
    fm.num_fields = fm.get_num_fields()
    fm.set_column_index()
    model = ref.DeepFM(fm, model_root="/tmp/b2_patch/", metrics=["AUC"], verbose=0, optimizer="adam",
                       loss="binary_crossentropy", task="binary_classification", gpu=-1, **g.meta["kwargs"])
    model.load_state_dict(g["w"])
    return fm, model


def test_enable_keeps_identity_and_cpu_results(ref):
    from fuxictr_b200 import patch
    g = Golden("model_DeepFM")
    cls_before = ref.L.FeatureEmbeddingDict
    patch.enable()
    try:
        assert ref.L.FeatureEmbeddingDict is cls_before                       # same class object
        fm, model = build_ref_deepfm(ref, g)
        assert list(model.state_dict().keys()) == list(g["w"].keys())
        assert type(model.embedding_layer.embedding_layer) == ref.L.FeatureEmbeddingDict   # rank_model.py:107
        B = g.meta["batch"]
        mat = g["in"]["matrix"][:B]
        batch = {c: mat[:, fm.get_column_index(c)] for c in list(fm.features.keys()) + fm.labels}
        y = model.forward(batch)["y_pred"]                                    # CPU tensors -> original forwards
        assert rel_err(y, g["out"]["y_pred"]) <= 1e-6
        assert patch.call_counts() == {}
    finally:
        patch.disable()


def test_cuda_tensors_are_routed_to_the_kernels(ref, monkeypatch):
    """No GPU here: pretend the tensors are CUDA and check that the patched forwards reach the
    kernel entry points (which then refuse the CPU tensors loudly)."""
    from fuxictr_b200 import patch
    g = Golden("model_DeepFM")
    patch.enable()
    try:
        fm, model = build_ref_deepfm(ref, g)
        B = g.meta["batch"]
        mat = g["in"]["matrix"][:B]
        batch = {c: mat[:, fm.get_column_index(c)] for c in list(fm.features.keys()) + fm.labels}
        monkeypatch.setattr(patch, "_on_cuda", lambda a, k: True)
        with pytest.raises(RuntimeError, match="CUDA"):
            model.forward(batch)
        assert patch.call_counts().get("FeatureEmbedding", 0) >= 1
    finally:
        patch.disable()


def test_evaluate_is_patched_but_cpu_models_use_the_reference_path(ref, monkeypatch):
    """BaseModel.evaluate / predict: a CPU model keeps the reference's sklearn path (identical
    numbers to fuxictr.metrics); a model that claims a CUDA device is routed to the device metrics
    (which refuse CPU tensors loudly here, where there is no GPU)."""
    import numpy as np
    from fuxictr_b200 import patch
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
    from oracle import fuxictr_oracle as O
    g = Golden("model_DeepFM")
    patch.enable()
    try:
        fm, model = build_ref_deepfm(ref, g)
        model._verbose = 0
        B = g.meta["batch"]
        mats = [g["in"]["matrix"][:B], g["in"]["matrix"][:B // 2]]
        cols = list(fm.features.keys()) + fm.labels
        gen = [{c: m[:, fm.get_column_index(c)] for c in cols} for m in mats]
        logs = model.evaluate(gen, metrics=["logloss", "AUC"])
        preds = model.predict(gen)
        assert patch.call_counts().get("evaluate", 0) == 0 and patch.call_counts().get("predict", 0) == 0
        y = np.concatenate([m[:, -1].numpy() for m in mats])
        want = O.evaluate_metrics(y, preds, ["logloss", "AUC"])
        assert abs(logs["logloss"] - want["logloss"]) <= 1e-12 and abs(logs["AUC"] - want["AUC"]) <= 1e-12
        monkeypatch.setattr(model, "device", torch.device("cuda:0"))
        with pytest.raises((RuntimeError, AssertionError)):
            model.evaluate(gen, metrics=["logloss", "AUC"])
        assert patch.call_counts().get("evaluate", 0) == 1
        # group metrics stay on the reference path even for a CUDA model
        fm.group_id = "C0"
        with pytest.raises(Exception):
            model.evaluate(gen, metrics=["gAUC"])
        assert patch.call_counts().get("evaluate", 0) == 1
    finally:
        patch.disable()

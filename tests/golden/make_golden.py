"""Generates tests/golden/*.npz by running the REAL reference (reczoo/FuxiCTR, read-only at
/root/reference) on seeded inputs.  Run in the build container only:

    python tests/golden/make_golden.py

The GPU box has no reference checkout; tests read the committed .npz files.  Each file
holds: "meta" (JSON: what was run), "in/<name>" inputs, "w/<key>" the module's
state_dict BEFORE the run, "out/<name>" forward outputs, "g/<key>" parameter gradients,
"gin/<name>" gradients w.r.t. float inputs, and for the model cases "w1/<key>" /
"w3/<key>" the state_dict after 1 / 3 reference train_step()s.
"""
import json
import os
import sys
import types

import numpy as np

REF = os.environ.get("FUXICTR_REFERENCE", "/root/reference")
HERE = os.path.dirname(os.path.abspath(__file__))


def import_reference():
    """SURVEY.md section 8(c): three import-time-only dependencies are stubbed."""
    for name in ["h5py", "polars", "keras_preprocessing", "keras_preprocessing.sequence"]:
        sys.modules[name] = types.ModuleType(name)
    sys.modules["keras_preprocessing.sequence"].pad_sequences = lambda *a, **k: None
    sys.modules["keras_preprocessing"].sequence = sys.modules["keras_preprocessing.sequence"]
    sys.path.insert(0, REF)
    import torch  # noqa
    import fuxictr.pytorch.layers as L
    from fuxictr.features import FeatureMap
    for name in ["h5py", "polars"]:
        sys.modules.pop(name, None)
    return L, FeatureMap


L, RefFeatureMap = import_reference()
import torch  # noqa: E402

torch.set_num_threads(1)
torch.use_deterministic_algorithms(True)


def load_model_class(rel_dir, name):
    import importlib
    path = os.path.join(REF, "model_zoo", rel_dir)
    sys.path.insert(0, path)
    for k in [k for k in sys.modules if k == "src" or k.startswith("src.")]:
        del sys.modules[k]
    mod = importlib.import_module("src." + name)
    sys.path.pop(0)
    return getattr(mod, name)


def save(name, meta, **groups):
    arrays = {"meta": np.array(json.dumps(meta))}
    for group, d in groups.items():
        for k, v in d.items():
            if isinstance(v, torch.Tensor):
                v = v.detach().cpu().numpy()
            arrays["%s/%s" % (group, k)] = np.asarray(v)
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **arrays)
    print("wrote", path, "%.1f KB" % (os.path.getsize(path) / 1024))


def sd(module):
    return {k: v.detach().clone() for k, v in module.state_dict().items()}


def grads(module):
    return {k: p.grad.detach().clone() for k, p in module.named_parameters() if p.grad is not None}


def tiny_batch(dataset, nrows, params):
    """What NpzDataLoader + BatchCollator hand to the model (npz_dataloader.py:63-66,111-125)."""
    fm = RefFeatureMap(dataset, os.path.join(REF, "data", dataset))
    fm.load(os.path.join(REF, "data", dataset, "feature_map.json"), params)
    data = np.load(os.path.join(REF, "data", dataset, "train.npz"))
    cols = list(fm.features.keys()) + fm.labels
    mat = np.column_stack([data[c] for c in cols])[:nrows]
    return fm, torch.from_numpy(mat)


def batch_dict(fm, mat):
    return {c: mat[:, fm.get_column_index(c)] for c in list(fm.features.keys()) + fm.labels}


def specs_json(fm):
    return [[k, v] for k, v in fm.features.items()]


def synthetic_fm(specs, labels=("label",), emb_dim=8, dataset_id="synthetic"):
    fm = RefFeatureMap(dataset_id, "/tmp")
    from collections import OrderedDict
    fm.features = OrderedDict((k, dict(v)) for k, v in specs)
    fm.labels = list(labels)
    fm.default_emb_dim = emb_dim
    fm.num_fields = fm.get_num_fields()
    fm.set_column_index()
    return fm


def synthetic_matrix(fm, batch, gen, seq_min=1):
    cols = []
    for name, spec in fm.features.items():
        if spec["type"] == "sequence":
            L_ = spec["max_len"]
            ids = torch.randint(1, spec["vocab_size"], (batch, L_), generator=gen)
            lens = torch.randint(seq_min, L_ + 1, (batch, 1), generator=gen)
            ids = ids * (torch.arange(L_).view(1, -1) < lens)
            cols.append(ids.double())
        else:
            ids = torch.randint(0, spec["vocab_size"], (batch, 1), generator=gen)  # includes padding id 0
            cols.append(ids.double())
    label = (torch.rand(batch, 1, generator=gen) < 0.3).double()
    return torch.cat(cols + [label], dim=1)


# ------------------------------------------------------------------------------------------
def case_feature_embedding_tiny_npz():
    torch.manual_seed(11)
    fm, mat = tiny_batch("tiny_npz", 48, {"embedding_dim": 4})
    X = {k: v for k, v in batch_dict(fm, mat).items() if k not in fm.labels}
    layer = L.FeatureEmbedding(fm, 4, embedding_initializer="partial(nn.init.normal_, std=0.1)")
    w = sd(layer)
    out = layer(X)
    gen = torch.Generator().manual_seed(5)
    gout = torch.randn(out.shape, generator=gen)
    out.backward(gout)
    flat = layer(X, flatten_emb=True)
    save("feature_embedding_tiny_npz",
         {"case": "FeatureEmbedding(tiny_npz, D=4)", "dataset": "tiny_npz", "embedding_dim": 4,
          "specs": specs_json(fm), "labels": fm.labels},
         **{"in": {"matrix": mat, "gout": gout}, "w": w, "out": {"stack": out, "flat": flat}, "g": grads(layer)})


def case_feature_embedding_dict_tiny_seq():
    for tag, override in [("plain", None),
                          ("avgpool", [{"name": "click_sequence", "feature_encoder": "layers.MaskedAveragePooling()"}]),
                          ("sumpool", [{"name": "click_sequence", "feature_encoder": "layers.MaskedSumPooling()"}])]:
        torch.manual_seed(12)
        fm, mat = tiny_batch("tiny_seq", 40, {"embedding_dim": 6, "feature_specs": override})
        X = {k: v for k, v in batch_dict(fm, mat).items() if k not in fm.labels}
        layer = L.FeatureEmbeddingDict(fm, 6, embedding_initializer="partial(nn.init.normal_, std=0.1)")
        w = sd(layer)
        emb = layer(X)
        gen = torch.Generator().manual_seed(6)
        gouts = {k: torch.randn(v.shape, generator=gen) for k, v in emb.items()}
        loss = sum((emb[k] * gouts[k]).sum() for k in emb)
        loss.backward()
        save("feature_embedding_dict_tiny_seq_" + tag,
             {"case": "FeatureEmbeddingDict(tiny_seq, D=6, %s)" % tag, "dataset": "tiny_seq", "embedding_dim": 6,
              "specs": specs_json(fm), "labels": fm.labels},
             **{"in": {"matrix": mat}, "gout": gouts, "w": w, "out": dict(emb), "g": grads(layer)})


def case_logistic_regression_tiny_seq():
    torch.manual_seed(13)
    fm, mat = tiny_batch("tiny_seq", 40, {"embedding_dim": 6})
    X = {k: v for k, v in batch_dict(fm, mat).items() if k not in fm.labels}
    layer = L.LogisticRegression(fm, use_bias=True)
    with torch.no_grad():
        for p in layer.parameters():
            p.copy_(torch.randn(p.shape) * 0.3)
        for m in layer.modules():
            if isinstance(m, torch.nn.Embedding) and m.padding_idx is not None:
                m.weight[m.padding_idx].zero_()
    w = sd(layer)
    out = layer(X)
    gen = torch.Generator().manual_seed(7)
    gout = torch.randn(out.shape, generator=gen)
    out.backward(gout)
    save("logistic_regression_tiny_seq",
         {"case": "LogisticRegression(tiny_seq)", "dataset": "tiny_seq", "specs": specs_json(fm), "labels": fm.labels},
         **{"in": {"matrix": mat, "gout": gout}, "w": w, "out": {"y": out}, "g": grads(layer)})


def case_inner_product():
    gen = torch.Generator().manual_seed(21)
    for (B, F_, D) in [(16, 7, 10), (9, 39, 16), (5, 27, 16)]:
        emb0 = torch.randn(B, F_, D, generator=gen) * 0.5
        ins, outs, gins = {"emb": emb0}, {}, {}
        modes = ["product_sum", "bi_interaction", "inner_product"] + (["elementwise_product"] if F_ <= 7 else [])
        for mode in modes:
            emb = emb0.clone().requires_grad_(True)
            layer = L.InnerProductInteraction(F_, output=mode)
            out = layer(emb)
            gout = torch.randn(out.shape, generator=gen)
            out.backward(gout)
            ins["gout_" + mode] = gout
            outs[mode] = out
            gins[mode] = emb.grad
        save("inner_product_B%d_F%d_D%d" % (B, F_, D), {"case": "InnerProductInteraction", "B": B, "F": F_, "D": D},
             **{"in": ins, "out": outs, "gin": gins})


def case_cross():
    gen = torch.Generator().manual_seed(22)
    B, d, nl = 24, 52, 3
    for name, cls in [("crossnet", L.CrossNet), ("crossnet_v2", L.CrossNetV2)]:
        torch.manual_seed(22)
        layer = cls(d, nl)
        with torch.no_grad():
            for p in layer.parameters():
                p.copy_(torch.randn(p.shape, generator=gen) * (0.2 if p.dim() > 1 else 0.1))
        x0 = (torch.randn(B, d, generator=gen) * 0.7).requires_grad_(True)
        w = sd(layer)
        out = layer(x0)
        gout = torch.randn(out.shape, generator=gen)
        out.backward(gout)
        save(name, {"case": name, "B": B, "input_dim": d, "num_layers": nl},
             **{"in": {"x0": x0, "gout": gout}, "w": w, "out": {"y": out}, "g": grads(layer), "gin": {"x0": x0.grad}})


def case_cin():
    gen = torch.Generator().manual_seed(23)
    B, F_, D, units = 12, 7, 10, [8, 6]
    torch.manual_seed(23)
    layer = L.CompressedInteractionNet(F_, units, output_dim=1)
    emb = (torch.randn(B, F_, D, generator=gen) * 0.5).requires_grad_(True)
    w = sd(layer)
    out = layer(emb)
    gout = torch.randn(out.shape, generator=gen)
    out.backward(gout)
    save("cin", {"case": "CompressedInteractionNet", "B": B, "F": F_, "D": D, "cin_hidden_units": units},
         **{"in": {"emb": emb, "gout": gout}, "w": w, "out": {"y": out}, "g": grads(layer), "gin": {"emb": emb.grad}})


def case_mlp_dice_din():
    gen = torch.Generator().manual_seed(24)
    # MLP_Block relu
    torch.manual_seed(24)
    mlp = L.MLP_Block(input_dim=20, hidden_units=[16, 12], hidden_activations="ReLU", output_dim=1)
    x = (torch.randn(33, 20, generator=gen)).requires_grad_(True)
    w = sd(mlp)
    out = mlp(x)
    gout = torch.randn(out.shape, generator=gen)
    out.backward(gout)
    save("mlp_relu", {"case": "MLP_Block(20,[16,12],ReLU,1)", "layout": ["linear", "relu", "linear", "relu", "linear"]},
         **{"in": {"x": x, "gout": gout}, "w": w, "out": {"y": out}, "g": grads(mlp), "gin": {"x": x.grad}})
    # Dice, train then eval
    torch.manual_seed(25)
    dice = L.Dice(12)
    with torch.no_grad():
        dice.alpha.copy_(torch.randn(12, generator=gen) * 0.3)
    x = (torch.randn(40, 12, generator=gen) * 2 + 0.5).requires_grad_(True)
    w = sd(dice)
    dice.train()
    out = dice(x)
    gout = torch.randn(out.shape, generator=gen)
    out.backward(gout)
    w_after = sd(dice)
    dice.eval()
    out_eval = dice(x.detach())
    save("dice", {"case": "Dice(12) train + eval"},
         **{"in": {"x": x, "gout": gout}, "w": w, "w1": w_after, "out": {"train": out, "eval": out_eval},
            "g": grads(dice), "gin": {"x": x.grad}})
    # DIN attention with Dice, both softmax settings
    for use_softmax in [False, True]:
        torch.manual_seed(26)
        att = L.DIN_Attention(embedding_dim=8, attention_units=[16], hidden_activations="Dice",
                              use_softmax=use_softmax)
        with torch.no_grad():
            for n, p in att.named_parameters():
                p.copy_(torch.randn(p.shape, generator=gen) * 0.3)
        B, Ls = 10, 6
        target = (torch.randn(B, 8, generator=gen)).requires_grad_(True)
        hist = (torch.randn(B, Ls, 8, generator=gen)).requires_grad_(True)
        lens = torch.randint(1, Ls + 1, (B, 1), generator=gen)
        mask = torch.arange(Ls).view(1, -1) < lens
        with torch.no_grad():
            hist.mul_(mask.unsqueeze(-1).float())
        w = sd(att)
        att.train()
        out = att(target, hist, mask)
        gout = torch.randn(out.shape, generator=gen)
        out.backward(gout)
        save("din_attention_softmax%d" % int(use_softmax),
             {"case": "DIN_Attention(8,[16],Dice)", "use_softmax": use_softmax,
              "layout": ["linear", "dice", "linear"]},
             **{"in": {"target": target, "history": hist, "mask": mask, "gout": gout}, "w": w,
                "out": {"y": out}, "g": grads(att), "gin": {"target": target.grad, "history": hist.grad}})


def model_params(**extra):
    p = dict(model_root="/tmp/b2_golden_ckpt/", metrics=["logloss", "AUC"], verbose=0, optimizer="adam",
             loss="binary_crossentropy", task="binary_classification", learning_rate=1e-3, gpu=-1)
    p.update(extra)
    return p


def run_model_case(name, model, fm, mat, meta):
    """Forward + loss + grads on batch 0, then 3 reference train_step()s on fixed batches."""
    model._max_gradient_norm = 10.0  # set by fit() in the reference (rank_model.py:236-248)
    model.train()
    B = mat.shape[0] // 3
    batches = [batch_dict(fm, mat[i * B:(i + 1) * B]) for i in range(3)]
    w0 = sd(model)
    model.optimizer.zero_grad()
    ret = model.forward(batches[0])
    y_true = model.get_labels(batches[0])
    loss = model.compute_loss(ret, y_true)
    loss.backward()
    g = grads(model)
    outs = {"y_pred": ret["y_pred"], "loss": loss}
    model.optimizer.zero_grad()
    losses = []
    states = {}
    for i in range(3):
        losses.append(model.train_step(batches[i]).detach())
        if i in (0, 2):
            states[i + 1] = sd(model)
    outs["step_losses"] = torch.stack(losses)
    meta = dict(meta, specs=specs_json(fm), labels=fm.labels, batch=B)
    save(name, meta, **{"in": {"matrix": mat}, "w": w0, "out": outs, "g": g, "w1": states[1], "w3": states[3]})


def criteo_like_specs(nf, vocab):
    return [("C%d" % i, {"type": "categorical", "source": "", "padding_idx": 0, "vocab_size": vocab + 3 * i})
            for i in range(nf)]


def case_models():
    gen = torch.Generator().manual_seed(31)
    # DeepFM / DCNv2 / DLRM / xDeepFM on a 10-field categorical map
    specs = criteo_like_specs(10, 40)
    for name, rel, kwargs in [
        ("DeepFM", "DeepFM/DeepFM_torch", dict(embedding_dim=8, hidden_units=[24, 16], hidden_activations="relu",
                                               net_dropout=0, batch_norm=False)),
        ("DCNv2", "DCNv2", dict(embedding_dim=8, model_structure="parallel", num_cross_layers=3,
                                parallel_dnn_hidden_units=[24, 16], dnn_activations="relu")),
        ("DLRM", "DLRM", dict(embedding_dim=8, top_mlp_units=[24, 16], interaction_op="dot")),
        ("xDeepFM", "xDeepFM", dict(embedding_dim=8, dnn_hidden_units=[24, 16], cin_hidden_units=[6, 5])),
    ]:
        torch.manual_seed(2023)
        fm = synthetic_fm(specs, emb_dim=8)
        cls = load_model_class(rel, name)
        model = cls(fm, **model_params(**kwargs))
        # larger-than-default embedding scale so every term of the logit matters numerically
        with torch.no_grad():
            for m in model.modules():
                if isinstance(m, torch.nn.Embedding):
                    m.weight[1:].copy_(torch.randn(m.weight[1:].shape, generator=gen) * 0.1)
        mat = synthetic_matrix(fm, 3 * 32, gen)
        run_model_case("model_" + name, model, fm, mat, {"case": name, "kwargs": kwargs, "seed": 2023})
    # DIN on a sequence map with shared tables (Taobao-like, tuple target/sequence fields)
    specs = [("user_id", {"type": "categorical", "source": "", "padding_idx": 0, "vocab_size": 30}),
             ("item_id", {"type": "categorical", "source": "", "padding_idx": 0, "vocab_size": 60}),
             ("cate_id", {"type": "categorical", "source": "", "padding_idx": 0, "vocab_size": 12}),
             ("click_history", {"type": "sequence", "source": "", "padding_idx": 0, "vocab_size": 60, "max_len": 7,
                                "share_embedding": "item_id", "feature_encoder": None}),
             ("cate_history", {"type": "sequence", "source": "", "padding_idx": 0, "vocab_size": 12, "max_len": 7,
                               "share_embedding": "cate_id", "feature_encoder": None})]
    kwargs = dict(embedding_dim=8, dnn_hidden_units=[24, 16], dnn_activations="relu", attention_hidden_units=[16],
                  attention_hidden_activations="Dice", din_use_softmax=False)
    torch.manual_seed(2023)
    fm = synthetic_fm(specs, emb_dim=8)
    cls = load_model_class("DIN", "DIN")
    model = cls(fm, **model_params(**kwargs))
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, torch.nn.Embedding):
                m.weight[1:].copy_(torch.randn(m.weight[1:].shape, generator=gen) * 0.1)
    mat = synthetic_matrix(fm, 3 * 32, gen)
    run_model_case("model_DIN", model, fm, mat, {"case": "DIN", "kwargs": kwargs, "seed": 2023})


def case_init_parity():
    """state_dict right after construction with a fixed seed: pins construction/RNG order."""
    specs = criteo_like_specs(6, 20)
    torch.manual_seed(777)
    fm = synthetic_fm(specs, emb_dim=4)
    cls = load_model_class("DeepFM/DeepFM_torch", "DeepFM")
    model = cls(fm, **model_params(embedding_dim=4, hidden_units=[8, 8]))
    save("init_DeepFM_seed777", {"case": "DeepFM init", "seed": 777, "specs": specs_json(fm), "labels": fm.labels,
                                  "kwargs": dict(embedding_dim=4, hidden_units=[8, 8])}, w=sd(model))


def case_mirror_constructors():
    """state_dict and module tree of the model_zoo classes right after construction with seed 4242,
    for every configuration of tests/test_host_logic.py:_MIRROR_CASES (one group per case)."""
    tests_dir = os.path.dirname(HERE)
    sys.path[:0] = [tests_dir, os.path.dirname(tests_dir)]
    from test_host_logic import _MIRROR_CASES, _mirror_case_ids
    rel = {"DeepFM": "DeepFM/DeepFM_torch", "DCNv2": "DCNv2", "DLRM": "DLRM", "DIN": "DIN", "xDeepFM": "xDeepFM"}
    meta, groups = {"seed": 4242, "cases": {}}, {}
    for case_id, (name, specs, kwargs) in zip(_mirror_case_ids(), _MIRROR_CASES):
        cls = load_model_class(rel[name], name)
        torch.manual_seed(4242)
        model = cls(synthetic_fm(specs, emb_dim=kwargs["embedding_dim"]), model_root="/tmp/b2_mirror/", metrics=["AUC"],
                    verbose=0, gpu=-1, optimizer="adam", loss="binary_crossentropy", **kwargs)
        w = sd(model)
        modules = [[m, "%s.%s" % (type(mod).__module__, type(mod).__qualname__)
                    if type(mod).__module__.startswith("torch.") else None] for m, mod in model.named_modules()]
        meta["cases"][case_id] = {"keys": list(w.keys()), "modules": modules}
        groups[case_id] = w
    save("mirror_constructors_seed4242", meta, **groups)


def case_next_layers():
    """Layers of the "next" row 8f-4 (kernels not built yet): pins the oracle restatement first."""
    import fuxictr.pytorch.layers as LL
    gen = torch.Generator().manual_seed(51)
    B, F_, D = 6, 5, 8
    emb0 = torch.randn(B, F_, D, generator=gen) * 0.5
    for cls_name in ("BilinearInteraction", "BilinearInteractionV2"):
        for btype in ("field_all", "field_each", "field_interaction"):
            torch.manual_seed(51)
            layer = getattr(LL, cls_name)(F_, D, bilinear_type=btype)
            emb = emb0.clone().requires_grad_(True)
            w0 = sd(layer)
            out = layer(emb)
            gout = torch.randn(out.shape, generator=gen)
            (out * gout).sum().backward()
            save("next_%s_%s" % (cls_name, btype), {"B": B, "F": F_, "D": D, "bilinear_type": btype},
                 **{"in": {"emb": emb0, "gout": gout}, "w": w0, "out": {"y": out}, "g": grads(layer),
                    "gin": {"emb": emb.grad}})
    for act in ("ReLU", "Sigmoid"):
        torch.manual_seed(52)
        layer = LL.SqueezeExcitation(F_, reduction_ratio=2, excitation_activation=act)
        emb = emb0.clone().requires_grad_(True)
        w0 = sd(layer)
        out = layer(emb)
        gout = torch.randn(out.shape, generator=gen)
        (out * gout).sum().backward()
        save("next_SqueezeExcitation_%s" % act, {"act": act}, **{"in": {"emb": emb0, "gout": gout}, "w": w0,
             "out": {"y": out}, "g": grads(layer), "gin": {"emb": emb.grad}})
    L_, d = 7, 12
    tgt0, hist0 = torch.randn(B, d, generator=gen), torch.randn(B, L_, d, generator=gen)
    lens = torch.randint(1, L_ + 1, (B,), generator=gen)
    mask = (torch.arange(L_)[None, :] < lens[:, None]).float()
    for heads, qkvo, scale in ((1, True, True), (3, True, True), (2, False, False)):
        torch.manual_seed(53)
        layer = LL.MultiHeadTargetAttention(input_dim=d, attention_dim=d, num_heads=heads, use_scale=scale,
                                            use_qkvo=qkvo)
        tgt, hist = tgt0.clone().requires_grad_(True), hist0.clone().requires_grad_(True)
        w0 = sd(layer)
        out = layer(tgt, hist, mask)
        gout = torch.randn(out.shape, generator=gen)
        (out * gout).sum().backward()
        save("next_MHTA_h%d_qkvo%d" % (heads, int(qkvo)), {"heads": heads, "use_qkvo": qkvo, "use_scale": scale},
             **{"in": {"target": tgt0, "history": hist0, "mask": mask, "gout": gout}, "w": w0,
                "out": {"y": out}, "g": grads(layer), "gin": {"target": tgt.grad, "history": hist.grad}})
    dd = 20
    x0 = torch.randn(B, dd, generator=gen)
    torch.manual_seed(54)
    layer = LL.CrossNetMix(dd, layer_num=2, low_rank=4, num_experts=3)
    with torch.no_grad():
        for b in layer.bias:
            b.normal_(0, 0.1)
    x = x0.clone().requires_grad_(True)
    w0 = sd(layer)
    out = layer(x)
    gout = torch.randn(out.shape, generator=gen)
    (out * gout).sum().backward()
    save("next_CrossNetMix", {"layer_num": 2, "low_rank": 4, "num_experts": 3},
         **{"in": {"x": x0, "gout": gout}, "w": w0, "out": {"y": out}, "g": grads(layer), "gin": {"x": x.grad}})


def case_metrics():
    """fuxictr.metrics.evaluate_metrics (metrics.py:26-48) as BaseModel.evaluate calls it: float64
    copies of fp32 predictions.  Three splits: smooth scores, heavy ties, saturated (0/1) scores."""
    import warnings
    from fuxictr.metrics import evaluate_metrics
    rng = np.random.default_rng(41)
    cases = {}
    n = 6000
    y = (rng.random(n) < 0.25).astype(np.float32)
    smooth = (1.0 / (1.0 + np.exp(-(rng.normal(size=n) + 1.5 * y - 1.0)))).astype(np.float32)
    ties = np.round(smooth, 2).astype(np.float32)
    sat = smooth.copy()
    sat[:50], sat[50:100] = 0.0, 1.0
    out, inp = {}, {}
    for name, p in [("smooth", smooth), ("ties", ties), ("saturated", sat)]:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            r = evaluate_metrics(np.array(y, np.float64), np.array(p, np.float64), ["logloss", "AUC"])
        inp["y_pred_" + name] = p
        out["logloss_" + name] = np.array(r["logloss"], np.float64)
        out["auc_" + name] = np.array(r["AUC"], np.float64)
    inp["y_true"] = y
    save("metrics_eval", {"what": "fuxictr.metrics.evaluate_metrics(['logloss','AUC'])", "n": n}, **{"in": inp, "out": out})


if __name__ == "__main__":
    if "--only-metrics" in sys.argv:
        case_metrics()
        sys.exit(0)
    if "--only-next" in sys.argv:
        case_next_layers()
        sys.exit(0)
    if "--only-mirror" in sys.argv:
        case_mirror_constructors()
        sys.exit(0)
    case_feature_embedding_tiny_npz()
    case_feature_embedding_dict_tiny_seq()
    case_logistic_regression_tiny_seq()
    case_inner_product()
    case_cross()
    case_cin()
    case_mlp_dice_din()
    case_models()
    case_init_parity()
    case_mirror_constructors()
    case_metrics()
    case_next_layers()

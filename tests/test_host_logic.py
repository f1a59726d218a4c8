"""Host-side mirror of the reference interface, CPU only: schema, construction order /
state_dict keys (pinned by reference goldens), launch plans, and the refusal to compute
on CPU tensors (there is no fallback path)."""

import pytest
import torch

from conftest import Golden, ROOT
from fuxictr_b200.schema import FeatureMap
from fuxictr_b200 import layers, zoo
from fuxictr_b200 import functional as F2
from fuxictr_b200._lib import B2_POOL_MEAN, B2_POOL_NONE, B2_POOL_SUM


def fm_from(g, emb_dim=None):
    return FeatureMap.from_specs(g.meta["specs"], labels=g.meta["labels"], embedding_dim=emb_dim)


def test_schema_matches_reference_json_layout():
    g = Golden("feature_embedding_dict_tiny_seq_plain")
    fm = fm_from(g, 6)
    assert fm.num_fields == 15 and fm.input_length == 19
    assert fm.column_index["click_sequence"] == [14, 15, 16, 17, 18]
    assert fm.column_index["clk"] == 19
    assert fm.sum_emb_out_dim() == 15 * 6
    batch = fm.batch_dict(g["in"]["matrix"])
    assert batch["userid"].stride() == (20,) and batch["click_sequence"].shape == (40, 5)


def test_init_matches_reference_seed_for_seed():
    g = Golden("init_DeepFM_seed777")
    torch.manual_seed(777)
    fm = fm_from(g, 4)
    model = zoo.DeepFM(fm, gpu=-1, **g.meta["kwargs"])
    sd = model.state_dict()
    assert list(sd.keys()) == list(g["w"].keys())
    for k, ref in g["w"].items():
        assert torch.equal(sd[k], ref), k


@pytest.mark.parametrize("name", ["DeepFM", "DCNv2", "DLRM", "xDeepFM", "DIN"])
def test_state_dict_keys_and_loading(name):
    g = Golden("model_" + name)
    fm = fm_from(g, g.meta["kwargs"]["embedding_dim"])
    model = getattr(zoo, name)(fm, gpu=-1, **g.meta["kwargs"])
    assert list(model.state_dict().keys()) == list(g["w"].keys())
    model.load_state_dict(g["w"])  # strict: shapes and names agree with the reference checkpoint


def test_shared_embedding_is_one_module():
    g = Golden("model_DIN")
    fm = fm_from(g, 8)
    model = zoo.DIN(fm, gpu=-1, **g.meta["kwargs"])
    el = model.embedding_layer.embedding_layers
    assert el["click_history"] is el["item_id"] and el["cate_history"] is el["cate_id"]
    # the regulariser of the reference selects by exact type (rank_model.py:107)
    assert type(model.embedding_layer) == layers.FeatureEmbeddingDict


def test_gather_plan_layout():
    g = Golden("feature_embedding_dict_tiny_seq_avgpool")
    fm = fm_from(g, 6)
    fed = layers.FeatureEmbeddingDict(fm, 6)
    names = list(fm.features.keys())
    assert all(fed._is_fusable(f) for f in names)
    plan, tables = fed._plan(names, names)
    seq = [f for f in plan.fields if f.name == "click_sequence"][0]
    assert seq.seq_len == 5 and seq.pool == B2_POOL_MEAN and seq.out_width == 6
    assert plan.width == 15 * 6 and plan.needs_count
    assert len(tables) == 14  # click_sequence shares adgroup_id's table
    assert seq.table_slot == [f for f in plan.fields if f.name == "adgroup_id"][0].table_slot
    # unpooled sequence: L*D wide slice
    g2 = Golden("feature_embedding_dict_tiny_seq_plain")
    fed2 = layers.FeatureEmbeddingDict(fm_from(g2, 6), 6)
    plan2, _ = fed2._plan(names, names)
    seq2 = [f for f in plan2.fields if f.name == "click_sequence"][0]
    assert seq2.pool == B2_POOL_NONE and seq2.out_width == 30 and plan2.width == 14 * 6 + 30
    # LR mode: MaskedSumPooling on sequences, separate (unshared) tables (feature_embedding.py:135-138)
    lr = layers.LogisticRegression(fm_from(g2, 6))
    plan3, tables3 = lr.embedding_layer.embedding_layer._plan(names, names)
    assert [f for f in plan3.fields if f.name == "click_sequence"][0].pool == B2_POOL_SUM
    assert len(tables3) == 15 and all(t.embedding_dim == 1 for t in tables3)


def test_cpu_tensors_are_refused():
    g = Golden("model_DeepFM")
    fm = fm_from(g, 8)
    model = zoo.DeepFM(fm, gpu=-1, **g.meta["kwargs"])
    batch = fm.batch_dict(g["in"]["matrix"][:8])
    with pytest.raises(RuntimeError, match="CUDA"):
        model.forward(batch)
    with pytest.raises(RuntimeError, match="CUDA"):
        F2.fm_interaction(torch.zeros(2, 3, 4), 0)
    with pytest.raises(RuntimeError, match="CUDA"):
        F2.linear_act(torch.zeros(2, 3), torch.zeros(4, 3))
    with pytest.raises(RuntimeError, match="CUDA"):
        zoo.ParamArena(model)


def test_unsupported_configs_fail_loudly():
    specs = [("a", {"type": "categorical", "source": "", "padding_idx": 0, "vocab_size": 5,
                    "pretrained_emb": "x.npz"})]
    fm = FeatureMap.from_specs(specs, embedding_dim=4)
    with pytest.raises(NotImplementedError):
        layers.FeatureEmbeddingDict(fm, 4)
    g = Golden("model_DCNv2")
    with pytest.raises(NotImplementedError):
        zoo.DCNv2(fm_from(g, 8), gpu=-1, use_low_rank_mixture=True, parallel_dnn_hidden_units=[8])
    with pytest.raises(ValueError):
        layers.InnerProductInteraction(4, output="nope")


def test_batch_views_alias_the_matrix_for_sequences_too():
    """schema.FeatureMap.batch_views: every entry (scalar columns AND sequence column ranges) is a
    view of the batch matrix, so a graph-captured static input stays live; values equal batch_dict."""
    import torch
    from fuxictr_b200.schema import FeatureMap
    specs = [("u", {"type": "categorical", "source": "", "vocab_size": 9}),
             ("hist", {"type": "sequence", "source": "", "vocab_size": 9, "max_len": 4}),
             ("i", {"type": "categorical", "source": "", "vocab_size": 9})]
    fm = FeatureMap.from_specs(specs, embedding_dim=4)
    mat = torch.arange(5 * 7, dtype=torch.float64).reshape(5, 7)
    views, copies = fm.batch_views(mat), fm.batch_dict(mat)
    assert list(views.keys()) == list(copies.keys()) == ["u", "hist", "i", "label"]
    for k in views:
        assert torch.equal(views[k], copies[k])
    mat.mul_(-1)
    assert torch.equal(views["hist"], mat[:, 1:5]) and views["hist"].stride() == (7, 1)
    assert not torch.equal(copies["hist"], mat[:, 1:5])        # the collator-style entry is a copy


# ---------------------------------------------------------------------------------------------
# Mirror constructors vs the LIVE reference (oracle/_ref): same seed => bit-identical state_dict
# (keys, shapes, registration order, RNG consumption order), over more configurations than the goldens.
# The same comparison against the stored reference state (mirror_constructors_seed4242.npz, made by
# tests/golden/make_golden.py) runs without the reference installed.
# ---------------------------------------------------------------------------------------------
_SEQ_SPECS = [
    ("user", {"type": "categorical", "source": "", "padding_idx": 0, "vocab_size": 30}),
    ("item_id", {"type": "categorical", "source": "", "padding_idx": 0, "vocab_size": 50}),
    ("cate_id", {"type": "categorical", "source": "", "padding_idx": 0, "vocab_size": 12, "embedding_dim": 8}),
    ("price", {"type": "numeric", "source": ""}),
    ("click_history", {"type": "sequence", "source": "", "padding_idx": 0, "vocab_size": 50, "max_len": 6,
                       "share_embedding": "item_id"}),
    ("cate_history", {"type": "sequence", "source": "", "padding_idx": 0, "vocab_size": 12, "max_len": 6,
                      "share_embedding": "cate_id", "embedding_dim": 8}),
    ("tags", {"type": "sequence", "source": "", "padding_idx": 0, "vocab_size": 20, "max_len": 4,
              "feature_encoder": "layers.MaskedAveragePooling()"}),
]
_CAT_SPECS = [("C%d" % i, {"type": "categorical", "source": "", "padding_idx": 0, "vocab_size": 11 + 3 * i})
              for i in range(5)]
_MIRROR_CASES = [
    ("DeepFM", _CAT_SPECS, dict(embedding_dim=4, hidden_units=[12, 8], hidden_activations="relu", net_dropout=0.1,
                                batch_norm=True)),
    ("DeepFM", _SEQ_SPECS[:3] + _SEQ_SPECS[6:], dict(embedding_dim=8, hidden_units=[6], hidden_activations=["PReLU"])),
    ("DCNv2", _CAT_SPECS, dict(embedding_dim=4, model_structure="stacked_parallel", num_cross_layers=2,
                               stacked_dnn_hidden_units=[10], parallel_dnn_hidden_units=[7, 5], dnn_activations="relu")),
    ("DCNv2", _CAT_SPECS, dict(embedding_dim=4, model_structure="crossnet_only", num_cross_layers=1)),
    ("DLRM", _CAT_SPECS, dict(embedding_dim=4, top_mlp_units=[9, 5], interaction_op="cat")),
    ("DLRM", _CAT_SPECS + [("price", {"type": "numeric", "source": ""})],
     dict(embedding_dim=4, top_mlp_units=[9], bottom_mlp_units=[6, 5], interaction_op="dot")),
    ("xDeepFM", _CAT_SPECS, dict(embedding_dim=4, dnn_hidden_units=[], cin_hidden_units=[3])),
    ("xDeepFM", _CAT_SPECS, dict(embedding_dim=4, dnn_hidden_units=[8, 4], cin_hidden_units=[4, 3, 2], batch_norm=True)),
    ("DIN", _SEQ_SPECS[:3] + _SEQ_SPECS[4:6], dict(embedding_dim=8, dnn_hidden_units=[10, 6], dnn_activations="Dice",
                                                   attention_hidden_units=[7, 5], attention_hidden_activations="Dice",
                                                   din_use_softmax=True, attention_dropout=0.2)),
    ("DIN", _SEQ_SPECS[:3] + _SEQ_SPECS[4:6], dict(embedding_dim=8, dnn_hidden_units=[10], dnn_activations="relu",
                                                   attention_hidden_units=[7], attention_hidden_activations="ReLU",
                                                   attention_output_activation="Sigmoid", batch_norm=True)),
]


def _mirror_case_ids():
    return ["%s-%d" % (c[0], i) for i, c in enumerate(_MIRROR_CASES)]


@pytest.mark.parametrize("name,specs,kwargs", _MIRROR_CASES, ids=_mirror_case_ids())
def test_mirror_constructors_match_the_live_reference_seed_for_seed(name, specs, kwargs):
    from baseline import refenv
    if not refenv.available():
        pytest.skip(refenv.why_unavailable())
    refenv.import_reference()
    ref_cls = refenv.load_model_class(name)
    emb_dim = kwargs["embedding_dim"]
    torch.manual_seed(4242)
    ref = ref_cls(refenv.synthetic_feature_map(specs, embedding_dim=emb_dim), model_root="/tmp/b2_mirror/",
                  metrics=["AUC"], verbose=0, gpu=-1, optimizer="adam", loss="binary_crossentropy", **kwargs)
    torch.manual_seed(4242)
    ours = getattr(zoo, name)(FeatureMap.from_specs(specs, embedding_dim=emb_dim), gpu=-1, **kwargs)
    sd_ref, sd = ref.state_dict(), ours.state_dict()
    assert list(sd.keys()) == list(sd_ref.keys())
    for k, v in sd_ref.items():
        assert sd[k].dtype == v.dtype and sd[k].shape == v.shape, k
        assert torch.equal(sd[k], v), k
    # module tree: same names, and the same torch module type wherever the reference uses a stock one
    ref_mods = dict(ref.named_modules())
    for mname, mod in ours.named_modules():
        assert mname in ref_mods, mname
        if type(ref_mods[mname]).__module__.startswith("torch."):
            assert type(mod) is type(ref_mods[mname]), mname
    assert set(ref_mods) == set(dict(ours.named_modules()))


@pytest.mark.parametrize("name,specs,kwargs", _MIRROR_CASES, ids=_mirror_case_ids())
def test_mirror_constructors_match_the_stored_reference_seed_for_seed(request, name, specs, kwargs):
    g = Golden("mirror_constructors_seed4242")
    case = g.meta["cases"][request.node.callspec.id]
    sd_ref = g[request.node.callspec.id]
    torch.manual_seed(g.meta["seed"])
    ours = getattr(zoo, name)(FeatureMap.from_specs(specs, embedding_dim=kwargs["embedding_dim"]), gpu=-1, **kwargs)
    sd = ours.state_dict()
    assert list(sd.keys()) == case["keys"]
    for k in case["keys"]:
        v = sd_ref[k]
        assert sd[k].dtype == v.dtype and sd[k].shape == v.shape, k
        assert torch.equal(sd[k], v), k
    # module tree: same names, and the same torch module type wherever the reference uses a stock one
    ref_mods = dict(case["modules"])
    for mname, mod in ours.named_modules():
        assert mname in ref_mods, mname
        if ref_mods[mname] is not None:
            assert "%s.%s" % (type(mod).__module__, type(mod).__qualname__) == ref_mods[mname], mname
    assert set(ref_mods) == set(dict(ours.named_modules()))

"""Locates and imports the UNMODIFIED reference for tests and bench.py's reference arms.

The reference lives under oracle/_ref/ (installed from a FuxiCTR checkout by oracle/install_ref.py,
which __graft_entry__.build() runs; git-ignored).  Test / benchmark infrastructure only: nothing under
fuxictr_b200/ imports this module, and nothing here reads the checkout itself.

SURVEY.md 8(c): `import fuxictr.pytorch.layers` needs three import-time-only dependencies that the
offline image lacks (h5py, polars, keras_preprocessing); empty stub modules are inserted for the
duration of the import and the h5py / polars stubs are removed again (sklearn -> narwhals probes
`polars.DataFrame` if it finds the name in sys.modules).
"""
import contextlib
import importlib
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
REF_ROOT = os.path.join(os.path.dirname(HERE), "oracle", "_ref")
EXTRAS = os.path.join(REF_ROOT, "extras")

MODEL_DIRS = {
    "DeepFM": os.path.join("DeepFM", "DeepFM_torch"),
    "DCNv2": "DCNv2",
    "DLRM": "DLRM",
    "DIN": "DIN",
    "xDeepFM": "xDeepFM",
}


def available():
    return os.path.isdir(os.path.join(REF_ROOT, "fuxictr")) and os.path.isdir(os.path.join(EXTRAS, "model_zoo"))


def why_unavailable():
    return "oracle/_ref is missing (build() installs it when a FuxiCTR checkout is found; see oracle/install_ref.py)"


_IMPORTED = {}


def import_reference():
    """Returns the namespace {layers, FeatureMap, BaseModel, utils, dataloaders, torch_utils} of the real reference."""
    if _IMPORTED:
        return types.SimpleNamespace(**_IMPORTED)
    if not available():
        raise ImportError(why_unavailable())
    stubs = ["h5py", "polars", "keras_preprocessing", "keras_preprocessing.sequence"]
    added = []
    for name in stubs:
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
            added.append(name)
    if "keras_preprocessing.sequence" in added:
        sys.modules["keras_preprocessing.sequence"].pad_sequences = lambda *a, **k: None
        sys.modules["keras_preprocessing"].sequence = sys.modules["keras_preprocessing.sequence"]
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    import fuxictr
    if not os.path.abspath(fuxictr.__file__).startswith(REF_ROOT):
        raise ImportError("another `fuxictr` (%s) shadows oracle/_ref" % fuxictr.__file__)
    import fuxictr.pytorch.layers as layers
    from fuxictr.features import FeatureMap
    from fuxictr.pytorch.models.rank_model import BaseModel
    from fuxictr import utils
    from fuxictr.pytorch import dataloaders, torch_utils
    for name in ("h5py", "polars"):
        if name in added:
            sys.modules.pop(name, None)
    _IMPORTED.update(layers=layers, FeatureMap=FeatureMap, BaseModel=BaseModel, utils=utils,
                     dataloaders=dataloaders, torch_utils=torch_utils)
    return types.SimpleNamespace(**_IMPORTED)


def model_dir(name):
    return os.path.join(EXTRAS, "model_zoo", MODEL_DIRS[name])


def load_model_class(name):
    """The unmodified model_zoo class, e.g. model_zoo/DeepFM/DeepFM_torch/src/DeepFM.py::DeepFM —
    imported exactly like the model's own run_expid.py does (`import src` from its directory)."""
    import_reference()
    path = model_dir(name)
    for k in [k for k in sys.modules if k == "src" or k.startswith("src.")]:
        del sys.modules[k]
    sys.path.insert(0, path)
    try:
        mod = importlib.import_module("src." + name)
    finally:
        sys.path.remove(path)
    return getattr(mod, name)


@contextlib.contextmanager
def chdir(path):
    """The reference's YAMLs hold paths relative to the model directory (run_expid.py chdirs there)."""
    old = os.getcwd()
    os.chdir(path)
    try:
        yield
    finally:
        os.chdir(old)


def load_params(name, expid, dataset_id=None, model_root=None):
    """load_config(model_zoo/<name>/config, expid) of the reference, with the data paths made
    absolute (relative to the model directory, as run_expid.py resolves them).  `dataset_id`
    overrides the experiment's dataset when the shipped dataset_config.yaml lacks it (DeepFM_test
    names tiny_parquet but DeepFM_torch/config only defines tiny_npz)."""
    R = import_reference()
    mdir = model_dir(name)
    with chdir(mdir):
        params = R.utils.load_model_config("./config/", expid)
        ds = dataset_id or params["dataset_id"]
        params["dataset_id"] = ds
        data_dir = os.path.join(EXTRAS, "data", ds)
        fmt = "npz" if os.path.exists(os.path.join(data_dir, "train.npz")) else "parquet"
        params.update(data_root=os.path.join(EXTRAS, "data") + os.sep, data_format=fmt,
                      train_data=os.path.join(data_dir, "train." + fmt),
                      valid_data=os.path.join(data_dir, "valid." + fmt),
                      test_data=os.path.join(data_dir, "test." + fmt))
    if model_root is not None:
        params["model_root"] = model_root
    return params


def load_feature_map(params):
    R = import_reference()
    data_dir = os.path.join(params["data_root"], params["dataset_id"])
    fm = R.FeatureMap(params["dataset_id"], data_dir)
    fm.load(os.path.join(data_dir, "feature_map.json"), params)
    return fm


def synthetic_feature_map(specs, labels=("label",), embedding_dim=None, dataset_id="synthetic"):
    """A reference FeatureMap built in memory from (name, spec) pairs (SURVEY.md 8d)."""
    from collections import OrderedDict
    R = import_reference()
    fm = R.FeatureMap(dataset_id, "/tmp")
    fm.features = OrderedDict((k, dict(v)) for k, v in specs)
    fm.labels = list(labels)
    fm.default_emb_dim = embedding_dim
    fm.num_fields = fm.get_num_fields()
    fm.total_features = sum(s.get("vocab_size", 0) for _, s in specs)
    fm.set_column_index()
    return fm

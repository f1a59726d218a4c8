"""Generates the data-loader fixtures and their golden digests.

    python tests/golden/make_loader_golden.py

1. writes small SYNTHETIC datasets (seeded) in the reference's on-disk formats under
   tests/golden/data/<dataset>/ : feature_map.json + {train,valid,test}.npz | .parquet
   (npz: one named array per column, sequences as (N, L) arrays; parquet: list-valued cells);
2. runs the REAL reference loaders (fuxictr.pytorch.dataloaders, imported from /root/reference —
   build container only) over them with a fixed torch seed and stores per-case SHA-256 digests of
   the batches (all of them, each one, and two further shuffled epochs), their keys, dtypes and shapes in
   tests/golden/loader_digests.json (cases: tests/test_dataloader.py:CASES).
"""
import hashlib
import json
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
DATA = os.path.join(HERE, "data")
REF = os.environ.get("FUXICTR_REFERENCE", "/root/reference")


def spec_cat(v):
    return {"source": "", "type": "categorical", "padding_idx": 0, "vocab_size": v}


def make_dataset(name, fmt, features, label, sizes, seed):
    rng = np.random.default_rng(seed)
    out_dir = os.path.join(DATA, name)
    os.makedirs(out_dir, exist_ok=True)
    input_length = sum(s.get("max_len", 1) for _, s in features)
    blob = {"dataset_id": name, "num_fields": len(features), "total_features": sum(s.get("vocab_size", 0) for _, s in features),
            "input_length": input_length, "labels": [label], "features": [{k: s} for k, s in features]}
    with open(os.path.join(out_dir, "feature_map.json"), "w") as fd:
        json.dump(blob, fd, separators=(",", ":"))
    for split, n in sizes.items():
        cols = {}
        for k, s in features:
            if s["type"] == "categorical":
                cols[k] = rng.integers(0, s["vocab_size"], n).astype(np.int64)
            elif s["type"] == "numeric":
                cols[k] = np.round(rng.random(n), 4)
            else:  # sequence, post-padded with 0
                L = s["max_len"]
                seq = rng.integers(1, s["vocab_size"], (n, L)).astype(np.int64)
                lens = rng.integers(0, L + 1, n)
                seq[np.arange(L)[None, :] >= lens[:, None]] = 0
                cols[k] = seq
        cols[label] = (rng.random(n) < 0.3).astype(np.float64)
        if fmt == "npz":
            np.savez(os.path.join(out_dir, split + ".npz"), **cols)
        else:
            import pandas as pd
            pd.DataFrame({k: (list(v) if v.ndim == 2 else v) for k, v in cols.items()}).to_parquet(
                os.path.join(out_dir, split + ".parquet"))


def write_fixtures():
    sizes = {"train": 203, "valid": 61, "test": 47}
    make_dataset("syn_cat", "npz", [("C%d" % i, spec_cat(20 + 7 * i)) for i in range(6)] +
                 [("price", {"source": "", "type": "numeric"})], "label", sizes, 1)
    make_dataset("syn_seq", "npz", [("userid", spec_cat(30)), ("item", spec_cat(90)),
                                     ("history", {"source": "", "type": "sequence", "share_embedding": "item",
                                                  "padding_idx": 0, "vocab_size": 90, "max_len": 5})],
                 "clk", sizes, 2)
    make_dataset("syn_pq", "parquet", [("userid", spec_cat(30)), ("item", spec_cat(90)),
                                             ("history", {"source": "", "type": "sequence", "share_embedding": "item",
                                                          "padding_idx": 0, "vocab_size": 90, "max_len": 4}),
                                             ("cate", spec_cat(12))], "label", sizes, 3)


def digest(batches):
    h = hashlib.sha256()
    for b in batches:
        for k in b:
            h.update(k.encode())
            h.update(np.ascontiguousarray(b[k].numpy()).tobytes())
    return h.hexdigest()


def reference_digests():
    for name in ["h5py", "polars", "keras_preprocessing", "keras_preprocessing.sequence"]:
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["keras_preprocessing.sequence"].pad_sequences = lambda *a, **k: None
    sys.modules["keras_preprocessing"].sequence = sys.modules["keras_preprocessing.sequence"]
    sys.path.insert(0, REF)
    import torch
    from fuxictr.features import FeatureMap
    from fuxictr.pytorch.dataloaders import rank_dataloader as RD   # re-exports the four loader classes
    sys.path.insert(0, os.path.join(os.path.dirname(HERE)))
    from test_dataloader import CASES
    out = {}
    for dataset, fmt, split, batch_size, shuffle in CASES:
        fm = FeatureMap(dataset, os.path.join(DATA, dataset))
        fm.load(os.path.join(DATA, dataset, "feature_map.json"), {})
        cls = RD.NpzDataLoader if fmt == "npz" else RD.ParquetDataLoader
        torch.manual_seed(7)
        loader = cls(fm, os.path.join(DATA, dataset, split), batch_size=batch_size, shuffle=shuffle, num_workers=0)
        batches = list(loader)
        entry = {"sha256": digest(batches), "num_batches": len(loader), "num_samples": loader.num_samples,
                 "dtype": str(batches[0][fm.labels[0]].dtype),
                 "keys": list(batches[0].keys()), "dtypes": {k: str(v.dtype) for k, v in batches[0].items()},
                 "batch_shapes": [[list(v.shape) for v in b.values()] for b in batches],
                 "batch_sha256": [digest([b]) for b in batches]}
        if shuffle:     # the next two epochs after reseeding: the permutation stream of the loader
            torch.manual_seed(11)
            entry["two_epochs_seed11_sha256"] = digest([b for _ in range(2) for b in loader])
        out["%s/%s/%s/%d/%d" % (dataset, fmt, split, batch_size, int(shuffle))] = entry
    with open(os.path.join(HERE, "loader_digests.json"), "w") as fd:
        json.dump(out, fd, indent=1, sort_keys=True)
    print("wrote", len(out), "digests")


if __name__ == "__main__":
    write_fixtures()
    reference_digests()

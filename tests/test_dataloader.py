"""fuxictr_b200.dataloader on the CPU: batches equal the REAL reference loaders' batches (where the
reference is installed), the stored digests of those batches (everywhere), and the structural contract
(num_samples / num_batches / len / RankDataLoader stages).  Pure host logic: no GPU."""
import hashlib
import json
import os
import sys
import types

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT

from baseline import refenv  # noqa: E402  (the unmodified reference under oracle/_ref)
HAVE_REF = refenv.available()
FIXTURES = os.path.join(ROOT, "tests", "golden", "data")


def FIXDIR(dataset):
    return os.path.join(FIXTURES, dataset)


def _feature_map(dataset):
    from fuxictr_b200.schema import FeatureMap
    fm = FeatureMap(dataset, os.path.join(FIXTURES, dataset))
    fm.load(os.path.join(FIXTURES, dataset, "feature_map.json"), {})
    return fm


def _digest(batches):
    h = hashlib.sha256()
    for b in batches:
        for k in b:
            h.update(k.encode())
            h.update(np.ascontiguousarray(b[k].numpy()).tobytes())
    return h.hexdigest()


def _ours(dataset, fmt, split, batch_size, shuffle, seed=7):
    from fuxictr_b200 import dataloader as DL
    cls = DL.NpzDataLoader if fmt == "npz" else DL.ParquetDataLoader
    torch.manual_seed(seed)
    loader = cls(_feature_map(dataset), os.path.join(FIXTURES, dataset, split), batch_size=batch_size,
                 shuffle=shuffle, pin=False)
    return loader, list(loader)


CASES = [("syn_cat", "npz", "train", 32, False), ("syn_cat", "npz", "train", 32, True),
         ("syn_cat", "npz", "valid", 7, False), ("syn_seq", "npz", "train", 16, True),
         ("syn_pq", "parquet", "train", 32, False), ("syn_pq", "parquet", "test", 10, True)]


@pytest.mark.parametrize("dataset,fmt,split,batch_size,shuffle", CASES)
def test_batches_match_golden_digest(dataset, fmt, split, batch_size, shuffle):
    """Digests were taken from the reference's own loaders (tests/golden/make_loader_golden.py)."""
    with open(os.path.join(GOLDEN, "loader_digests.json")) as fd:
        want = json.load(fd)["%s/%s/%s/%d/%d" % (dataset, fmt, split, batch_size, int(shuffle))]
    loader, batches = _ours(dataset, fmt, split, batch_size, shuffle)
    assert len(batches) == len(loader) == want["num_batches"]
    assert loader.num_samples == want["num_samples"] and loader.num_blocks == 1
    assert str(batches[0][loader.feature_map.labels[0]].dtype) == want["dtype"]
    assert _digest(batches) == want["sha256"]


@pytest.fixture(scope="module")
def ref_loaders():
    if not HAVE_REF:
        pytest.skip(refenv.why_unavailable())
    R = refenv.import_reference()
    from fuxictr.pytorch.dataloaders import rank_dataloader as RD   # re-exports the four loader classes
    return types.SimpleNamespace(FeatureMap=R.FeatureMap, RD=RD)


@pytest.mark.parametrize("dataset,fmt,split,batch_size,shuffle", CASES)
def test_batches_match_the_live_reference(ref_loaders, dataset, fmt, split, batch_size, shuffle):
    rfm = ref_loaders.FeatureMap(dataset, FIXDIR(dataset))
    rfm.load(os.path.join(FIXDIR(dataset), "feature_map.json"), {})
    cls = ref_loaders.RD.NpzDataLoader if fmt == "npz" else ref_loaders.RD.ParquetDataLoader
    torch.manual_seed(7)
    rloader = cls(rfm, os.path.join(FIXDIR(dataset), split), batch_size=batch_size, shuffle=shuffle,
                  num_workers=0)
    want = list(rloader)
    loader, got = _ours(dataset, fmt, split, batch_size, shuffle)
    assert len(got) == len(want) == len(loader) == len(rloader)
    for a, b in zip(got, want):
        assert list(a.keys()) == list(b.keys())
        for k in a:
            assert a[k].dtype == b[k].dtype and torch.equal(a[k], b[k]), k
    # a second epoch draws the next permutation from the same RNG stream on both sides
    if shuffle:
        torch.manual_seed(11)
        want2 = [b for _ in range(2) for b in rloader]
        torch.manual_seed(11)
        got2 = [b for _ in range(2) for b in loader]
        assert _digest(got2) == _digest(want2)


@pytest.mark.parametrize("dataset,fmt,split,batch_size,shuffle", CASES)
def test_batches_match_the_stored_reference_batches(dataset, fmt, split, batch_size, shuffle):
    """The live comparison above, against what the reference's own loaders yielded when the goldens
    were made (keys, dtypes, shapes and SHA-256 of every batch; make_loader_golden.py): runs without
    the reference installed."""
    with open(os.path.join(GOLDEN, "loader_digests.json")) as fd:
        want = json.load(fd)["%s/%s/%s/%d/%d" % (dataset, fmt, split, batch_size, int(shuffle))]
    loader, got = _ours(dataset, fmt, split, batch_size, shuffle)
    assert len(got) == len(want["batch_sha256"]) == len(loader) == want["num_batches"]
    for a, shapes, digest in zip(got, want["batch_shapes"], want["batch_sha256"]):
        assert list(a.keys()) == want["keys"]
        assert {k: str(v.dtype) for k, v in a.items()} == want["dtypes"]
        assert [list(v.shape) for v in a.values()] == shapes
        assert _digest([a]) == digest
    # a second epoch draws the next permutation from the same RNG stream on both sides
    if shuffle:
        torch.manual_seed(11)
        got2 = [b for _ in range(2) for b in loader]
        assert _digest(got2) == want["two_epochs_seed11_sha256"]


def test_matrices_are_the_collators_matrix():
    """`.matrices()` yields the (B, W) matrix whose column views the batch dict holds."""
    loader, batches = _ours("syn_cat", "npz", "train", 32, False)
    fm = loader.feature_map
    for mat, b in zip(loader.matrices(), batches):
        assert mat.shape[1] == fm.input_length + len(fm.labels)
        for k, v in fm.batch_dict(mat).items():
            assert torch.equal(v, b[k])
    assert loader.matrix.shape[0] == loader.num_samples


def _write_blocks(tmp_path, fmt, sizes, seed=0):
    fm = _feature_map("syn_cat" if fmt == "npz" else "syn_pq")
    src = os.path.join(FIXTURES, fm.dataset_id, "train." + fmt)
    from fuxictr_b200 import dataloader as DL
    full = (DL.load_npz_matrix if fmt == "npz" else DL.load_parquet_matrix)(fm, src)
    cols = list(fm.features.keys()) + list(fm.labels)
    lo = 0
    for i, n in enumerate(sizes):
        part = full[lo:lo + n]
        lo += n
        path = os.path.join(str(tmp_path), "part_%03d.%s" % (i, fmt))
        if fmt == "npz":
            np.savez(path, **{c: part[:, fm.get_column_index(c)] for c in cols})
        else:
            import pandas as pd
            frame = {}
            for c in cols:
                v = part[:, fm.get_column_index(c)]
                frame[c] = list(v) if v.ndim == 2 else v
            pd.DataFrame(frame).to_parquet(path)
    return fm, full[:lo]


@pytest.mark.parametrize("fmt", ["npz", "parquet"])
def test_block_loader_runs_batches_across_block_boundaries(tmp_path, fmt):
    from fuxictr_b200 import dataloader as DL
    fm, full = _write_blocks(tmp_path, fmt, [30, 1, 45, 24])
    cls = DL.NpzBlockDataLoader if fmt == "npz" else DL.ParquetBlockDataLoader
    loader = cls(fm, str(tmp_path), split="train", batch_size=16, shuffle=False, pin=False)
    assert (loader.num_blocks, loader.num_samples, len(loader)) == (4, 100, 7)
    got = torch.cat([m.clone() for m in loader.matrices()])
    assert np.array_equal(got.numpy(), full)
    batches = list(loader)                      # dict protocol hands out copies, safe to keep
    assert [b[fm.labels[0]].shape[0] for b in batches] == [16] * 6 + [4]
    assert np.array_equal(torch.cat([b[fm.labels[0]] for b in batches]).numpy(), full[:, -1])


def test_block_loader_shuffle_is_a_permutation_and_seeded(tmp_path):
    from fuxictr_b200 import dataloader as DL
    fm, full = _write_blocks(tmp_path, "npz", [40, 40, 20])
    loader = DL.NpzBlockDataLoader(fm, str(tmp_path), batch_size=16, shuffle=True, buffer_size=24, pin=False)
    torch.manual_seed(3)
    a = torch.cat([m.clone() for m in loader.matrices()]).numpy()
    torch.manual_seed(3)
    b = torch.cat([m.clone() for m in loader.matrices()]).numpy()
    assert np.array_equal(a, b) and not np.array_equal(a, full)
    key = lambda m: sorted(map(tuple, m.tolist()))   # noqa: E731
    assert key(a) == key(full)


def test_rank_dataloader_stages():
    from fuxictr_b200 import dataloader as DL
    fm = _feature_map("syn_cat")
    base = os.path.join(FIXTURES, "syn_cat")
    kw = dict(train_data=os.path.join(base, "train"), valid_data=os.path.join(base, "valid"),
              test_data=os.path.join(base, "test"), batch_size=64, data_format="npz", pin=False)
    train, valid, test = DL.RankDataLoader(fm, stage="both", **kw).make_iterator()
    assert train.shuffle and not valid.shuffle and not test.shuffle
    assert isinstance(train, DL.NpzDataLoader) and len(train) == int(np.ceil(train.num_samples / 64))
    train, valid = DL.RankDataLoader(fm, stage="train", **kw).make_iterator()
    assert train is not None and valid is not None
    only_test = DL.RankDataLoader(fm, stage="test", **kw).make_iterator()
    assert isinstance(only_test, DL.NpzDataLoader) and not only_test.shuffle
    rd = DL.RankDataLoader(fm, stage="train", train_data=kw["train_data"], batch_size=8, shuffle=False, pin=False)
    assert rd.valid_gen is None and rd.test_gen is None and not rd.train_gen.shuffle


def test_prefetcher_surfaces_producer_errors():
    from fuxictr_b200.dataloader import _Prefetcher

    def bad():
        yield 1
        raise ValueError("boom")
    it = iter(_Prefetcher(bad, 2))
    assert next(it) == 1
    with pytest.raises(ValueError, match="boom"):
        next(it)


@pytest.mark.parametrize("shuffle", [False, True])
@pytest.mark.parametrize("world", [2, 3])
def test_sharded_loader_is_a_partition_of_the_global_batches(world, shuffle):
    """shard=(rank, world): rank r holds rows [r*B, (r+1)*B) of every global batch of B*world rows —
    concatenating the ranks rebuilds the unsharded loader's batches (same seed on every rank)."""
    from fuxictr_b200 import dataloader as DL
    fm = _feature_map("syn_cat")
    path = os.path.join(FIXTURES, "syn_cat", "train")
    B = 16
    torch.manual_seed(9)
    whole = [m.clone() for m in DL.NpzDataLoader(fm, path, batch_size=B * world, shuffle=shuffle, pin=False).matrices()]
    parts = []
    for r in range(world):
        torch.manual_seed(9)
        loader = DL.NpzDataLoader(fm, path, batch_size=B, shuffle=shuffle, pin=False, shard=(r, world))
        parts.append([m.clone() for m in loader.matrices()])
        assert len(parts[-1]) == len(loader) == 203 // (B * world)          # incomplete last global batch dropped
        assert all(m.shape[0] == B for m in parts[-1])
    for g in range(len(parts[0])):
        assert torch.equal(torch.cat([parts[r][g] for r in range(world)]), whole[g])
    # drop_last=False: the tail is split in rank order, short or empty shares allowed
    tails = []
    for r in range(world):
        torch.manual_seed(9)
        loader = DL.NpzDataLoader(fm, path, batch_size=B, shuffle=shuffle, pin=False, shard=(r, world), drop_last=False)
        ms = [m.clone() for m in loader.matrices()]
        assert len(ms) == len(loader) == len(whole)
        tails.append(ms[-1])
    assert torch.equal(torch.cat(tails), whole[-1])
    with pytest.raises(ValueError):
        DL.NpzDataLoader(fm, path, batch_size=B, pin=False, shard=(world, world))

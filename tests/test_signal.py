"""Data-feed parity (CPU): the signal iterator and index-batching follow the reference's semantics;
indexing is BIT-EXACT (mirrors test/index_test.py:93-114 and test/dataset_test.py:74-171,717-735)."""
import os

import numpy as np
import pytest
import torch

from oracle import signal as OS
from pytorch_geometric_temporal_b200.dataset import ChickenpoxDatasetLoader
from pytorch_geometric_temporal_b200.signal import (IndexDataset, StaticGraphTemporalSignal, index_splits, shard_indices,
                                                    temporal_signal_split)


def _random_signal(T=7, n=5, e=9, f=3, seed=0):
    rng = np.random.RandomState(seed)
    ei = rng.randint(0, n, size=(2, e))
    ew = rng.rand(e)
    feats = [rng.rand(n, f) for _ in range(T)]
    tg = [rng.rand(n) for _ in range(T)]
    return ei, ew, feats, tg


def test_iterator_two_epochs_and_types():
    ei, ew, feats, tg = _random_signal()
    sig = StaticGraphTemporalSignal(ei, ew, feats, tg)
    for _ in range(2):  # __iter__ resets (static_graph_temporal_signal.py:123-134)
        n = 0
        for t, snap in enumerate(sig):
            want = OS.snapshot(ei, ew, feats, tg, t)
            for k in ("x", "edge_index", "edge_attr", "y"):
                assert torch.equal(getattr(snap, k), want[k])
            assert snap.x.dtype == torch.float32 and snap.edge_index.dtype == torch.int64
            n += 1
        assert n == 7


def test_none_passthrough_int_targets_and_kwargs():
    ei, ew, feats, tg = _random_signal()
    sig = StaticGraphTemporalSignal(None, None, [None] * 7, [None] * 7)
    s = sig[0]
    assert s.x is None and s.edge_index is None and s.edge_attr is None and s.y is None
    ints = [np.arange(5) for _ in range(7)]
    extra = [np.ones((5, 2)) for _ in range(7)]
    sig = StaticGraphTemporalSignal(ei, ew, feats, ints, optional=extra, labels=ints)
    s = sig[3]
    assert s.y.dtype == torch.int64 and s.optional.dtype == torch.float32 and s.labels.dtype == torch.int64
    assert sig.additional_feature_keys == ["optional", "labels"]
    with pytest.raises(AssertionError):
        StaticGraphTemporalSignal(ei, ew, feats, tg[:-1])


def test_split_and_slice():
    ei, ew, feats, tg = _random_signal(T=10)
    sig = StaticGraphTemporalSignal(ei, ew, feats, tg)
    tr, te = temporal_signal_split(sig, 0.8)
    assert (tr.snapshot_count, te.snapshot_count) == OS.split_counts(10, 0.8) == (8, 2)
    assert torch.equal(te[0].x, sig[8].x)
    sub = sig[2:5]
    assert sub.snapshot_count == 3 and torch.equal(sub[0].x, sig[2].x)


def test_index_batching_equals_snapshot_iterator_chickenpox():
    """The reference's only value-level test (test/index_test.py:93-114), on the in-tree fixture."""
    loader = ChickenpoxDatasetLoader()
    dataset = loader.get_dataset()
    train, _, _, edges, edge_weights = ChickenpoxDatasetLoader(index=True).get_index_dataset(batch_size=1, shuffle=False)
    for _ in range(2):
        n = 0
        for snapshot, (x, y) in zip(dataset, train):
            x = torch.squeeze(x).permute(1, 0).float()
            y = torch.squeeze(y).float()[0, ...]
            assert torch.equal(snapshot.x, x) and torch.equal(snapshot.y, y)
            assert torch.equal(snapshot.edge_index, edges) and torch.equal(snapshot.edge_attr, edge_weights)
            assert edges.shape == (2, 102) and edge_weights.shape == (102,) and x.shape == (20, 4) and y.shape == (20,)
            n += 1
        assert n == len(train)
    assert dataset.snapshot_count == 517


def test_index_dataset_matches_oracle_and_reference(golden_dir):
    rng = np.random.RandomState(0)
    data = rng.rand(60, 7, 2).astype(np.float32)
    tr, va, te = index_splits(60, 12)
    otr, ova, ote = OS.index_splits(60, 12)
    assert np.array_equal(tr, otr) and np.array_equal(va, ova) and np.array_equal(te, ote)
    ds = IndexDataset(tr, data, 12)
    for i in (0, 3, len(ds) - 1):
        x, y = ds[i]
        ox, oy = OS.index_window(data, tr, i, 12)
        assert np.array_equal(x.numpy(), ox) and np.array_equal(y.numpy(), oy)
    # what the unmodified reference IndexDataset returns for every window (tests/golden/make_goldens_parity.py)
    ref = torch.load(os.path.join(golden_dir, "reference_data.pt"), weights_only=False)["index_dataset"]
    assert len(ds) == len(ref["x"])
    for i in range(len(ds)):
        assert torch.equal(ds[i][0], ref["x"][i]) and torch.equal(ds[i][1], ref["y"][i])
    with pytest.raises(ValueError):
        IndexDataset(tr, data, 12, lazy=True)


@pytest.mark.parametrize("n,world,shuffle", [(23, 4, False), (23, 4, True), (8, 8, True), (5, 8, False), (100, 2, True)])
def test_shard_indices_is_distributed_sampler(n, world, shuffle):
    from torch.utils.data import DistributedSampler
    ds = list(range(n))
    for epoch in (0, 3):
        for rank in range(world):
            s = DistributedSampler(ds, num_replicas=world, rank=rank, shuffle=shuffle, seed=7)
            s.set_epoch(epoch)
            assert list(s) == shard_indices(n, world, rank, shuffle, 7, epoch)


def test_snapshot_to_device_reuses_static_graph_tensors():
    """`.to(device)` on successive snapshots must hand the layers the SAME edge tensors (plan-cache identity)."""
    ei, ew, feats, tg = _random_signal()
    sig = StaticGraphTemporalSignal(ei, ew, feats, tg)
    a, b = sig[0].to("cpu"), sig[1].to("cpu")
    assert a.edge_index is b.edge_index and a.edge_attr is b.edge_attr
    assert a.x is not b.x and torch.equal(a.edge_index, torch.LongTensor(ei))

"""Host-side tests of the SURVEY 8f rank 2/3 rows: StaticGraphTemporalSignalBatch (mirrors test/batch_test.py:120-134,
:181-190) and the offline METR-LA / PEMS-BAY loaders (mirrors test/index_test.py:18-66 on synthetic archives; what the
unmodified reference loaders and iterators return on the same inputs is stored in tests/golden/reference_data.pt by
tests/golden/make_goldens_parity.py and must be matched bit for bit)."""
import hashlib
import os

import numpy as np
import pytest
import torch

from pytorch_geometric_temporal_b200.dataset import METRLADatasetLoader, PemsBayDatasetLoader, dense_to_sparse
from pytorch_geometric_temporal_b200.signal import StaticGraphTemporalSignalBatch, temporal_signal_split


def _archive(tmp, n, f, t, prefix=""):
    rng = np.random.default_rng(7)
    A = (rng.random((n, n)) < 0.2) * rng.random((n, n)).astype(np.float32)
    np.fill_diagonal(A, 1.0)
    np.save(os.path.join(tmp, prefix + "adj_mat.npy"), A.astype(np.float32))
    np.save(os.path.join(tmp, prefix + "node_values.npy"), (rng.normal(size=(t, n, f)) * 10 + 50))   # float64, like the archive
    return A


def test_static_graph_temporal_signal_batch_none_and_typing():
    ds = StaticGraphTemporalSignalBatch(None, None, [None, None], [None, None], None)
    n = 0
    for snap in ds:
        assert snap.edge_index is None and snap.edge_attr is None and snap.x is None and snap.y is None and snap.batch is None
        n += 1
    assert n == 2
    ds = StaticGraphTemporalSignalBatch(None, None, [np.array([1])], [np.array([2])], None)
    for snap in ds:
        assert snap.x.shape == (1,) and snap.y.shape == (1,) and snap.batch is None


def test_static_graph_temporal_signal_batch_iteration_and_split():
    rng = np.random.default_rng(0)
    # two graphs of 5 and 7 nodes, block-diagonal edge list
    e1, e2 = rng.integers(0, 5, (2, 12)), rng.integers(0, 7, (2, 20)) + 5
    ei = np.concatenate([e1, e2], axis=1)
    ew = rng.random(ei.shape[1])
    batches = np.array([0] * 5 + [1] * 7)
    feats = [rng.random((12, 3)) for _ in range(10)]
    targs = [rng.random((12,)) for _ in range(10)]
    extra = [rng.integers(0, 4, (12,)) for _ in range(10)]
    ds = StaticGraphTemporalSignalBatch(ei, ew, feats, targs, batches, marks=extra)
    for epoch in range(2):
        seen = 0
        for t, snap in enumerate(ds):
            assert snap.x.shape == (12, 3) and snap.x.dtype == torch.float32
            assert snap.edge_index.dtype == torch.int64 and torch.equal(snap.edge_index, torch.from_numpy(ei))
            assert torch.equal(snap.batch, torch.from_numpy(batches)) and snap.batch.dtype == torch.int64
            assert torch.equal(snap.marks, torch.from_numpy(extra[t]))
            assert "batch" in snap.keys()
            seen += 1
        assert seen == 10
    a, b = ds[0], ds[1]
    assert a.edge_index is b.edge_index and a.batch is b.batch        # static tensors are shared, not re-wrapped
    tr, te = temporal_signal_split(ds, 0.8)
    assert isinstance(tr, StaticGraphTemporalSignalBatch) and tr.snapshot_count == 8 and te.snapshot_count == 2
    assert torch.equal(te[0].batch, torch.from_numpy(batches))
    assert isinstance(ds[2:5], StaticGraphTemporalSignalBatch) and len(ds[2:5].features) == 3


def test_dense_to_sparse_row_major():
    A = torch.tensor([[0.0, 2.0, 0.0], [3.0, 0.0, 0.0], [0.0, 4.0, 5.0]])
    ei, w = dense_to_sparse(A)
    assert ei.tolist() == [[0, 1, 2, 2], [1, 0, 1, 2]] and w.tolist() == [2.0, 3.0, 4.0, 5.0]


@pytest.mark.parametrize("cls,prefix,lags", [(METRLADatasetLoader, "", 6), (PemsBayDatasetLoader, "pems_", 4)])
def test_index_batching_equals_snapshot_iterator(tmp_path, cls, prefix, lags):
    """test/index_test.py:18-66 on a synthetic archive: windows served by index batching are the snapshots, bit for bit."""
    tmp = str(tmp_path)
    A = _archive(tmp, 9, 2, 60, prefix)
    dataset = cls(raw_data_dir=tmp).get_dataset(num_timesteps_in=lags, num_timesteps_out=lags)
    train, val, test, edges, weights, means, stds = cls(raw_data_dir=tmp, index=True).get_index_dataset(batch_size=1, shuffle=False, lags=lags)
    n_windows = 60 - (2 * lags - 1)
    assert len(train.dataset) == round(n_windows * 0.7) and len(test.dataset) == round(n_windows * 0.2)
    assert len(train.dataset) + len(val.dataset) + len(test.dataset) == n_windows
    assert edges.shape == (2, int((A != 0).sum())) and means.shape == (2,) and stds.shape == (2,)
    for epoch in range(2):
        k = 0
        for snap, (x, y) in zip(dataset, train):
            x = torch.squeeze(x).permute(1, 2, 0)
            y = torch.squeeze(y)[..., 0].permute(1, 0) if cls is METRLADatasetLoader else torch.squeeze(y).permute(1, 2, 0)
            assert torch.equal(snap.x, x) and torch.equal(snap.y, y)
            assert torch.equal(snap.edge_index, edges) and torch.equal(snap.edge_attr, weights)
            k += 1
        assert k == len(train.dataset)


def test_offline_loader_errors(tmp_path):
    with pytest.raises(FileNotFoundError):
        METRLADatasetLoader(raw_data_dir=str(tmp_path))
    _archive(str(tmp_path), 5, 2, 40)
    with pytest.raises(ValueError):
        METRLADatasetLoader(raw_data_dir=str(tmp_path)).get_index_dataset()


def _digest(t):
    """SHA-256 of a tensor's dtype, shape and bytes: equal digests <=> bit-identical tensors of one dtype and shape."""
    t = t.contiguous()
    return hashlib.sha256(f"{t.dtype}{tuple(t.shape)}".encode() + t.numpy().tobytes()).hexdigest()


@pytest.fixture(scope="module")
def ref(golden_dir):
    return torch.load(os.path.join(golden_dir, "reference_data.pt"), weights_only=False)


@pytest.mark.parametrize("mod,name,prefix", [("dataset.metr_la", "METRLADatasetLoader", ""), ("dataset.pems_bay", "PemsBayDatasetLoader", "pems_")])
def test_offline_loaders_match_reference(tmp_path, mod, name, prefix, ref):
    """Our loaders against the outputs of the unmodified reference loaders on the same archive, stored as `_digest`s."""
    tmp = str(tmp_path)
    _archive(tmp, 9, 2, 30, prefix)
    want = ref["loaders"][prefix]
    ours_cls = METRLADatasetLoader if prefix == "" else PemsBayDatasetLoader
    got = [[_digest(getattr(b, k)) for k in ("x", "y", "edge_index", "edge_attr")] for b in ours_cls(raw_data_dir=tmp).get_dataset(6, 6)]
    assert got == want["snapshots"]
    g = ours_cls(raw_data_dir=tmp, index=True).get_index_dataset(lags=6, batch_size=4)
    for i in range(3):
        assert [[_digest(x), _digest(y)] for x, y in g[i]] == want["index_batches"][i]
    assert [_digest(t) for t in g[3:7]] == want["index_tensors"]
    # DistributedSampler shards
    g = ours_cls(raw_data_dir=tmp, index=True).get_index_dataset(lags=6, batch_size=4, shuffle=True, world_size=2, ddp_rank=1)
    assert [[_digest(x), _digest(y)] for x, y in g[0]] == want["shard_batches"]


# ---- SURVEY 8f rank 4: dynamic-graph iterators ------------------------------------------------------------------------
from pytorch_geometric_temporal_b200.signal import (DynamicGraphStaticSignal, DynamicGraphStaticSignalBatch,  # noqa: E402
                                                     DynamicGraphTemporalSignal, DynamicGraphTemporalSignalBatch)


def _dynamic_case(T=6, n=9, seed=0):
    rng = np.random.default_rng(seed)
    eis = [rng.integers(0, n, (2, int(rng.integers(5, 15)))) for _ in range(T)]
    ews = [rng.random(e.shape[1]) for e in eis]
    xs = [rng.random((n, 3)) for _ in range(T)]
    ys = [rng.integers(0, 5, (n,)) if t % 2 else rng.random((n,)) for t in range(T)]
    bs = [np.array([0] * 4 + [1] * (n - 4)) for _ in range(T)]
    marks = [rng.random((n, 2)) for _ in range(T)]
    return eis, ews, xs, ys, bs, marks


def test_dynamic_signals_none_passthrough():
    for snap in DynamicGraphTemporalSignal([None, None], [None, None], [None, None], [None, None]):       # dataset_test.py:117-125
        assert snap.edge_index is None and snap.edge_attr is None and snap.x is None and snap.y is None
    for snap in DynamicGraphStaticSignal([None], [None], None, [None]):                                    # :137-143
        assert snap.edge_index is None and snap.edge_attr is None and snap.x is None and snap.y is None
    for snap in DynamicGraphTemporalSignalBatch([None, None], [None, None], [None, None], [None, None], [None, None]):
        assert snap.x is None and snap.batch is None
    for snap in DynamicGraphStaticSignalBatch([None], [None], None, [None], [None]):
        assert snap.x is None and snap.batch is None
    with pytest.raises(AssertionError):
        DynamicGraphTemporalSignal([None, None], [None], [None, None], [None, None])


def test_dynamic_signals_iteration_typing_slicing():
    eis, ews, xs, ys, bs, marks = _dynamic_case()
    ds = DynamicGraphTemporalSignal(eis, ews, xs, ys, marks=marks)
    for epoch in range(2):
        for t, snap in enumerate(ds):
            assert torch.equal(snap.edge_index, torch.from_numpy(eis[t])) and snap.edge_index.dtype == torch.int64
            assert torch.equal(snap.edge_attr, torch.from_numpy(ews[t]).float())
            assert torch.equal(snap.x, torch.from_numpy(xs[t]).float())
            assert snap.y.dtype == (torch.int64 if t % 2 else torch.float32)
            assert torch.equal(snap.marks, torch.from_numpy(marks[t]).float())
        assert t == 5
    tr, te = temporal_signal_split(ds, 0.5)
    assert isinstance(tr, DynamicGraphTemporalSignal) and tr.snapshot_count == 3 and te.snapshot_count == 3
    assert torch.equal(te[0].edge_index, torch.from_numpy(eis[3])) and torch.equal(te[0].marks, torch.from_numpy(marks[3]).float())
    st = DynamicGraphStaticSignal(eis, ews, xs[0], ys)
    assert len(st) == 6 and st[2].x is st[4].x and torch.equal(st[2].x, torch.from_numpy(xs[0]).float())   # static field converted once
    assert isinstance(st[1:3], DynamicGraphStaticSignal) and st[1:3].snapshot_count == 2
    bt = DynamicGraphTemporalSignalBatch(eis, ews, xs, ys, bs)
    assert torch.equal(bt[3].batch, torch.from_numpy(bs[3])) and "batch" in bt[3].keys()
    sb = DynamicGraphStaticSignalBatch(eis, ews, xs[0], ys, bs)
    assert torch.equal(sb[5].batch, torch.from_numpy(bs[5])) and sb[0:2].snapshot_count == 2
    # a piecewise-constant graph handing in the same array object twice shares the converted tensor (=> one cached plan)
    pc = DynamicGraphTemporalSignal([eis[0], eis[0], eis[1]], [ews[0], ews[0], ews[1]], xs[:3], ys[:3])
    assert pc[0].edge_index is pc[1].edge_index and pc[1].edge_index is not pc[2].edge_index


def test_dynamic_signals_match_reference(ref):
    eis, ews, xs, ys, bs, marks = _dynamic_case(seed=3)
    pairs = [
        (DynamicGraphTemporalSignal, (eis, ews, xs, ys)),
        (DynamicGraphStaticSignal, (eis, ews, xs[0], ys)),
        (DynamicGraphTemporalSignalBatch, (eis, ews, xs, ys, bs)),
        (DynamicGraphStaticSignalBatch, (eis, ews, xs[0], ys, bs)),
        (StaticGraphTemporalSignalBatch, (eis[0], ews[0], xs, ys, bs[0])),
    ]
    for our_cls, args in pairs:
        want, got = ref["dynamic_signals"][our_cls.__name__], our_cls(*args, marks=marks)
        keys = ("x", "edge_index", "edge_attr", "y", "marks") + (("batch",) if "Batch" in our_cls.__name__ else ())
        assert [[_digest(getattr(b, k)) for k in keys] for b in got] == want["snapshots"]
        ga = got[1:4]
        assert [ga.snapshot_count, _digest(ga[0].x), _digest(ga[2].edge_index)] == want["slice"]


# ---- host-side algebra of the hand-written DCRNN backward ---------------------------------------------------------------
@pytest.mark.parametrize("K", [1, 2, 3, 4])
def test_unstack_weight_grad_is_the_adjoint_of_stack_weight(K):
    """dL/dW from dL/d(stacked W): block 0 of the stacked basis feeds BOTH W[0,0] and W[1,0] (dcrnn.py:81-84 adds the two
    k=0 products of the same X), block 1+2(k-1)+o feeds W[o,k].  Checked against autograd of `_stack_weight`."""
    from pytorch_geometric_temporal_b200.nn.recurrent.dcrnn import _stack_weight, _unstack_weight_grad
    C, O = 5, 3
    W = torch.randn(2, K, C, O, requires_grad=True)
    G = torch.randn((2 * K - 1) * C, O)
    (_stack_weight(W) * G).sum().backward()
    assert torch.equal(W.grad, _unstack_weight_grad(G, K, C))

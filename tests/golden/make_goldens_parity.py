"""Golden vectors for the parity tests that compare with the UNMODIFIED reference: the module checks of
tests/test_oracle_vs_reference.py and the data-feed checks of tests/test_next_rows_cpu.py, tests/test_signal.py and
tests/test_distributed_cpu.py.  Each case runs the reference (imported through oracle/refload.py on top of oracle/stubs)
on the inputs its test builds and stores what the reference returned, so the tests need no reference checkout.

Module parameters and inputs are not stored: both sides draw them with `_seeded` (numpy's RandomState, a stream numpy
keeps fixed across releases) from the seed and shapes stored with each case.

Run where the reference checkout is present:   python tests/golden/make_goldens_parity.py
Writes tests/golden/reference_modules.pt and tests/golden/reference_data.pt."""
import importlib.util
import os
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
from oracle import refload  # noqa: E402
from make_goldens import save  # noqa: E402
from test_distributed_cpu import _mae_inputs  # noqa: E402
from test_next_rows_cpu import _archive, _digest, _dynamic_case  # noqa: E402
from test_oracle_vs_reference import _seeded  # noqa: E402

NORMS = ["sym", "rw", None]


def _graph(n=12, e=40, seed=0):
    g = torch.Generator().manual_seed(seed)
    row = torch.randint(0, n, (e,), generator=g)
    col = torch.randint(0, n, (e,), generator=g)
    pairs = {(int(r), int(c)) for r, c in zip(row, col)} | {(i, i) for i in range(n)} | {(i, (i + 1) % n) for i in range(n)}
    ei = torch.tensor(sorted(pairs)).t().contiguous()
    return ei, torch.rand(ei.size(1), generator=g) * 0.9 + 0.1


def _case(ref, seed, **inputs):
    """Set `ref`'s parameters to `_seeded(seed, ...)` and draw its inputs from seed + 1; returns (case dict, inputs)."""
    params = {k: tuple(p.shape) for k, p in ref.named_parameters()}
    res = ref.load_state_dict(_seeded(seed, params), strict=False)
    assert not res.unexpected_keys and all(k.rsplit(".", 1)[-1] in ("running_mean", "running_var", "num_batches_tracked")
                                           for k in res.missing_keys), res
    return dict(seed=seed, params=params, inputs=inputs), _seeded(seed + 1, inputs)


def modules():
    ei, ew = _graph()
    eiu = sorted({(a, b) for a, b in ei.t().tolist() if a != b} | {(b, a) for a, b in ei.t().tolist() if a != b})
    eiu = torch.tensor(eiu).t().contiguous()
    out = {"edge_index": ei, "edge_weight": ew, "edge_index_undirected": eiu}
    torch.set_grad_enabled(False)

    dc = refload.load("nn.recurrent.dcrnn")
    out["dcrnn"] = {}
    for K in (1, 2, 3, 4):
        ref = dc.DCRNN(2, 8, K)
        cell, x = _case(ref, 100 + 10 * K, X=(12, 2), H=(12, 8))
        cell.update(out=ref(x["X"], ei, ew, x["H"]), out_noew_noh=ref(x["X"], ei))
        ref = dc.BatchedDCRNN(2, 8, K)
        batched, x = _case(ref, 105 + 10 * K, X=(3, 4, 12, 2))
        batched.update(out=ref(x["X"], ei, ew))
        out["dcrnn"][K] = dict(cell=cell, batched=batched)

    gg, gl = refload.load("nn.recurrent.gconv_gru"), refload.load("nn.recurrent.gconv_lstm")
    out["gconv"] = {}
    for K in (1, 2, 3, 4):
        for i, norm in enumerate(NORMS):
            lm = None if norm == "sym" else torch.tensor(2.3)
            ref = gg.GConvGRU(4, 8, K, normalization=norm)
            gru, x = _case(ref, 200 + 10 * K + 2 * i, X=(12, 4), H=(12, 8))
            gru.update(lambda_max=lm, out=ref(x["X"], ei, ew, x["H"], lm))
            ref = gl.GConvLSTM(4, 8, K, normalization=norm)
            lstm, x = _case(ref, 300 + 10 * K + 2 * i, X=(12, 4), H=(12, 8), C=(12, 8))
            lstm.update(lambda_max=lm, out=ref(x["X"], ei, ew, x["H"], x["C"], lm))
            out["gconv"][(K, norm)] = dict(gru=gru, lstm=lstm)

    tg, at = refload.load("nn.recurrent.temporalgcn"), refload.load("nn.recurrent.attentiontemporalgcn")
    t = {"tgcn": {}}
    for i, (improved, asl) in enumerate([(False, True), (False, False), (True, True), (True, False)]):
        ref = tg.TGCN(4, 8, improved=improved, add_self_loops=asl)
        c, x = _case(ref, 400 + 2 * i, X=(12, 4), H=(12, 8))
        c.update(out=ref(x["X"], ei, ew, x["H"]))
        t["tgcn"][(improved, asl)] = c
    ref = tg.TGCN2(4, 8, 3)
    t["tgcn2"], x = _case(ref, 410, X=(3, 12, 4), H=(3, 12, 8))
    t["tgcn2"]["out"] = ref(x["X"], ei, ew, x["H"])
    ref = at.A3TGCN2(4, 8, 6, 3)
    t["a3tgcn2"], x = _case(ref, 412, X=(3, 12, 4, 6))
    t["a3tgcn2"]["out"] = ref(x["X"], ei, ew)
    ref = at.A3TGCN(4, 8, 6)
    t["a3tgcn"], x = _case(ref, 414, X=(12, 4, 6))
    t["a3tgcn"]["out"] = ref(x["X"], ei, ew)
    out["tgcn_family"] = t

    ag = refload.load("nn.attention.astgcn")
    out["astgcn"], out["chebconv_attention"] = {}, {}
    for i, norm in enumerate(NORMS):
        ref = ag.ASTGCN(2, 1, 3, 8, 8, 2, 4, 6, 12, normalization=norm)
        c, x = _case(ref, 500 + 2 * i, X=(3, 12, 1, 6))
        c["out"] = ref(x["X"], eiu)
        out["astgcn"][norm] = c
        # the multi-graph mini-batch call of the reference's own test (test/attention_test.py:205-218): a node->graph
        # `batch` vector and one lambda_max per graph
        ref = ag.ChebConvAttention(5, 7, K=3, normalization=norm)
        c, x = _case(ref, 510 + 2 * i, x=(3, 7, 5))
        g = torch.Generator().manual_seed(i)
        c.update(batch=torch.tensor([0, 0, 0, 1, 1, 1, 1]), edge_index=torch.tensor([[0, 1, 1, 2, 3, 4, 5, 6, 3, 6], [1, 0, 2, 1, 4, 3, 6, 5, 6, 3]]),
                 lambda_max=torch.tensor([2.0, 3.0]))
        c.update(edge_weight=torch.rand(10, generator=g) + 0.1, S=torch.softmax(torch.rand(3, 7, 7, generator=g), dim=1))
        c.update(out=ref(x["x"], c["edge_index"], c["S"], c["edge_weight"], c["batch"], c["lambda_max"]),
                 out_one_lambda=ref(x["x"], c["edge_index"], c["S"], c["edge_weight"], None, 2.0))
        out["chebconv_attention"][norm] = c

    gc = refload.load("nn.recurrent.gc_lstm")
    out["gc_lstm"] = {}
    for K in (1, 2, 3):
        for i, norm in enumerate(NORMS):
            lm = None if norm == "sym" else torch.tensor(2.3)
            ref = gc.GCLSTM(4, 8, K, normalization=norm)
            c, x = _case(ref, 600 + 10 * K + 2 * i, X=(12, 4), H=(12, 8), C=(12, 8))
            c.update(lambda_max=lm, out=ref(x["X"], ei, ew, x["H"], x["C"], lm), out_noew_nohc=ref(x["X"], ei, lambda_max=lm))
            out["gc_lstm"][(K, norm)] = c

    st = refload.load("nn.attention.stgcn")
    out["stconv"] = {}
    for K in (1, 2, 3):
        ref = st.STConv(12, 3, 8, 6, 3, K)
        c, x = _case(ref, 700 + 2 * K, X=(2, 9, 12, 3))
        c["out_train"] = ref(x["X"], ei, ew)                    # module default: training-mode BatchNorm, updates the running stats
        c["buffers"] = {k: v.clone() for k, v in ref.state_dict().items() if k.endswith(("running_mean", "running_var"))}
        ref.eval()
        c.update(out_eval=ref(x["X"], ei, ew), out_temporal_conv1=ref._temporal_conv1(x["X"]))
        out["stconv"][K] = c

    ms = refload.load("nn.attention.mstgcn")
    out["mstgcn"] = {}
    for strides in (1, 2):
        ref = ms.MSTGCN(2, 2, 3, 8, 8, strides, 4, 6)
        c, x = _case(ref, 800 + 2 * strides, X=(3, 12, 2, 6))
        c.update(out=ref(x["X"], eiu), out_list=ref(x["X"], [eiu] * 6))
        out["mstgcn"][strides] = c
    torch.set_grad_enabled(True)
    save("reference_modules", **out)


def data():
    out = {"loaders": {}, "dynamic_signals": {}}
    # offline METR-LA / PEMS-BAY loaders on the synthetic archive of test_next_rows_cpu.py::test_offline_loaders_match_reference;
    # they only window and z-score the archive, so their outputs are stored as digests of the exact bits
    sig = refload.load("signal.static_graph_temporal_signal")
    # the reference loader does `from ..signal import StaticGraphTemporalSignal`; its signal/__init__ pulls every iterator
    # (PyG Batch/HeteroData), so expose just that one unmodified class on the path-only parent package refload registers
    sys.modules["torch_geometric_temporal.signal"].StaticGraphTemporalSignal = sig.StaticGraphTemporalSignal
    for mod, name, prefix in [("dataset.metr_la", "METRLADatasetLoader", ""), ("dataset.pems_bay", "PemsBayDatasetLoader", "pems_")]:
        ref_cls = getattr(refload.load(mod), name)
        with tempfile.TemporaryDirectory() as tmp:
            _archive(tmp, 9, 2, 30, prefix)
            open(os.path.join(tmp, "METR-LA.zip" if prefix == "" else "PEMS-BAY.zip"), "wb").close()   # the reference checks the zip exists
            c = dict(snapshots=[[_digest(getattr(s, k)) for k in ("x", "y", "edge_index", "edge_attr")]
                                for s in ref_cls(raw_data_dir=tmp).get_dataset(6, 6)])
            w = ref_cls(raw_data_dir=tmp, index=True).get_index_dataset(lags=6, batch_size=4)
            c.update(index_batches=[[[_digest(x), _digest(y)] for x, y in w[i]] for i in range(3)], index_tensors=[_digest(t) for t in w[3:7]])
            w = ref_cls(raw_data_dir=tmp, index=True).get_index_dataset(lags=6, batch_size=4, shuffle=True, world_size=2, ddp_rank=1)
            c["shard_batches"] = [[_digest(x), _digest(y)] for x, y in w[0]]
        out["loaders"][prefix] = c

    # dynamic-graph iterators (data conversion only, digests as above), test_next_rows_cpu.py::test_dynamic_signals_match_reference
    eis, ews, xs, ys, bs, marks = _dynamic_case(seed=3)
    for mod, name, args in [("signal.dynamic_graph_temporal_signal", "DynamicGraphTemporalSignal", (eis, ews, xs, ys)),
                            ("signal.dynamic_graph_static_signal", "DynamicGraphStaticSignal", (eis, ews, xs[0], ys)),
                            ("signal.dynamic_graph_temporal_signal_batch", "DynamicGraphTemporalSignalBatch", (eis, ews, xs, ys, bs)),
                            ("signal.dynamic_graph_static_signal_batch", "DynamicGraphStaticSignalBatch", (eis, ews, xs[0], ys, bs)),
                            ("signal.static_graph_temporal_signal_batch", "StaticGraphTemporalSignalBatch", (eis[0], ews[0], xs, ys, bs[0]))]:
        want = getattr(refload.load(mod), name)(*args, marks=marks)
        keys = ("x", "edge_index", "edge_attr", "y", "marks") + (("batch",) if "Batch" in name else ())
        sl = want[1:4]
        out["dynamic_signals"][name] = dict(snapshots=[[_digest(getattr(s, k)) for k in keys] for s in want],
                                            slice=[sl.snapshot_count, _digest(sl[0].x), _digest(sl[2].edge_index)])

    # IndexDataset, test_signal.py::test_index_dataset_matches_oracle_and_reference
    from pytorch_geometric_temporal_b200.signal import index_splits
    series = np.random.RandomState(0).rand(60, 7, 2).astype(np.float32)
    tr, _, _ = index_splits(60, 12)
    ref = refload.load("signal.index_dataset").IndexDataset(tr, series, 12)
    out["index_dataset"] = dict(x=torch.stack([ref[i][0] for i in range(len(ref))]), y=torch.stack([ref[i][1] for i in range(len(ref))]))

    # masked MAE of examples/indexBatching/DCRNN/utils.py, test_distributed_cpu.py::test_masked_mae_matches_reference_example_util
    path = os.path.join(refload.REFERENCE_ROOT, "examples", "indexBatching", "DCRNN", "utils.py")
    spec = importlib.util.spec_from_file_location("ref_dcrnn_utils", path)
    utils = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(utils)
    out["masked_mae"] = {zero_frac: utils.masked_mae_loss(*_mae_inputs(zero_frac)) for zero_frac in (0.0, 0.3, 1.0)}
    save("reference_data", **out)


if __name__ == "__main__":
    modules()
    data()

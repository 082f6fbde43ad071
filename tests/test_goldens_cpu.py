"""The oracle must reproduce every committed golden vector (generated from the unmodified reference by
tests/golden/make_goldens.py).  This is what pins the oracle on machines without /root/reference."""
import os

import pytest
import torch

from oracle import recurrent as R, attention as A


def _load(golden_dir, name):
    return torch.load(os.path.join(golden_dir, name + ".pt"), weights_only=False)


def test_dcrnn_goldens(golden_dir):
    g = _load(golden_dir, "dcrnn_cfg2_batched")
    assert g["edge_index"].shape == (2, 1722) and g["X"].shape == (2, 12, 207, 2)
    assert torch.equal(R.batched_dcrnn(g["state"], g["X"], g["edge_index"], g["edge_weight"]), g["out"])
    g = _load(golden_dir, "dcrnn_cfg2_cell")
    # one thread, as the vector was generated: MKL splits the reduction of the (1 x 207) @ (207 x 207) in-degree product
    # by thread count, so the last bit of this output depends on it
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        assert torch.equal(R.dcrnn_cell(g["state"], g["X"], g["edge_index"], g["edge_weight"], g["H"]), g["out"])
        assert torch.equal(R.dcrnn_cell(g["state"], g["X"], g["edge_index"]), g["out_noew_noh"])
    finally:
        torch.set_num_threads(threads)
    for K in (1, 3, 4):
        g = _load(golden_dir, f"dcrnn_small_K{K}")
        assert torch.equal(R.dcrnn_cell(g["state"], g["X"], g["edge_index"], g["edge_weight"], g["H"]), g["out"])
    g = _load(golden_dir, "dcrnn_small_batched_K3")
    assert torch.equal(R.batched_dcrnn(g["state"], g["X"], g["edge_index"], g["edge_weight"]), g["out"])


def test_cheb_goldens(golden_dir):
    g = _load(golden_dir, "gconv_gru_small")
    for c in g["cases"].values():
        got = R.gconv_gru_cell(c["state"], c["X"], g["edge_index"], g["edge_weight"], c["H"], c["lambda_max"], c["normalization"])
        assert torch.equal(got, c["out"])
    g = _load(golden_dir, "gconv_lstm_small")
    for c in g["cases"].values():
        h, cc = R.gconv_lstm_cell(c["state"], c["X"], g["edge_index"], g["edge_weight"], c["H"], c["C"])
        assert torch.equal(h, c["outH"]) and torch.equal(cc, c["outC"])
        h, cc = R.gconv_lstm_cell(c["state"], c["X"], g["edge_index"])
        assert torch.equal(h, c["outH0"]) and torch.equal(cc, c["outC0"])


def test_tgcn_goldens(golden_dir):
    g = _load(golden_dir, "tgcn_small")
    for c in g["cases"].values():
        assert torch.equal(R.tgcn_cell(c["state"], c["X"], g["edge_index"], g["edge_weight"], c["H"], c["improved"], c["add_self_loops"]), c["out"])
        assert torch.equal(R.tgcn_cell(c["state2"], c["X2"], g["edge_index"], g["edge_weight"], c["H2"], c["improved"], c["add_self_loops"]), c["out2"])
    g = _load(golden_dir, "a3tgcn_small")
    assert torch.equal(R.a3tgcn(g["state"], g["X"], g["edge_index"], g["edge_weight"]), g["out"])
    assert torch.equal(R.a3tgcn(g["state"], g["X"], g["edge_index"], g["edge_weight"], torch.ones(3, 40, 16) * 0.3), g["outH"])
    assert torch.equal(R.a3tgcn(g["state1"], g["X1"], g["edge_index"], g["edge_weight"]), g["out1"])


def test_astgcn_goldens(golden_dir):
    g = _load(golden_dir, "astgcn_small")
    for c in g["cases"].values():
        got = A.astgcn(c["state"], c["X"], g["edge_index"], g["ctor"]["nb_block"], c["normalization"],
                       g["ctor"]["time_strides"], c["lambda_max"])
        assert torch.allclose(got, c["out"], rtol=1e-6, atol=1e-6)


def test_gc_lstm_goldens(golden_dir):
    g = _load(golden_dir, "gc_lstm_small")
    for c in g["cases"].values():
        h, cc = R.gc_lstm_cell(c["state"], c["X"], g["edge_index"], g["edge_weight"], c["H"], c["C"], c["lambda_max"], c["normalization"])
        assert torch.equal(h, c["outH"]) and torch.equal(cc, c["outC"])
        if "outH0" in c:
            h, cc = R.gc_lstm_cell(c["state"], c["X"], g["edge_index"], lambda_max=c["lambda_max"], normalization=c["normalization"])
            assert torch.equal(h, c["outH0"]) and torch.equal(cc, c["outC0"])


def test_stconv_goldens(golden_dir):
    g = _load(golden_dir, "stconv_small")
    for c in g["cases"].values():
        got = A.stconv(c["state"], c["X"], g["edge_index"], g["edge_weight"], c["normalization"], training=True)
        assert torch.equal(got, c["out_train"])                # batch statistics do not depend on the running buffers
        assert torch.equal(A.stconv(c["state"], c["X"], g["edge_index"], g["edge_weight"], c["normalization"], training=False), c["out_eval"])
        assert torch.equal(A.stconv(c["state"], c["X"], g["edge_index"], None, c["normalization"], training=False), c["out_eval_noew"])


def test_mstgcn_goldens(golden_dir):
    g = _load(golden_dir, "mstgcn_small")
    for c in g["cases"].values():
        got = A.mstgcn(c["state"], c["X"], g["edge_index"], g["ctor"]["nb_block"], c["time_strides"], g["lambda_max"])
        assert torch.allclose(got, c["out"], rtol=1e-6, atol=1e-6)      # ARPACK start vector: lambda_max moves in the last bits
        got = A.mstgcn(c["state"], c["X"], [g["edge_index"]] * 6, g["ctor"]["nb_block"], c["time_strides"], g["lambda_max"])
        assert torch.allclose(got, c["out_list"], rtol=1e-6, atol=1e-6)  # list path: a different function (no reshape scramble)

"""Pin of the oracle's MODULE logic: the functional restatement (oracle/recurrent.py, oracle/attention.py) must reproduce
the UNMODIFIED reference modules bit for bit.  What the reference modules returned is stored in
tests/golden/reference_modules.pt (tests/golden/make_goldens_parity.py); their parameters and inputs are drawn here
again by `_seeded` from the seed and shapes stored with each case."""
import os

import numpy as np
import pytest
import torch

from oracle import recurrent as R, attention as A, pyg


def _seeded(seed, shapes):
    """{name: float32 tensor uniform in [-1, 1)} for {name: shape}, drawn in order from numpy's RandomState (whose stream
    numpy keeps fixed across releases, so the stored reference outputs stay valid)."""
    rs = np.random.RandomState(seed)
    return {k: torch.from_numpy(rs.uniform(-1.0, 1.0, s).astype(np.float32)) for k, s in shapes.items()}


def _case(c):
    """(parameters, inputs) the reference module of stored case `c` ran with."""
    return _seeded(c["seed"], c["params"]), _seeded(c["seed"] + 1, c["inputs"])


@pytest.fixture(scope="module")
def ref(golden_dir):
    return torch.load(os.path.join(golden_dir, "reference_modules.pt"), weights_only=False)


@pytest.mark.parametrize("K", [1, 2, 3, 4])
def test_dcrnn(K, ref):
    ei, ew = ref["edge_index"], ref["edge_weight"]
    c = ref["dcrnn"][K]
    with torch.no_grad():
        p, x = _case(c["cell"])
        assert torch.equal(c["cell"]["out"], R.dcrnn_cell(p, x["X"], ei, ew, x["H"]))
        assert torch.equal(c["cell"]["out_noew_noh"], R.dcrnn_cell(p, x["X"], ei))
        p, x = _case(c["batched"])
        assert torch.equal(c["batched"]["out"], R.batched_dcrnn(p, x["X"], ei, ew))


@pytest.mark.parametrize("K", [1, 2, 3, 4])
@pytest.mark.parametrize("norm", ["sym", "rw", None])
def test_gconv(K, norm, ref):
    ei, ew = ref["edge_index"], ref["edge_weight"]
    c = ref["gconv"][(K, norm)]
    with torch.no_grad():
        p, x = _case(c["gru"])
        assert torch.equal(c["gru"]["out"], R.gconv_gru_cell(p, x["X"], ei, ew, x["H"], c["gru"]["lambda_max"], norm))
        p, x = _case(c["lstm"])
        a, b = c["lstm"]["out"], R.gconv_lstm_cell(p, x["X"], ei, ew, x["H"], x["C"], c["lstm"]["lambda_max"], norm)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_tgcn_family(ref):
    ei, ew = ref["edge_index"], ref["edge_weight"]
    t = ref["tgcn_family"]
    with torch.no_grad():
        for improved in (False, True):
            for asl in (True, False):
                c = t["tgcn"][(improved, asl)]
                p, x = _case(c)
                assert torch.equal(c["out"], R.tgcn_cell(p, x["X"], ei, ew, x["H"], improved, asl))
        p, x = _case(t["tgcn2"])
        assert torch.equal(t["tgcn2"]["out"], R.tgcn_cell(p, x["X"], ei, ew, x["H"]))
        p, x = _case(t["a3tgcn2"])
        assert torch.equal(t["a3tgcn2"]["out"], R.a3tgcn(p, x["X"], ei, ew))
        p, x = _case(t["a3tgcn"])
        assert torch.equal(t["a3tgcn"]["out"], R.a3tgcn(p, x["X"], ei, ew))


@pytest.mark.parametrize("norm", ["sym", None, "rw"])
def test_astgcn(norm, ref):
    eiu = ref["edge_index_undirected"]
    c = ref["astgcn"][norm]
    p, x = _case(c)
    lm = None
    if norm != "sym":
        lm = pyg.LaplacianLambdaMax()(pyg.Data(edge_index=eiu, edge_attr=None, num_nodes=12)).lambda_max
    with torch.no_grad():
        got = A.astgcn(p, x["X"], eiu, 2, norm, 2, lm)
    assert torch.allclose(c["out"], got, rtol=1e-6, atol=1e-6)  # diag-scale vs dense matmul: 1 ulp


@pytest.mark.parametrize("norm", ["sym", None, "rw"])
def test_chebconv_attention_per_graph_lambda_max(norm, ref):
    """The multi-graph mini-batch call of the reference's own test (test/attention_test.py:205-218): a node->graph `batch`
    vector and one lambda_max per graph."""
    c = ref["chebconv_attention"][norm]
    p, x = _case(c)
    with torch.no_grad():
        got = A.cheb_conv_attention(p, x["x"], c["edge_index"], c["S"], norm, c["edge_weight"], c["lambda_max"], c["batch"])
        assert torch.allclose(c["out"], got, rtol=1e-6, atol=1e-6)
        assert not torch.allclose(c["out"], c["out_one_lambda"], rtol=1e-3, atol=1e-4)   # the second graph really uses 3.0


# ---- SURVEY 8f rank 1: GCLSTM, STConv, MSTGCN ---------------------------------------------------------------
@pytest.mark.parametrize("K", [1, 2, 3])
@pytest.mark.parametrize("norm", ["sym", "rw", None])
def test_gc_lstm(K, norm, ref):
    ei, ew = ref["edge_index"], ref["edge_weight"]
    c = ref["gc_lstm"][(K, norm)]
    p, x = _case(c)
    lm = c["lambda_max"]
    with torch.no_grad():
        a, b = c["out"], R.gc_lstm_cell(p, x["X"], ei, ew, x["H"], x["C"], lm, norm)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
        a, b = c["out_noew_nohc"], R.gc_lstm_cell(p, x["X"], ei, lambda_max=lm, normalization=norm)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.parametrize("K", [1, 2, 3])
def test_stconv(K, ref):
    ei, ew = ref["edge_index"], ref["edge_weight"]
    c = ref["stconv"][K]
    p, x = _case(c)
    X = x["X"]
    with torch.no_grad():
        assert torch.equal(c["out_train"], A.stconv(p, X, ei, ew))      # module default: training-mode BatchNorm
        # eval mode reads the running statistics the reference's training-mode call left behind
        assert torch.equal(c["out_eval"], A.stconv({**p, **c["buffers"]}, X, ei, ew, training=False))
        assert torch.equal(c["out_temporal_conv1"], A.temporal_conv({k[len("_temporal_conv1."):]: v for k, v in p.items()
                                                                      if k.startswith("_temporal_conv1.")}, X))


@pytest.mark.parametrize("strides", [1, 2])
def test_mstgcn(strides, ref):
    eiu = ref["edge_index_undirected"]
    c = ref["mstgcn"][strides]
    p, x = _case(c)
    with torch.no_grad():
        assert torch.allclose(c["out"], A.mstgcn(p, x["X"], eiu, 2, strides), rtol=1e-6, atol=1e-6)  # ARPACK seed
        assert torch.allclose(c["out_list"], A.mstgcn(p, x["X"], [eiu] * 6, 2, strides), rtol=1e-6, atol=1e-6)

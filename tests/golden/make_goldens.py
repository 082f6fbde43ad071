"""Generate the committed golden vectors by running the UNMODIFIED reference modules
(/root/reference, imported through oracle/refload.py on top of oracle/stubs) on seeded inputs.

Run in the build container only:   python tests/golden/make_goldens.py
Each .pt holds inputs, the reference module's state_dict and the reference outputs (+ input/param
grads where noted).  The GPU parity tests load these; /root/reference is never read at test time.
"""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import refload, pyg  # noqa: E402
from pytorch_geometric_temporal_b200.dataset import synthetic  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def save(name, **kw):
    torch.save(kw, os.path.join(OUT, name + ".pt"))
    sz = os.path.getsize(os.path.join(OUT, name + ".pt"))
    print(f"{name}.pt  {sz / 1024:.0f} KB")


def sd(m):
    return {k: v.detach().clone() for k, v in m.state_dict().items()}


def small_graph(n, e, seed, loops=True):
    g = torch.Generator().manual_seed(seed)
    pairs = set()
    while len(pairs) < e:
        r, c = int(torch.randint(0, n, (1,), generator=g)), int(torch.randint(0, n, (1,), generator=g))
        if r != c:
            pairs.add((r, c))
    if loops:
        pairs |= {(i, i) for i in range(n)}
    pairs |= {(i, (i + 1) % n) for i in range(n)}  # every node has in/out degree >= 1
    pairs = sorted(pairs)
    ei = torch.tensor(pairs, dtype=torch.long).t().contiguous()
    ew = torch.rand(ei.size(1), generator=g) * 0.9 + 0.1
    return ei, ew


def main():
    dc = refload.load("nn.recurrent.dcrnn")
    # ---- cfg2: BatchedDCRNN(2,32,K=2) on the METR-LA-shaped graph, B=2 windows of 12 -------------------
    ei, ew, series = synthetic.metr_la_like(seed=0, t_total=64)
    ei_t, ew_t = torch.from_numpy(ei), torch.from_numpy(ew)
    torch.manual_seed(0)
    m = dc.BatchedDCRNN(2, 32, 2)
    X = torch.from_numpy(np.stack([series[0:12], series[7:19]]))  # (2,12,207,2)
    with torch.no_grad():
        out = m(X, ei_t, ew_t)
    save("dcrnn_cfg2_batched", edge_index=ei_t, edge_weight=ew_t, X=X, state=sd(m), out=out, K=2)
    # single-step DCRNN (dense-adjacency degrees) on the same graph, with an incoming H
    torch.manual_seed(1)
    m1 = dc.DCRNN(2, 32, 2)
    x1, h1 = torch.randn(207, 2), torch.randn(207, 32) * 0.5
    # one thread: the dense-adjacency in-degrees are a (1 x 207) @ (207 x 207) product whose reduction MKL splits by thread
    # count, so only a fixed count reproduces these bits on another machine (tests/test_goldens_cpu.py runs it the same way)
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    with torch.no_grad():
        o1 = m1(x1, ei_t, ew_t, h1)
        o1_now = m1(x1, ei_t)  # edge_weight None, H None
    torch.set_num_threads(threads)
    save("dcrnn_cfg2_cell", edge_index=ei_t, edge_weight=ew_t, X=x1, H=h1, state=sd(m1), out=o1, out_noew_noh=o1_now, K=2)
    # K=1,3,4 on a small asymmetric graph (exercises the positional norm_in pairing and the Tx_0 quirk)
    ei_s, ew_s = small_graph(40, 150, 3)
    for K in (1, 3, 4):
        torch.manual_seed(10 + K)
        mk = dc.DCRNN(3, 16, K)
        xs, hs = torch.randn(40, 3), torch.randn(40, 16) * 0.5
        xs.requires_grad_(True)
        hs.requires_grad_(True)
        o = mk(xs, ei_s, ew_s, hs)
        loss = (o * torch.linspace(-1, 1, o.numel()).view_as(o)).sum()
        loss.backward()
        grads = {k: p.grad.detach().clone() for k, p in mk.named_parameters()}
        save(f"dcrnn_small_K{K}", edge_index=ei_s, edge_weight=ew_s, X=xs.detach(), H=hs.detach(), state=sd(mk),
             out=o.detach(), gX=xs.grad.clone(), gH=hs.grad.clone(), grads=grads, K=K)
    torch.manual_seed(20)
    mb = dc.BatchedDCRNN(3, 16, 3)
    Xb = torch.randn(3, 5, 40, 3)
    with torch.no_grad():
        ob = mb(Xb, ei_s, ew_s)
    save("dcrnn_small_batched_K3", edge_index=ei_s, edge_weight=ew_s, X=Xb, state=sd(mb), out=ob, K=3)

    # ---- ChebConv cells ----------------------------------------------------------------------------------
    gg = refload.load("nn.recurrent.gconv_gru")
    gl = refload.load("nn.recurrent.gconv_lstm")
    cases = {}
    for K in (1, 2, 3):
        for norm in ("sym", "rw", None):
            torch.manual_seed(30 + K)
            m = gg.GConvGRU(4, 16, K, normalization=norm)
            x, h = torch.randn(40, 4), torch.randn(40, 16) * 0.5
            lm = None if norm == "sym" else torch.tensor(2.5)
            with torch.no_grad():
                o = m(x, ei_s, ew_s, h, lm)
            cases[f"K{K}_{norm}"] = dict(state=sd(m), X=x, H=h, lambda_max=lm, out=o, K=K, normalization=norm)
    save("gconv_gru_small", edge_index=ei_s, edge_weight=ew_s, cases=cases)
    cases = {}
    for K in (1, 2, 3):
        torch.manual_seed(40 + K)
        m = gl.GConvLSTM(4, 16, K)
        x, h, c = torch.randn(40, 4), torch.randn(40, 16) * 0.5, torch.randn(40, 16) * 0.5
        with torch.no_grad():
            ho, co = m(x, ei_s, ew_s, h, c)
            ho0, co0 = m(x, ei_s)
        cases[f"K{K}"] = dict(state=sd(m), X=x, H=h, C=c, outH=ho, outC=co, outH0=ho0, outC0=co0, K=K)
    save("gconv_lstm_small", edge_index=ei_s, edge_weight=ew_s, cases=cases)

    # ---- TGCN / A3TGCN2 ------------------------------------------------------------------------------------
    tg = refload.load("nn.recurrent.temporalgcn")
    at = refload.load("nn.recurrent.attentiontemporalgcn")
    cases = {}
    for improved in (False, True):
        for asl in (True, False):
            torch.manual_seed(50)
            m = tg.TGCN(4, 16, improved=improved, add_self_loops=asl)
            x, h = torch.randn(40, 4), torch.randn(40, 16) * 0.5
            with torch.no_grad():
                o = m(x, ei_s, ew_s, h)
            m2 = tg.TGCN2(4, 16, 3, improved=improved, add_self_loops=asl)
            xb, hb = torch.randn(3, 40, 4), torch.randn(3, 40, 16) * 0.5
            with torch.no_grad():
                o2 = m2(xb, ei_s, ew_s, hb)
            cases[f"imp{int(improved)}_asl{int(asl)}"] = dict(state=sd(m), X=x, H=h, out=o, state2=sd(m2), X2=xb, H2=hb, out2=o2,
                                                            improved=improved, add_self_loops=asl)
    save("tgcn_small", edge_index=ei_s, edge_weight=ew_s, cases=cases)
    torch.manual_seed(60)
    m = at.A3TGCN2(2, 16, 6, 3)
    xp = torch.randn(3, 40, 2, 6)
    with torch.no_grad():
        o = m(xp, ei_s, ew_s)
        oh = m(xp, ei_s, ew_s, torch.ones(3, 40, 16) * 0.3)
    m1 = at.A3TGCN(2, 16, 6)
    xp1 = torch.randn(40, 2, 6)
    with torch.no_grad():
        o1 = m1(xp1, ei_s, ew_s)
    save("a3tgcn_small", edge_index=ei_s, edge_weight=ew_s, state=sd(m), X=xp, out=o, outH=oh, state1=sd(m1), X1=xp1, out1=o1)

    # ---- ASTGCN ------------------------------------------------------------------------------------------------
    ag = refload.load("nn.attention.astgcn")
    und = sorted({(a, b) for a, b in ei_s.t().tolist() if a != b} | {(b, a) for a, b in ei_s.t().tolist() if a != b})
    eiu = torch.tensor(und, dtype=torch.long).t().contiguous()
    cases = {}
    for norm in ("sym", None, "rw"):
        torch.manual_seed(70)
        m = ag.ASTGCN(2, 1, 3, 8, 8, 2, 4, 6, 40, normalization=norm)
        xa = torch.randn(3, 40, 1, 6)
        lm = None
        if norm != "sym":
            lm = pyg.LaplacianLambdaMax()(pyg.Data(edge_index=eiu, edge_attr=None, num_nodes=40)).lambda_max
        with torch.no_grad():
            o = m(xa, eiu)
        cases[str(norm)] = dict(state=sd(m), X=xa, out=o, lambda_max=lm, normalization=norm)
    save("astgcn_small", edge_index=eiu, cases=cases,
         ctor=dict(nb_block=2, in_channels=1, K=3, nb_chev_filter=8, nb_time_filter=8, time_strides=2,
                   num_for_predict=4, len_input=6, num_of_vertices=40))

    # ---- chickenpox fixture (in-tree JSON of the reference, dataset/chickenpox.json) -> npz ------------------
    with open(os.path.join(refload.REFERENCE_ROOT, "dataset", "chickenpox.json")) as f:
        d = json.load(f)
    pkg_data = os.path.join(os.path.dirname(os.path.dirname(OUT)), "pytorch_geometric_temporal_b200", "dataset", "data")
    os.makedirs(pkg_data, exist_ok=True)       # the dataset ships INSIDE the package (ChickenpoxDatasetLoader's default)
    np.savez_compressed(os.path.join(pkg_data, "chickenpox.npz"), edges=np.array(d["edges"], dtype=np.int64),
                        FX=np.array(d["FX"], dtype=np.float64))
    print("chickenpox.npz", os.path.getsize(os.path.join(pkg_data, "chickenpox.npz")) // 1024, "KB")


if __name__ == "__main__":
    main()

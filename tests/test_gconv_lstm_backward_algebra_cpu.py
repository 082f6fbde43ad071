"""Host-side algebra of the hand-written GConvLSTM cell backward (`nn/recurrent/gconv_lstm.py::_LstmCellFn`) checked on the CPU
against autograd through the op-for-op path and against the reference module's gradients: the CUDA entry points are replaced by
dense torch stand-ins that follow the contracts of include/stmp.h (stmp_spmm on column blocks, stmp_gemm_lstm_f32, stmp_gemm_f32
with a strided `out` and `a_row_scale`, stmp_lstm_gate_bwd).  Pins, without a GPU: the recompute-in-backward scheme, the gate
derivatives' call shapes, dS = dpre W^T in two column halves on power-of-two row-scaled dpre, the in-place adjoint of the Chebyshev
recurrence, the chunked weight gradient, the peephole / bias reductions and the reuse of one (W, bias) graph across the steps of a
sequence."""
import pytest
import torch

import pytorch_geometric_temporal_b200.nn.recurrent._cheb as cheb_mod
import pytorch_geometric_temporal_b200.nn.recurrent.gconv_lstm as L
from oracle import pyg, recurrent as R
from pytorch_geometric_temporal_b200 import ops


class _Plan(object):
    def __init__(self, Lm):
        self.L = Lm


def _install(monkeypatch):
    def spmm_cols(plan, op, buf, src, dst, width, alpha=1.0, z_col=None, beta=0.0, transposed=False):
        A = plan.L.t() if transposed else plan.L
        y = alpha * torch.matmul(A, buf[..., src:src + width])
        if z_col is not None:
            y = y + beta * buf[..., z_col:z_col + width]
        buf[..., dst:dst + width] = y

    def spmm(plan, op, x, alpha=1.0, z=None, beta=0.0, att=None):
        y = alpha * torch.matmul(plan.L, x)
        return y if z is None else y + beta * z

    def gemm_prepack(W):
        return W.clone()                                  # "packed" = the fp32 matrix itself

    def gemm(A, packed, K, N, bias=None, out=None, row_scale=None):
        A2 = A.reshape(-1, K)
        if row_scale is None:
            C = A2 @ packed
        else:                                             # a_row_scale: one power of two per row of A, undone on the product
            assert row_scale.shape == (A2.size(0),) and (torch.frexp(row_scale).mantissa == 0.5).all()
            row_scaled_calls.append(A2.size(0))
            C = ((A2 * row_scale[:, None]) @ packed) / row_scale[:, None]
        if bias is not None:
            C = C + bias
        if out is not None:
            out.copy_(C)
            return out
        return C.reshape(*A.shape[:-1], N)

    def gemm_lstm(A, packed, K, cout, cb, cell, wci, wcf, wco, bi, bf, bc, bo):
        pre = A @ packed + (0 if cb is None else cb)
        pi, pf, pc, po = (pre[..., j * cout:(j + 1) * cout] for j in range(4))
        I, Fg = torch.sigmoid(pi + wci * cell + bi), torch.sigmoid(pf + wcf * cell + bf)
        Cn = Fg * cell + I * torch.tanh(pc + bc)
        return torch.sigmoid(po + wco * Cn + bo) * torch.tanh(Cn), Cn

    def lstm_gate_bwd(pre, c_old, c_new, gh, gc, wci, wcf, wco, bi, bf, bc, bo):
        Co = c_old.size(-1)
        pi, pf, pc, po = (pre[:, j * Co:(j + 1) * Co] for j in range(4))
        iv, fv = torch.sigmoid(pi + wci * c_old + bi), torch.sigmoid(pf + wcf * c_old + bf)
        tv, ov, tc = torch.tanh(pc + bc), torch.sigmoid(po + wco * c_new + bo), torch.tanh(c_new)
        g = torch.zeros_like(c_old) if gh is None else gh
        dpo = g * tc * ov * (1 - ov)
        dcn = (0 if gc is None else gc) + g * ov * (1 - tc * tc) + dpo * wco
        dpi, dpf, dpc = dcn * tv * iv * (1 - iv), dcn * c_old * fv * (1 - fv), dcn * iv * (1 - tv * tv)
        return torch.cat([dpi, dpf, dpc, dpo], dim=1), dcn * fv + dpi * wci + dpf * wcf

    row_scaled_calls = []
    for name, fn in dict(spmm_cols=spmm_cols, spmm=spmm, gemm_prepack=gemm_prepack, gemm=gemm, gemm_lstm=gemm_lstm,
                         lstm_gate_bwd=lstm_gate_bwd).items():
        monkeypatch.setattr(ops, name, fn)
    monkeypatch.setattr(L, "_require_cuda", lambda *a, **k: None)

    def plan(self, edge_index, edge_weight, num_nodes, normalization, lambda_max, batch=None):
        e, w = pyg.cheb_norm(edge_index, num_nodes, edge_weight, normalization, self._lambda_value(lambda_max))
        M = torch.zeros(num_nodes, num_nodes)
        M.index_put_((e[1], e[0]), w, accumulate=True)
        return _Plan(M)
    monkeypatch.setattr(cheb_mod.ChebPlanMixin, "_cheb_plan", plan)
    return row_scaled_calls


@pytest.mark.parametrize("K,batched", [(3, False), (2, True), (1, False)])
def test_lstm_cell_backward_row_scaled_matches_autograd_and_reference(monkeypatch, K, batched):
    row_scaled_calls = _install(monkeypatch)
    torch.manual_seed(K)
    n, Ci, Co, T = 24, 32, 32, 3
    ei = torch.stack([torch.randint(0, n, (90,)), torch.randint(0, n, (90,))])
    ei = torch.unique(ei[:, ei[0] != ei[1]], dim=1)
    ew = torch.rand(ei.size(1)) + 0.1
    lead = (2, n) if batched else (n,)
    X = (torch.randn(T, *lead, Ci) * 0.5)
    a, b = L.GConvLSTM(Ci, Co, K), L.GConvLSTM(Ci, Co, K)
    for p in a.parameters():                      # zero biases would hide bias-gradient mistakes
        if p.dim() == 1 or p.size(0) == 1:
            torch.nn.init.normal_(p, std=0.2)
    b.load_state_dict(a.state_dict())
    b.fused_training = False
    outs = {}
    for name, m in (("fused", a), ("autograd", b)):
        x = X.clone().requires_grad_(True)
        H = C = None
        loss = 0
        for t in range(T):
            H, C = m(x[t], ei, ew, H, C)
            loss = loss + (H * torch.linspace(-1, 1, H.numel()).view_as(H)).sum() + 0.3 * C.square().sum()
        loss.backward()
        outs[name] = (H.detach(), C.detach(), x.grad, {k: p.grad.clone() for k, p in m.named_parameters()})
    assert a._train_cache is None                                   # the shared (W, bias) graph was dropped by the backward pass
    assert len(row_scaled_calls) == 2 * T                           # every step's dS = dpre W^T (two halves) took row-scaled dpre
    fH, fC, fx, fp = outs["fused"]
    aH, aC, ax, ap = outs["autograd"]
    assert torch.allclose(fH, aH, rtol=1e-5, atol=1e-6) and torch.allclose(fC, aC, rtol=1e-5, atol=1e-6)
    assert torch.allclose(fx, ax, rtol=1e-4, atol=1e-5), float((fx - ax).abs().max())
    for k in ap:
        assert torch.allclose(fp[k], ap[k], rtol=1e-4, atol=1e-4 * float(ap[k].abs().max()) + 1e-6), (k, float((fp[k] - ap[k]).abs().max()))
    if not batched:
        # and the reference's own cell (oracle restatement, pinned bit-exactly to the unmodified module) gives the same gradients
        p = {k: v.detach().clone().requires_grad_(True) for k, v in a.state_dict().items()}
        x = X.clone().requires_grad_(True)
        H = C = None
        loss = 0
        for t in range(T):
            H, C = R.gconv_lstm_cell(p, x[t], ei, ew, H, C)
            loss = loss + (H * torch.linspace(-1, 1, H.numel()).view_as(H)).sum() + 0.3 * C.square().sum()
        loss.backward()
        assert torch.allclose(fx, x.grad, rtol=1e-4, atol=1e-5)
        for k in fp:
            assert torch.allclose(fp[k], p[k].grad, rtol=1e-4, atol=1e-4 * float(p[k].grad.abs().max()) + 1e-6), k

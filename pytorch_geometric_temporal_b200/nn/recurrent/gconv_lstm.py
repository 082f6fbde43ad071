"""GConvLSTM -- drop-in for torch_geometric_temporal/nn/recurrent/gconv_lstm.py (:9-238): constructor
`(in_channels, out_channels, K, normalization="sym", bias=True)`, `forward(X, edge_index, edge_weight,
H, C, lambda_max) -> (H, C)`, state_dict keys `conv_{x,h}_{i,f,c,o}.lins.{k}.weight/.bias`,
`w_c_{i,f,o} (1,out)` (glorot), `b_{i,f,c,o} (1,out)` (zeros).  Eight ChebConvs per step in the
reference = 8(K-1) propagations; here T_k([X|H]) is computed once (K-1 SpMMs on Ci+Co channels) and one
GEMM produces all four gate pre-activations."""
import torch

from ... import _lib, ops
from ...plan import _require_cuda
from ._cheb import ChebParams, ChebPlanMixin, cheb_basis, glorot_


def _chunked_tn(A: torch.Tensor, B: torch.Tensor) -> torch.Tensor:
    """A^T @ B for tall-skinny A (rows, a), B (rows, b): a single GEMM has a handful of output tiles, so the row axis is cut into
    chunks that every SM can take a partial product of (as the DCRNN backward does for its weight gradients)."""
    rows = A.size(0)
    chunks = 1
    for c in (128, 96, 64, 48, 32, 16, 8, 4, 2):
        if rows % c == 0 and rows // c >= 256:
            chunks = c
            break
    per = rows // chunks
    return torch.bmm(A.view(chunks, per, -1).transpose(1, 2), B.view(chunks, per, -1)).sum(0)


class _LstmCellFn(torch.autograd.Function):
    """Training path of one GConvLSTM step on a large graph (gconv_lstm.py:204-238) with a hand-written backward.

    forward : Chebyshev basis S = [T_0|..|T_{K-1}]([X|H]) built in place by `stmp_spmm`, then ONE tcgen05 launch computes S @ W and
              the whole peephole gate chain in its epilogue (`stmp_gemm_lstm_f32`).  Only S, C_{t-1}, C_t are kept.
    backward: pre = S @ W recomputed on tcgen05 -> `stmp_lstm_gate_bwd` (gate derivatives) -> dS = dpre @ W^T (tcgen05, two column
              halves, rows of dpre scaled by powers of two into the split's range) -> adjoint of the Chebyshev recurrence by TRANSPOSED SpMMs in place -> dX, dH;  dW = S^T dpre as a chunked
              GEMM; peephole / bias gradients as column reductions.  ~14 launches instead of the ~90 autograd records."""

    @staticmethod
    def forward(ctx, X, H, C, W, cb, wci, wcf, wco, bi, bf, bc, bo, plan, K, packed, packedT):
        Ci, Co = X.size(-1), H.size(-1)
        Cw = Ci + Co
        S = torch.empty(*X.shape[:-1], K * Cw, device=X.device, dtype=torch.float32)
        S[..., :Ci] = X
        S[..., Ci:Cw] = H
        for k in range(1, K):
            if k == 1:
                ops.spmm_cols(plan, 0, S, 0, Cw, Cw)
            else:
                ops.spmm_cols(plan, 0, S, (k - 1) * Cw, k * Cw, Cw, alpha=2.0, z_col=(k - 2) * Cw, beta=-1.0)
        Cc = C.contiguous()
        Hn, Cn = ops.gemm_lstm(S, packed, K * Cw, Co, cb, Cc, wci, wcf, wco, bi, bf, bc, bo)
        ctx.plan, ctx.K, ctx.Ci, ctx.Co, ctx.packed, ctx.packedT, ctx.has_cb = plan, K, Ci, Co, packed, packedT, cb is not None
        ctx.save_for_backward(S, Cc, Cn, cb, wci, wcf, wco, bi, bf, bc, bo)
        return Hn, Cn

    @staticmethod
    def backward(ctx, gH, gC):
        S, C, Cn, cb, wci, wcf, wco, bi, bf, bc, bo = ctx.saved_tensors
        plan, K, Ci, Co = ctx.plan, ctx.K, ctx.Ci, ctx.Co
        Cw, KCw = Ci + Co, K * (Ci + Co)
        S2 = S.reshape(-1, KCw)
        rows = S2.size(0)
        pre = ops.gemm(S2, ctx.packed, KCw, 4 * Co, cb)                                    # recompute the pre-activations
        dpre, dC = ops.lstm_gate_bwd(pre, C.reshape(rows, Co), Cn.reshape(rows, Co), None if gH is None else gH.reshape(rows, Co),
                                     None if gC is None else gC.reshape(rows, Co), wci, wcf, wco, bi, bf, bc, bo)
        dS = torch.empty_like(S)
        dS2 = dS.view(rows, KCw)
        half = KCw // 2
        # dS = dpre @ W^T, N split in two (N <= 256).  dpre is a gradient: its magnitude follows the loss (a mean over 10^6 terms, a
        # loss scale), so every row is scaled by a power of two into the range of the fp16 hi/lo split and back (exact).
        rs = ops.pow2_row_scale(dpre)
        for j in range(2):
            ops.gemm(dpre, ctx.packedT[j], 4 * Co, half, None, out=dS2[:, j * half:(j + 1) * half], row_scale=rs)
        dW = _chunked_tn(S2, dpre) if ctx.needs_input_grad[3] else None
        colsum = dpre.sum(0)
        dcb = colsum if ctx.has_cb else None
        Cf, Cnf = C.reshape(rows, Co), Cn.reshape(rows, Co)
        dwci = (dpre[:, :Co] * Cf).sum(0, keepdim=True)
        dwcf = (dpre[:, Co:2 * Co] * Cf).sum(0, keepdim=True)
        dwco = (dpre[:, 3 * Co:] * Cnf).sum(0, keepdim=True)
        dbi, dbf, dbc, dbo = (colsum[j * Co:(j + 1) * Co].view(1, Co) for j in range(4))
        # adjoint of T_0 = U, T_1 = L U, T_k = 2 L T_{k-1} - T_{k-2}, in place on the column blocks of dS
        for k in range(K - 1, 1, -1):
            ops.spmm_cols(plan, 0, dS, k * Cw, (k - 1) * Cw, Cw, alpha=2.0, z_col=(k - 1) * Cw, beta=1.0, transposed=True)
            dS[..., (k - 2) * Cw:(k - 1) * Cw].sub_(dS[..., k * Cw:(k + 1) * Cw])
        if K > 1:
            ops.spmm_cols(plan, 0, dS, Cw, 0, Cw, z_col=0, beta=1.0, transposed=True)
        dX = dS[..., :Ci] if ctx.needs_input_grad[0] else None
        dH = dS[..., Ci:Cw] if ctx.needs_input_grad[1] else None
        return (dX, dH, dC.view_as(C), dW, dcb, dwci, dwcf, dwco, dbi, dbf, dbc, dbo, None, None, None, None)


class GConvLSTM(torch.nn.Module, ChebPlanMixin):
    def __init__(self, in_channels: int, out_channels: int, K: int, normalization: str = "sym", bias: bool = True):
        super().__init__()
        self.in_channels, self.out_channels, self.K = in_channels, out_channels, K
        self.normalization, self.bias = normalization, bias
        P = torch.nn.Parameter
        # creation order mirrors the reference (gconv_lstm.py:60-147) so seeded init consumes the RNG identically
        for g in "ifco":
            setattr(self, f"conv_x_{g}", ChebParams(in_channels, out_channels, K, bias))
            setattr(self, f"conv_h_{g}", ChebParams(out_channels, out_channels, K, bias))
            if g != "c":
                setattr(self, f"w_c_{g}", P(torch.empty(1, out_channels)))
            setattr(self, f"b_{g}", P(torch.empty(1, out_channels)))
        for g in "ifo":
            glorot_(getattr(self, f"w_c_{g}"))
        for g in "ifco":
            torch.nn.init.zeros_(getattr(self, f"b_{g}"))
        self._init_plans()
        self._pack = ops.PackCache()
        self._train_cache = None
        self.fused_training = True      # False: op-for-op autograd path (tests compare the two)

    def _train_weights(self):
        """(W, conv bias) WITH their autograd graph plus the packed operands of the hand-written backward, shared by all steps of
        a sequence: rebuilt when a parameter changes, and dropped as soon as a backward pass has consumed the graph."""
        key = tuple((p.data_ptr(), p._version) for p in self.parameters())
        if self._train_cache is not None and self._train_cache[0] == key:
            return self._train_cache[1]
        W, cb = self._weight(), self._conv_bias()
        with torch.no_grad():
            Wd = W.detach()
            half = Wd.size(0) // 2
            WT = Wd.t().contiguous()
            packs = (ops.gemm_prepack(Wd), [ops.gemm_prepack(WT[:, :half].contiguous()), ops.gemm_prepack(WT[:, half:].contiguous())])

        def drop(_g):
            self._train_cache = None
        if W.requires_grad:
            W.register_hook(drop)
        val = (W, cb, packs)
        self._train_cache = (key, val)
        return val

    def _weight(self):
        cols = []
        for g in "ifco":
            cx, ch = getattr(self, f"conv_x_{g}"), getattr(self, f"conv_h_{g}")
            cols.append(torch.cat([torch.cat([cx.lins[k].weight.t(), ch.lins[k].weight.t()], dim=0) for k in range(self.K)], dim=0))
        return torch.cat(cols, dim=1)

    def _conv_bias(self):
        if self.conv_x_i.bias is None:
            return None
        return torch.cat([getattr(self, f"conv_x_{g}").bias + getattr(self, f"conv_h_{g}").bias for g in "ifco"])

    def forward(self, X: torch.FloatTensor, edge_index: torch.LongTensor, edge_weight: torch.FloatTensor = None,
                H: torch.FloatTensor = None, C: torch.FloatTensor = None, lambda_max: torch.Tensor = None):
        _require_cuda(X, "X")
        N, Co = X.size(-2), self.out_channels
        if H is None:
            H = torch.zeros(*X.shape[:-1], Co, device=X.device, dtype=X.dtype)
        if C is None:
            C = torch.zeros(*X.shape[:-1], Co, device=X.device, dtype=X.dtype)
        plan = self._cheb_plan(edge_index, edge_weight, N, self.normalization, lambda_max)
        needs_grad = torch.is_grad_enabled() and (any(p.requires_grad for p in self.parameters()) or X.requires_grad
                                                  or H.requires_grad or C.requires_grad)
        Cw = self.in_channels + Co
        if not needs_grad and Co in (32, 64) and (self.K * Cw) % 4 == 0 and Cw % 4 == 0:
            # large-graph inference: T_k written in place into S = [T_0|T_1|..] by the SpMM kernel, then ONE tcgen05
            # launch does S @ W and the whole peephole-LSTM gate chain in its epilogue (stmp_gemm_lstm_f32)
            S = torch.empty(*X.shape[:-1], self.K * Cw, device=X.device, dtype=torch.float32)
            S[..., :self.in_channels] = X
            S[..., self.in_channels:Cw] = H
            for k in range(1, self.K):
                if k == 1:
                    ops.spmm_cols(plan, 0, S, 0, Cw, Cw)
                else:
                    ops.spmm_cols(plan, 0, S, (k - 1) * Cw, k * Cw, Cw, alpha=2.0, z_col=(k - 2) * Cw, beta=-1.0)
            packed, cb = self._pack.get(list(self.parameters()), lambda: (ops.gemm_prepack(self._weight()), self._conv_bias()))
            try:
                return ops.gemm_lstm(S, packed, self.K * Cw, Co, cb, C.contiguous(), self.w_c_i, self.w_c_f, self.w_c_o,
                                     self.b_i, self.b_f, self.b_c, self.b_o)
            except _lib.StmpUnsupported:
                pass
        if (needs_grad and self.fused_training and Co in (32, 64) and Cw % 4 == 0 and (self.K * Cw) % 64 == 0 and self.K * Cw // 2 <= 256
                and 4 * Co <= 256):
            W, cb, (packed, packedT) = self._train_weights()
            try:
                return _LstmCellFn.apply(X, H, C, W, cb, self.w_c_i, self.w_c_f, self.w_c_o, self.b_i, self.b_f, self.b_c, self.b_o,
                                         plan, self.K, packed, packedT)
            except _lib.StmpUnsupported:
                pass
        S = torch.cat(cheb_basis(plan, torch.cat([X, H], dim=-1), self.K), dim=-1)
        pre = torch.matmul(S, self._weight())
        cb = self._conv_bias()
        if cb is not None:
            pre = pre + cb
        pi, pf, pc, po = (pre[..., j * Co:(j + 1) * Co] for j in range(4))
        grad = needs_grad
        if grad:
            I = torch.sigmoid(pi + self.w_c_i * C + self.b_i)
            Fg = torch.sigmoid(pf + self.w_c_f * C + self.b_f)
            Cn = Fg * C + I * torch.tanh(pc + self.b_c)
            O = torch.sigmoid(po + self.w_c_o * Cn + self.b_o)          # uses the NEW cell state (:235-236)
            return O * torch.tanh(Cn), Cn
        Cn = ops.lstm_ifc(pi.contiguous(), pf.contiguous(), pc.contiguous(), C, self.w_c_i, self.w_c_f, self.b_i, self.b_f, self.b_c)
        Hn = ops.lstm_oh(po.contiguous(), Cn, self.w_c_o, self.b_o)
        return Hn, Cn

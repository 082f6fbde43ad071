"""Autograd-aware wrappers over the C ABI (stmp_spmm, fused DCRNN sequence, gate epilogues)."""
import ctypes
from typing import Optional

import torch

from . import _lib
from .plan import GraphPlan, _require_cuda


def _f32c(t: torch.Tensor, name: str) -> torch.Tensor:
    _require_cuda(t, name)
    if t.dtype != torch.float32:
        raise RuntimeError(f"{name} must be float32, got {t.dtype}")
    return t.contiguous()


def spmm_raw(plan: GraphPlan, op: int, x: torch.Tensor, transposed: bool = False, alpha: float = 1.0,
             z: Optional[torch.Tensor] = None, beta: float = 0.0, att: Optional[torch.Tensor] = None,
             out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """y = alpha * A_op x + beta * z on (N,F) or (B,N,F) tensors; no autograd."""
    x = _f32c(x, "x")
    squeeze = x.dim() == 2
    x3 = x.unsqueeze(0) if squeeze else x
    if x3.dim() != 3 or x3.size(1) != plan.num_nodes:
        raise RuntimeError(f"expected (..., {plan.num_nodes}, F) features, got {tuple(x.shape)}")
    B, N, F = x3.shape
    y = torch.empty_like(x3) if out is None else out
    z3 = None
    if z is not None:
        z3 = _f32c(z, "z")
        z3 = z3.unsqueeze(0) if z3.dim() == 2 else z3
    a3 = None
    if att is not None:
        a3 = _f32c(att, "att")
        if a3.shape != (B, N, N):
            raise RuntimeError(f"attention must be ({B},{N},{N}), got {tuple(a3.shape)}")
    with torch.cuda.device(x.device):
        rc = _lib.lib().stmp_spmm(plan.handle, op, int(transposed), B, F, _lib.ptr(x3), F, N * F, _lib.ptr(y), F, N * F,
                                  alpha, _lib.ptr(z3), F, N * F, beta, _lib.ptr(a3), _lib.stream_ptr())
    _lib.check(rc)
    return y.squeeze(0) if squeeze else y


class _SpMM(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, z, att, plan, op, alpha, beta):
        ctx.plan, ctx.op, ctx.alpha, ctx.beta = plan, op, alpha, beta
        ctx.has_z, ctx.has_att = z is not None, att is not None
        ctx.save_for_backward(x if att is not None else None, att)
        return spmm_raw(plan, op, x, False, alpha, z, beta, att)

    @staticmethod
    def backward(ctx, gy):
        x, att = ctx.saved_tensors
        gy = gy.contiguous()
        gx = gz = gatt = None
        if ctx.needs_input_grad[0]:
            gx = spmm_raw(ctx.plan, ctx.op, gy, True, ctx.alpha, None, 0.0, att)
        if ctx.has_z and ctx.needs_input_grad[1]:
            gz = gy * ctx.beta
        if ctx.has_att and ctx.needs_input_grad[2]:
            B, N, F = gy.shape
            gatt = torch.zeros_like(att)
            with torch.cuda.device(gy.device):
                rc = _lib.lib().stmp_spmm_att_grad(ctx.plan.handle, ctx.op, B, F, _lib.ptr(gy), F, N * F,
                                                   _lib.ptr(x.contiguous()), F, N * F, _lib.ptr(gatt), _lib.stream_ptr())
            _lib.check(rc)
            if ctx.alpha != 1.0:
                gatt = gatt * ctx.alpha
        return gx, gz, gatt, None, None, None, None


def spmm(plan: GraphPlan, op: int, x: torch.Tensor, alpha: float = 1.0, z: Optional[torch.Tensor] = None,
         beta: float = 0.0, att: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Differentiable y = alpha * A_op x + beta * z (gather -> weighted scatter-add, K1/K3)."""
    return _SpMM.apply(x, z, att, plan, op, float(alpha), float(beta))


_SEQ_WS = {}


def _seq_workspace(plan: GraphPlan, T: int, cin: int, device) -> torch.Tensor:
    """Per-(device, stream) workspace of the fused sequence kernels (stmp_seq_workspace_bytes), grown on demand and reused: launches on
    one stream are ordered, so consecutive calls may share it."""
    need = int(_lib.lib().stmp_seq_workspace_bytes(plan.handle, T, cin))
    key = (torch.device(device).index, torch.cuda.current_stream(device).cuda_stream)
    buf = _SEQ_WS.get(key)
    if buf is None or buf.numel() < need:
        buf = torch.empty(max(need, 1), dtype=torch.uint8, device=device)
        _SEQ_WS[key] = buf
    return buf


def dcrnn_seq_supported(plan: GraphPlan, cin: int, cout: int, K: int) -> bool:
    return bool(_lib.lib().stmp_dcrnn_seq_supported(plan.handle, cin, cout, K))


def dcrnn_seq_fwd(plan: GraphPlan, x: torch.Tensor, wz, wr, wh, bz, br, bh, K: int, h0=None,
                  win_start: Optional[torch.Tensor] = None, horizon: Optional[int] = None, stash: bool = False,
                  wimage: Optional[torch.Tensor] = None):
    """Fused DCRNN recurrence.  x: (B,T,N,Cin) windows, or -- with win_start (int64 [B]) and horizon --
    the resident series (T_total,N,Cin) from which window b = series[win_start[b]:win_start[b]+horizon]
    is read in-kernel (index-batching).  Returns out (B,T,N,Cout) [, stash (B,T,3,N,Cout)]."""
    x = _f32c(x, "X")
    N = plan.num_nodes
    cout = wz.size(-1)
    if win_start is None:
        if x.dim() != 4 or x.size(2) != N:
            raise RuntimeError(f"X must be (B,T,{N},Cin), got {tuple(x.shape)}")
        B, T, _, cin = x.shape
        bstride, tstride = T * N * cin, N * cin
        ws = None
    else:
        if x.dim() != 3 or x.size(1) != N:
            raise RuntimeError(f"series must be (T_total,{N},Cin), got {tuple(x.shape)}")
        _require_cuda(win_start, "win_start")
        ws = win_start.to(torch.int64).contiguous()
        B, T, cin = ws.numel(), int(horizon), x.size(2)
        bstride, tstride = 0, N * cin
    if wz.size(2) != cin + cout:
        raise RuntimeError(f"DConv weight expects {wz.size(2)} input channels, got Cin+Cout={cin + cout}")
    out = torch.empty((B, T, N, cout), dtype=torch.float32, device=x.device)
    st = torch.empty((B, T, 3, N, cout), dtype=torch.float32, device=x.device) if stash else None
    if B == 0 or T == 0:   # nothing to launch (empty tensors have NULL data pointers)
        return (out, st) if stash else out
    h0c = None if h0 is None else _f32c(h0, "H")
    args = [_f32c(w.detach(), "weight") for w in (wz, wr, wh)]
    bs = [None if b is None else _f32c(b.detach(), "bias") for b in (bz, br, bh)]
    with torch.cuda.device(x.device):
        rc = _lib.lib().stmp_dcrnn_seq_fwd(plan.handle, B, T, cin, cout, K, _lib.ptr(x), _lib.ptr(ws), bstride, tstride,
                                           _lib.ptr(args[0]), _lib.ptr(args[1]), _lib.ptr(args[2]), _lib.ptr(bs[0]),
                                           _lib.ptr(bs[1]), _lib.ptr(bs[2]), _lib.ptr(h0c), _lib.ptr(out), _lib.ptr(st),
                                           _lib.ptr(wimage), _lib.ptr(_seq_workspace(plan, T, cin, x.device)), _lib.stream_ptr())
    _lib.check(rc)
    return (out, st) if stash else out


def gru_seq_supported(plan: GraphPlan, n_ops: int, cin: int, cout: int) -> bool:
    return bool(_lib.lib().stmp_gru_seq_supported(plan.handle, n_ops, cin, cout))


def gru_seq_fwd(plan: GraphPlan, n_ops: int, x: torch.Tensor, wcat: torch.Tensor, bcat: torch.Tensor, h0=None,
                h0_shared: bool = False, wimage: Optional[torch.Tensor] = None):
    """Generic fused graph-GRU recurrence (stmp_gru_seq_fwd).  x (B,T,N,Cin) -> (B,T,N,32).
    h0: (B,N,32), or (N,32)/(1,N,32) with h0_shared=True (every window starts from the same state), or None."""
    x = _f32c(x, "X")
    N = plan.num_nodes
    if x.dim() != 4 or x.size(2) != N:
        raise RuntimeError(f"X must be (B,T,{N},Cin), got {tuple(x.shape)}")
    B, T, _, cin = x.shape
    wcat, bcat = _f32c(wcat, "wcat"), _f32c(bcat, "bcat")
    if wcat.shape != (96, 112) or bcat.numel() != 96:
        raise RuntimeError("wcat must be (96,112) and bcat (96,)")
    out = torch.empty((B, T, N, 32), dtype=torch.float32, device=x.device)
    if B == 0 or T == 0:
        return out
    h0c, hs = None, 0
    if h0 is not None:
        h0c = _f32c(h0, "H")
        hs = 0 if h0_shared else N * 32
    with torch.cuda.device(x.device):
        rc = _lib.lib().stmp_gru_seq_fwd(plan.handle, n_ops, B, T, cin, _lib.ptr(x), None, T * N * cin, N * cin, _lib.ptr(wcat),
                                         _lib.ptr(bcat), _lib.ptr(h0c), hs, _lib.ptr(out), None, _lib.ptr(wimage),
                                         _lib.ptr(_seq_workspace(plan, T, cin, x.device)), _lib.stream_ptr())
    _lib.check(rc)
    return out


def tgcn_attn_fwd(plan: GraphPlan, x: torch.Tensor, A: torch.Tensor, Bm: torch.Tensor, c: torch.Tensor,
                  probs: Optional[torch.Tensor] = None, h: Optional[torch.Tensor] = None, h_shared: bool = False) -> torch.Tensor:
    """Fused A3TGCN(2) / TGCN(2) forward (stmp_tgcn_attn_fwd).  x (B,N,Fin,P) -> (B,N,32); h (B,N,32), or (N,32) with
    h_shared=True (the same state for every batch row), or None (zeros)."""
    x = _f32c(x, "X")
    if x.dim() != 4 or x.size(1) != plan.num_nodes:
        raise RuntimeError(f"X must be (B,{plan.num_nodes},Fin,P), got {tuple(x.shape)}")
    B, N, fin, P = x.shape
    A, Bm, c = _f32c(A, "A"), _f32c(Bm, "Bm"), _f32c(c, "c")
    if A.shape != (fin, 96) or Bm.shape != (32, 96) or c.numel() != 96:
        raise RuntimeError("folded weights must be A (Fin,96), Bm (32,96), c (96,)")
    out = torch.empty((B, N, 32), dtype=torch.float32, device=x.device)
    if B == 0:
        return out
    hc, hs = None, 0
    if h is not None:
        hc = _f32c(h, "H")
        hs = 0 if h_shared else N * 32
    pr = None if probs is None else _f32c(probs.detach(), "probs")
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().stmp_tgcn_attn_fwd(plan.handle, B, fin, P, _lib.ptr(x), _lib.ptr(hc), hs, _lib.ptr(A), _lib.ptr(Bm),
                                                 _lib.ptr(c), _lib.ptr(pr), _lib.ptr(out), _lib.stream_ptr()))
    return out


class _TgcnAttnFn(torch.autograd.Function):
    """Training form of the fused A3TGCN(2) / TGCN(2) forward for H = None: forward = `stmp_tgcn_attn_fwd`, backward =
    `stmp_tgcn_attn_bwd` (gates recomputed, gradients of the folded weights A, c and of the attention probabilities reduced on the
    device).  No gradient w.r.t. X."""

    @staticmethod
    def forward(ctx, plan, x, A, Bm, c, probs):
        out = tgcn_attn_fwd(plan, x, A.detach(), Bm.detach(), c.detach(), None if probs is None else probs.detach(), None)
        ctx.plan, ctx.has_probs = plan, probs is not None
        ctx.save_for_backward(x, A.detach(), c.detach(), probs.detach() if probs is not None else x.new_empty(0))
        return out

    @staticmethod
    def backward(ctx, gout):
        x, A, c, probs = ctx.saved_tensors
        plan = ctx.plan
        B, N, fin, P = x.shape
        gout = _f32c(gout, "gout")
        dev = x.device
        ws = torch.empty(int(_lib.lib().stmp_tgcn_attn_bwd_workspace_bytes(plan.handle, B)), dtype=torch.uint8, device=dev)
        dA = torch.empty(fin, 96, dtype=torch.float32, device=dev)
        dc = torch.empty(96, dtype=torch.float32, device=dev)
        dprobs = torch.empty(P, dtype=torch.float32, device=dev) if ctx.has_probs else None
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().stmp_tgcn_attn_bwd(plan.handle, B, fin, P, _lib.ptr(_f32c(x, "X")), _lib.ptr(_f32c(A, "A")), _lib.ptr(_f32c(c, "c")),
                                                     _lib.ptr(_f32c(probs, "probs")) if ctx.has_probs else None, _lib.ptr(gout), _lib.ptr(ws),
                                                     _lib.ptr(dA), _lib.ptr(dc), _lib.ptr(dprobs), _lib.stream_ptr()))
        return None, None, dA, None, dc, dprobs


def tgcn_attn_train(plan: GraphPlan, x, A, Bm, c, probs=None) -> torch.Tensor:
    """Differentiable (w.r.t. A, c, probs) fused A3TGCN(2) / TGCN(2) forward for H = None."""
    return _TgcnAttnFn.apply(plan, x, A, Bm, c, probs)


def spmm_cols(plan: GraphPlan, op: int, buf: torch.Tensor, src_col: int, dst_col: int, width: int, alpha: float = 1.0,
              z_col: Optional[int] = None, beta: float = 0.0, transposed: bool = False):
    """In-place column-block product inside one basis buffer `buf` (..., N, LD):
    buf[..., dst_col:dst_col+width] = alpha * A_op buf[..., src_col:+width] + beta * buf[..., z_col:+width].
    Lets T_k be written straight into its slot of S = [T_0 | T_1 | ...] (no torch.cat of large tensors); with
    `transposed` (A_op^T) and z_col == dst_col it is the accumulate step of the basis adjoint.  src and dst blocks must
    not overlap; z may alias dst exactly (each output element reads its own z before it is written)."""
    _require_cuda(buf, "buf")
    b3 = buf if buf.dim() == 3 else buf.unsqueeze(0)
    B, N, LD = b3.shape
    if not b3.is_contiguous() or N != plan.num_nodes:
        raise RuntimeError("basis buffer must be contiguous (..., N, LD)")
    base, es = b3.data_ptr(), 4
    pz = None if z_col is None else ctypes.c_void_p(base + z_col * es)
    with torch.cuda.device(buf.device):
        rc = _lib.lib().stmp_spmm(plan.handle, op, 1 if transposed else 0, B, width, ctypes.c_void_p(base + src_col * es), LD, N * LD,
                                  ctypes.c_void_p(base + dst_col * es), LD, N * LD, alpha, pz, LD, N * LD, beta, None,
                                  _lib.stream_ptr())
    _lib.check(rc)


def gemm_prepack(W: torch.Tensor) -> torch.Tensor:
    """Split a (K,N) fp32 weight into the packed fp16 hi/lo buffer of stmp_gemm_f32 (once per weight update)."""
    W = _f32c(W, "W")
    K, N = W.shape
    packed = torch.empty(int(_lib.lib().stmp_gemm_packed_elems(K, N)), dtype=torch.float16, device=W.device)
    with torch.cuda.device(W.device):
        _lib.check(_lib.lib().stmp_gemm_prepack(_lib.ptr(W), N, K, N, _lib.ptr(packed), _lib.stream_ptr()))
    return packed


def pow2_row_scale(A: torch.Tensor) -> torch.Tensor:
    """Per-row powers of two s_r = 2^(12 - E_r), E_r the binary exponent of max|A_r|, for `gemm(..., row_scale=)`: they bring each
    row's largest magnitude into [2^12, 2^13), where the fp16 hi/lo split keeps its relative 2^-22.  The shift is clamped to +-126 so
    s_r and 1/s_r are normal fp32 (zero and subnormal rows get 2^126; zero rows stay zero), and a row holding inf / NaN gets a finite
    scale (and stays non-finite).  Read off the exponent bits of the row max: one reduction and four elementwise launches on
    (M,) values.  A (M, K) fp32 on any device -> (M,) fp32."""
    amax = torch.linalg.vector_norm(A, float("inf"), dim=-1)
    biased = amax.view(torch.int32) >> 23                           # E + 127; 0 for zero / subnormal, 255 for inf / NaN
    return ((266 - biased).clamp_(1, 253) << 23).view(torch.float32)   # the IEEE bits of 2^(12 - E), E + 127 in [1, 253]


def gemm(A: torch.Tensor, packed: torch.Tensor, K: int, N: int, bias: Optional[torch.Tensor] = None,
         out: Optional[torch.Tensor] = None, row_scale: Optional[torch.Tensor] = None) -> torch.Tensor:
    """C = A @ W + bias on tcgen05 with the fp16 hi/lo operand split (fp32-class accuracy).  A (..., K) contiguous.
    `out`: a 2-D (M, N) view with unit column stride (e.g. a column block of a wider buffer) to write into.
    The split is exact to a relative 2^-22 only for 2^-3 <= |a| < 65520; below that its error is an absolute ~2^-25 (values under
    ~3e-8 vanish) and from 65520 up the operand is inf.  For an A of arbitrary magnitude (a gradient) pass
    `row_scale = pow2_row_scale(A)`: every row is scaled into that range before the split and back after the product, exactly, so
    the result is the same for any power-of-two scaling of A."""
    A = _f32c(A, "A")
    M = A.numel() // K
    if row_scale is not None:
        row_scale = _f32c(row_scale, "row_scale")
        if row_scale.numel() != M:
            raise RuntimeError(f"gemm: row_scale must have one entry per row of A ({M}), got {row_scale.numel()}")
    if out is None:
        C = torch.empty(*A.shape[:-1], N, dtype=torch.float32, device=A.device)
        ldc = N
    else:
        C = out
        if C.dim() != 2 or C.size(0) != M or C.size(1) != N or C.stride(1) != 1 or C.dtype != torch.float32:
            raise RuntimeError("gemm: `out` must be a float32 (M, N) view with unit column stride")
        ldc = C.stride(0)
    b = None if bias is None else _f32c(bias.detach(), "bias")
    with torch.cuda.device(A.device):
        _lib.check(_lib.lib().stmp_gemm_f32(_lib.ptr(A), K, M, K, N, _lib.ptr(packed), _lib.ptr(b), _lib.ptr(row_scale), _lib.ptr(C), ldc,
                                            _lib.stream_ptr()))
    return C


EPI_BIAS, EPI_RELU, EPI_RELU_LN = 0, 1, 2


def _weight_image(packed: torch.Tensor, N: int, nblk: int) -> torch.Tensor:
    img = torch.empty(int(_lib.lib().stmp_gemm_blocks_image_bytes(N, nblk)), dtype=torch.uint8, device=packed.device)
    with torch.cuda.device(packed.device):
        _lib.check(_lib.lib().stmp_gemm_blocks_image(_lib.ptr(packed), N, nblk, _lib.ptr(img), _lib.stream_ptr()))
    return img


def gemm_blocks_prepack(blocks):
    """Pack the per-block weights [(width_i, N) fp32 ...] of a blocked GEMM: every block is zero-padded to 64 rows, the stack
    (nblk*64, N) is split into fp16 hi/lo (stmp_gemm_prepack) and rewritten as the per-k-block shared-memory image the kernel
    fetches by TMA (stmp_gemm_blocks_image).  Returns (packed, image)."""
    N = blocks[0].size(1)
    W = torch.zeros(64 * len(blocks), N, device=blocks[0].device, dtype=torch.float32)
    for i, w in enumerate(blocks):
        if w.size(0) > 64 or w.size(1) != N:
            raise RuntimeError("blocked GEMM: weight blocks must be (<=64, N)")
        W[64 * i:64 * i + w.size(0)] = w
    packed = gemm_prepack(W)
    return packed, _weight_image(packed, N, len(blocks))


def gemm_blocks(blocks, packed: torch.Tensor, N: int, ncols: int, bias: Optional[torch.Tensor] = None, epilogue: int = EPI_BIAS,
                gamma=None, beta=None, eps: float = 1e-5, seq: int = 1, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """C[m, :ncols] = epilogue(sum_i A_i[m + shift_i, :width_i] @ W_i + bias)  (stmp_gemm_blocks_f32).
    blocks: list of (tensor, width, shift): `tensor` is a 2-D fp32 CUDA view (M, >=width) with unit column stride."""
    M = blocks[0][0].size(0)
    dev = blocks[0][0].device
    n = len(blocks)
    ptrs = (ctypes.c_void_p * n)()
    lds = (ctypes.c_int64 * n)()
    widths = (ctypes.c_int32 * n)()
    shifts = (ctypes.c_int32 * n)()
    for i, (t, width, shift) in enumerate(blocks):
        _require_cuda(t, "block")
        if t.dtype != torch.float32 or t.dim() != 2 or t.size(0) != M or (t.size(1) > 1 and t.stride(1) != 1) or t.size(1) < width:
            raise RuntimeError("blocked GEMM: every block must be a float32 (M, >=width) view with unit column stride")
        ptrs[i], lds[i], widths[i], shifts[i] = t.data_ptr(), t.stride(0), width, shift
    C = torch.empty((M, ncols), dtype=torch.float32, device=dev) if out is None else out
    v = [None if t is None else _f32c(t.detach(), "param") for t in (bias, gamma, beta)]
    packed, image = packed if isinstance(packed, tuple) else (packed, None)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().stmp_gemm_blocks_f32(M, N, ncols, n, ctypes.cast(ptrs, ctypes.c_void_p), ctypes.cast(lds, ctypes.c_void_p),
                                                   ctypes.cast(widths, ctypes.c_void_p), ctypes.cast(shifts, ctypes.c_void_p), seq,
                                                   _lib.ptr(packed), _lib.ptr(image), _lib.ptr(v[0]), epilogue, _lib.ptr(v[1]), _lib.ptr(v[2]), eps,
                                                   _lib.ptr(C), C.stride(0), _lib.stream_ptr()))
    return C


def astgcn_factors(Xc, U1, U2, U3, be, Ve, W1, W2, W3, want_E: bool = False):
    """(lhs_s (B,N,T), rhs_s (B,T,N) [, E (B,T,T)]) of an ASTGCN block from channels-last X (B,N,T,F): temporal attention, X~ = X E and
    the spatial-attention factors in one launch (stmp_astgcn_factors_fwd)."""
    Xc = _f32c(Xc, "X")
    B, N, T, Fi = Xc.shape
    lhs = torch.empty((B, N, T), dtype=torch.float32, device=Xc.device)
    rhs = torch.empty((B, T, N), dtype=torch.float32, device=Xc.device)
    E = torch.empty((B, T, T), dtype=torch.float32, device=Xc.device) if want_E else None
    v = [_f32c(t.detach(), "param") for t in (U1, U2, U3, be.reshape(T, T), Ve, W1, W2, W3)]
    with torch.cuda.device(Xc.device):
        _lib.check(_lib.lib().stmp_astgcn_factors_fwd(B, N, T, Fi, _lib.ptr(Xc), *[_lib.ptr(t) for t in v], _lib.ptr(lhs), _lib.ptr(rhs),
                                                      _lib.ptr(E), _lib.stream_ptr()))
    return (lhs, rhs, E) if want_E else (lhs, rhs)


def spatial_attention_prepack(Vs: torch.Tensor) -> torch.Tensor:
    """Vs (N,N) -> packed fp16 hi/lo of Vs^T zero-padded to (P,P), P = N rounded up to 64."""
    n = Vs.size(0)
    P = (n + 63) // 64 * 64
    W = torch.zeros(P, P, device=Vs.device, dtype=torch.float32)
    W[:n, :n] = Vs.detach().t()
    packed = gemm_prepack(W)
    return packed, _weight_image(packed, P, P // 64)


def spatial_attention(lhs: torch.Tensor, rhs: torch.Tensor, bsT: torch.Tensor, vsT_packed: torch.Tensor) -> torch.Tensor:
    """ST (B, N, P) with ST[b, j, i] = softmax_dim1(Vs @ sigmoid(lhs @ rhs + bs))[b, i, j]; columns >= N are zero."""
    lhs, rhs, bsT = _f32c(lhs, "lhs"), _f32c(rhs, "rhs"), _f32c(bsT, "bsT")
    B, n, T = lhs.shape
    P = (n + 63) // 64 * 64
    st = torch.empty((B, n, P), dtype=torch.float32, device=lhs.device)
    packed, image = vsT_packed if isinstance(vsT_packed, tuple) else (vsT_packed, None)
    with torch.cuda.device(lhs.device):
        _lib.check(_lib.lib().stmp_spatial_attention_fwd(B, n, T, _lib.ptr(lhs), _lib.ptr(rhs), _lib.ptr(bsT), _lib.ptr(packed),
                                                         _lib.ptr(image), _lib.ptr(st), P, _lib.stream_ptr()))
    return st


def spmm_attT(plan: GraphPlan, op: int, x: torch.Tensor, attT: torch.Tensor, alpha: float = 1.0) -> torch.Tensor:
    """y = alpha * (A_op * att) x with the attention given transposed / row-padded (B, N, ld) as `spatial_attention` writes it."""
    x = _f32c(x, "x")
    B, N, F = x.shape
    y = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().stmp_spmm_att_t(plan.handle, op, B, F, _lib.ptr(x), F, N * F, _lib.ptr(y), F, N * F, alpha, None, F, N * F, 0.0,
                                             _lib.ptr(attT), attT.stride(1), _lib.stream_ptr()))
    return y


def gemm_lstm(A: torch.Tensor, packed: torch.Tensor, K: int, cout: int, conv_bias, cell, wci, wcf, wco, bi, bf, bc, bo):
    """(H', C') = peephole-LSTM gates of (A @ W + conv_bias), fused in the GEMM epilogue (stmp_gemm_lstm_f32)."""
    A, cell = _f32c(A, "A"), _f32c(cell, "C")
    M = A.numel() // K
    h = torch.empty_like(cell)
    c = torch.empty_like(cell)
    v = [None if t is None else _f32c(t.detach().reshape(-1), "param") for t in (conv_bias, wci, wcf, wco, bi, bf, bc, bo)]
    with torch.cuda.device(A.device):
        _lib.check(_lib.lib().stmp_gemm_lstm_f32(_lib.ptr(A), K, M, K, cout, _lib.ptr(packed), _lib.ptr(v[0]), _lib.ptr(cell),
                                                 _lib.ptr(v[1]), _lib.ptr(v[2]), _lib.ptr(v[3]), _lib.ptr(v[4]), _lib.ptr(v[5]),
                                                 _lib.ptr(v[6]), _lib.ptr(v[7]), _lib.ptr(h), _lib.ptr(c), _lib.stream_ptr()))
    return h, c


def dcrnn_weight_image(wz, wr, wh, bz, br, bh, cin: int, K: int) -> Optional[torch.Tensor]:
    """B-operand image of the tcgen05 kernel for DConv weights (None when the configuration has no tensor kernel)."""
    cout = wz.size(-1)
    if cout != 32 or K != 2 or not (1 <= cin <= 4):
        return None
    img = torch.empty(int(_lib.lib().stmp_gru_weight_image_bytes()), dtype=torch.uint8, device=wz.device)
    args = [_f32c(w.detach(), "weight") for w in (wz, wr, wh)]
    bs = [None if b is None else _f32c(b.detach(), "bias") for b in (bz, br, bh)]
    with torch.cuda.device(wz.device):
        _lib.check(_lib.lib().stmp_dcrnn_pack_weights(cin, cout, K, _lib.ptr(args[0]), _lib.ptr(args[1]), _lib.ptr(args[2]),
                                                      _lib.ptr(bs[0]), _lib.ptr(bs[1]), _lib.ptr(bs[2]), _lib.ptr(img), _lib.stream_ptr()))
    return img


def gru_weight_image(wcat: torch.Tensor, bcat: torch.Tensor) -> torch.Tensor:
    img = torch.empty(int(_lib.lib().stmp_gru_weight_image_bytes()), dtype=torch.uint8, device=wcat.device)
    with torch.cuda.device(wcat.device):
        _lib.check(_lib.lib().stmp_gru_pack_weights(_lib.ptr(_f32c(wcat, "wcat")), _lib.ptr(_f32c(bcat, "bcat")), _lib.ptr(img),
                                                    _lib.stream_ptr()))
    return img


class PackCache(object):
    """Caches the packed (wcat, bcat) of a module until one of its parameters changes (host-side `_version`
    check, no device sync), so inference pays the packing once."""

    def __init__(self):
        self._key, self._val = None, None

    def get(self, params, build):
        key = tuple((p.data_ptr(), p._version) for p in params)
        if key != self._key:
            with torch.no_grad():
                self._val = build()
            self._key = key
        return self._val


def gru_zr(pz, pr, h):
    pz, pr, h = _f32c(pz, "pz"), _f32c(pr, "pr"), _f32c(h, "h")
    z, r, hr = torch.empty_like(pz), torch.empty_like(pz), torch.empty_like(pz)
    with torch.cuda.device(pz.device):
        _lib.check(_lib.lib().stmp_gru_zr(pz.numel(), _lib.ptr(pz), _lib.ptr(pr), _lib.ptr(h), _lib.ptr(z), _lib.ptr(r),
                                          _lib.ptr(hr), _lib.stream_ptr()))
    return z, r, hr


def gru_out(ph, z, h):
    ph, z, h = _f32c(ph, "ph"), _f32c(z, "z"), _f32c(h, "h")
    hn = torch.empty_like(ph)
    with torch.cuda.device(ph.device):
        _lib.check(_lib.lib().stmp_gru_out(ph.numel(), _lib.ptr(ph), _lib.ptr(z), _lib.ptr(h), None, _lib.ptr(hn),
                                           _lib.stream_ptr()))
    return hn


def dcrnn_bwd_supported(plan: GraphPlan, cin: int, cout: int, K: int) -> bool:
    return bool(_lib.lib().stmp_dcrnn_bwd_supported(plan.handle, cin, cout, K))


def dcrnn_bwd_basis(plan: GraphPlan, x, out, h0, stash, S1, S2):
    """S1/S2 (T*B, N, ld) <- bases of [X_t | H_{t-1}] and [X_t | H_{t-1}*R_t] for every (t, b): one launch."""
    x, out, stash = _f32c(x, "x"), _f32c(out, "out"), _f32c(stash, "stash")
    B, T, N, Ci = x.shape
    h0 = None if h0 is None else _f32c(h0, "h0")
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().stmp_dcrnn_bwd_basis(plan.handle, B, T, Ci, out.size(-1), _lib.ptr(x), T * N * Ci, N * Ci, _lib.ptr(out),
                                                   _lib.ptr(h0), _lib.ptr(stash), _lib.ptr(S1), _lib.ptr(S2), S1.size(-1), _lib.stream_ptr()))


def dcrnn_bwd_seq(plan: GraphPlan, cin: int, gout, out, h0, stash, whsT, wzrT, dph_all, dpzr_all, dx, dh0):
    """The reverse-time recurrence of the DCRNN backward in one persistent launch (one CTA per window)."""
    gout, out, stash = _f32c(gout, "gout"), _f32c(out, "out"), _f32c(stash, "stash")
    B, T, N, Co = gout.shape
    h0 = None if h0 is None else _f32c(h0, "h0")
    with torch.cuda.device(gout.device):
        _lib.check(_lib.lib().stmp_dcrnn_bwd_seq(plan.handle, B, T, cin, Co, _lib.ptr(gout), _lib.ptr(out), _lib.ptr(h0), _lib.ptr(stash),
                                                 _lib.ptr(_f32c(whsT, "whsT")), _lib.ptr(_f32c(wzrT, "wzrT")), _lib.ptr(dph_all),
                                                 _lib.ptr(dpzr_all), _lib.ptr(dx), _lib.ptr(dh0), _lib.stream_ptr()))


def dcrnn_bwd_basis_ld(cin: int, cout: int, K: int) -> int:
    """Row pitch of the stacked bases: (2K-1)(cin+cout) rounded up to 8 floats (16-byte rows for the weight-gradient kernel's tiles)."""
    return ((2 * K - 1) * (cin + cout) + 7) // 8 * 8


_WGRAD_WS = {}


def dcrnn_bwd_wgrad(cin: int, K: int, S1, S2, dpzr_all, dph_all, has_bias: bool):
    """(gz, gr, gh, gbz, gbr, gbh): weight / bias gradients of the three gates over all (t, b, n) rows in two launches
    (`stmp_dcrnn_bwd_wgrad`); S1 / S2 (T*B, N, ld) from dcrnn_bwd_basis with ld = dcrnn_bwd_basis_ld(...)."""
    Co = dph_all.size(-1)
    C = cin + Co
    dev = S1.device
    rows = S1.size(0) * S1.size(1)
    key = (dev, torch.cuda.current_stream(dev).cuda_stream, cin)
    ws = _WGRAD_WS.get(key)
    if ws is None:
        ws = torch.empty(int(_lib.lib().stmp_dcrnn_bwd_wgrad_workspace_bytes(cin)), device=dev, dtype=torch.uint8)
        _WGRAD_WS[key] = ws
    g = torch.empty(3, 2, K, C, Co, device=dev, dtype=torch.float32)
    gb = torch.empty(3, Co, device=dev, dtype=torch.float32) if has_bias else None
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().stmp_dcrnn_bwd_wgrad(cin, Co, K, rows, S1.size(-1), _lib.ptr(S1), _lib.ptr(S2), _lib.ptr(dpzr_all), _lib.ptr(dph_all),
                                                   _lib.ptr(ws), _lib.ptr(g[0]), _lib.ptr(g[1]), _lib.ptr(g[2]),
                                                   _lib.ptr(None if gb is None else gb[0]), _lib.ptr(None if gb is None else gb[1]),
                                                   _lib.ptr(None if gb is None else gb[2]), _lib.stream_ptr()))
    if gb is None:
        return g[0], g[1], g[2], None, None, None
    return g[0], g[1], g[2], gb[0], gb[1], gb[2]


def adam_flat(param, grad, exp_avg, exp_avg_sq, step, ticket, lr, beta1, beta2, eps, weight_decay=0.0, grad_scale=1.0, zero_grad=True):
    """One-launch Adam over flat fp32 buffers (`stmp_adam_flat`); `step` (1 float) and `ticket` (1 int32, zero) are device tensors."""
    for t, nm in ((param, "param"), (grad, "grad"), (exp_avg, "exp_avg"), (exp_avg_sq, "exp_avg_sq")):
        if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.numel() == param.numel()):
            raise RuntimeError(f"adam_flat: {nm} must be a contiguous CUDA fp32 buffer of {param.numel()} elements")
    with torch.cuda.device(param.device):
        _lib.check(_lib.lib().stmp_adam_flat(param.numel(), _lib.ptr(param), _lib.ptr(grad), _lib.ptr(exp_avg), _lib.ptr(exp_avg_sq), _lib.ptr(step),
                                             _lib.ptr(ticket), lr, beta1, beta2, eps, weight_decay, grad_scale, 1 if zero_grad else 0,
                                             _lib.stream_ptr()))


def dcrnn_pack_bwd_weights(wz, wr, wh, cin: int, K: int):
    """(whsT (Co, (2K-1)C), wzrT (2Co, (2K-1)C)): transposed stacked weights of the backward GEMMs, one launch."""
    Co = wz.size(-1)
    nbC = (2 * K - 1) * (cin + Co)
    whsT = torch.empty(Co, nbC, device=wz.device, dtype=torch.float32)
    wzrT = torch.empty(2 * Co, nbC, device=wz.device, dtype=torch.float32)
    with torch.cuda.device(wz.device):
        _lib.check(_lib.lib().stmp_dcrnn_pack_bwd_weights(cin, Co, K, _lib.ptr(_f32c(wz.detach(), "wz")), _lib.ptr(_f32c(wr.detach(), "wr")),
                                                          _lib.ptr(_f32c(wh.detach(), "wh")), _lib.ptr(whsT), _lib.ptr(wzrT), _lib.stream_ptr()))
    return whsT, wzrT


class _MaskedMAE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, target):
        pred, target = _f32c(pred, "pred"), _f32c(target, "target")
        if pred.shape != target.shape:
            raise RuntimeError(f"masked_mae: shape mismatch {tuple(pred.shape)} vs {tuple(target.shape)}")
        ws = torch.empty(int(_lib.lib().stmp_masked_mae_workspace_floats()), device=pred.device, dtype=torch.float32)
        out = torch.empty(2, device=pred.device, dtype=torch.float32)           # [loss, sum(mask)]
        with torch.cuda.device(pred.device):
            _lib.check(_lib.lib().stmp_masked_mae_fwd(pred.numel(), _lib.ptr(pred), _lib.ptr(target), _lib.ptr(ws), ctypes.c_void_p(out.data_ptr()),
                                                      ctypes.c_void_p(out.data_ptr() + 4), _lib.stream_ptr()))
        ctx.save_for_backward(pred, target, out)
        return out[0].clone()

    @staticmethod
    def backward(ctx, gout):
        pred, target, out = ctx.saved_tensors
        gp = torch.empty_like(pred)
        gout = gout.contiguous().to(torch.float32)
        with torch.cuda.device(pred.device):
            _lib.check(_lib.lib().stmp_masked_mae_bwd(pred.numel(), _lib.ptr(pred), _lib.ptr(target), ctypes.c_void_p(out.data_ptr() + 4),
                                                      _lib.ptr(gout), _lib.ptr(gp), _lib.stream_ptr()))
        return gp, None


def masked_mae(pred: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
    """Fused masked MAE (forward 2 launches, backward 1) with the semantics of examples/indexBatching/DCRNN/utils.py:10-18."""
    return _MaskedMAE.apply(pred, target)


def _slice_ptr(t: Optional[torch.Tensor]):
    """(pointer, batch stride in elements) of a (B, N, C) fp32 slice whose trailing two dims are dense."""
    if t is None:
        return None, 0
    if t.dtype != torch.float32 or t.dim() != 3 or t.stride(2) != 1 or t.stride(1) != t.size(2):
        raise RuntimeError("expected a float32 (B, N, C) slice with dense trailing dims")
    return ctypes.c_void_p(t.data_ptr()), t.stride(0)


def gru_bwd_carry(cin: int, cout: int, du2, du1, g_prev=None, z_prev=None, r_prev=None, dx=None, gout=None, z=None, ht=None,
                  g=None, dph=None, dh_out=None):
    """stmp_gru_bwd_carry: close step t+1 (g_prev, z_prev, r_prev, du2, du1 [, dx]) and/or open step t (gout, z, ht -> g, dph)."""
    ref = g_prev if g_prev is not None else gout
    B, N = ref.size(0), ref.size(1)
    du_ld = du2.size(-1)
    zp, s1 = _slice_ptr(z_prev)
    rp, _ = _slice_ptr(r_prev)
    zz, s2 = _slice_ptr(z)
    hh, _ = _slice_ptr(ht)
    go, gs = _slice_ptr(gout)
    dxp, dxs = _slice_ptr(dx)
    stash_bs = s1 if z_prev is not None else s2
    if z_prev is not None and z is not None and s1 != s2:
        raise RuntimeError("stash slices of one call must share their batch stride")
    with torch.cuda.device(ref.device):
        _lib.check(_lib.lib().stmp_gru_bwd_carry(B, N, cin, cout, du_ld, _lib.ptr(g_prev), zp, rp, _lib.ptr(du2), _lib.ptr(du1), dxp, dxs,
                                                 go, gs, zz, hh, stash_bs, _lib.ptr(g), _lib.ptr(dph), _lib.ptr(dh_out), _lib.stream_ptr()))


def gru_bwd_zr(cin: int, cout: int, g, hprev, z, r, ht, du2, dpzr):
    B, N = g.size(0), g.size(1)
    hp, hs = _slice_ptr(hprev)
    zz, ss = _slice_ptr(z)
    rr, _ = _slice_ptr(r)
    hh, _ = _slice_ptr(ht)
    with torch.cuda.device(g.device):
        _lib.check(_lib.lib().stmp_gru_bwd_zr(B, N, cin, cout, du2.size(-1), _lib.ptr(g), hp, hs, zz, rr, hh, ss, _lib.ptr(du2),
                                              _lib.ptr(dpzr), _lib.stream_ptr()))


def lstm_ifc(pi, pf, pc, c, wci, wcf, bi, bf, bc):
    pi, pf, pc, c = (_f32c(t, "gate") for t in (pi, pf, pc, c))
    cout = pi.size(-1)
    rows = pi.numel() // cout
    cn = torch.empty_like(pi)
    v = [_f32c(t.detach().reshape(-1), "param") for t in (wci, wcf, bi, bf, bc)]
    with torch.cuda.device(pi.device):
        _lib.check(_lib.lib().stmp_lstm_ifc(rows, cout, _lib.ptr(pi), _lib.ptr(pf), _lib.ptr(pc), _lib.ptr(c), _lib.ptr(v[0]),
                                            _lib.ptr(v[1]), _lib.ptr(v[2]), _lib.ptr(v[3]), _lib.ptr(v[4]), None, None, None,
                                            _lib.ptr(cn), _lib.stream_ptr()))
    return cn


def lstm_oh(po, cnew, wco, bo):
    po, cnew = _f32c(po, "po"), _f32c(cnew, "cnew")
    cout = po.size(-1)
    rows = po.numel() // cout
    hn = torch.empty_like(po)
    v = [_f32c(t.detach().reshape(-1), "param") for t in (wco, bo)]
    with torch.cuda.device(po.device):
        _lib.check(_lib.lib().stmp_lstm_oh(rows, cout, _lib.ptr(po), _lib.ptr(cnew), _lib.ptr(v[0]), _lib.ptr(v[1]), None,
                                           _lib.ptr(hn), _lib.stream_ptr()))
    return hn


def lstm_gate_bwd(pre, c_old, c_new, gh, gc, wci, wcf, wco, bi, bf, bc, bo):
    """(dpre (rows,4Co), dC_old (rows,Co)) of the peephole-LSTM gate chain (stmp_lstm_gate_bwd); gh / gc may be None."""
    pre, c_old, c_new = _f32c(pre, "pre"), _f32c(c_old, "c_old"), _f32c(c_new, "c_new")
    cout = c_old.size(-1)
    rows = c_old.numel() // cout
    dpre = torch.empty_like(pre)
    dco = torch.empty_like(c_old)
    gh = None if gh is None else _f32c(gh, "gh")
    gc = None if gc is None else _f32c(gc, "gc")
    v = [_f32c(t.detach().reshape(-1), "param") for t in (wci, wcf, wco, bi, bf, bc, bo)]
    with torch.cuda.device(pre.device):
        _lib.check(_lib.lib().stmp_lstm_gate_bwd(rows, cout, _lib.ptr(pre), _lib.ptr(c_old), _lib.ptr(c_new), _lib.ptr(gh), _lib.ptr(gc),
                                                 *[_lib.ptr(t) for t in v], _lib.ptr(dpre), _lib.ptr(dco), _lib.stream_ptr()))
    return dpre, dco


def window_gather(series: torch.Tensor, start: torch.Tensor, horizon: int, with_target: bool = True):
    """x[b] = series[start[b]:start[b]+h], y[b] = series[start[b]+h:start[b]+2h] (index_dataset.py:49-57)."""
    series = _f32c(series, "series")
    _require_cuda(start, "start")
    start = start.to(torch.int64).contiguous()
    B = start.numel()
    row = series[0].numel()
    shape = (B, horizon) + tuple(series.shape[1:])
    x = torch.empty(shape, dtype=torch.float32, device=series.device)
    y = torch.empty(shape, dtype=torch.float32, device=series.device) if with_target else None
    with torch.cuda.device(series.device):
        _lib.check(_lib.lib().stmp_window_gather(_lib.ptr(series), series.size(0), row, _lib.ptr(start), B, horizon,
                                                 _lib.ptr(x), _lib.ptr(y), _lib.stream_ptr()))
    return (x, y) if with_target else x

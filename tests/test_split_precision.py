"""Accuracy envelope of the fp16 hi/lo split behind every tcgen05 GEMM (`gemm_tc.cu`, `gemm_blocks.cu`, `dcrnn_seq_tc.cu`).

An fp32 operand v is split into hi = fp16(v), lo = fp16(v - hi) and the product is accumulated as lo*hi + hi*lo + hi*hi in fp32.
That keeps a relative 2^-22 only for 2^-3 <= |v| < 65520: below 2^-3 `lo` is subnormal and the split's error is an absolute ~2^-25,
values under ~3e-8 are 0 in both halves, and |v| >= 65520 is inf.  The tests here

* state that error model element by element (`bound`) and show on the CPU that it accepts correct arithmetic with a 2x margin and
  rejects kernels that drop a pass or the lo halves (so a kernel that passes the GPU tests is not just "close");
* hold every split-GEMM entry point to that bound against float64 across operand scales 2^-20 .. 2^15, rows of mixed scale in one
  launch, and weight scales 2^-8 .. 2^4;
* pin the power-of-two row scaling of gradient operands (`ops.pow2_row_scale`, `ops.gemm(row_scale=)`) and the GConvLSTM cell
  backward that uses it under a mean loss, and check that every hand-written backward is equivariant under power-of-two loss scaling.
"""
import math

import pytest
import torch

from oracle import recurrent as R
from pytorch_geometric_temporal_b200 import _lib, ops
from pytorch_geometric_temporal_b200.dataset import synthetic

DEV = "cuda"
C_ACC = 16                                    # fp32 accumulation term of the bound, in units of 2^-24 * (|A| @ |W|)
A_SCALES = [2.0 ** e for e in (-20, -12, -6, 0, 6, 12, 15)]
W_SCALES = [2.0 ** e for e in (-8, 0, 4)]
SHAPES = [(K, N) for K in (4, 36, 128, 256, 384) for N in (32, 64, 96, 128, 256)]


# ---- the error model -----------------------------------------------------------------------------------------------------------------
def split16(v: torch.Tensor):
    """(hi, lo) of the device split, as fp32: torch's CPU conversion rounds to nearest and keeps subnormals, like __float2half_rn."""
    v = v.float()
    hi = v.half().float()
    return hi, (v - hi).half().float()


def emulate(A: torch.Tensor, W: torch.Tensor) -> torch.Tensor:
    """ahi@whi + ahi@wlo + alo@whi in float64: the split's value of A @ W without accumulation error."""
    ah, al = (t.double() for t in split16(A))
    wh, wl = (t.double() for t in split16(W))
    return ah @ wh + ah @ wl + al @ wh


def bound(A: torch.Tensor, W: torch.Tensor, c: float = C_ACC) -> torch.Tensor:
    """Per-element tolerance of a split GEMM against the exact float64 product: twice the split's representation error (which the
    tensor core reproduces exactly -- fp16 x fp16 products are exact in fp32) plus c * 2^-24 * (|A| @ |W|) for fp32 accumulation."""
    A64, W64 = A.double(), W.double()
    return 2 * (emulate(A, W) - A64 @ W64).abs() + c * 2.0 ** -24 * (A64.abs() @ W64.abs())


def _mutants(A, W):
    ah, al = split16(A)
    wh, wl = split16(W)
    return {"drop lo*hi": ah @ wh + ah @ wl, "drop hi*lo": ah @ wh + al @ wh, "hi only": ah @ wh}


def _ratio(got: torch.Tensor, A: torch.Tensor, W: torch.Tensor) -> float:
    return float(((got.double() - A.double() @ W.double()).abs() / bound(A, W)).max())


@pytest.mark.parametrize("K,N", SHAPES)
def test_bound_accepts_fp32_accumulated_split_with_margin(K, N):
    g = torch.Generator().manual_seed(K * 1000 + N)
    A, W = torch.randn(256, K, generator=g), torch.randn(K, N, generator=g)
    ah, al = split16(A)
    wh, wl = split16(W)
    got = (ah @ wh + ah @ wl) + al @ wh                # three fp32-accumulated passes
    assert _ratio(got, A, W) <= 0.5


@pytest.mark.parametrize("K,N", SHAPES)
def test_bound_rejects_broken_split_kernels(K, N):
    """A kernel that drops the lo*hi or the hi*lo pass, or uses the hi halves only, exceeds the bound by far (> 20x) at operand
    scale 1.  Not listed: rounding lo toward zero instead of to nearest.  It doubles only the split's representation error
    (~2^-22 |a||w| per term), which stays below the fp32 accumulation term from K = 36 up, so no tolerance that admits fp32
    accumulation can reject it."""
    g = torch.Generator().manual_seed(K * 1000 + N)
    A, W = torch.randn(256, K, generator=g), torch.randn(K, N, generator=g)
    for name, got in _mutants(A, W).items():
        assert _ratio(got, A, W) > 20.0, name


def test_pow2_row_scale_edges():
    """Zero, subnormal, tiny, ordinary, near-fp32-max, inf and NaN rows: every scale is a finite power of two whose reciprocal is
    normal, every finite row's max lands in [2^12, 2^13) unless the shift is clamped, zero rows stay zero and non-finite rows stay
    non-finite."""
    fmax, tiny = torch.finfo(torch.float32).max, torch.finfo(torch.float32).tiny
    rows = torch.tensor([[0.0, 0.0, 0.0, 0.0],
                         [1e-45, -3e-45, 0.0, 1e-45],          # subnormal
                         [tiny, -2 * tiny, 0.0, tiny],
                         [1e-30, 3e-31, -2e-30, 0.0],
                         [1.0, -0.5, 0.25, 0.0],
                         [4096.0, 8191.0, -1.0, 2.0],
                         [-8192.0, 1.0, 0.0, 0.0],
                         [fmax, -fmax / 3, 1.0, 0.0],
                         [float("inf"), 1.0, 2.0, 3.0],
                         [1.0, float("nan"), 2.0, 3.0]], dtype=torch.float32)
    s = ops.pow2_row_scale(rows)
    assert s.dtype == torch.float32 and s.shape == (rows.size(0),)
    m, e = torch.frexp(s)
    assert torch.isfinite(s).all() and (m == 0.5).all()                     # powers of two ...
    assert (e - 1).min() >= -126 and (e - 1).max() <= 126                    # ... with normal reciprocals
    assert torch.equal((1.0 / s) * s, torch.ones_like(s))
    scaled = rows * s[:, None]
    amax = scaled.abs().amax(1)
    shift = (e - 1).double()
    for r in range(rows.size(0)):
        if not torch.isfinite(rows[r]).all():
            assert not torch.isfinite(scaled[r]).all()
        elif rows[r].abs().max() == 0:
            assert (scaled[r] == 0).all()
        elif abs(shift[r]) < 126:
            assert 2.0 ** 12 <= amax[r] < 2.0 ** 13, (r, float(amax[r]))
        else:                                                                # clamped: as close to the range as fp32 allows
            assert amax[r] < 2.0 ** 13 and shift[r] == 126
    assert torch.equal(rows[5:7] * s[5:7, None] / s[5:7, None], rows[5:7])    # scaling is exact


# ---- GPU: the split GEMM entry points against float64 -------------------------------------------------------------------------------
def _operand(M, K, scale, g):
    """Rows of magnitude `scale` (uniform in (-scale, scale), so 2^15 rows stay below 65520); scale=None mixes every A_SCALES scale
    row by row in one matrix."""
    u = torch.rand(M, K, generator=g) * 2 - 1
    if scale is None:
        s = torch.tensor(A_SCALES)[torch.arange(M) % len(A_SCALES)]
        return u * s[:, None]
    return u * scale


def _assert_within(got, want, tol, what):
    err = (got.double().cpu() - want).abs()
    bad = ~(err <= tol)
    assert not bad.any(), f"{what}: {int(bad.sum())} elements out of bound, worst err/bound {float((err / tol).max()):.3g}"


@pytest.mark.gpu
@pytest.mark.parametrize("K,N", [(4, 32), (36, 96), (384, 256)])
@pytest.mark.parametrize("a_scale", A_SCALES + [None], ids=[f"a2^{int(math.log2(s))}" for s in A_SCALES] + ["mixed"])
def test_gemm_split_vs_fp64_across_scales(K, N, a_scale):
    """stmp_gemm_f32 with and without bias, into a strided column block, M = 300 (not a multiple of the 128-row tile).  The 2^-20
    rows have fp16-subnormal hi and lo halves: passing the bound built from `split16` (which keeps subnormals) shows the tensor core
    does not flush them."""
    g = torch.Generator().manual_seed(K + N)
    M = 300
    A = _operand(M, K, a_scale, g)
    for w_scale in W_SCALES:
        W = torch.randn(K, N, generator=g) * w_scale
        bias = torch.randn(N, generator=g) * w_scale
        exact = A.double() @ W.double()
        tol = bound(A, W)
        packed = ops.gemm_prepack(W.to(DEV))
        Ad = A.to(DEV)
        _assert_within(ops.gemm(Ad, packed, K, N), exact, tol, f"w2^{math.log2(w_scale):.0f}")
        want_b = exact + bias.double()
        _assert_within(ops.gemm(Ad, packed, K, N, bias.to(DEV)), want_b, tol + 2.0 ** -24 * want_b.abs(), "bias")
        wide = torch.full((M, N + 64), float("nan"), device=DEV)
        ops.gemm(Ad, packed, K, N, bias.to(DEV), out=wide[:, 32:32 + N])
        _assert_within(wide[:, 32:32 + N], want_b, tol + 2.0 ** -24 * want_b.abs(), "out= column block")
        assert torch.isnan(wide[:, :32]).all() and torch.isnan(wide[:, 32 + N:]).all()


def _lstm_gates64(pre, C, wci, wcf, wco, bi, bf, bc, bo):
    Co = C.size(1)
    pi, pf, pc, po = (pre[:, j * Co:(j + 1) * Co] for j in range(4))
    I, Fg = torch.sigmoid(pi + wci * C + bi), torch.sigmoid(pf + wcf * C + bf)
    Cn = Fg * C + I * torch.tanh(pc + bc)
    return torch.sigmoid(po + wco * Cn + bo) * torch.tanh(Cn), Cn


@pytest.mark.gpu
@pytest.mark.parametrize("K,Co", [(384, 64), (128, 32)])
@pytest.mark.parametrize("a_scale", A_SCALES + [None], ids=[f"a2^{int(math.log2(s))}" for s in A_SCALES] + ["mixed"])
def test_gemm_lstm_split_vs_fp64_across_scales(K, Co, a_scale):
    """stmp_gemm_lstm_f32: the fp64 peephole gate chain on the exact pre-activations.  Sigmoid and tanh are 1-Lipschitz, so a
    pre-activation error e moves C' by at most (|C|/4 + 5/4) e and H' by at most e/4 + (1 + |w_co|/4) of C''s; plus a few fp32 ulps of
    gate rounding."""
    g = torch.Generator().manual_seed(K + Co)
    M = 333
    A = _operand(M, K, a_scale, g)
    for w_scale in W_SCALES:
        W = torch.randn(K, 4 * Co, generator=g) * w_scale
        cb = torch.randn(4 * Co, generator=g) * 0.5
        C = torch.randn(M, Co, generator=g)
        peep = [torch.randn(Co, generator=g) * 0.5 for _ in range(3)]
        gb = [torch.randn(Co, generator=g) * 0.5 for _ in range(4)]
        pre = A.double() @ W.double() + cb.double()
        e = bound(A, W) + 2.0 ** -24 * pre.abs()
        e = torch.stack([e[:, j * Co:(j + 1) * Co] for j in range(4)]).amax(0)       # worst gate per (row, channel)
        H64, C64 = _lstm_gates64(pre, C.double(), *(t.double() for t in peep + gb))
        tol_c = (C.double().abs() / 4 + 1.25) * e + 8 * 2.0 ** -24 * (1 + C.double().abs() + C64.abs())
        tol_h = e / 4 + (1 + peep[2].double().abs() / 4) * tol_c + 8 * 2.0 ** -24
        d = lambda t: t.to(DEV)
        h, c = ops.gemm_lstm(d(A), ops.gemm_prepack(d(W)), K, Co, d(cb), d(C), *(d(t) for t in peep + gb))
        _assert_within(c, C64, tol_c, f"C' w2^{math.log2(w_scale):.0f}")
        _assert_within(h, H64, tol_h, f"H' w2^{math.log2(w_scale):.0f}")


@pytest.mark.gpu
@pytest.mark.parametrize("a_scale", A_SCALES + [None], ids=[f"a2^{int(math.log2(s))}" for s in A_SCALES] + ["mixed"])
def test_gemm_blocks_split_vs_fp64_across_scales(a_scale):
    """stmp_gemm_blocks_f32: blocks X[t-1] | X[t] | X[t+1] (row shifts -1, 0, +1 inside sequences of 12, zero outside) with the bias,
    ReLU and ReLU + LayerNorm epilogues.  LayerNorm is checked after normalisation against fp64 LN of the fp64 product: a
    pre-LN error e moves the normalised value z by at most (2 + |z|) max(e) / std of the row."""
    g = torch.Generator().manual_seed(7)
    B, T, Cc, N = 25, 12, 64, 64                                   # 300 rows
    M = B * T
    X = _operand(M, Cc, a_scale, g)
    Xs = X.view(B, T, Cc)
    z = torch.zeros(B, 1, Cc)
    A = torch.cat([torch.cat([z, Xs[:, :-1]], 1), Xs, torch.cat([Xs[:, 1:], z], 1)], 2).reshape(M, 3 * Cc)   # the gathered operand
    for w_scale in W_SCALES:
        Wb = [torch.randn(Cc, N, generator=g) * w_scale for _ in range(3)]
        W = torch.cat(Wb, 0)
        bias = torch.randn(N, generator=g) * w_scale * (float(X.abs().max()) + 1e-30) ** 0.5
        gamma, beta = torch.rand(N, generator=g) + 0.5, torch.randn(N, generator=g)
        pre = A.double() @ W.double() + bias.double()
        e = bound(A, W) + 2.0 ** -24 * pre.abs()
        packed = ops.gemm_blocks_prepack([w.to(DEV) for w in Wb])
        xd = X.to(DEV)
        blocks = [(xd, Cc, -1), (xd, Cc, 0), (xd, Cc, 1)]
        _assert_within(ops.gemm_blocks(blocks, packed, N, N, bias.to(DEV), ops.EPI_BIAS, seq=T), pre, e, "bias")
        _assert_within(ops.gemm_blocks(blocks, packed, N, N, bias.to(DEV), ops.EPI_RELU, seq=T), pre.clamp(min=0), e, "relu")
        r = pre.clamp(min=0)
        mu, var = r.mean(1, keepdim=True), r.var(1, unbiased=False, keepdim=True)
        sd = (var + 1e-5).sqrt()
        zn = (r - mu) / sd
        want = zn * gamma.double() + beta.double()
        tol = gamma.double() * (2 + zn.abs()) * e.amax(1, keepdim=True) / sd + 256 * 2.0 ** -24 * (gamma.double() * (1 + zn.abs()) + beta.double().abs())
        got = ops.gemm_blocks(blocks, packed, N, N, bias.to(DEV), ops.EPI_RELU_LN, gamma.to(DEV), beta.to(DEV), 1e-5, seq=T)
        _assert_within(got, want, tol, f"relu+LN w2^{math.log2(w_scale):.0f}")


@pytest.mark.gpu
@pytest.mark.parametrize("x_exp", [-8, -4, 0, 6, 10])
def test_dcrnn_fused_forward_across_input_scales(x_exp):
    """The tcgen05 DCRNN sequence kernel (split X and H operands) with inputs scaled by 2^-8 .. 2^10 (raw METR-LA speeds reach ~2^6)
    against the FFMA fp32 kernel and the float64 oracle, at rtol 1e-4 / atol 1e-5 of the output's magnitude up to 2^6."""
    ei, ew, _ = synthetic.metr_la_like(0, 16)
    ei_t, ew_t = torch.from_numpy(ei), torch.from_numpy(ew)
    torch.manual_seed(x_exp + 100)
    from pytorch_geometric_temporal_b200.nn.recurrent import BatchedDCRNN
    m = BatchedDCRNN(2, 32, 2)
    for p in m.parameters():
        if p.dim() == 1:
            torch.nn.init.uniform_(p, -0.5, 0.5)
    X = torch.randn(3, 12, 207, 2) * 2.0 ** x_exp
    sd64 = {k: v.double() for k, v in m.state_dict().items()}
    want = R.batched_dcrnn(sd64, X.double(), ei_t, ew_t)
    assert want.dtype == torch.float64
    mg = m.to(DEV)
    try:
        with torch.no_grad():
            _lib.set_option("dcrnn_tc", 1)
            c0 = _lib.path_counters()
            out_tc = mg(X.to(DEV), ei_t.to(DEV), ew_t.to(DEV))
            assert _lib.path_counters().get("k_dcrnn_seq_tc", 0) == c0.get("k_dcrnn_seq_tc", 0) + 1
            _lib.set_option("dcrnn_tc", 0)
            out_ff = mg(X.to(DEV), ei_t.to(DEV), ew_t.to(DEV))
    finally:
        _lib.set_option("dcrnn_tc", 1)
    scale = float(want.abs().max())
    if x_exp > 6:
        # beyond the raw-speed range the pre-activations reach ~2^14: even exact fp32 arithmetic (the FFMA kernel) is off by more
        # than 1e-5 of the gated output, and the split kernel by more again (B200: 1.4e-4 vs 2.1e-5 at 2^10).  Pinned, not strict.
        err_tc, err_ff = (float((o.double().cpu() - want).abs().max()) for o in (out_tc, out_ff))
        assert err_ff <= 2e-4 * scale and err_tc <= 1e-3 * scale, (err_tc, err_ff)
    else:
        for got in (out_tc, out_ff):
            _assert_within(got, want, 1e-4 * want.abs() + 1e-5 * scale, "vs fp64 oracle")
        _assert_within(out_tc, out_ff.double().cpu(), 1e-4 * out_ff.double().abs().cpu() + 1e-5 * scale, "tc vs ffma")


# ---- GPU: power-of-two row scaling of gradient operands -----------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("N", [192, 384])
def test_gemm_row_scaled_gradient_operand_vs_fp64(N):
    """dS = dpre @ W^T as the GConvLSTM backward runs it (M = 20 000, K = 256, two column halves of N/2) with rows from 2^-40 to
    2^14 mixed in one launch, zero rows and one NaN row.  Each row is held to the bound of its scaled copy, scaled back: the error
    is relative to the row, whatever its magnitude.  The NaN row stays NaN and does not reach other rows."""
    g = torch.Generator().manual_seed(N)
    M, K = 20000, 256
    exps = torch.linspace(-40, 14, M, dtype=torch.float64)[torch.randperm(M, generator=g)]
    A = (torch.randn(M, K, generator=g).double() * torch.pow(2.0, exps)[:, None]).float()
    A[17::997] = 0.0
    nan_row = 4242
    A[nan_row, 5] = float("nan")
    Wt = torch.randn(K, N, generator=g) * 0.1
    half = N // 2
    packs = [ops.gemm_prepack(Wt[:, j * half:(j + 1) * half].contiguous().to(DEV)) for j in range(2)]
    Ad = A.to(DEV)
    rs = ops.pow2_row_scale(Ad)
    out = torch.empty(M, N, device=DEV)
    for j in range(2):
        ops.gemm(Ad, packs[j], K, half, out=out[:, j * half:(j + 1) * half], row_scale=rs)
    got = out.cpu()
    assert torch.isnan(got[nan_row]).all()
    keep = torch.ones(M, dtype=torch.bool)
    keep[nan_row] = False
    assert torch.isfinite(got[keep]).all()
    s = rs.cpu().double()[keep]
    As = (A[keep].double() * s[:, None]).float()                  # exact: powers of two
    assert torch.equal(As.double() / s[:, None], A[keep].double())
    tol = bound(As, Wt) / s[:, None]
    _assert_within(got[keep], A[keep].double() @ Wt.double(), tol, "row-scaled dS")
    zero = A[keep].abs().amax(1) == 0
    assert zero.any() and (got[keep][zero] == 0).all()


def _gconv_lstm_setup(Ci, Co, K):
    from pytorch_geometric_temporal_b200.nn.recurrent import GConvLSTM
    ei, ew = synthetic.large_graph(2000, 20000, 1)
    ei, ew = torch.from_numpy(ei), torch.from_numpy(ew)
    torch.manual_seed(Ci + Co + K)
    m = GConvLSTM(Ci, Co, K)
    for p in m.parameters():                                    # non-zero biases and peepholes
        if p.dim() == 1 or p.size(0) == 1:
            torch.nn.init.normal_(p, std=0.2)
    head = torch.nn.Linear(Co, 8)
    X = torch.randn(6, 2000, Ci)
    Y = torch.randn(2000, 8)
    return m, head, X, Y, ei, ew


def _gconv_lstm_grads(m, head, X, Y, ei, ew, loss_scale=1.0):
    """X.grad and every parameter gradient (cell + head) of a 6-step unroll under the MEAN squared error of a linear head."""
    X = X.clone().requires_grad_(True)
    H = C = None
    for t in range(X.size(0)):
        H, C = m(X[t], ei, ew, H, C)
    loss = torch.nn.functional.mse_loss(head(H), Y) * loss_scale
    loss.backward()
    grads = {"X": X.grad}
    grads.update({k: p.grad.clone() for k, p in list(m.named_parameters()) + [("head." + k, p) for k, p in head.named_parameters()]})
    for p in list(m.parameters()) + list(head.parameters()):
        p.grad = None
    return grads


@pytest.mark.gpu
@pytest.mark.parametrize("Ci,Co,K", [(64, 64, 3), (32, 32, 2), (32, 64, 2)])
def test_gconv_lstm_fused_backward_mean_loss_vs_fp64(Ci, Co, K):
    """The hand-written cell backward (_LstmCellFn) under a mean loss, where the gate gradients dpre are ~1e-6: X.grad and every
    parameter gradient against the float64 CPU oracle's autograd and against the op-for-op path, to 1e-3 of the largest reference
    gradient.  Without the row scaling of dpre, most of dS = dpre @ W^T is lost in fp16 subnormals."""
    m, head, X, Y, ei, ew = _gconv_lstm_setup(Ci, Co, K)
    p64 = {k: v.double().requires_grad_(True) for k, v in m.state_dict().items()}
    h64 = torch.nn.Linear(Co, 8).double()
    h64.load_state_dict({k: v.double() for k, v in head.state_dict().items()})
    x64 = X.double().requires_grad_(True)
    H = C = torch.zeros(2000, Co, dtype=torch.float64)
    for t in range(6):
        H, C = R.gconv_lstm_cell(p64, x64[t], ei, ew.double(), H, C)
    torch.nn.functional.mse_loss(h64(H), Y.double()).backward()
    ref = {"X": x64.grad}
    ref.update({k: p64[k].grad for k in p64})
    ref.update({"head." + k: p.grad for k, p in h64.named_parameters()})

    md, hd = m.to(DEV), head.to(DEV)
    args = (X.to(DEV), Y.to(DEV), ei.to(DEV), ew.to(DEV))
    c0 = _lib.path_counters()
    fused = _gconv_lstm_grads(md, hd, *args)
    assert _lib.path_counters().get("k_lstm_gate_bwd", 0) - c0.get("k_lstm_gate_bwd", 0) == 6
    md.fused_training = False
    plain = _gconv_lstm_grads(md, hd, *args)
    for k, want in ref.items():
        tol = 1e-3 * float(want.abs().max())
        for name, got in (("fused", fused[k]), ("op-for-op", plain[k])):
            err = float((got.double().cpu() - want).abs().max())
            assert err <= tol, f"{name} {k}: max err {err:.3e} > {tol:.3e}"


# ---- GPU: every hand-written backward is equivariant under power-of-two loss scaling ---------------------------------------------------
def _equivariant(grads_of, what):
    """grads_of(scale) -> {name: gradient}.  g(2^k L) 2^-k must equal g(L) for k = -20 and 16 (a mean loss over 10^6 terms, an AMP loss
    scale); exact equality is expected -- every operation involved commutes with power-of-two scaling."""
    base = grads_of(1.0)
    exact = True
    for k in (-20, 16):
        got = grads_of(2.0 ** k)
        for name, g0 in base.items():
            g1 = got[name] * 2.0 ** -k
            assert torch.isfinite(g1).all(), f"{what} k={k} {name}: non-finite gradient"
            err = float((g1 - g0).abs().max())
            assert err <= 1e-6 * float(g0.abs().max()), f"{what} k={k} {name}: max err {err:.3e} vs max|g| {float(g0.abs().max()):.3e}"
            exact = exact and torch.equal(g1, g0)
    print(f"loss-scale equivariance of {what}: {'bit-exact' if exact else 'within 1e-6, not bit-exact'}")


@pytest.mark.gpu
def test_loss_scale_equivariance_gconv_lstm_cell_backward():
    m, head, X, Y, ei, ew = _gconv_lstm_setup(64, 64, 3)
    md, hd = m.to(DEV), head.to(DEV)
    Xd, ed, wd = X.to(DEV), ei.to(DEV), ew.to(DEV)
    wt = torch.linspace(-1, 1, 2000 * 64, device=DEV).view(2000, 64)

    def grads(scale):
        x = Xd.clone().requires_grad_(True)
        H = C = None
        loss = 0
        for t in range(6):
            H, C = md(x[t], ed, wd, H, C)
            loss = loss + (H * wt).sum() + 0.3 * C.square().sum()          # O(1) gate gradients: 2^16 of them pass 65504
        c0 = _lib.path_counters()
        (loss * scale).backward()
        assert _lib.path_counters().get("k_lstm_gate_bwd", 0) - c0.get("k_lstm_gate_bwd", 0) == 6
        out = {"X": x.grad}
        out.update({k: p.grad.clone() for k, p in md.named_parameters()})
        md.zero_grad(set_to_none=True)
        return out
    _equivariant(grads, "GConvLSTM _LstmCellFn")


@pytest.mark.gpu
def test_loss_scale_equivariance_dcrnn_fused_training():
    from pytorch_geometric_temporal_b200.nn.recurrent import BatchedDCRNN
    ei, ew, series = synthetic.metr_la_like(2, 64)
    ed, wd = torch.from_numpy(ei).to(DEV), torch.from_numpy(ew).to(DEV)
    X = torch.from_numpy(series[:48]).reshape(4, 12, 207, 2).to(DEV)
    torch.manual_seed(2)
    m = BatchedDCRNN(2, 32, 2).to(DEV)
    w = torch.randn(4, 12, 207, 32, device=DEV)

    def grads(scale):
        x = X.clone().requires_grad_(True)
        c0 = _lib.path_counters()
        ((m(x, ed, wd) * w).sum() * scale).backward()
        c1 = _lib.path_counters()
        assert c1.get("k_dcrnn_seq_tc", 0) > c0.get("k_dcrnn_seq_tc", 0) and c1.get("k_dcrnn_bwd_seq", 0) > c0.get("k_dcrnn_bwd_seq", 0)
        out = {"X": x.grad}
        out.update({k: p.grad.clone() for k, p in m.named_parameters()})
        m.zero_grad(set_to_none=True)
        return out
    _equivariant(grads, "DCRNN fused forward + persistent backward")


@pytest.mark.gpu
def test_loss_scale_equivariance_a3tgcn2_fused_training():
    from pytorch_geometric_temporal_b200.nn.recurrent import A3TGCN2
    ei, ew, _ = synthetic.pems_bay_like(0, 16)
    ed, wd = torch.from_numpy(ei).to(DEV), torch.from_numpy(ew).to(DEV)
    torch.manual_seed(3)
    m = A3TGCN2(2, 32, 12, 8).to(DEV)
    X = torch.randn(8, 325, 2, 12, device=DEV)
    w = torch.randn(8, 325, 32, device=DEV)

    def grads(scale):
        c0 = _lib.path_counters()
        ((m(X, ed, wd) * w).sum() * scale).backward()
        assert _lib.path_counters().get("k_tgcn_attn_bwd", 0) == c0.get("k_tgcn_attn_bwd", 0) + 1
        out = {k: p.grad.clone() for k, p in m.named_parameters()}
        m.zero_grad(set_to_none=True)
        return out
    _equivariant(grads, "A3TGCN2 tgcn_attn_train")


@pytest.mark.gpu
def test_loss_scale_equivariance_masked_mae():
    from pytorch_geometric_temporal_b200 import distributed as D
    g = torch.Generator(device=DEV).manual_seed(4)
    y = torch.randn(8, 10000, 8, device=DEV, generator=g)
    y[torch.rand(y.shape, device=DEV, generator=g) < 0.1] = 0.0
    p = torch.randn(y.shape, device=DEV, generator=g)

    def grads(scale):
        q = p.clone().requires_grad_(True)
        (D.masked_mae_loss(q, y) * scale).backward()
        return {"pred": q.grad}
    _equivariant(grads, "masked_mae")

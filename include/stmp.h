/*
 * stmp.h -- C ABI of libstmp.so, the sm_100a spatiotemporal message-passing engine.
 *
 * The reference (benedekrozemberczki/pytorch_geometric_temporal @ adefe44) is pure Python and has no
 * FFI layer: its hot path is `torch.nn.Module.forward` -> torch_geometric `MessagePassing.propagate`
 * (index_select + scatter_add_) + ATen matmul/pointwise.  This header is therefore the boundary a
 * maintainer would bind with ctypes from those modules (INTEGRATION.md shows the stub).  Each entry
 * point cites the reference code it replaces, relative to /root/reference/torch_geometric_temporal/.
 *
 * Conventions
 *  - plain C types only; all data pointers are DEVICE pointers unless a name ends in `_host`;
 *  - tensors are fp32, row-major, indices int64 on input (torch LongTensor) and int32 inside a plan;
 *  - every call enqueues on the caller's `stream` (a cudaStream_t passed as void*), never
 *    synchronises the device and never allocates, except stmp_plan_create/destroy/export (setup path);
 *  - return value: 0 = STMP_OK, otherwise an stmp_status code; the message is available from
 *    stmp_last_error() (thread-local);
 *  - entry points are re-entrant (autograd / DDP call backward from worker threads); a plan is
 *    immutable after creation.
 */
#ifndef STMP_H_
#define STMP_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct stmp_plan stmp_plan;

enum stmp_status {
  STMP_OK = 0,
  STMP_EINVAL = 1,       /* bad argument (null pointer, negative size, unknown enum)  -> ValueError   */
  STMP_ESHAPE = 2,       /* shape/stride/alignment the kernels cannot take            -> RuntimeError */
  STMP_EGRAPH = 3,       /* edge_index out of range / duplicate edges where the reference would fail */
  STMP_ECUDA = 4,        /* CUDA runtime error (message carries cudaGetErrorString)                   */
  STMP_EUNSUPPORTED = 5, /* configuration does not fit the fused kernel; caller must use the tiled path */
  STMP_ENOMEM = 6
};

/* Which normalised operator(s) a plan holds. */
enum stmp_flavor {
  /* DConv / BatchedDConv (nn/recurrent/dcrnn.py:59-77, :277-290): two operators,
   *   op 0 "out": dst=col[e], src=row[e], val = 1/deg_out[row[e]]
   *   op 1 "in" : p-th entry of the (col,row)-sorted reverse list: dst=row[q_p], src=col[q_p],
   *               val = 1/deg_in[row[p]]   (positional pairing, quirk preserved)
   * degrees are weighted sums; messages never multiply by edge_weight. */
  STMP_FLAVOR_DCONV = 0,
  /* PyG ChebConv.__norm__ (used by gconv_gru.py:57-107, gconv_lstm.py:62-138): scaled Laplacian
   *   2L/lambda_max - I, self-loop entries appended after the non-loop edges. */
  STMP_FLAVOR_CHEB = 1,
  /* PyG gcn_norm (used by temporalgcn.py:38-68,162-173): D^-1/2 (A+I) D^-1/2 with remaining self loops. */
  STMP_FLAVOR_GCN = 2,
  /* ChebConvAttention.__norm__ (nn/attention/astgcn.py:82-110), propagated on the TRANSPOSED index
   * (:167): dst=row', src=col', E'+2N entries. */
  STMP_FLAVOR_CHEB_ATT = 3
};

enum stmp_norm { STMP_NORM_NONE = 0, STMP_NORM_SYM = 1, STMP_NORM_RW = 2 };

enum stmp_plan_flags {
  STMP_GCN_IMPROVED = 1u << 0,      /* GCNConv(improved=True): self-loop fill 2 instead of 1 */
  STMP_GCN_NO_SELF_LOOPS = 1u << 1, /* GCNConv(add_self_loops=False) */
  STMP_DCONV_ALLOW_DUPLICATES = 1u << 2 /* BatchedDConv semantics (scatter degrees, no dense adjacency):
                                           duplicate edges are legal; DConv proper raises on them */
};

/* ---- plan ------------------------------------------------------------------------------------ */

/* Build the cached operator(s) for a static graph on the device (stable radix sort to CSR by
 * destination + CSR by source for the transposed/backward product, degree/Laplacian/GCN norms).
 * Replaces the per-call renormalisation of dcrnn.py:59-77, PyG get_laplacian / gcn_norm and
 * astgcn.py:82-110.  edge_index: int64 [2,E] row-major; edge_weight: [E] or NULL (=> ones).
 * lambda_max: >0 to use it, <=0 / NaN => PyG default (CHEB: 2*max(w_hat); CHEB_ATT: 2.0).
 * Setup path: allocates, and synchronises `stream` once to read validation flags. */
int stmp_plan_create(int flavor, int64_t num_nodes, int64_t num_edges, const int64_t* edge_index,
                     const float* edge_weight, int normalization, float lambda_max, uint32_t flags,
                     void* stream, stmp_plan** out);
/* Multi-graph mini-batches (StaticGraphTemporalSignalBatch; PyG ChebConv `lambda_max[batch[edge_index[0]]]`, and
 * ChebConvAttention.__norm__, astgcn.py:98-99; exercised by the reference's test/attention_test.py:205-218): the scaling
 * 2 w / lambda uses the lambda_max of the entry's ROW node.  lambda_node: device float [num_nodes] = lambda_max[batch].
 * Flavors CHEB and CHEB_ATT only. */
int stmp_plan_create_pergraph(int flavor, int64_t num_nodes, int64_t num_edges, const int64_t* edge_index,
                              const float* edge_weight, int normalization, const float* lambda_node, uint32_t flags,
                              void* stream, stmp_plan** out);
void stmp_plan_destroy(stmp_plan* plan);

/* Introspection (tests, bit-exact index parity): number of operators, nodes, entries of operator `op`. */
int stmp_plan_num_ops(const stmp_plan* plan);
int64_t stmp_plan_num_nodes(const stmp_plan* plan);
int64_t stmp_plan_nnz(const stmp_plan* plan, int op);
/* Copy operator `op` (transposed=0: CSR by destination; 1: CSR by source) into caller device buffers:
 * rowptr[N+1], col[nnz], val[nnz], eid[nnz] (eid = position of the entry in the reference-order
 * COO list, i.e. the order the reference's scatter_add_ visits it).  Any output may be NULL. */
int stmp_plan_export(const stmp_plan* plan, int op, int transposed, int32_t* rowptr, int32_t* col,
                     float* val, int32_t* eid, void* stream);

/* ---- K1/K3: gather -> weighted scatter-add (SpMM) with fused Chebyshev axpby -------------------
 * y[b,i,:] = alpha * sum_k val_k * x[b, col_k, :] + beta * z[b,i,:]        (z may be NULL)
 * Replaces MessagePassing.propagate (x_j = index_select; norm*x_j; scatter_add_) at
 * dcrnn.py:86-87,95-99,300-313, astgcn.py:169-175 and inside ChebConv/GCNConv, plus the
 * `2*prop - T0` recurrence (dcrnn.py:96,100; astgcn.py:176).  Per destination the products are summed
 * in the reference's edge order with separate multiply and add (no FMA), so results are bit-identical
 * to the CPU scatter_add_ path.  x,y,z: [batch, N, f] with row strides ld* and batch strides bs*
 * (elements).  att (nullable): [batch, N, N] spatial attention; the entry value becomes
 * val * att[b, dst, src] (astgcn.py:156-157, first hop only).  transposed=1 applies A^T (backward). */
int stmp_spmm(const stmp_plan* plan, int op, int transposed, int64_t batch, int64_t f,
              const float* x, int64_t ldx, int64_t bsx, float* y, int64_t ldy, int64_t bsy,
              float alpha, const float* z, int64_t ldz, int64_t bsz, float beta,
              const float* att, void* stream);

/* The forward product with the attention handed in TRANSPOSED and row-padded: entry (dst, src) uses attT[b, src, dst], rows att_ld
 * floats apart (the layout stmp_spatial_attention_fwd writes: softmax over dim 1 of S is a row softmax of S^T). */
int stmp_spmm_att_t(const stmp_plan* plan, int op, int64_t batch, int64_t f, const float* x, int64_t ldx, int64_t bsx, float* y,
                   int64_t ldy, int64_t bsy, float alpha, const float* z, int64_t ldz, int64_t bsz, float beta, const float* attT,
                   int64_t att_ld, void* stream);

/* d(att)[b,dst,src] += val * <gy[b,dst,:], x[b,src,:]> for every entry of `op` (backward of the
 * attention-weighted first hop, astgcn.py:156-170).  datt must be zero-initialised by the caller. */
int stmp_spmm_att_grad(const stmp_plan* plan, int op, int64_t batch, int64_t f, const float* gy,
                       int64_t ldg, int64_t bsg, const float* x, int64_t ldx, int64_t bsx, float* datt,
                       void* stream);

/* ---- K1-K5 fused: the DCRNN recurrence ---------------------------------------------------------
 * For each window b: H_0 = h0[b] (or 0); for t in [0,T): H_t = DCRNN_cell(X[b,t], H_{t-1});
 * out[b,t] = H_t.  One persistent CTA per window keeps graph, weights, [X|H] and both diffusion
 * products in shared memory across all T steps.  Replaces BatchedDCRNN.forward (dcrnn.py:429-475)
 * and, with B=T=1, DCRNN.forward (:194-219).  plan: STMP_FLAVOR_DCONV.
 *   x: window b, step t starts at x + (win_start ? win_start[b] : b*x_bstride) ... see x_tstride:
 *      addr = x + base_b + t*x_tstride, base_b = win_start ? win_start[b]*x_tstride : b*x_bstride
 *      (win_start: int64 [B] device, index-batching over a resident series, signal/index_dataset.py:49-57)
 *   w_z,w_r,w_h: DConv.weight [2,K,cin+cout,cout]; b_*: [cout] or NULL (dcrnn.py:26-37)
 *   h0: [B,N,cout] or NULL; out: [B,T,N,cout]
 *   stash (nullable): [B,T,3,N,cout] receives (Z,R,Htilde) per step for the backward pass.
 * Returns STMP_EUNSUPPORTED when (N, nnz, cin, cout, K) do not fit the fused kernel. */
int stmp_dcrnn_seq_fwd(const stmp_plan* plan, int64_t B, int64_t T, int64_t cin, int64_t cout, int64_t K,
                       const float* x, const int64_t* win_start, int64_t x_bstride, int64_t x_tstride,
                       const float* w_z, const float* w_r, const float* w_h, const float* b_z,
                       const float* b_r, const float* b_h, const float* h0, float* out, float* stash,
                       const void* wimage, void* workspace, void* stream);
/* 1 if stmp_dcrnn_seq_fwd can take this configuration on the current device, else 0. */
int stmp_dcrnn_seq_supported(const stmp_plan* plan, int64_t cin, int64_t cout, int64_t K);

/* Generic fused graph-GRU recurrence on the tensor cores (tcgen05, fp16 hi/lo operand split = fp32-class accuracy):
 *   pre_g = [H' | Op0 H' | Op1 H' | X | Op0 X | Op1 X] @ wcat_g^T + bcat_g      g in {z, r, h};  H' = H (z, r) or H*R (h)
 *   Z = sigmoid(pre_z); R = sigmoid(pre_r); Ht = tanh(pre_h); H_t = Z*H + (1-Z)*Ht
 * with the first `n_ops` (0..2) operators of `plan` (any flavor).  This one kernel serves DCRNN K=2 (DConv plan, 2 ops),
 * GConvGRU K<=2 (gconv_gru.py:119-139; CHEB plan, 1 op) and TGCN / A3TGCN(2) (temporalgcn.py:82-102; GCN plan, 1 op:
 * the GCNConv weight and the gate Linear are folded into wcat on the host side).  Cout = 32, cin <= 4, N <= 207.
 *   wcat: [96][112] fp32, row = gate*32 + out channel, columns = H(32) | Op0 H(32) | Op1 H(32) | X(4) | Op0 X(4) | Op1 X(4) | 0(4)
 *   bcat: [96];  h0: [B,N,32] (h0_bstride = N*32), one shared [N,32] (h0_bstride = 0) or NULL (zeros)
 * x / win_start / strides / out / stash as stmp_dcrnn_seq_fwd.  STMP_EUNSUPPORTED outside the envelope. */
int stmp_gru_seq_fwd(const stmp_plan* plan, int n_ops, int64_t B, int64_t T, int64_t cin, const float* x,
                     const int64_t* win_start, int64_t x_bstride, int64_t x_tstride, const float* wcat,
                     const float* bcat, const float* h0, int64_t h0_bstride, float* out, float* stash,
                     const void* wimage, void* workspace, void* stream);
/* Optional weight image for the tcgen05 kernel: the B operand (fp16 hi/lo halves, SWIZZLE_128B, + biases) exactly as the kernel
 * holds it in shared memory, so every CTA fetches it with one TMA bulk copy instead of converting the fp32 weights itself.
 * Build it once per weight update into a device buffer of stmp_gru_weight_image_bytes() bytes and pass it as `wimage`
 * (NULL => the kernel converts in place).  The plan carries the analogous graph image. */
int64_t stmp_gru_weight_image_bytes(void);
/* Optional workspace of the tcgen05 kernel (both entries): stmp_seq_workspace_bytes(plan, T, cin) bytes of device memory, reusable across
 * calls on one stream.  The window prologue parks P_o X_t / P_i X_t of all steps there (per-CTA rows, rewritten every window => L2-resident,
 * full-sector stores).  NULL => they are parked in the window's own not-yet-written output rows instead (same results; partial-sector
 * writes cost extra DRAM traffic: 1.7x the algorithmic bytes measured). */
int64_t stmp_seq_workspace_bytes(const stmp_plan* plan, int64_t T, int64_t cin);
int stmp_dcrnn_pack_weights(int64_t cin, int64_t cout, int64_t K, const float* w_z, const float* w_r, const float* w_h,
                            const float* b_z, const float* b_r, const float* b_h, void* image, void* stream);
int stmp_gru_pack_weights(const float* wcat, const float* bcat, void* image, void* stream);
int stmp_gru_seq_supported(const stmp_plan* plan, int n_ops, int64_t cin, int64_t cout);

/* ---- fused temporal-attention + GCN-GRU: A3TGCN / A3TGCN2 (attentiontemporalgcn.py:51-79,130-157) and, with periods = 1 and
 * probs = NULL, a TGCN / TGCN2 cell (temporalgcn.py:104-130,212-233) -- graphs of any size, out_channels = 32.
 *   out[b,n,:] = sum_t probs[t] * GRU(A^ X[b,:,:,t], H[b])        A^ = operator 0 of `plan` (GCN flavor: gcn_norm)
 * with GCNConv's Linear and the gate Linear folded on the host:  pre_g = (A^X_t) A[:, g] + H' Bm[:, g] + c[g],  g in z|r|h
 *   x: [B][N][fin][periods] contiguous;  h: [B][N][32] with batch stride h_bstride (0: one state shared by all rows) or NULL (zeros)
 *   A: [fin][96], Bm: [32][96], c: [96] (columns z | r | h);  probs: [periods] = softmax(attention) or NULL;  out: [B][N][32]
 * One gather per node serves every period (A^(XW) = (A^X)W); X[b] is staged in shared memory by one TMA bulk copy per CTA.
 * STMP_EUNSUPPORTED unless fin <= 4 and fin * periods <= 128. */
int stmp_tgcn_attn_fwd(const stmp_plan* plan, int64_t B, int64_t fin, int64_t periods, const float* x, const float* h,
                       int64_t h_bstride, const float* A, const float* Bm, const float* c, const float* probs, float* out,
                       void* stream);

/* ---- K5: gate epilogues for the tiled path -------------------------------------------------------
 * GRU (dcrnn.py:172-192, gconv_gru.py:119-139, temporalgcn.py:82-102), n = number of elements:
 *   stmp_gru_zr:   z = sigmoid(pz); r = sigmoid(pr); hr = h * r
 *   stmp_gru_out:  ht = tanh(ph); hnew = z*h + (1-z)*ht
 * LSTM with peepholes (gconv_lstm.py:168-202), rows x cout, w_c*, b_* are [cout]:
 *   stmp_lstm_ifc: i = sig(pi + wci*c + bi); f = sig(pf + wcf*c + bf); t = tanh(pc + bc); cnew = f*c + i*t
 *   stmp_lstm_oh:  o = sig(po + wco*cnew + bo); hnew = o * tanh(cnew)
 */
int stmp_gru_zr(int64_t n, const float* pz, const float* pr, const float* h, float* z, float* r, float* hr,
                void* stream);
int stmp_gru_out(int64_t n, const float* ph, const float* z, const float* h, float* ht, float* hnew,
                 void* stream);
int stmp_lstm_ifc(int64_t rows, int64_t cout, const float* pi, const float* pf, const float* pc,
                  const float* c, const float* wci, const float* wcf, const float* bi, const float* bf,
                  const float* bc, float* i, float* f, float* t, float* cnew, void* stream);
int stmp_lstm_oh(int64_t rows, int64_t cout, const float* po, const float* cnew, const float* wco,
                 const float* bo, float* o, float* hnew, void* stream);

/* Backward of the peephole-LSTM gate chain (what autograd records for gconv_lstm.py:168-202): pre [rows][4*cout] = i|f|c|o pre-activations
 * of the contraction incl. the ChebConv biases, c_old / c_new [rows][cout], gh = dL/dH', gc = dL/dC' (either may be NULL = zeros)
 * -> dpre [rows][4*cout], dc_old [rows][cout].  The gates are recomputed from `pre` (nothing but S, C_{t-1}, C_t is kept by the forward). */
int stmp_lstm_gate_bwd(int64_t rows, int64_t cout, const float* pre, const float* c_old, const float* c_new, const float* gh,
                       const float* gc, const float* wci, const float* wcf, const float* wco, const float* bi, const float* bf,
                       const float* bc, const float* bo, float* dpre, float* dc_old, void* stream);

/* ---- backward of the fused DCRNN sequence (what autograd replays for dcrnn.py:429-475 / :172-219), small graphs ----
 * Served when stmp_dcrnn_bwd_supported(plan, cin, cout, K) != 0 (DCONV plan, K = 2, cout = 32, cin <= 4, graph + tiles
 * fit one SM's shared memory: N <= ~235); otherwise callers use the per-step path (stmp_gru_bwd_* + stmp_spmm).
 *   stmp_dcrnn_bwd_basis: for every (t, b) rebuild S1[t*B+b] = [U | P_o U | P_i U], U = [X_t | H_{t-1}] and S2 with
 *                         U = [X_t | H_{t-1} * R_t] (row pitch ld >= 3(cin+cout)) from x, the forward output `out`
 *                         (B,T,N,cout), h0 (nullable) and the gate stash (B,T,3,N,cout).  One launch.
 *   stmp_dcrnn_bwd_seq:   the reverse-time recurrence, one CTA per window: consumes gout (B,T,N,cout), whsT (cout, 3C),
 *                         wzrT (2cout, 3C) [transposed stacked weights]; writes d pre-activations dph_all (T,B,N,cout),
 *                         dpzr_all (T,B,N,2cout) for the weight-gradient GEMMs, dx (B,T,N,cin; nullable), dh0 (B,N,cout).
 */
int stmp_dcrnn_bwd_supported(const stmp_plan* plan, int64_t cin, int64_t cout, int64_t K);
int stmp_dcrnn_bwd_basis(const stmp_plan* plan, int64_t B, int64_t T, int64_t cin, int64_t cout, const float* x,
                         int64_t x_bstride, int64_t x_tstride, const float* out, const float* h0, const float* stash,
                         float* S1, float* S2, int64_t ld, void* stream);
int stmp_dcrnn_bwd_seq(const stmp_plan* plan, int64_t B, int64_t T, int64_t cin, int64_t cout, const float* gout,
                       const float* out, const float* h0, const float* stash, const float* whsT, const float* wzrT,
                       float* dph_all, float* dpzr_all, float* dx, float* dh0, void* stream);

/* Backward of stmp_tgcn_attn_fwd for H = NULL (the training configuration of the reference's A3TGCN2 example; what autograd records for
 * attentiontemporalgcn.py:130-157 / temporalgcn.py:187-233 over all periods): given gout (B, N, 32) it recomputes A^X and the gates and
 * reduces dA (fin, 96; the r-gate columns are zero: R multiplies H = 0), dc (96) and dprobs (periods; nullable when probs is NULL) over all
 * (batch row, node, period).  The gradients of the module parameters follow from the (differentiable, host-side) folding A = (L1 W)^T,
 * c = L1 b + l and probs = softmax(attention).  No gradient w.r.t. X.  Two launches (per-CTA partials, fixed-order reduction);
 * workspace of stmp_tgcn_attn_bwd_workspace_bytes(plan, B) bytes. */
int64_t stmp_tgcn_attn_bwd_workspace_bytes(const stmp_plan* plan, int64_t B);
int stmp_tgcn_attn_bwd(const stmp_plan* plan, int64_t B, int64_t fin, int64_t periods, const float* x, const float* A,
                       const float* c, const float* probs, const float* gout, void* workspace, float* dA, float* dc,
                       float* dprobs, void* stream);

/* Weight / bias gradients of the three DCRNN gates over all (t, b, n) rows (what autograd accumulates for the `matmul(basis, W)` and
 * `+ bias` of dcrnn.py:86-111 across steps, gates and hops): S1 / S2 (rows, ld) are stmp_dcrnn_bwd_basis' bases (ld = 3(cin+cout) rounded
 * up to 8), dpzr (rows, 2cout) / dph (rows, cout) stmp_dcrnn_bwd_seq's d pre-activations.  Writes gz / gr / gh in the module's
 * (2, K, cin+cout, cout) layout and the bias gradients (nullable).  Two launches (per-CTA partials, fixed-order reduction: deterministic);
 * the contraction runs on tcgen05 (kind::tf32, MN-major operands, TF32 hi/lo split; stmp_set_option("dcrnn_wgrad_tc", 0) selects the
 * fp32 FFMA kernel).  Workspace of stmp_dcrnn_bwd_wgrad_workspace_bytes(cin) bytes.  K = 2, cout = 32, cin <= 4. */
int64_t stmp_dcrnn_bwd_wgrad_workspace_bytes(int64_t cin);
int stmp_dcrnn_bwd_wgrad(int64_t cin, int64_t cout, int64_t K, int64_t rows, int64_t ld, const float* S1, const float* S2,
                         const float* dpzr, const float* dph, void* workspace, float* gz, float* gr, float* gh, float* gbz,
                         float* gbr, float* gbh, void* stream);

/* torch.optim.Adam's update (the optimizer of examples/indexBatching/DCRNN/pems_ddp.py:90) over ONE flat fp32 buffer of n parameters:
 * g' = grad * grad_scale (+ weight_decay * param); exp_avg.lerp(g', 1-beta1); exp_avg_sq = beta2 exp_avg_sq + (1-beta2) g'^2;
 * param -= lr / (1-beta1^t) * exp_avg / (sqrt(exp_avg_sq) / sqrt(1-beta2^t) + eps), t = *step + 1.  `step` (one float) and `ticket`
 * (one zero-initialised uint32) live on the device: the last block to finish bumps the counter, so a captured CUDA graph replays
 * correctly.  zero_grad != 0 clears the gradient buffer in the same pass.  One launch. */
int stmp_adam_flat(int64_t n, float* param, float* grad, float* exp_avg, float* exp_avg_sq, float* step, void* ticket, float lr,
                   float beta1, float beta2, float eps, float weight_decay, float grad_scale, int zero_grad, void* stream);

/* Transposed stacked DConv weights for the backward kernels, one launch: whsT (cout, (2K-1)C) from wh, wzrT (2cout, (2K-1)C)
 * from wz | wr; C = cin + cout; stacked block 0 = W[0,0] + W[1,0], block 1+2(k-1)+o = W[o,k] (the order of the basis). */
int stmp_dcrnn_pack_bwd_weights(int64_t cin, int64_t cout, int64_t K, const float* wz, const float* wr, const float* wh,
                                float* whsT, float* wzrT, void* stream);

/* Masked MAE of the index-batching training loops (examples/indexBatching/DCRNN/utils.py:10-18, used at pems_ddp.py:104-121):
 * loss = mean(nan_to_zero(|pred - y| * mask / mean(mask))), mask = (y != 0) == sum_i nz(|p_i - y_i| m_i) / sum_i m_i.
 * fwd writes the scalar loss and s0 = sum(mask) (device scalars; deterministic two-stage reduction, workspace of
 * stmp_masked_mae_workspace_floats() floats); bwd writes gpred = gout * sign(pred - y) * mask / s0. */
int64_t stmp_masked_mae_workspace_floats(void);
int stmp_masked_mae_fwd(int64_t n, const float* pred, const float* target, float* workspace, float* loss, float* s0, void* stream);
int stmp_masked_mae_bwd(int64_t n, const float* pred, const float* target, const float* s0, const float* gout, float* gpred,
                        void* stream);

/* GRU reverse-time gate derivatives: the pointwise part of the hand-written backward of the DCRNN sequence (what
 * autograd records for dcrnn.py:172-192, once per step).  Tensors are (B, N, cout) with a batch stride in elements
 * (slices of gout (B,T,N,cout) and of the forward stash (B,T,3,N,cout)); du2/du1 are (B, N, du_ld) buffers whose
 * first cin+cout columns hold dL/d[X | H*R] and dL/d[X | H_{t-1}] of the step being closed.
 *   stmp_gru_bwd_carry: close step t+1 (all of g_prev.. or none): dH = g_prev*Z + dU2[...,cin:]*R + dU1[...,cin:],
 *                       dX_{t+1} = dU2[...,:cin] + dU1[...,:cin] (dx nullable), dh_out = dH (nullable);
 *                       open step t (gout.. or none): g = gout_t + dH, dph = g (1-Z_t)(1-Ht_t^2).
 *   stmp_gru_bwd_zr:    dpzr[..., :cout] = g (H_{t-1} - Ht) Z (1-Z);  dpzr[..., cout:] = dU2[...,cin:] H_{t-1} R (1-R);
 *                       hprev NULL = zeros (first step without H0).
 */
int stmp_gru_bwd_carry(int64_t B, int64_t N, int64_t cin, int64_t cout, int64_t du_ld, const float* g_prev,
                       const float* z_prev, const float* r_prev, const float* du2, const float* du1, float* dx,
                       int64_t dx_bstride, const float* gout, int64_t gout_bstride, const float* z, const float* ht,
                       int64_t stash_bstride, float* g, float* dph, float* dh_out, void* stream);
int stmp_gru_bwd_zr(int64_t B, int64_t N, int64_t cin, int64_t cout, int64_t du_ld, const float* g, const float* hprev,
                    int64_t hprev_bstride, const float* z, const float* r, const float* ht, int64_t stash_bstride,
                    const float* du2, float* dpzr, void* stream);

/* ---- K4: dense node-feature x weight contraction on the tensor cores (tcgen05), fp32 in / fp32 out ------------------
 * C[M,N] = A[M,K] @ W[K,N] + bias.  Replaces `torch.matmul(Tx_k, weight[..][k])` / ChebConv `lins[k](Tx_k)` / GCNConv
 * `lin(x)` (dcrnn.py:81-105; PyG) for the large-graph (tiled) path.  fp32-class accuracy: operands are split into fp16
 * hi/lo halves and multiplied in three tcgen05.mma passes with an fp32 TMEM accumulator.
 *   stmp_gemm_packed_elems(K,N): number of fp16 elements of the packed weight buffer
 *   stmp_gemm_prepack: W [K,N] row-major (row stride ldw) -> packed (hi/lo, K-major, K padded to 64); once per weight update
 *   stmp_gemm_f32: A row-major (row stride lda), C row-major (ldc); needs N <= 256, N % 32 == 0, K % 4 == 0, 16-byte aligned
 *                  rows; otherwise STMP_EUNSUPPORTED (callers use cuBLAS).  The split holds a relative 2^-22 only for operands in
 *                  2^-3 <= |v| < 65520 (absolute ~2^-25 below, inf above).  a_row_scale (optional, [M] powers of two that fp32
 *                  holds together with their reciprocals): row r of A is multiplied by a_row_scale[r] before the split and the
 *                  row of the product by 1/a_row_scale[r] before the bias -- both exact; lets a caller bring every row of an
 *                  operand of arbitrary magnitude into the split's range.
 *   stmp_gemm_lstm_f32: same contraction with N = 4*cout (column blocks i|f|c|o) fused with the peephole-LSTM gate epilogue
 *                  of GConvLSTM (gconv_lstm.py:168-202): conv_bias [4*cout] (ChebConv biases), cell C_{t-1} [M,cout],
 *                  peepholes w_c{i,f,o} [cout], gate biases b_{i,f,c,o} [cout] -> h_out, c_out [M,cout]; cout in {32, 64}. */
int64_t stmp_gemm_packed_elems(int64_t K, int64_t N);
int stmp_gemm_prepack(const float* W, int64_t ldw, int64_t K, int64_t N, void* packed, void* stream);
int stmp_gemm_f32(const float* A, int64_t lda, int64_t M, int64_t K, int64_t N, const void* packed, const float* bias,
                  const float* a_row_scale, float* C, int64_t ldc, void* stream);
int stmp_gemm_lstm_f32(const float* A, int64_t lda, int64_t M, int64_t K, int64_t cout, const void* packed,
                       const float* conv_bias, const float* cell, const float* wci, const float* wcf, const float* wco,
                       const float* bi, const float* bf, const float* bc, const float* bo, float* h_out, float* c_out,
                       void* stream);

/* ---- ASTGCN block (nn/attention/astgcn.py:408-481): the dense products on tcgen05 with their operand gathers and pointwise tails fused
 * stmp_gemm_blocks_f32:  C[m, 0:ncols] = epilogue( sum_i A_i[m + shift_i, 0:width_i] @ W_i + bias )
 *   the A operand is a list of nblk (<= 12) K-blocks of <= 64 columns: blk_ptr[i] (device pointer, HOST array), row stride blk_ld[i],
 *   valid columns blk_width[i], row shift blk_shift[i] inside sequences of `seq` consecutive rows (rows shifted out of their sequence read
 *   as zero).  packed = stmp_gemm_prepack of the stacked weight [nblk*64][N] (rows of a block beyond its width are zero), N % 16 == 0,
 *   N <= 320.  epilogue 0: + bias; 1: + bias, ReLU; 2: + bias, ReLU, LayerNorm(gamma, beta, eps) over the row (N == ncols == 64).
 *   With channels-last activations (B, nodes, T, F) this is: the Chebyshev contraction sum_k T_k W_k + ReLU (astgcn.py:166-178,448) with
 *   blocks T_0|T_1|T_2; time convolution (1x3, padding 1) + residual 1x1 convolution + ReLU + LayerNorm (:473-480) with blocks
 *   X^[t-1] | X^[t] | X^[t+1] | X[t], seq = T; the final (1 x F) convolution (:604-610) with the T blocks of a row.
 * stmp_spatial_attention_fwd:  S = softmax_dim1(Vs @ sigmoid(LHS @ RHS + bs)) (astgcn.py:245-262), written TRANSPOSED:
 *   st_out[b, j, i] = S[b, i, j], rows ld_out (>= nodes rounded up to 64, % 4 == 0) floats apart, padding columns zero.
 *   lhs [B][nodes][T] = (X~ W1) W2, rhs [B][T][nodes] = (W3 X~)^T, bsT [nodes][nodes] = bs^T, vsT_packed = stmp_gemm_prepack of Vs^T
 *   zero-padded to [P][P], P = nodes rounded up to 64 (<= 320).  The N x N sigmoid is generated inside the GEMM's operand stage and the
 *   softmax is the GEMM epilogue: neither ever reaches HBM.
 *   nodes <= 320, T <= 12.
 * Optional weight IMAGE (both entries; NULL = the kernel swizzles the packed weights itself): stmp_gemm_blocks_image rewrites a packed weight
 * into the per-k-block shared-memory image (hi | lo tile, SWIZZLE_128B) of stmp_gemm_blocks_image_bytes(N, nblk) bytes, which every CTA then
 * fetches with ONE TMA bulk copy per k-block while it loads / generates its A tile. */
int stmp_gemm_blocks_f32(int64_t M, int64_t N, int64_t ncols, int64_t nblk, const float* const* blk_ptr, const int64_t* blk_ld,
                         const int32_t* blk_width, const int32_t* blk_shift, int64_t seq, const void* packed, const void* image,
                         const float* bias, int epilogue, const float* gamma, const float* beta, float eps, float* C, int64_t ldc, void* stream);
int stmp_spatial_attention_fwd(int64_t B, int64_t n_nodes, int64_t n_steps, const float* lhs, const float* rhs, const float* bsT,
                               const void* vsT_packed, const void* vsT_image, float* st_out, int64_t ld_out, void* stream);
/* The small-matrix front of an ASTGCN block in one launch (astgcn.py:311-328 temporal attention, :427-430 X~ = X E, :245-256 the spatial
 * attention factors): x [B][nodes][T][F] channels-last; TemporalAttention parameters U1 [nodes], U2 [F][nodes], U3 [F], be [T][T],
 * Ve [T][T]; SpatialAttention parameters W1 [T], W2 [F][T], W3 [F]  ->  lhs_s [B][nodes][T] = (X~ W1) W2, rhs_s [B][T][nodes] = (W3 X~)^T
 * (the inputs of stmp_spatial_attention_fwd) and optionally E [B][T][T].  X~ is never materialised.  T <= 12, F in {1,2,4,...,64}. */
int stmp_astgcn_factors_fwd(int64_t B, int64_t n_nodes, int64_t n_steps, int64_t f_in, const float* x, const float* U1, const float* U2,
                            const float* U3, const float* be, const float* Ve, const float* W1, const float* W2, const float* W3,
                            float* lhs_s, float* rhs_s, float* E_out, void* stream);
int64_t stmp_gemm_blocks_image_bytes(int64_t N, int64_t nblk);
int stmp_gemm_blocks_image(const void* packed, int64_t N, int64_t nblk, void* image, void* stream);

/* ---- K8: index-batching window gather -----------------------------------------------------------
 * x[b] = series[start[b] : start[b]+h], y[b] = series[start[b]+h : start[b]+2h]   (index_dataset.py:49-57
 * + DataLoader default collate), series [T_total, row_elems] resident on the device.  y may be NULL. */
int stmp_window_gather(const float* series, int64_t t_total, int64_t row_elems, const int64_t* start,
                       int64_t B, int64_t horizon, float* x, float* y, void* stream);

/* Run-time switches for tests: "dcrnn_tc" = 1 (tcgen05 kernel, default) / 0 (FFMA kernel) behind stmp_dcrnn_seq_fwd; "spmm_variant" = 0
 * (register gather, default) / 1, 2 (TMA-staged rows, 8 / 16 per warp); "dcrnn_bwd_all_cin" = 1 (default) / 0 (persistent backward only for cin == 2); "dcrnn_bwd_split" = 1 (default: a 2-CTA cluster per window
 * when 2 B <= SM count) / 0 (one CTA per window); "dcrnn_fwd_split" = 1 (default: the fused forward also runs on a 2-CTA cluster per window when 2 B <= SM count and N > 128) / 0;
 * "dcrnn_wgrad_tc" = 1 (default, tcgen05) / 0 (FFMA); "spmm_rows_per_group" (default 8) and
 * "spmm_block" (256 / 1024): the SpMM's row blocking. */
int stmp_set_option(const char* name, int value);

/* ---- misc ---------------------------------------------------------------------------------------- */
const char* stmp_last_error(void);
/* "stmp <version> sm_100a" */
const char* stmp_version(void);
/* Number of kernels this library has launched in the calling process (bench.py's gpu_launches). */
int64_t stmp_launch_count(void);
/* Which kernels served the calls so far ("did the fused tcgen05 path run, or the tiled one?" -- the dispatchers fall back
 * silently on STMP_EUNSUPPORTED, e.g. dcrnn.py:429-475 at N > 207).  Fills up to max_entries (kernel name, launches) pairs,
 * names are static strings such as "k_dcrnn_seq_tc"; returns the number of distinct kernels launched. */
int stmp_path_counters(const char** names, int64_t* counts, int max_entries);

#ifdef __cplusplus
}
#endif
#endif /* STMP_H_ */

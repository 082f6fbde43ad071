// gemm_tc.cu -- K4 (+K5): the dense node-feature x weight contraction of the tiled (large-graph) path on the
// 5th-gen tensor cores, fp32 in / fp32 out:   C[M,N] = A[M,K] @ W[K,N] + bias
// optionally fused with the peephole-LSTM gate epilogue of GConvLSTM (gconv_lstm.py:168-202), so the gate
// pre-activations never reach HBM.
//
// fp32-class accuracy from fp16 tensor cores: every operand is split into hi = fp16(v), lo = fp16(v - hi) and the
// product is accumulated as lo*hi + hi*lo + hi*hi in the fp32 TMEM accumulator (three tcgen05.mma.kind::f16 passes;
// validated in tools/tc_probe.cu).  The weights are split ONCE (stmp_gemm_prepack); activations are split on the
// fly while they are staged: 256 threads stream a 128 x 64 fp32 tile from HBM (coalesced float4), convert, and
// write both halves into the hand-swizzled K-major SWIZZLE_128B layout the UMMA descriptors expect.  Two stages:
// the tile of k-block i+1 is loaded/converted while the MMAs of k-block i run (tcgen05.commit -> mbarrier).
//
// The split keeps a relative 2^-22 only while an operand lies in 2^-3 <= |v| < 65520: below 2^-3 `lo` is subnormal and the
// error of the split is an absolute ~2^-25, below ~3e-8 a value is 0 in both halves, and |v| >= 65520 becomes inf.  Operands of
// unknown magnitude (gradients) go through `a_row_scale`: row r of A is multiplied by the power of two a_row_scale[r] while it is
// staged and the row of the product by its reciprocal in the epilogue -- both exact, so the result does not depend on the scale of
// the row as long as fp32 holds it.
//
// One CTA = 128 rows x all N (<= 256) columns, so A is read from HBM exactly once: algorithmic bytes
// 4*M*K + 4*M*N (+ the L2-resident weights).  This is a true dense GEMM (cfg5: 80 000 x 384 x 256), the one place on
// the path where tensor cores are the right tool (north_star).
#include "common.cuh"
#include "tc_common.cuh"

namespace stmp {
namespace {

constexpr int GM_NT = 256;
constexpr int GM_BM = 128;
constexpr int GM_BK = 64;
constexpr int GM_A_BYTES = GM_BM * 128;   // one K-block of A (hi or lo): 128 rows x 128 B

struct GemmParams {
  const float* A; long long lda;
  int M, K, N, Kpad;
  const __half* w_hi;   // [N][Kpad]
  const __half* w_lo;
  const float* bias;    // [N] or null
  const float* a_scale; // [M] powers of two or null (EPI == 0 only): C[r] = ((a_scale[r] * A[r]) @ W) / a_scale[r] + bias
  float* C; long long ldc;
  // LSTM epilogue (EPI == 1): N = 4*Co, column blocks i|f|c|o
  int Co;
  const float* cell; long long ldcell;     // C_{t-1} [M][Co]
  const float* wci; const float* wcf; const float* wco;   // peepholes [Co]
  const float* bi; const float* bf; const float* bc; const float* bo;   // gate biases [Co]
  float* h_out; long long ldh;             // H_t  [M][Co]
  float* c_out; long long ldco;            // C_t  [M][Co]
};

__global__ void k_split_weights(const float* __restrict__ W, long long ldw, int K, int N, int Kpad, __half* __restrict__ hi,
                                __half* __restrict__ lo) {
  const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (idx >= (long long)N * Kpad) return;
  const int n = (int)(idx / Kpad), k = (int)(idx - (long long)n * Kpad);
  const float v = k < K ? W[(long long)k * ldw + n] : 0.f;
  const __half h = __float2half_rn(v);
  hi[idx] = h;
  lo[idx] = __float2half_rn(v - __half2float(h));
}

template <int EPI>
__global__ void __launch_bounds__(GM_NT, 1) k_gemm_split(const GemmParams p) {
  extern __shared__ __align__(1024) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = p.N;
  const int b_bytes = N * 128;                       // one K-block of B (hi or lo)
  const int stage_bytes = 2 * GM_A_BYTES + 2 * b_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 2 * stage_bytes);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);

  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(256));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    fence_mbar_init();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const long long m0 = (long long)blockIdx.x * GM_BM;
  const int nkb = p.Kpad / GM_BK;
  const uint32_t idesc = umma_idesc_f16(128, N);

  float4 av[8];
  float ascale[8];   // the row scale of each of this thread's 8 staging rows (row idx >> 4 = tid / 16 + 16 j)
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const long long row = m0 + ((tid + j * GM_NT) >> 4);
    ascale[j] = (EPI == 0 && p.a_scale && row < p.M) ? __ldg(p.a_scale + row) : 1.f;
  }
  auto load_a = [&](int kb) {
    const int k0 = kb * GM_BK;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int idx = tid + j * GM_NT;
      const int r = idx >> 4, c4 = idx & 15;
      const long long row = m0 + r;
      const int k = k0 + 4 * c4;
      av[j] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row < p.M && k < p.K) av[j] = __ldg(reinterpret_cast<const float4*>(p.A + row * p.lda + k));   // K % 4 == 0
      if (EPI == 0 && p.a_scale) { av[j].x *= ascale[j]; av[j].y *= ascale[j]; av[j].z *= ascale[j]; av[j].w *= ascale[j]; }
    }
  };

  for (int kb = 0; kb < nkb; ++kb) {
    const int s = kb & 1;
    unsigned char* a_hi = smem + s * stage_bytes;
    unsigned char* a_lo = a_hi + GM_A_BYTES;
    unsigned char* b_hi = a_lo + GM_A_BYTES;
    unsigned char* b_lo = b_hi + b_bytes;
    if (kb >= 2) {  // the MMAs of k-block kb-2 must have drained this stage
      mbar_wait(&bars[s], (uint32_t)((kb >> 1) - 1) & 1u);
      tc_fence_after();
    }
    const int k0 = kb * GM_BK;
    // A: 128 x 64 fp32 -> hi/lo fp16, swizzled.  16 lanes cover one row's 256 B contiguously.  The 8 loads of k-block kb+1 are
    // issued into registers right after k-block kb's tile is stored, i.e. before its barrier and MMAs: a k-block no longer costs a
    // full HBM round trip (the kernel is bound by HBM latency, not by math).
    if (kb == 0) load_a(0);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int idx = tid + j * GM_NT;
      store_split4(a_hi, a_lo, idx >> 4, 4 * (idx & 15), av[j]);
    }
    if (kb + 1 < nkb) load_a(kb + 1);
    // B: N x 64 fp16 (already split, L2-resident) -> swizzled; 4 x (hi, lo) 128-bit loads in flight per thread
    for (int base = 0; base < N * 8; base += 4 * GM_NT) {
      uint4 h[4], l[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int idx = base + tid + j * GM_NT;
        if (idx < N * 8) {
          const long long g = (long long)(idx >> 3) * p.Kpad + k0 + 8 * (idx & 7);
          h[j] = __ldg(reinterpret_cast<const uint4*>(p.w_hi + g));
          l[j] = __ldg(reinterpret_cast<const uint4*>(p.w_lo + g));
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int idx = base + tid + j * GM_NT;
        if (idx < N * 8) {
          const int n = idx >> 3, c = idx & 7;
          const int off = n * 128 + ((c ^ (n & 7)) << 4);
          *reinterpret_cast<uint4*>(b_hi + off) = h[j];
          *reinterpret_cast<uint4*>(b_lo + off) = l[j];
        }
      }
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (tid == 0) {
      const uint32_t ah = smem_u32(a_hi), al = smem_u32(a_lo), bh = smem_u32(b_hi), bl = smem_u32(b_lo);
#pragma unroll
      for (int pass = 0; pass < 3; ++pass) {          // lo*hi, hi*lo, hi*hi
        const uint32_t ab = pass == 0 ? al : ah, bb = pass == 1 ? bl : bh;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks)
          umma_f16(tmem, umma_desc(ab + ks * 32), umma_desc(bb + ks * 32), idesc, (kb | pass | ks) ? 1u : 0u);
      }
      umma_commit(&bars[s]);
    }
  }
  {  // all MMAs complete in order: waiting for the last commit is enough
    const int last = nkb - 1;
    mbar_wait(&bars[last & 1], (uint32_t)(last >> 1) & 1u);
    tc_fence_after();
  }

  // ---- epilogue: TMEM lane == row; warps 0-3 / 4-7 split the columns ------------------------------------------
  const int q = warp & 3, half = warp >> 2;
  const long long row = m0 + q * 32 + lane;
  const bool live = row < p.M;
  const uint32_t trow = tmem + ((uint32_t)(q * 32) << 16);
  if (EPI == 0) {
    const int ncol = N / 2;   // N % 32 == 0 on this path
    const float unscale = (p.a_scale && live) ? __frcp_rn(__ldg(p.a_scale + row)) : 1.f;   // exact: a power of two
    for (int c0 = half * ncol; c0 < (half + 1) * ncol; c0 += 16) {
      uint32_t v[16];
      tmem_ld16(trow + c0, v);
      tmem_ld_wait();
      if (live) {
        float* dst = p.C + row * p.ldc + c0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float4 o = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]),
                                 __uint_as_float(v[4 * j + 3]));
          if (p.a_scale) { o.x *= unscale; o.y *= unscale; o.z *= unscale; o.w *= unscale; }
          if (p.bias) {
            const float4 bq = __ldg(reinterpret_cast<const float4*>(p.bias + c0 + 4 * j));
            o.x += bq.x; o.y += bq.y; o.z += bq.z; o.w += bq.w;
          }
          *reinterpret_cast<float4*>(dst + 4 * j) = o;
        }
      }
    }
  } else {
    // peephole LSTM (gconv_lstm.py:168-202): I = sig(pi + wci*C + bi); F = sig(pf + wcf*C + bf); T = tanh(pc + bc);
    // C' = F*C + I*T; O = sig(po + wco*C' + bo); H' = O*tanh(C').   p.bias carries the ChebConv biases (x + h) per column.
    const int Co = p.Co, nch = Co / 2;
    for (int ch = half * nch; ch < (half + 1) * nch; ch += 16) {
      uint32_t vi[16], vf[16], vc[16], vo[16];
      tmem_ld16(trow + ch, vi);
      tmem_ld16(trow + Co + ch, vf);
      tmem_ld16(trow + 2 * Co + ch, vc);
      tmem_ld16(trow + 3 * Co + ch, vo);
      tmem_ld_wait();
      if (live) {
        float cold[16], hn[16], cn[16];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 cq = __ldg(reinterpret_cast<const float4*>(p.cell + row * p.ldcell + ch + 4 * j));
          cold[4 * j] = cq.x; cold[4 * j + 1] = cq.y; cold[4 * j + 2] = cq.z; cold[4 * j + 3] = cq.w;
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int c = ch + j;
          const float cb_i = p.bias ? __ldg(p.bias + c) : 0.f, cb_f = p.bias ? __ldg(p.bias + Co + c) : 0.f;
          const float cb_c = p.bias ? __ldg(p.bias + 2 * Co + c) : 0.f, cb_o = p.bias ? __ldg(p.bias + 3 * Co + c) : 0.f;
          const float ig = sigmoidf_acc(__uint_as_float(vi[j]) + cb_i + __ldg(p.wci + c) * cold[j] + __ldg(p.bi + c));
          const float fg = sigmoidf_acc(__uint_as_float(vf[j]) + cb_f + __ldg(p.wcf + c) * cold[j] + __ldg(p.bf + c));
          const float tg = tanhf(__uint_as_float(vc[j]) + cb_c + __ldg(p.bc + c));
          cn[j] = fg * cold[j] + ig * tg;
          const float og = sigmoidf_acc(__uint_as_float(vo[j]) + cb_o + __ldg(p.wco + c) * cn[j] + __ldg(p.bo + c));
          hn[j] = og * tanhf(cn[j]);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          *reinterpret_cast<float4*>(p.h_out + row * p.ldh + ch + 4 * j) = make_float4(hn[4 * j], hn[4 * j + 1], hn[4 * j + 2], hn[4 * j + 3]);
          *reinterpret_cast<float4*>(p.c_out + row * p.ldco + ch + 4 * j) = make_float4(cn[4 * j], cn[4 * j + 1], cn[4 * j + 2], cn[4 * j + 3]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(256));
}

inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

int gemm_check(int64_t M, int64_t K, int64_t N, const float* A, int64_t lda) {
  STMP_REQUIRE(M >= 0 && K > 0 && N > 0, STMP_EINVAL, "stmp_gemm: bad sizes");
  if (N > 256 || N % 32 != 0 || K % 4 != 0 || lda % 4 != 0 || !al16(A) || M >= (1ll << 31) - 128)
    return set_error(STMP_EUNSUPPORTED, "tcgen05 GEMM needs N<=256, N%%32==0, K%%4==0 and 16-byte aligned rows (M=%lld K=%lld N=%lld)",
                     (long long)M, (long long)K, (long long)N);
  return STMP_OK;
}

template <int EPI>
int gemm_launch(GemmParams& p, cudaStream_t st) {
  const int smem = 2 * (2 * GM_A_BYTES + 2 * p.N * 128) + 64;
  STMP_CUDA_OK(cudaFuncSetAttribute(k_gemm_split<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  const unsigned grid = (unsigned)((p.M + GM_BM - 1) / GM_BM);
  k_gemm_split<EPI><<<grid, GM_NT, smem, st>>>(p);
  STMP_LAUNCH_OK("k_gemm_split");
  return STMP_OK;
}

}  // namespace
}  // namespace stmp

using namespace stmp;

extern "C" int64_t stmp_gemm_packed_elems(int64_t K, int64_t N) {
  const int64_t kpad = (K + GM_BK - 1) / GM_BK * GM_BK;
  return 2 * N * kpad;   // fp16 elements: hi [N][Kpad] followed by lo [N][Kpad]
}

extern "C" int stmp_gemm_prepack(const float* W, int64_t ldw, int64_t K, int64_t N, void* packed, void* stream) {
  STMP_REQUIRE(W && packed && K > 0 && N > 0 && ldw >= N, STMP_EINVAL, "stmp_gemm_prepack: bad argument");
  const int kpad = (int)((K + GM_BK - 1) / GM_BK * GM_BK);
  __half* hi = reinterpret_cast<__half*>(packed);
  __half* lo = hi + N * kpad;
  const long long total = (long long)N * kpad;
  k_split_weights<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(W, ldw, (int)K, (int)N, kpad, hi, lo);
  STMP_LAUNCH_OK("k_split_weights");
  return STMP_OK;
}

extern "C" int stmp_gemm_f32(const float* A, int64_t lda, int64_t M, int64_t K, int64_t N, const void* packed, const float* bias,
                             const float* a_row_scale, float* C, int64_t ldc, void* stream) {
  STMP_REQUIRE(A && packed && C, STMP_EINVAL, "stmp_gemm_f32: NULL pointer");
  int rc = gemm_check(M, K, N, A, lda);
  if (rc) return rc;
  if (ldc % 4 != 0 || !al16(C) || (bias && !al16(bias))) return set_error(STMP_EUNSUPPORTED, "stmp_gemm_f32: C/bias must be 16-byte aligned");
  if (M == 0) return STMP_OK;
  GemmParams p = {};
  p.A = A; p.lda = lda; p.M = (int)M; p.K = (int)K; p.N = (int)N; p.Kpad = (int)((K + GM_BK - 1) / GM_BK * GM_BK);
  p.w_hi = reinterpret_cast<const __half*>(packed); p.w_lo = p.w_hi + N * p.Kpad;
  p.bias = bias; p.a_scale = a_row_scale; p.C = C; p.ldc = ldc;
  return gemm_launch<0>(p, (cudaStream_t)stream);
}

extern "C" int stmp_gemm_lstm_f32(const float* A, int64_t lda, int64_t M, int64_t K, int64_t cout, const void* packed,
                                  const float* conv_bias, const float* cell, const float* wci, const float* wcf, const float* wco,
                                  const float* bi, const float* bf, const float* bc, const float* bo, float* h_out, float* c_out,
                                  void* stream) {
  STMP_REQUIRE(A && packed && cell && wci && wcf && wco && bi && bf && bc && bo && h_out && c_out, STMP_EINVAL,
               "stmp_gemm_lstm_f32: NULL pointer");
  int rc = gemm_check(M, K, 4 * cout, A, lda);
  if (rc) return rc;
  if (cout % 32 != 0 || !al16(cell) || !al16(h_out) || !al16(c_out))
    return set_error(STMP_EUNSUPPORTED, "stmp_gemm_lstm_f32: cout must be a multiple of 32 (<= 64) and state tensors 16-byte aligned");
  if (M == 0) return STMP_OK;
  GemmParams p = {};
  p.A = A; p.lda = lda; p.M = (int)M; p.K = (int)K; p.N = (int)(4 * cout); p.Kpad = (int)((K + GM_BK - 1) / GM_BK * GM_BK);
  p.w_hi = reinterpret_cast<const __half*>(packed); p.w_lo = p.w_hi + (long long)p.N * p.Kpad;
  p.bias = conv_bias; p.Co = (int)cout;
  p.cell = cell; p.ldcell = cout; p.wci = wci; p.wcf = wcf; p.wco = wco; p.bi = bi; p.bf = bf; p.bc = bc; p.bo = bo;
  p.h_out = h_out; p.ldh = cout; p.c_out = c_out; p.ldco = cout;
  return gemm_launch<1>(p, (cudaStream_t)stream);
}

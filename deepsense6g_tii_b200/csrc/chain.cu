// Row-local forward chain of the transformer block for the narrow stages (n_embd 64 / 128), one launch per block.
//
// At n_embd <= 128 every Linear of model2_seq.py:113-134 is a few microseconds of tensor work and each separate kernel of the
// chain  proj -> +residual -> LayerNorm -> mlp.0 -> ReLU -> mlp.2 -> +residual -> LayerNorm(next block) -> QKV(next block)
// runs at its launch / fill / drain floor.  All of these operators are ROW-local (a token row never meets another row
// between two attention calls), so one CTA can carry a tile of rows through the whole chain with the activations in
// registers: the accumulator fragment of one warp-level MMA is, element for element, the A-operand fragment of the next one
// (m16n8k16: C rows g / g+8, columns 2t, 2t+1 of n-tile j <-> A rows g / g+8, k = 2t, 2t+1 (+8) of k-step j/2), so LayerNorm,
// bias, ReLU and the bf16 rounding happen in place and nothing but the tensors the backward needs is written to HBM.
// The weights (0.1-0.4 MB per block, L2-resident) stream through a double-buffered shared-memory ring with cp.async.
//
// These stages sit far below the tensor-core ridge (SURVEY.md §8d: 32-100 flop/B): the kernel is bound by the HBM / L2 bytes of
// the saved activations and by instruction issue, not by MMA throughput, which is why it uses register-fragment
// mma.sync.m16n8k16 (no TMEM round trip between the chained GEMMs) rather than tcgen05; the n_embd >= 256 stages keep the
// TMA + tcgen05 kernels of gemm_tc2.cu.
#include <algorithm>

#include "common.cuh"

namespace dsf {

struct ChainFwdArgs {
  const __nv_bfloat16* y;      // (M, C)  attention output of this block
  const float* x_in;           // (M, C)  residual stream entering the block
  const __nv_bfloat16 *wp, *w1, *w2, *wqkv;   // bf16 shadows: proj (C,C), mlp.0 (F,C), mlp.2 (C,F), next block's fused QKV (3C,C) or NULL
  const float *bp, *b1, *b2, *bqkv;
  const float *g2, *be2;       // ln2 of this block
  const float *gn, *ben;       // ln1 of the next block, or ln_f after the last block
  float *x_mid, *x_out;        // (M, C) fp32, saved for the backward / handed to the next block
  __nv_bfloat16 *h2, *a;       // (M, C), (M, F) saved GEMM operands
  __nv_bfloat16 *hn, *qkv;     // next block: ln1 output (M, C) and fused QKV (M, 3C); unused when wqkv == NULL
  float* yf;                   // last block: ln_f output (M, C) fp32
  float *mean2, *rstd2, *meann, *rstdn;
  int M;
  float eps;
};

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void* smem_row) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem_row);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(s));
}
// D (16x8 fp32) += A (16x16 bf16, row) * B (16x8 bf16, col)
__device__ __forceinline__ void mma_bf16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&v);
}

// acc[j] (j < NTL n-tiles) += A-fragments afr[kk] (kk < KSL k-steps) x W^T, W = [n rows][k] bf16 in shared memory with row stride
// ldw elements (rows n0.., columns k0..).  B fragments of two adjacent n-tiles come from one ldmatrix.x4.
template <int NTL, int KSL>
__device__ __forceinline__ void warp_gemm(float (&acc)[NTL][4], const uint32_t (&afr)[KSL][4], const __nv_bfloat16* w, int ldw, int lane) {
  const int r_in = (lane & 7) + ((lane >> 4) << 3);   // row within the 16-row (two n-tile) group
  const int k_in = ((lane >> 3) & 1) << 3;            // 0 / 8: low / high half of the k-step
#pragma unroll
  for (int kk = 0; kk < KSL; ++kk) {
#pragma unroll
    for (int j = 0; j < NTL; j += 2) {
      uint32_t b[4];
      ldmatrix_x4(b, w + (size_t)(j * 8 + r_in) * ldw + kk * 16 + k_in);
      mma_bf16(acc[j], afr[kk], b[0], b[1]);
      mma_bf16(acc[j + 1], afr[kk], b[2], b[3]);
    }
  }
}

// LayerNorm of the 16 rows a warp holds in accumulator layout (v[j][0..1]: row g, v[j][2..3]: row g + 8): returns the
// normalised values in place (gamma / beta applied) and the row statistics of the two rows of this lane.
template <int NT>
__device__ __forceinline__ void warp_layernorm(float (&v)[NT][4], const float* __restrict__ gamma, const float* __restrict__ beta, int t, float eps,
                                               float& mean_lo, float& rstd_lo, float& mean_hi, float& rstd_hi) {
  constexpr float inv_c = 1.0f / (float)(NT * 8);
  float s_lo = 0.f, s_hi = 0.f;
#pragma unroll
  for (int j = 0; j < NT; ++j) { s_lo += v[j][0] + v[j][1]; s_hi += v[j][2] + v[j][3]; }
  s_lo += __shfl_xor_sync(0xffffffffu, s_lo, 1); s_lo += __shfl_xor_sync(0xffffffffu, s_lo, 2);
  s_hi += __shfl_xor_sync(0xffffffffu, s_hi, 1); s_hi += __shfl_xor_sync(0xffffffffu, s_hi, 2);
  mean_lo = s_lo * inv_c; mean_hi = s_hi * inv_c;
  float q_lo = 0.f, q_hi = 0.f;
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const float a0 = v[j][0] - mean_lo, a1 = v[j][1] - mean_lo, a2 = v[j][2] - mean_hi, a3 = v[j][3] - mean_hi;
    q_lo += a0 * a0 + a1 * a1; q_hi += a2 * a2 + a3 * a3;
  }
  q_lo += __shfl_xor_sync(0xffffffffu, q_lo, 1); q_lo += __shfl_xor_sync(0xffffffffu, q_lo, 2);
  q_hi += __shfl_xor_sync(0xffffffffu, q_hi, 1); q_hi += __shfl_xor_sync(0xffffffffu, q_hi, 2);
  rstd_lo = rsqrtf(q_lo * inv_c + eps); rstd_hi = rsqrtf(q_hi * inv_c + eps);
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const float2 gm = *reinterpret_cast<const float2*>(gamma + j * 8 + 2 * t);
    const float2 bt = *reinterpret_cast<const float2*>(beta + j * 8 + 2 * t);
    v[j][0] = (v[j][0] - mean_lo) * rstd_lo * gm.x + bt.x; v[j][1] = (v[j][1] - mean_lo) * rstd_lo * gm.y + bt.y;
    v[j][2] = (v[j][2] - mean_hi) * rstd_hi * gm.x + bt.x; v[j][3] = (v[j][3] - mean_hi) * rstd_hi * gm.y + bt.y;
  }
}

// CTA = CH_WARPS warps x 16 rows = 80 token rows, one tile per CTA: 11544 rows -> 145 CTAs = one wave on the 148 SMs.
// The weight chunks ride in a ring of NS slots filled NS - 1 steps ahead (cp.async groups): at n_embd = 64 the ring holds the whole
// block (the weights are fetched once, up front), at 128 it runs four 36 KB chunks deep, so a step never waits for L2 latency.
constexpr int CH_WARPS = 5, CH_THREADS = CH_WARPS * 32, CH_ROWS = CH_WARPS * 16;
template <int C> struct ChainCfg {
  static constexpr int NS_FWD = C == 64 ? 8 : 4;
};

template <int C>
__global__ void __launch_bounds__(CH_THREADS, 1) chain_fwd_kernel(ChainFwdArgs p) {
  constexpr int NS = ChainCfg<C>::NS_FWD;
  constexpr int F = 4 * C, NT = C / 8, KS = C / 16;
  constexpr int LDW = C + 8;        // padded row stride of [rows][C] chunks (ldmatrix rows land in distinct banks)
  constexpr int LDW2 = 64 + 8;      // row stride of the mlp.2 chunk [C rows][64 hidden columns]
  constexpr int CHUNK = (C * LDW > 64 * LDW + C * LDW2) ? C * LDW : 64 * LDW + C * LDW2;   // elements per ring slot
  constexpr int N_MLP = F / 64, N_QKV = 3 * C / 64;
  extern __shared__ __align__(16) uint8_t smem_raw[];
  __nv_bfloat16* ring = reinterpret_cast<__nv_bfloat16*>(smem_raw);             // [NS][CHUNK]
  __nv_bfloat16* ybuf = ring + NS * CHUNK;                                       // [CH_WARPS][16][LDW]
  // Every operand an epilogue needs is staged in shared memory by the same cp.async group as the first weight chunk: with five
  // warps per SM nothing hides a global-load round trip inside the dependent chain (ncu: 52 % of the stall samples of the first
  // version sat on the FADDs consuming bias / residual loads).
  constexpr int LDX = C + 8;
  float* xbuf = reinterpret_cast<float*>(ybuf + CH_WARPS * 16 * LDW);           // [CH_WARPS][16][LDX]: x_in, then x_mid in place
  float* vec = xbuf + CH_WARPS * 16 * LDX;                                       // bp | b2 | g2 | be2 | gn | ben | b1 | bqkv
  const float *v_bp = vec, *v_b2 = vec + C, *v_g2 = vec + 2 * C, *v_be2 = vec + 3 * C, *v_gn = vec + 4 * C, *v_ben = vec + 5 * C,
              *v_b1 = vec + 6 * C, *v_bqkv = vec + 6 * C + F;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int row0 = blockIdx.x * CH_ROWS + warp * 16;
  const int r_lo = row0 + g, r_hi = r_lo + 8;
  const bool ok_lo = r_lo < p.M, ok_hi = r_hi < p.M;
  const int n_steps = 1 + N_MLP + (p.wqkv ? N_QKV : 0);
  pdl_trigger();
  pdl_wait();

  auto prefetch = [&](int s) {   // weight chunk of step s -> ring slot s % NS (all threads, 16-byte pieces)
    __nv_bfloat16* dst = ring + (s % NS) * CHUNK;
    if (s == 0) {
      for (int i = tid; i < C * (C / 8); i += CH_THREADS) { const int r = i / (C / 8), c8 = i % (C / 8); cp_async16(dst + r * LDW + c8 * 8, p.wp + (size_t)r * C + c8 * 8); }
    } else if (s <= N_MLP) {
      const int hc = s - 1;
      for (int i = tid; i < 64 * (C / 8); i += CH_THREADS) { const int r = i / (C / 8), c8 = i % (C / 8); cp_async16(dst + r * LDW + c8 * 8, p.w1 + (size_t)(hc * 64 + r) * C + c8 * 8); }
      __nv_bfloat16* d2 = dst + 64 * LDW;
      for (int i = tid; i < C * 8; i += CH_THREADS) { const int r = i >> 3, c8 = i & 7; cp_async16(d2 + r * LDW2 + c8 * 8, p.w2 + (size_t)r * F + hc * 64 + c8 * 8); }
    } else {
      const int qc = s - 1 - N_MLP;
      for (int i = tid; i < 64 * (C / 8); i += CH_THREADS) { const int r = i / (C / 8), c8 = i % (C / 8); cp_async16(dst + r * LDW + c8 * 8, p.wqkv + (size_t)(qc * 64 + r) * C + c8 * 8); }
    }
    cp_async_commit();
  };
  // step boundary: refill the slot step s - 1 has released with the chunk of step s + NS - 1 (one cp.async group per step, empty
  // past the end, so that "all but the newest NS - 1 groups have landed" always means "chunk s has landed")
  auto acquire = [&](int s) {
    if (s + NS - 1 < n_steps) prefetch(s + NS - 1); else cp_async_commit();
    cp_async_wait<NS - 1>();
    __syncthreads();
  };
  auto release = [&](int s) {   // every warp is done with slot s % NS before chunk s + NS may overwrite it
    if (s + NS < n_steps) __syncthreads();
  };

  // this warp's 16 rows of y and x_in and the bias / LayerNorm vectors -> shared memory (same cp.async group as the first weight chunk)
  {
    float* xb = xbuf + warp * 16 * LDX;
    for (int i = lane; i < 16 * (C / 4); i += 32) {
      const int r = i / (C / 4), c4 = i % (C / 4);
      if (row0 + r < p.M) cp_async16(xb + r * LDX + c4 * 4, p.x_in + (size_t)(row0 + r) * C + c4 * 4);
      else *reinterpret_cast<float4*>(xb + r * LDX + c4 * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    const float* srcs[6] = {p.bp, p.b2, p.g2, p.be2, p.gn, p.ben};
    for (int i = tid; i < 6 * (C / 4); i += CH_THREADS) cp_async16(vec + i * 4, srcs[i / (C / 4)] + (i % (C / 4)) * 4);
    for (int i = tid; i < F / 4; i += CH_THREADS) cp_async16(vec + 6 * C + i * 4, p.b1 + i * 4);
    if (p.wqkv) { for (int i = tid; i < 3 * C / 4; i += CH_THREADS) cp_async16(vec + 6 * C + F + i * 4, p.bqkv + i * 4); }
  }
  {
    __nv_bfloat16* yb = ybuf + warp * 16 * LDW;
    for (int i = lane; i < 16 * (C / 8); i += 32) {
      const int r = i / (C / 8), c8 = i % (C / 8);
      if (row0 + r < p.M) cp_async16(yb + r * LDW + c8 * 8, p.y + (size_t)(row0 + r) * C + c8 * 8);
      else *reinterpret_cast<uint4*>(yb + r * LDW + c8 * 8) = make_uint4(0u, 0u, 0u, 0u);
    }
  }
  for (int s = 0; s < NS - 1; ++s) { if (s < n_steps) prefetch(s); else cp_async_commit(); }
  acquire(0);

  uint32_t hfr[KS][4];   // A fragments of the current LayerNorm output (h2, later the next block's h1)
  // ---------------------------------------------------------------- step 0: proj + residual, ln2
  {
    uint32_t yfr[KS][4];
    const __nv_bfloat16* yb = ybuf + warp * 16 * LDW;
#pragma unroll
    for (int kk = 0; kk < KS; ++kk) ldmatrix_x4(yfr[kk], yb + (size_t)((lane & 7) + (((lane >> 3) & 1) << 3)) * LDW + kk * 16 + ((lane >> 4) << 3));
    float xm[NT][4];
#pragma unroll
    for (int j = 0; j < NT; ++j) { xm[j][0] = xm[j][1] = xm[j][2] = xm[j][3] = 0.f; }
    warp_gemm<NT, KS>(xm, yfr, ring, LDW, lane);
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      const int n = j * 8 + 2 * t;
      const float2 b = *reinterpret_cast<const float2*>(v_bp + n);
      float* xs_lo = xbuf + (warp * 16 + g) * LDX + n;
      float* xs_hi = xs_lo + 8 * LDX;
      const float2 x0 = *reinterpret_cast<const float2*>(xs_lo), x1 = *reinterpret_cast<const float2*>(xs_hi);
      xm[j][0] += b.x + x0.x; xm[j][1] += b.y + x0.y; xm[j][2] += b.x + x1.x; xm[j][3] += b.y + x1.y;
      *reinterpret_cast<float2*>(xs_lo) = make_float2(xm[j][0], xm[j][1]);   // x_mid stays on chip for the mlp.2 epilogue
      *reinterpret_cast<float2*>(xs_hi) = make_float2(xm[j][2], xm[j][3]);
      if (ok_lo) *reinterpret_cast<float2*>(p.x_mid + (size_t)r_lo * C + n) = make_float2(xm[j][0], xm[j][1]);
      if (ok_hi) *reinterpret_cast<float2*>(p.x_mid + (size_t)r_hi * C + n) = make_float2(xm[j][2], xm[j][3]);
    }
    float m_lo, s_lo, m_hi, s_hi;
    warp_layernorm<NT>(xm, v_g2, v_be2, t, p.eps, m_lo, s_lo, m_hi, s_hi);
    if (t == 0) {
      if (ok_lo) { p.mean2[r_lo] = m_lo; p.rstd2[r_lo] = s_lo; }
      if (ok_hi) { p.mean2[r_hi] = m_hi; p.rstd2[r_hi] = s_hi; }
    }
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      const uint32_t lo = pack2(xm[j][0], xm[j][1]), hi = pack2(xm[j][2], xm[j][3]);
      hfr[j >> 1][(j & 1) * 2] = lo;
      hfr[j >> 1][(j & 1) * 2 + 1] = hi;
      const int n = j * 8 + 2 * t;
      if (ok_lo) *reinterpret_cast<uint32_t*>(p.h2 + (size_t)r_lo * C + n) = lo;
      if (ok_hi) *reinterpret_cast<uint32_t*>(p.h2 + (size_t)r_hi * C + n) = hi;
    }
  }
  release(0);

  // ---------------------------------------------------------------- steps 1 .. F/64: mlp.0 + ReLU + mlp.2, 64 hidden units at a time
  float acc2[NT][4];
#pragma unroll
  for (int j = 0; j < NT; ++j) { acc2[j][0] = acc2[j][1] = acc2[j][2] = acc2[j][3] = 0.f; }
  for (int hc = 0; hc < N_MLP; ++hc) {
    const int s = 1 + hc;
    acquire(s);
    const __nv_bfloat16* w1c = ring + (s % NS) * CHUNK;
    const __nv_bfloat16* w2c = w1c + 64 * LDW;
    float aa[8][4];
#pragma unroll
    for (int j = 0; j < 8; ++j) { aa[j][0] = aa[j][1] = aa[j][2] = aa[j][3] = 0.f; }
    warp_gemm<8, KS>(aa, hfr, w1c, LDW, lane);
    uint32_t afr[4][4];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int n = hc * 64 + j * 8 + 2 * t;
      const float2 b = *reinterpret_cast<const float2*>(v_b1 + n);
      const uint32_t lo = pack2(fmaxf(aa[j][0] + b.x, 0.f), fmaxf(aa[j][1] + b.y, 0.f));
      const uint32_t hi = pack2(fmaxf(aa[j][2] + b.x, 0.f), fmaxf(aa[j][3] + b.y, 0.f));
      afr[j >> 1][(j & 1) * 2] = lo;
      afr[j >> 1][(j & 1) * 2 + 1] = hi;
      if (ok_lo) *reinterpret_cast<uint32_t*>(p.a + (size_t)r_lo * F + n) = lo;
      if (ok_hi) *reinterpret_cast<uint32_t*>(p.a + (size_t)r_hi * F + n) = hi;
    }
    warp_gemm<NT, 4>(acc2, afr, w2c, LDW2, lane);
    release(s);
  }

  // ---------------------------------------------------------------- mlp.2 epilogue: + bias + x_mid, next LayerNorm
  float m_lo, s_lo, m_hi, s_hi;
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const int n = j * 8 + 2 * t;
    const float2 b = *reinterpret_cast<const float2*>(v_b2 + n);
    const float* xs_lo = xbuf + (warp * 16 + g) * LDX + n;   // x_mid, written by this thread above
    const float2 x0 = *reinterpret_cast<const float2*>(xs_lo), x1 = *reinterpret_cast<const float2*>(xs_lo + 8 * LDX);
    acc2[j][0] += b.x + x0.x; acc2[j][1] += b.y + x0.y; acc2[j][2] += b.x + x1.x; acc2[j][3] += b.y + x1.y;
    if (ok_lo) *reinterpret_cast<float2*>(p.x_out + (size_t)r_lo * C + n) = make_float2(acc2[j][0], acc2[j][1]);
    if (ok_hi) *reinterpret_cast<float2*>(p.x_out + (size_t)r_hi * C + n) = make_float2(acc2[j][2], acc2[j][3]);
  }
  warp_layernorm<NT>(acc2, v_gn, v_ben, t, p.eps, m_lo, s_lo, m_hi, s_hi);
  if (t == 0) {
    if (ok_lo) { p.meann[r_lo] = m_lo; p.rstdn[r_lo] = s_lo; }
    if (ok_hi) { p.meann[r_hi] = m_hi; p.rstdn[r_hi] = s_hi; }
  }
  if (p.wqkv == nullptr) {   // last block: ln_f output in fp32 (model2_seq.py:274)
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      const int n = j * 8 + 2 * t;
      if (ok_lo) *reinterpret_cast<float2*>(p.yf + (size_t)r_lo * C + n) = make_float2(acc2[j][0], acc2[j][1]);
      if (ok_hi) *reinterpret_cast<float2*>(p.yf + (size_t)r_hi * C + n) = make_float2(acc2[j][2], acc2[j][3]);
    }
    return;
  }
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const uint32_t lo = pack2(acc2[j][0], acc2[j][1]), hi = pack2(acc2[j][2], acc2[j][3]);
    hfr[j >> 1][(j & 1) * 2] = lo;
    hfr[j >> 1][(j & 1) * 2 + 1] = hi;
    const int n = j * 8 + 2 * t;
    if (ok_lo) *reinterpret_cast<uint32_t*>(p.hn + (size_t)r_lo * C + n) = lo;
    if (ok_hi) *reinterpret_cast<uint32_t*>(p.hn + (size_t)r_hi * C + n) = hi;
  }
  // ---------------------------------------------------------------- next block's fused QKV, 64 output columns at a time
  for (int qc = 0; qc < N_QKV; ++qc) {
    const int s = 1 + N_MLP + qc;
    acquire(s);
    const __nv_bfloat16* wq = ring + (s % NS) * CHUNK;
    float qa[8][4];
#pragma unroll
    for (int j = 0; j < 8; ++j) { qa[j][0] = qa[j][1] = qa[j][2] = qa[j][3] = 0.f; }
    warp_gemm<8, KS>(qa, hfr, wq, LDW, lane);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int n = qc * 64 + j * 8 + 2 * t;
      const float2 b = *reinterpret_cast<const float2*>(v_bqkv + n);
      if (ok_lo) *reinterpret_cast<uint32_t*>(p.qkv + (size_t)r_lo * (3 * C) + n) = pack2(qa[j][0] + b.x, qa[j][1] + b.y);
      if (ok_hi) *reinterpret_cast<uint32_t*>(p.qkv + (size_t)r_hi * (3 * C) + n) = pack2(qa[j][2] + b.x, qa[j][3] + b.y);
    }
    release(s);
  }
}

template <int C>
static int launch_chain_fwd(const ChainFwdArgs& a, cudaStream_t st) {
  constexpr int LDW = C + 8, LDW2 = 72;
  constexpr int CHUNK = (C * LDW > 64 * LDW + C * LDW2) ? C * LDW : 64 * LDW + C * LDW2;
  constexpr int SMEM = (ChainCfg<C>::NS_FWD * CHUNK + CH_WARPS * 16 * LDW) * 2 + (CH_WARPS * 16 * (C + 8) + 13 * C) * 4;
  static_assert(SMEM <= 232448, "shared memory budget");
  static bool configured_on[64] = {};
  bool& configured = per_device_flag(configured_on);
  if (!configured) {
    if (cudaFuncSetAttribute(chain_fwd_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM) != cudaSuccess) return check_launch("chain_fwd/attr");
    configured = true;
  }
  launch_pdl(chain_fwd_kernel<C>, dim3(cdiv(a.M, CH_ROWS)), dim3(CH_THREADS), (size_t)SMEM, st, a);
  return check_launch("chain_fwd");
}

}  // namespace dsf

using namespace dsf;

extern "C" int dsf_chain_fwd(const void* y, const float* x_in, const void* wp, const void* w1, const void* w2, const void* wqkv_next,
                             const float* bp, const float* b1, const float* b2, const float* bqkv_next, const float* ln2_g,
                             const float* ln2_b, const float* lnn_g, const float* lnn_b, float* x_mid, float* x_out, void* h2, void* a,
                             void* h_next, void* qkv_next, float* yf, float* mean2, float* rstd2, float* mean_next, float* rstd_next,
                             int32_t M, int32_t C, float eps, void* stream) {
  DSF_REQUIRE(C == 64 || C == 128, "chain_fwd: n_embd must be 64 or 128 (wider stages use the tcgen05 GEMM kernels), got %d", C);
  DSF_REQUIRE(M > 0, "chain_fwd: M must be positive");
  DSF_REQUIRE(y && x_in && wp && w1 && w2 && bp && b1 && b2 && ln2_g && ln2_b && lnn_g && lnn_b && x_mid && x_out && h2 && a && mean2 && rstd2 &&
                  mean_next && rstd_next, "chain_fwd: NULL pointer");
  DSF_REQUIRE(wqkv_next ? (bqkv_next && h_next && qkv_next) : (yf != nullptr),
              "chain_fwd: the next block's QKV needs bqkv / h_next / qkv_next; the last block needs yf");
  DSF_REQUIRE(aligned16(y) && aligned16(x_in) && aligned16(wp) && aligned16(w1) && aligned16(w2) && aligned16(wqkv_next) && aligned16(x_mid) &&
                  aligned16(x_out) && aligned16(h2) && aligned16(a) && aligned16(h_next) && aligned16(qkv_next) && aligned16(yf) && aligned16(bp) &&
                  aligned16(b1) && aligned16(b2) && aligned16(bqkv_next) && aligned16(ln2_g) && aligned16(ln2_b) && aligned16(lnn_g) && aligned16(lnn_b),
              "chain_fwd: 16-byte alignment required");
  ChainFwdArgs p{(const __nv_bfloat16*)y, x_in, (const __nv_bfloat16*)wp, (const __nv_bfloat16*)w1, (const __nv_bfloat16*)w2,
                 (const __nv_bfloat16*)wqkv_next, bp, b1, b2, bqkv_next, ln2_g, ln2_b, lnn_g, lnn_b, x_mid, x_out, (__nv_bfloat16*)h2,
                 (__nv_bfloat16*)a, (__nv_bfloat16*)h_next, (__nv_bfloat16*)qkv_next, yf, mean2, rstd2, mean_next, rstd_next, M, eps};
  return C == 64 ? launch_chain_fwd<64>(p, (cudaStream_t)stream) : launch_chain_fwd<128>(p, (cudaStream_t)stream);
}

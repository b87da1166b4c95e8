// K4 (v2): warp-specialised, TMA-fed flash attention forward / backward on tcgen05 + TMEM.
// Same math and I/O contract as attn_tc.cu (model2_seq.py:102-106 and its autograd); the difference is
// the schedule:
//   * a producer warp streams Q / K / V / dO tiles with 3-D TMA (tensor maps over (3C, T, B), out-of-range
//     token rows zero-filled) into swizzled shared memory through an mbarrier ring,
//   * one elected thread issues every tcgen05.mma, running ahead of the math warps (S(j+1) is issued before
//     softmax(j) finishes; the P.V / dV / dK / dQ MMAs are issued as soon as the bf16 tile lands in smem),
//   * forward: one softmax warpgroup per 128 query rows, two CTAs per SM; S and P are double-buffered in TMEM,
//   * backward: accumulators (dK, dV / dQ) stay in TMEM across the whole loop, S/dP are double-buffered.
// Shared-memory operand images: TMA tiles are [half][row][ROWB bytes] with the hardware swizzle that matches
// ROWB (128/64/32 B for head sizes >=64/32/16); the same image is read as a K-major operand (rows = M/N)
// or an MN-major operand (rows = K).  P / dS are written by the math warps back into tensor memory (bf16, two
// per column) and feed the next MMA as TS-mode A operands.
#include <algorithm>

#include "tc_common.cuh"

namespace dsf {

using namespace tc;

__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// ---- optional in-kernel timeline (make trace -> libdsfuse_trace.so, scripts/attn_trace.py): CTA (0,0,0) of the forward and
// dK/dV kernels stamps clock64() at the hand-over points of one warp per math warpgroup (rows 0, 1; the forward has one) and
// of its MMA warp (row 2).
#ifdef DSF_ATTN_TRACE
__device__ long long g_attn_trace[3][64][6];
#define TRACE(who, it, slot)                                                                               \
  do {                                                                                                     \
    if (blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && (threadIdx.x & 31) == 0 && (it) < 64)     \
      g_attn_trace[who][it][slot] = clock64();                                                             \
  } while (0)
#else
#define TRACE(who, it, slot) do {} while (0)
#endif

__device__ __forceinline__ float ex2_approx(float x) {  // 2^x, MUFU.EX2 without the denormal fix-up of exp2f()
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// ---- packed fp32 pairs (sm_100 FFMA2 / FADD2: two lanes of fp32 per instruction, half the issue slots of the scalar forms)
__device__ __forceinline__ uint64_t pack2(float lo, float hi) { uint64_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void unpack2(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) { uint64_t d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) { uint64_t d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) { uint64_t d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
// 2^x for a pair on the FMA / ALU pipes instead of MUFU.EX2 (the forward kernel's softmax is MUFU-bound: 64 exponentials per
// row and tile against 16 per clock and SM).  Cody-Waite: n = round(x) via the 1.5 * 2^23 trick, f = x - n in [-0.5, 0.5],
// 2^f by a cubic (max relative error 7.5e-5 — the result is rounded to bf16, 2e-3, right after), n added into the exponent field.
__device__ __forceinline__ void ex2_poly2(uint64_t x, float& p0, float& p1) {
  float x0, x1;
  unpack2(x, x0, x1);
  const uint64_t xc = pack2(fmaxf(x0, -126.f), fmaxf(x1, -126.f));
  const uint64_t t = add2(xc, pack2(12582912.f, 12582912.f));
  const uint64_t r = add2(t, pack2(-12582912.f, -12582912.f));
  const uint64_t f = fma2(r, pack2(-1.f, -1.f), xc);
  uint64_t q = fma2(f, pack2(0.05517164617776871f, 0.05517164617776871f), pack2(0.2426111251115799f, 0.2426111251115799f));
  q = fma2(q, f, pack2(0.6932609677314758f, 0.6932609677314758f));
  q = fma2(q, f, pack2(0.9999280571937561f, 0.9999280571937561f));
  float q0, q1, t0, t1;
  unpack2(q, q0, q1);
  unpack2(t, t0, t1);
  p0 = __int_as_float(__float_as_int(q0) + (__float_as_int(t0) << 23));
  p1 = __int_as_float(__float_as_int(q1) + (__float_as_int(t1) << 23));
}

// 2^x of a packed pair on MUFU.EX2
__device__ __forceinline__ uint64_t ex2_pair(uint64_t x) {
  float x0, x1;
  unpack2(x, x0, x1);
  return pack2(ex2_approx(x0), ex2_approx(x1));
}
// (Packing on the ALU pipe instead of cvt.rn.bf16x2 — bit pattern + 0x8000, then one byte permute per pair — measured slower in all
// three kernels: forward 24.4 -> 25.7 us, dK/dV 28.7 -> 30.7 us at head size 16; profiles/r02al_attn_pack_alu.txt.)
__device__ __forceinline__ uint32_t pack_bf16x2_pair(uint64_t v) {
  float lo, hi;
  unpack2(v, lo, hi);
  return pack_bf16x2(lo, hi);
}

// Attention-probability dropout (attn_drop, model2_seq.py:104).  Decisions use 8-bit thresholds (p is quantised to
// k/256, scale = 256/(256-k)) so that one Philox4x32 call yields 16 of them; the forward kernel writes the keep
// bits of every (b, h, q) row to a bitmap (Tw 32-bit words per row) and the backward kernels read them back.
struct AttnDrop {
  uint32_t thresh8;  // drop iff random byte < thresh8; 0 = disabled
  float scale;
  uint32_t k0, k1, site;
  uint32_t* bits;    // (B, nh, T, Tw)
  int Tw;
  const unsigned long long* seed_dev;  // nullable device word XOR-ed into the Philox key (graph-safe reseeding)
};
// keep bits of keys 32*word .. 32*word+31 of row `rowid`
__device__ __forceinline__ uint32_t attn_keep_word(const AttnDrop& a, uint64_t rowid, uint32_t word) {
  uint32_t out = 0;
  const uint32_t t4 = a.thresh8 * 0x01010101u;
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const uint4 r = philox4x32(a.k0, a.k1, (uint32_t)rowid, (uint32_t)(rowid >> 32), word * 2 + c, a.site);
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t ge = __vcmpgeu4(w[k], t4) & 0x01010101u;           // one flag bit per byte
      out |= (((ge * 0x01020408u) >> 24) & 0xFu) << (c * 16 + k * 4);   // gather the 4 flags into a nibble
    }
  }
  return out;
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

template <int HS>
struct HeadCfg {
  static constexpr int BOXC = HS < 64 ? HS : 64;  // TMA box columns (elements)
  static constexpr int ROWB = BOXC * 2;           // bytes per shared-memory row of one box
  static constexpr int NHALF = HS / BOXC;         // boxes per tile along the head dimension
  static constexpr uint32_t SWZ = ROWB == 128 ? SWZ_128B : (ROWB == 64 ? SWZ_64B : SWZ_32B);
  static constexpr int KPH = ROWB / 32;           // UMMA K-steps (16 elements) per box
};

// K-major operand over a TMA tile of R rows (rows = M or N index); k-step kk covers head dims 16kk..16kk+15
template <int HS>
__device__ __forceinline__ uint64_t kmaj_desc(uint32_t tile, int R, int kk) {
  using H = HeadCfg<HS>;
  const uint32_t off = (uint32_t)(kk / H::KPH) * R * H::ROWB + (uint32_t)(kk % H::KPH) * 32;
  return make_smem_desc(tile + off, 16, 8 * H::ROWB, H::SWZ);
}
// MN-major operand over a TMA tile of R rows (rows = K index, N = HS); k-step kk covers rows 16kk..16kk+15
template <int HS>
__device__ __forceinline__ uint64_t mnmaj_desc(uint32_t tile, int R, int kk) {
  using H = HeadCfg<HS>;
  return make_smem_desc(tile + (uint32_t)kk * 16 * H::ROWB, (uint32_t)R * H::ROWB, 8 * H::ROWB, H::SWZ);
}
// The MMA-issuing helpers below are WARP-COLLECTIVE: all 32 lanes of the issuer warp call them with uniform
// arguments.  Base descriptors are computed in warp-uniform control flow (so they live in uniform registers) and
// per-k-step offsets are compile-time immediates; only the tcgen05.mma / tcgen05.commit themselves run under
// elect.sync.  (Computing descriptors inside a divergent `if (lane == 0)` costs ~13 SASS instructions and a
// BRA.U.ANY uniformity loop per MMA — more than the 32-64 cycles one 128xNx16 MMA occupies the tensor pipe.)
__device__ __forceinline__ void tc_commit_elect(uint32_t bar) {
  if (elect_one()) tc::tc_commit(bar);
  __syncwarp();
}
// D[128 x NB] (+)= A(tile, RA rows, K-major) . B(tile, RB rows, K-major)^T, contraction over the head dim
template <int HS>
__device__ __forceinline__ void mma_over_head(uint32_t tmem_d, uint32_t a_tile, int RA, uint32_t b_tile, int RB, uint32_t idesc) {
  using H = HeadCfg<HS>;
  const uint64_t da = make_smem_desc(a_tile, 16, 8 * H::ROWB, H::SWZ), db = make_smem_desc(b_tile, 16, 8 * H::ROWB, H::SWZ);
  if (elect_one()) {
#pragma unroll
    for (int kk = 0; kk < HS / 16; ++kk) {
      const uint32_t oa = (uint32_t)(kk / H::KPH) * RA * H::ROWB + (uint32_t)(kk % H::KPH) * 32;
      const uint32_t ob = (uint32_t)(kk / H::KPH) * RB * H::ROWB + (uint32_t)(kk % H::KPH) * 32;
      tc_mma_bf16(tmem_d, da + (oa >> 4), db + (ob >> 4), idesc, kk != 0);
    }
  }
  __syncwarp();
}
// D[128 x HS] (+)= P(tensor memory, [128 x KC] bf16 packed two per column at p_tmem) . B(tile with KC rows, MN-major)
// CW = 0 (forward): the packed columns are contiguous (8 per K = 16 step).  CW = 32 (backward kernels): every math warpgroup owns
// 32 fp32 columns of the tile and overwrites the first 16 of them with its packed values, so K-step kk (16 values = 8 packed
// columns) sits at column (16 kk / CW) * CW + (16 kk % CW) / 2: 0, 8, 32, 40.
template <int HS, int KC, int CW = 0>
__device__ __forceinline__ void mma_over_rows_ts(uint32_t tmem_d, uint32_t p_tmem, uint32_t b_tile, uint32_t idesc, bool accumulate) {
  using H = HeadCfg<HS>;
  const uint64_t db = make_smem_desc(b_tile, (uint32_t)KC * H::ROWB, 8 * H::ROWB, H::SWZ);
  const uint32_t acc = accumulate ? 1u : 0u;
  if (elect_one()) {
#pragma unroll
    for (int kk = 0; kk < KC / 16; ++kk) {
      const uint32_t col = CW > 0 ? (uint32_t)((kk * 16 / (CW > 0 ? CW : 1)) * CW + (kk * 16 % (CW > 0 ? CW : 1)) / 2) : (uint32_t)(kk * 8);
      tc_mma_bf16_ts(tmem_d, p_tmem + col, db + (uint32_t)((kk * 16 * H::ROWB) >> 4), idesc, kk == 0 ? acc : 1u);
    }
  }
  __syncwarp();
}

// D[128 x NB] (+)= A(tensor memory: 128 rows x HS bf16, packed two per column at a_tmem) . B(tile, RB rows, K-major)^T
template <int HS>
__device__ __forceinline__ void mma_over_head_ts(uint32_t tmem_d, uint32_t a_tmem, uint32_t b_tile, int RB, uint32_t idesc) {
  using H = HeadCfg<HS>;
  const uint64_t db = make_smem_desc(b_tile, 16, 8 * H::ROWB, H::SWZ);
  if (elect_one()) {
#pragma unroll
    for (int kk = 0; kk < HS / 16; ++kk) {
      const uint32_t ob = (uint32_t)(kk / H::KPH) * RB * H::ROWB + (uint32_t)(kk % H::KPH) * 32;
      tc_mma_bf16_ts(tmem_d, a_tmem + (uint32_t)(kk * 8), db + (ob >> 4), idesc, kk != 0);
    }
  }
  __syncwarp();
}

template <int HS>
__device__ __forceinline__ void tma_tile(uint32_t dst, const CUtensorMap* m, uint32_t bar, int col0, int row0, int b, int R) {
  using H = HeadCfg<HS>;
#pragma unroll
  for (int hf = 0; hf < H::NHALF; ++hf) tma_load_3d(dst + hf * R * H::ROWB, m, bar, col0 + hf * H::BOXC, row0, b);
}

__device__ __forceinline__ void store_row16_bf16(__nv_bfloat16* dst, const uint32_t (&a)[16], float scale) {
#pragma unroll
  for (int e = 0; e < 16; e += 8)
    *reinterpret_cast<uint4*>(dst + e) =
        make_uint4(pack_bf16x2(__uint_as_float(a[e]) * scale, __uint_as_float(a[e + 1]) * scale),
                   pack_bf16x2(__uint_as_float(a[e + 2]) * scale, __uint_as_float(a[e + 3]) * scale),
                   pack_bf16x2(__uint_as_float(a[e + 4]) * scale, __uint_as_float(a[e + 5]) * scale),
                   pack_bf16x2(__uint_as_float(a[e + 6]) * scale, __uint_as_float(a[e + 7]) * scale));
}

// =============================================================================================== forward
// =============================================================================================== backward: dK, dV
// CTA = 128 keys (K, V resident); loop over BQ-query tiles.  Threads own key rows:
//   S^T = K Q^T, dP^T = V dO^T -> P^T = exp2(S^T*c - lse), dS^T = P^T (dP^T - delta) * scale -> dV += P^T dO, dK += dS^T Q
// P^T / dS^T are written back (bf16, two per column) over the S^T / dP^T tiles in tensor memory and feed the dV / dK MMAs as
// TS-mode A operands; per-query statistics (lse, delta) are staged per WARP in shared memory (each lane fetches one pair a
// tile ahead, a __syncwarp publishes them), so the math warps never meet at a CTA-wide barrier inside the loop.
// Two math warpgroups of 128 threads split a tile's 64 query columns, 32 each (both work on EVERY tile); the note above
// launch_bwd_kv has the measurements of the four-warpgroup variant that was removed.
template <int HS, int BQ, int ST>
struct BwdKV2 {
  static constexpr int KV_BYTES = 128 * HS * 2, Q_BYTES = BQ * HS * 2;
  static constexpr int K_OFF = 0, V_OFF = KV_BYTES, Q_OFF = 2 * KV_BYTES, DO_OFF = Q_OFF + ST * Q_BYTES;
  static constexpr int BAR_OFF = DO_OFF + ST * Q_BYTES;
  static constexpr int NBAR = 2 + 2 * ST + 4;
  static constexpr int STAT_OFF = BAR_OFF + NBAR * 8 + 16;  // lse (log2 units) | delta of ALL queries of this (batch, head), padded to tiles
  static constexpr int THREADS = 256 + 64;
  static_assert(4 * BQ + 2 * HS <= 512, "TMEM budget");
  static_assert(STAT_OFF % 16 == 0, "float4 reads of the statistics");
  static int dyn_bytes(int T) { return STAT_OFF + 2 * cdiv(T, BQ) * BQ * 4 + 1024; }
};

// The dropout-free math runs on packed fp32 pairs.
template <int HS, int BQ, int ST, bool DROP>
__global__ void __launch_bounds__(256 + 64, 1)
attn_bwd_kv2_kernel(const __grid_constant__ CUtensorMap tmKV, const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmDO,
                    const float* __restrict__ lse, const float* __restrict__ delta, __nv_bfloat16* __restrict__ dqkv, int T, int C, int nh,
                    float scale, AttnDrop ad) {
  using L = BwdKV2<HS, BQ, ST>;
  constexpr int MMAW = 8, TMAW = 9;  // warp roles: 0 .. 7 math, then MMA issuer, TMA producer
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (sbase - smem_u32(smem_raw));
  const uint32_t bar0 = sbase + L::BAR_OFF;
  const uint32_t kv_full = bar0, acc_done = bar0 + 8, q_full = bar0 + 16, q_empty = q_full + 8 * ST, s_full = q_empty + 8 * ST,
                 ds_full = s_full + 16, tmem_slot = ds_full + 16;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;  // warp-uniform for the compiler
  const int kv0 = blockIdx.x * 128, h = blockIdx.y, b = blockIdx.z;
  const int n_q = (T + BQ - 1) / BQ;

  pdl_trigger();
  if (threadIdx.x == 0) {
    mbar_init(kv_full, 1);
    mbar_init(acc_done, 1);
    for (int s = 0; s < ST; ++s) { mbar_init(q_full + 8 * s, 1); mbar_init(q_empty + 8 * s, 1); }
    for (int w = 0; w < 2; ++w) { mbar_init(s_full + 8 * w, 1); mbar_init(ds_full + 8 * w, 256); }
    fence_barrier_init();
  }
  if (warp == MMAW) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  if (warp == TMAW && lane == 0) { tma_prefetch_desc(&tmKV); tma_prefetch_desc(&tmQ); tma_prefetch_desc(&tmDO); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  pdl_wait();  // set-up above overlaps the previous kernel's tail
  const uint32_t tm_dv = tmem_base + 4 * BQ, tm_dk = tm_dv + HS;

  if (warp == TMAW) {
    if (lane == 0) {
      mbar_expect_tx(kv_full, 2 * L::KV_BYTES);
      tma_tile<HS>(sbase + L::K_OFF, &tmKV, kv_full, C + h * HS, kv0, b, 128);
      tma_tile<HS>(sbase + L::V_OFF, &tmKV, kv_full, 2 * C + h * HS, kv0, b, 128);
      for (int i = 0; i < n_q; ++i) {
        const int st = i % ST;
        if (i >= ST) mbar_wait(q_empty + 8 * st, ((i / ST) - 1) & 1);
        mbar_expect_tx(q_full + 8 * st, 2 * L::Q_BYTES);
        tma_tile<HS>(sbase + L::Q_OFF + st * L::Q_BYTES, &tmQ, q_full + 8 * st, h * HS, i * BQ, b, BQ);
        tma_tile<HS>(sbase + L::DO_OFF + st * L::Q_BYTES, &tmDO, q_full + 8 * st, h * HS, i * BQ, b, BQ);
      }
    }
  } else if (warp == MMAW) {
    {  // MMA issuer: all 32 lanes walk the schedule (uniform control flow); single lanes are elected per instruction
      constexpr uint32_t idesc_s = make_idesc_bf16(128, BQ, 0, 0);
      constexpr uint32_t idesc_g = make_idesc_bf16(128, HS, 0, 1);
      mbar_wait(kv_full, 0);
      mbar_wait(q_full, 0);
      tc_fence_after();
      mma_over_head<HS>(tmem_base, sbase + L::K_OFF, 128, sbase + L::Q_OFF, BQ, idesc_s);
      mma_over_head<HS>(tmem_base + BQ, sbase + L::V_OFF, 128, sbase + L::DO_OFF, BQ, idesc_s);
      tc_commit_elect(s_full);
      for (int i = 0; i < n_q; ++i) {
        const int bf = i & 1, st = i % ST;
        TRACE(2, i, 0);
        if (i + 1 < n_q) {
          // buffer bn is free: dV / dK (i-1) were issued after its math warps arrived at ds_full, and the tensor pipe runs in order
          const int sn = (i + 1) % ST, bn = (i + 1) & 1;
          mbar_wait(q_full + 8 * sn, ((i + 1) / ST) & 1);
          TRACE(2, i, 1);
          tc_fence_after();
          mma_over_head<HS>(tmem_base + bn * 2 * BQ, sbase + L::K_OFF, 128, sbase + L::Q_OFF + sn * L::Q_BYTES, BQ, idesc_s);
          mma_over_head<HS>(tmem_base + bn * 2 * BQ + BQ, sbase + L::V_OFF, 128, sbase + L::DO_OFF + sn * L::Q_BYTES, BQ, idesc_s);
          tc_commit_elect(s_full + 8 * bn);
        }
        TRACE(2, i, 2);
        mbar_wait(ds_full + 8 * bf, (i >> 1) & 1);
        TRACE(2, i, 3);
        tc_fence_after();
        mma_over_rows_ts<HS, BQ, 32>(tm_dv, tmem_base + bf * 2 * BQ, sbase + L::DO_OFF + st * L::Q_BYTES, idesc_g, i > 0);
        mma_over_rows_ts<HS, BQ, 32>(tm_dk, tmem_base + bf * 2 * BQ + BQ, sbase + L::Q_OFF + st * L::Q_BYTES, idesc_g, i > 0);
        tc_commit_elect(q_empty + 8 * st);
        TRACE(2, i, 4);
      }
      tc_commit_elect(acc_done);
    }
  } else {
    constexpr int CW = BQ / 2;  // query columns of a tile per warpgroup
    const int wgi = warp >> 2;  // warpgroup 0 / 1: columns wgi * CW ..
    const int row = (warp & 3) * 32 + lane;
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    const bool key_ok = (kv0 + row) < T;
    const float scale_log2 = scale * 1.4426950408889634f;
    const float* lse_g = lse + ((size_t)b * nh + h) * T;
    const float* delta_g = delta + ((size_t)b * nh + h) * T;
    static_assert(BQ == 64, "a 64-query tile in two 32-column shares");
    const size_t bh = (size_t)b * nh + h;
    const int kw = kv0 / 32 + (warp & 3);  // bitmap word holding this warp's 32 keys
    // lse (log2 units) and delta of every query of this (batch, head) are copied to shared memory ONCE by the math warps
    // (2 x 4 B x T: 7.7 KB at T = 962, 31 KB at T = 3842); tiles then read them with broadcast 16-byte loads.  (Staging them per
    // tile and warp cost ~250 of the ~1200 cycles a math warp spends on a tile.)  Padding queries get lse = +inf -> P = 0.  Both are stored negated.
    float* s_lse = reinterpret_cast<float*>(smem + L::STAT_OFF);
    float* s_delta = s_lse + n_q * BQ;
    for (int idx = threadIdx.x; idx < n_q * BQ; idx += 256) {
      s_lse[idx] = idx < T ? __ldg(lse_g + idx) * -1.4426950408889634f : -INFINITY;  // NEGATED: x = s * c + (-lse), d = p * (dp + (-delta))
      s_delta[idx] = idx < T ? -__ldg(delta_g + idx) : 0.f;
    }
    // attn-dropout: keep word of query (tile * BQ + wgi * CW + lane % CW) over this warp's 32 keys, fetched one tile ahead
    uint32_t wv = 0xFFFFFFFFu;
    auto fetch_w = [&](int it) {
      const int qq = it * BQ + wgi * CW + (lane % CW);
      wv = qq < T ? ad.bits[(bh * T + qq) * ad.Tw + kw] : 0u;
    };
    if (DROP) fetch_w(0);
    named_bar_sync(1, 256);  // statistics visible to all math warps
    for (int i = 0; i < n_q; ++i) {
      const int bf = i & 1;
      const float* wst = s_lse + i * BQ + wgi * CW;
      const float* wsd = s_delta + i * BQ + wgi * CW;
      const uint32_t myw = wv;
      if ((warp & 3) == 0) TRACE(wgi, i, 0);
      if (DROP && i + 1 < n_q) fetch_w(i + 1);
      if ((warp & 3) == 0) TRACE(wgi, i, 1);
      // s_full(i) also says that buffer bf is free: S^T / dP^T (i) were issued after dV / dK (i-2), the MMAs of one thread
      // complete in order, and the commit covers every MMA issued before it
      mbar_wait(s_full + 8 * bf, (i >> 1) & 1);
      if ((warp & 3) == 0) TRACE(wgi, i, 2);
      tc_fence_after();
      const uint32_t tm_s = tmem_base + bf * 2 * BQ + lane_off + wgi * CW, tm_dp = tm_s + BQ;
      uint32_t rs[CW], rp[CW];
      tmem_ld32(tm_s, rs);
      tmem_ld32(tm_dp, rp);
      tmem_wait_ld();
      if ((warp & 3) == 0) TRACE(wgi, i, 3);
      const uint64_t sc2 = pack2(scale_log2, scale_log2);
#pragma unroll
      for (int c = 0; c < CW; c += 16) {
        uint32_t pk[8], dk[8];
#pragma unroll
        for (int e = 0; e < 16; e += 4) {
          // rows of keys >= T hold finite garbage (K, V rows are zero-filled): they only reach the dK / dV rows of those
          // keys, which are never stored.  The 1/sqrt(hs) factor of dS is applied once when dK is drained.
          if (!DROP) {  // packed pairs: FFMA2 / FADD2 / FMUL2, two queries per instruction
            const ulonglong2 nl = *reinterpret_cast<const ulonglong2*>(wst + c + e);  // -lse of queries c+e .. c+e+3
            const ulonglong2 nd = *reinterpret_cast<const ulonglong2*>(wsd + c + e);  // -delta
#pragma unroll
            for (int u = 0; u < 4; u += 2) {
              const uint64_t x = fma2(pack2(__uint_as_float(rs[c + e + u]), __uint_as_float(rs[c + e + u + 1])), sc2, u ? nl.y : nl.x);
              const uint64_t p2 = ex2_pair(x);
              const uint64_t t2 = add2(pack2(__uint_as_float(rp[c + e + u]), __uint_as_float(rp[c + e + u + 1])), u ? nd.y : nd.x);
              pk[(e + u) / 2] = pack_bf16x2_pair(p2);
              dk[(e + u) / 2] = pack_bf16x2_pair(mul2(p2, t2));
            }
            continue;
          }
          const float4 l4 = *reinterpret_cast<const float4*>(wst + c + e);
          const float4 d4 = *reinterpret_cast<const float4*>(wsd + c + e);
          const float ls[4] = {l4.x, l4.y, l4.z, l4.w}, dl[4] = {d4.x, d4.y, d4.z, d4.w};
          float p[4], d[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            p[u] = ex2_approx(fmaf(__uint_as_float(rs[c + e + u]), scale_log2, ls[u]));
            float dp = __uint_as_float(rp[c + e + u]);
            // attn_drop: dV sees P*mask/(1-p); dP = dP_drop*mask/(1-p)
            const float m = (__shfl_sync(0xffffffffu, myw, c + e + u) >> lane) & 1u ? ad.scale : 0.f;
            dp *= m;
            d[u] = p[u] * (dp + dl[u]);
            p[u] *= m;
          }
          pk[e / 2] = pack_bf16x2(p[0], p[1]);
          pk[e / 2 + 1] = pack_bf16x2(p[2], p[3]);
          dk[e / 2] = pack_bf16x2(d[0], d[1]);
          dk[e / 2 + 1] = pack_bf16x2(d[2], d[3]);
        }
        // packed pairs of columns c .. c+15 -> 8 columns at c/2 of this warpgroup's CW-column region (mma_over_rows_ts CW layout);
        // the first store only overwrites columns whose values already sit in registers
        tmem_st8(tm_s + c / 2, pk);
        tmem_st8(tm_dp + c / 2, dk);
      }
      if ((warp & 3) == 0) TRACE(wgi, i, 4);
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(ds_full + 8 * bf);
      if ((warp & 3) == 0) TRACE(wgi, i, 5);
    }
    mbar_wait(acc_done, 0);
    tc_fence_after();
    const int ld = 3 * C;
    __nv_bfloat16* dk_row = dqkv + ((size_t)b * T + kv0 + row) * ld + C + h * HS;
    __nv_bfloat16* dv_row = dk_row + C;
    // warpgroup 0 drains dK, warpgroup 1 dV.  (wgi is 0 or 1, but the compiler cannot tell: `which` and `part` keep the
    // instructions this kernel was measured with.)
    const int which = wgi & 1, part = wgi >> 1;
    if (part < 1) {
#pragma unroll 1
      for (int c = part * HS; c < (part + 1) * HS; c += 16) {
        uint32_t a[16];
        tmem_ld16((which == 0 ? tm_dk : tm_dv) + lane_off + c, a);
        tmem_wait_ld();
        if (key_ok) store_row16_bf16((which == 0 ? dk_row : dv_row) + c, a, which == 0 ? scale : 1.0f);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == MMAW) tmem_dealloc(tmem_base, 512);
}

// =============================================================================================== backward: dQ
// CTA = 128 queries (Q, dO resident); loop over 64-key tiles.  Threads own query rows:
//   S = Q K^T, dP = dO V^T -> dS = exp2(S*c - lse) (dP - delta) * scale -> dQ += dS K
// dS (bf16) is written back over the dP tile in tensor memory and feeds dQ += dS K as a TS-mode A operand.
// The two stationary operands, the Q and dO rows of the CTA's 128 queries, live in tensor memory (written once by the math
// warps straight from global memory) and feed the S = Q K^T and dP = dO V^T MMAs as TS-mode A operands.  A tcgen05.mma whose A
// operand comes from shared memory spends ~128 cycles fetching its 128 x 16 slice whatever N is, so the 64-wide S / dP MMAs ran
// at a quarter of the tensor pipe's rate; from tensor memory they are N-bound (measured +-0 at T = 962, +6 % at T = 3842; the
// shared-memory variant was removed).
template <int HS, int ST>
struct BwdQ2 {
  static constexpr int BKV = 64;
  static constexpr int Q_BYTES = 128 * HS * 2, KV_BYTES = BKV * HS * 2;
  // the K / V rings start after 2 * Q_BYTES that nothing reads (where the shared-memory Q / dO tiles were): the layout as measured
  static constexpr int K_OFF = 2 * Q_BYTES, V_OFF = K_OFF + ST * KV_BYTES;
  static constexpr int BAR_OFF = V_OFF + ST * KV_BYTES;
  static constexpr int NBAR = 2 + 2 * ST + 4;
  static constexpr int DYN = BAR_OFF + NBAR * 8 + 16 + 1024;
  static_assert(4 * BKV + HS <= 512, "TMEM budget");
};

// Two math warpgroups share every key tile (32 columns each), as in the dK/dV kernel.
template <int HS, int ST, bool DROP>
__global__ void __launch_bounds__(256 + 64, 1)
attn_bwd_q2_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmDO, const __grid_constant__ CUtensorMap tmKV,
                   const float* __restrict__ lse, const float* __restrict__ delta, __nv_bfloat16* __restrict__ dqkv, int T, int C, int nh,
                   float scale, AttnDrop ad, const __nv_bfloat16* __restrict__ qkv, const __nv_bfloat16* __restrict__ dy) {
  using L = BwdQ2<HS, ST>;
  constexpr int BKV = L::BKV;
  constexpr int MMAW = 8, TMAW = 9;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar0 = sbase + L::BAR_OFF;
  const uint32_t q_full = bar0, acc_done = bar0 + 8, kv_full = bar0 + 16, kv_empty = kv_full + 8 * ST, s_full = kv_empty + 8 * ST,
                 ds_full = s_full + 16, tmem_slot = ds_full + 16;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;  // warp-uniform for the compiler
  const int q0 = blockIdx.x * 128, h = blockIdx.y, b = blockIdx.z;
  const int n_kv = (T + BKV - 1) / BKV;
  constexpr uint32_t TMEM_COLS = (4 * BKV + HS + (HS >= 32 ? HS : 32)) <= 256 ? 256 : 512;
  static_assert(4 * BKV + 2 * HS <= 512, "TMEM budget (S/dP double-buffered, dQ, Q and dO rows)");

  pdl_trigger();
  if (threadIdx.x == 0) {
    mbar_init(q_full, 256);
    mbar_init(acc_done, 1);
    for (int s = 0; s < ST; ++s) { mbar_init(kv_full + 8 * s, 1); mbar_init(kv_empty + 8 * s, 1); }
    for (int w = 0; w < 2; ++w) { mbar_init(s_full + 8 * w, 1); mbar_init(ds_full + 8 * w, 256); }
    fence_barrier_init();
  }
  if (warp == MMAW) { tmem_alloc(tmem_slot, TMEM_COLS); tmem_relinquish(); }
  if (warp == TMAW && lane == 0) { tma_prefetch_desc(&tmKV); tma_prefetch_desc(&tmQ); tma_prefetch_desc(&tmDO); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  pdl_wait();  // set-up above overlaps the previous kernel's tail
  const uint32_t tm_dq = tmem_base + 4 * BKV;
  const uint32_t tm_q = tm_dq + HS, tm_do = tm_q + (HS >= 32 ? HS / 2 : 16);  // packed Q / dO rows (HS/2 columns each, >= 16 apart)

  if (warp == TMAW) {
    if (lane == 0) {
      for (int j = 0; j < n_kv; ++j) {
        const int st = j % ST;
        if (j >= ST) mbar_wait(kv_empty + 8 * st, ((j / ST) - 1) & 1);
        mbar_expect_tx(kv_full + 8 * st, 2 * L::KV_BYTES);
        tma_tile<HS>(sbase + L::K_OFF + st * L::KV_BYTES, &tmKV, kv_full + 8 * st, C + h * HS, j * BKV, b, BKV);
        tma_tile<HS>(sbase + L::V_OFF + st * L::KV_BYTES, &tmKV, kv_full + 8 * st, 2 * C + h * HS, j * BKV, b, BKV);
      }
    }
  } else if (warp == MMAW) {
    {  // MMA issuer: all 32 lanes walk the schedule (uniform control flow); single lanes are elected per instruction
      constexpr uint32_t idesc_s = make_idesc_bf16(128, BKV, 0, 0);
      constexpr uint32_t idesc_q = make_idesc_bf16(128, HS, 0, 1);
      mbar_wait(q_full, 0);
      mbar_wait(kv_full, 0);
      tc_fence_after();
      mma_over_head_ts<HS>(tmem_base, tm_q, sbase + L::K_OFF, BKV, idesc_s);
      mma_over_head_ts<HS>(tmem_base + BKV, tm_do, sbase + L::V_OFF, BKV, idesc_s);
      tc_commit_elect(s_full);
      for (int j = 0; j < n_kv; ++j) {
        const int bf = j & 1, st = j % ST;
        if (j + 1 < n_kv) {
          const int sn = (j + 1) % ST, bn = (j + 1) & 1;
          mbar_wait(kv_full + 8 * sn, ((j + 1) / ST) & 1);
          tc_fence_after();
          mma_over_head_ts<HS>(tmem_base + bn * 2 * BKV, tm_q, sbase + L::K_OFF + sn * L::KV_BYTES, BKV, idesc_s);
          mma_over_head_ts<HS>(tmem_base + bn * 2 * BKV + BKV, tm_do, sbase + L::V_OFF + sn * L::KV_BYTES, BKV, idesc_s);
          tc_commit_elect(s_full + 8 * bn);
        }
        mbar_wait(ds_full + 8 * bf, (j >> 1) & 1);
        tc_fence_after();
        mma_over_rows_ts<HS, BKV, 32>(tm_dq, tmem_base + bf * 2 * BKV + BKV, sbase + L::K_OFF + st * L::KV_BYTES, idesc_q, j > 0);
        tc_commit_elect(kv_empty + 8 * st);
      }
      tc_commit_elect(acc_done);
    }
  } else {
    constexpr int CW = BKV / 2;  // key columns of a tile per warpgroup
    static_assert(BKV == 64, "a 64-key tile in two 32-column shares");
    const int wgi = warp >> 2;   // warpgroup 0 / 1: columns wgi * CW ..
    const int row = (warp & 3) * 32 + lane;
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    const int q = q0 + row;
    const bool q_ok = q < T;
    const float scale_log2 = scale * 1.4426950408889634f;
    const float my_lse = q_ok ? lse[((size_t)b * nh + h) * T + q] * 1.4426950408889634f : INFINITY;
    const float my_delta = q_ok ? delta[((size_t)b * nh + h) * T + q] : 0.f;
    if (wgi < 2) {  // warpgroup 0 parks the Q row of its query in tensor memory, warpgroup 1 the dO row (two bf16 per column)
      const __nv_bfloat16* src = wgi == 0 ? qkv + ((size_t)b * T + q) * (3 * C) + h * HS : dy + ((size_t)b * T + q) * C + h * HS;
      const uint32_t dst = (wgi == 0 ? tm_q : tm_do) + lane_off;
#pragma unroll 1
      for (int c = 0; c < HS; c += 32) {
        uint32_t wds[16];
#pragma unroll
        for (int k = 0; k < 4; ++k) {  // head size 16: the row is only 32 bytes (2 x 16 B); the upper 8 columns are padding
          const bool real = q_ok && (HS >= 32 || k < 2);
          const uint4 v = real ? __ldg(reinterpret_cast<const uint4*>(src + c) + k) : make_uint4(0u, 0u, 0u, 0u);
          wds[4 * k] = v.x; wds[4 * k + 1] = v.y; wds[4 * k + 2] = v.z; wds[4 * k + 3] = v.w;
        }
        tmem_st16(dst + c / 2, wds);
      }
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(q_full);
    }
    // attn-dropout keep bits of (my query row, keys kv0 + wgi * CW ..): word 2j + wgi * CW / 32 of the row, fetched one tile ahead
    const uint32_t* my_bits = (DROP && q_ok) ? ad.bits + (((size_t)b * nh + h) * T + q) * ad.Tw + (wgi * CW) / 32 : nullptr;
    uint32_t wnext = my_bits ? my_bits[0] : 0xFFFFFFFFu;
    for (int j = 0; j < n_kv; ++j) {
      const int bf = j & 1, kv0 = j * BKV;
      const uint32_t keepw = wnext >> ((wgi * CW) % 32);
      if (my_bits && j + 1 < n_kv) wnext = my_bits[2 * (j + 1)];
      // s_full(j) also says that buffer bf is free: S / dP (j) were issued after dQ += dS K (j-2), one thread's MMAs complete in order
      mbar_wait(s_full + 8 * bf, (j >> 1) & 1);
      tc_fence_after();
      const uint32_t tm_s = tmem_base + bf * 2 * BKV + lane_off + wgi * CW, tm_dp = tm_s + BKV;
      const bool full = kv0 + BKV <= T;  // only the last key tile needs the column mask
      uint32_t rs[CW], rp[CW];
      tmem_ld32(tm_s, rs);
      tmem_ld32(tm_dp, rp);
      tmem_wait_ld();
#pragma unroll
      for (int c = 0; c < CW; c += 16) {
        uint32_t dk[8];
        // the 1/sqrt(hs) factor of dS is applied once when dQ is drained
        if (full && !DROP) {  // packed pairs: FFMA2 / FADD2 / FMUL2, two keys per instruction
          const uint64_t sc2 = pack2(scale_log2, scale_log2), nl2 = pack2(-my_lse, -my_lse), nd2 = pack2(-my_delta, -my_delta);
#pragma unroll
          for (int e = 0; e < 16; e += 2) {
            const uint64_t x = fma2(pack2(__uint_as_float(rs[c + e]), __uint_as_float(rs[c + e + 1])), sc2, nl2);
            const uint64_t p2 = ex2_pair(x);
            const uint64_t t2 = add2(pack2(__uint_as_float(rp[c + e]), __uint_as_float(rp[c + e + 1])), nd2);
            dk[e / 2] = pack_bf16x2_pair(mul2(p2, t2));
          }
        } else {
          const int k0 = kv0 + wgi * CW + c;  // first key of this sub-chunk
#pragma unroll
          for (int e = 0; e < 16; e += 2) {
            float p0 = (k0 + e < T) ? ex2_approx(fmaf(__uint_as_float(rs[c + e]), scale_log2, -my_lse)) : 0.f;
            float p1 = (k0 + e + 1 < T) ? ex2_approx(fmaf(__uint_as_float(rs[c + e + 1]), scale_log2, -my_lse)) : 0.f;
            float dp0 = __uint_as_float(rp[c + e]), dp1 = __uint_as_float(rp[c + e + 1]);
            if (DROP) {  // dP = dP_drop * mask/(1-p)
              dp0 *= (keepw >> (c + e)) & 1u ? ad.scale : 0.f;
              dp1 *= (keepw >> (c + e + 1)) & 1u ? ad.scale : 0.f;
            }
            dk[e / 2] = pack_bf16x2(p0 * (dp0 - my_delta), p1 * (dp1 - my_delta));
          }
        }
        tmem_st8(tm_dp + c / 2, dk);  // dS over the dP tile it came from (mma_over_rows_ts CW layout)
      }
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(ds_full + 8 * bf);
    }
    mbar_wait(acc_done, 0);
    tc_fence_after();
    __nv_bfloat16* dq_row = dqkv + ((size_t)b * T + q) * (3 * C) + h * HS;
    // the head's columns are drained in 16-column groups by as many warpgroups as there are groups (at most 2)
    constexpr int NG = (HS / 16) < 2 ? (HS / 16) : 2;
    constexpr int CH = HS / NG;
    const int g = wgi;
    if (g < NG) {
#pragma unroll 1
      for (int c = g * CH; c < (g + 1) * CH; c += 16) {
        uint32_t a[16];
        tmem_ld16(tm_dq + lane_off + c, a);
        tmem_wait_ld();
        if (q_ok) store_row16_bf16(dq_row + c, a, scale);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == MMAW) tmem_dealloc(tmem_base, TMEM_COLS);
}

// =============================================================================================== forward (v3 schedule)
// One softmax warpgroup owns the CTA's 128 query rows.  S and P are double-buffered so the softmax warps never wait for the
// tensor pipe: S(j+2) is issued as soon as softmax(j) has drained its S buffer, and softmax(j+1) may write its P tile while
// P.V(j) is still reading the other one.  K and V ride in separate TMA rings because K(j+2) is consumed two iterations ahead
// of V(j).  BKV = 64.  A CTA needs 192 threads, 256 TMEM columns and <= 113 KB of shared memory, so TWO of them share an SM
// (see attn_fwd_run for the measured alternative).
// The bf16 probabilities never touch shared memory: the softmax warps write them back (packed two per column) over the S tile
// they came from and P.V runs with its A operand in tensor memory (tcgen05.mma [d], [a], b-desc).
// POLY: every POLY-th pair of probabilities of a full, dropout-free tile is exponentiated by ex2_poly2 instead of MUFU.EX2
// (see attn_fwd_run for the measurements).
template <int HS, int KST, int VST>
struct Fwd3 {
  static constexpr int BKV = 64;
  static constexpr int POLY = HS >= 128 ? 4 : 3;
  static constexpr int Q_BYTES = 128 * HS * 2, KV_BYTES = BKV * HS * 2;
  static constexpr int Q_OFF = 0, K_OFF = Q_BYTES, V_OFF = K_OFF + KST * KV_BYTES, BAR_OFF = V_OFF + VST * KV_BYTES;
  static constexpr int NBAR = 1 + 2 * KST + 2 * VST + 12;
  static constexpr int DYN = BAR_OFF + NBAR * 8 + 16 + 1024;
  static constexpr int THREADS = 128 + 64;
  static constexpr uint32_t TMEM_COLS = 256;
  static_assert(2 * BKV + HS <= (int)TMEM_COLS, "TMEM budget");
  static_assert(DYN <= 232448 / 2 - 1024, "shared memory budget of two CTAs per SM");
};

template <int HS, int KST, int VST>
__global__ void __launch_bounds__(128 + 64, 2)
attn_fwd3_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV, __nv_bfloat16* __restrict__ y,
                 float* __restrict__ lse, int T, int C, int nh, float scale_log2, AttnDrop ad) {
  using L = Fwd3<HS, KST, VST>;
  constexpr int BKV = L::BKV, POLY = L::POLY;
  constexpr int MMAW = 4, TMAW = 5;  // warp roles: 0 .. 3 softmax, then MMA issuer, TMA producer
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar0 = sbase + L::BAR_OFF;
  // s_full / p_full / p_empty: two barriers (one per buffer) in 32-byte slots
  const uint32_t q_full = bar0, k_full = bar0 + 8, k_empty = k_full + 8 * KST, v_full = k_empty + 8 * KST, v_empty = v_full + 8 * VST,
                 s_full = v_empty + 8 * VST, p_full = s_full + 32, p_empty = p_full + 32, tmem_slot = p_empty + 32;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;  // warp-uniform for the compiler
  const int q0 = blockIdx.x * 128, h = blockIdx.y, b = blockIdx.z;
  const int n_kv = (T + BKV - 1) / BKV;

  pdl_trigger();
  if (threadIdx.x == 0) {
    mbar_init(q_full, 1);
    for (int s = 0; s < KST; ++s) { mbar_init(k_full + 8 * s, 1); mbar_init(k_empty + 8 * s, 1); }
    for (int s = 0; s < VST; ++s) { mbar_init(v_full + 8 * s, 1); mbar_init(v_empty + 8 * s, 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(s_full + 8 * i, 1); mbar_init(p_full + 8 * i, 128); mbar_init(p_empty + 8 * i, 1); }
    fence_barrier_init();
  }
  if (warp == MMAW) { tmem_alloc(tmem_slot, L::TMEM_COLS); tmem_relinquish(); }
  if (warp == TMAW && lane == 0) { tma_prefetch_desc(&tmQ); tma_prefetch_desc(&tmKV); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  pdl_wait();  // set-up above overlaps the previous kernel's tail
  if (ad.thresh8 && ad.seed_dev != nullptr) {  // graph-safe reseeding: fold the device word into the Philox key
    const unsigned long long sd = __ldg(ad.seed_dev);
    ad.k0 ^= (uint32_t)(sd & 0xFFFFFFFFull);
    ad.k1 ^= (uint32_t)(sd >> 32);
  }

  if (warp == TMAW) {
    if (lane == 0) {
      mbar_expect_tx(q_full, L::Q_BYTES);
      tma_tile<HS>(sbase + L::Q_OFF, &tmQ, q_full, h * HS, q0, b, 128);
      for (int j = 0; j < n_kv; ++j) {
        const int ks = j % KST, vs = j % VST;
        if (j >= KST) mbar_wait(k_empty + 8 * ks, ((j / KST) - 1) & 1);
        mbar_expect_tx(k_full + 8 * ks, L::KV_BYTES);
        tma_tile<HS>(sbase + L::K_OFF + ks * L::KV_BYTES, &tmKV, k_full + 8 * ks, C + h * HS, j * BKV, b, BKV);
        if (j >= VST) mbar_wait(v_empty + 8 * vs, ((j / VST) - 1) & 1);
        mbar_expect_tx(v_full + 8 * vs, L::KV_BYTES);
        tma_tile<HS>(sbase + L::V_OFF + vs * L::KV_BYTES, &tmKV, v_full + 8 * vs, 2 * C + h * HS, j * BKV, b, BKV);
      }
    }
  } else if (warp == MMAW) {
    {  // MMA issuer: all 32 lanes walk the schedule (uniform control flow); single lanes are elected per instruction
      constexpr uint32_t idesc_s = make_idesc_bf16(128, BKV, 0, 0);
      constexpr uint32_t idesc_o = make_idesc_bf16(128, HS, 0, 1);
      mbar_wait(q_full, 0);
      for (int jj = 0; jj < 2 && jj < n_kv; ++jj) {
        mbar_wait(k_full + 8 * (jj % KST), (jj / KST) & 1);
        tc_fence_after();
        mma_over_head<HS>(tmem_base + jj * BKV, sbase + L::Q_OFF, 128, sbase + L::K_OFF + (jj % KST) * L::KV_BYTES, BKV, idesc_s);
        tc_commit_elect(s_full + 8 * jj);
        tc_commit_elect(k_empty + 8 * (jj % KST));
      }
      for (int j = 0; j < n_kv; ++j) {
        const int buf = j & 1, vs = j % VST;
        TRACE(2, j, 0);
        mbar_wait(v_full + 8 * vs, (j / VST) & 1);
        TRACE(2, j, 1);
        mbar_wait(p_full + 8 * buf, (j >> 1) & 1);
        TRACE(2, j, 2);
        tc_fence_after();
        mma_over_rows_ts<HS, BKV>(tmem_base + 2 * BKV, tmem_base + buf * BKV, sbase + L::V_OFF + vs * L::KV_BYTES, idesc_o, j > 0);
        tc_commit_elect(p_empty + 8 * buf);
        tc_commit_elect(v_empty + 8 * vs);
        if (j + 2 < n_kv) {
          const int ks = (j + 2) % KST;
          mbar_wait(k_full + 8 * ks, ((j + 2) / KST) & 1);
          tc_fence_after();
          mma_over_head<HS>(tmem_base + buf * BKV, sbase + L::Q_OFF, 128, sbase + L::K_OFF + ks * L::KV_BYTES, BKV, idesc_s);
          tc_commit_elect(s_full + 8 * buf);
          tc_commit_elect(k_empty + 8 * ks);
        }
      }
    }
  } else {
    // w = warp >> 2 is 0 for every softmax warp, but the compiler cannot tell: the terms in w keep the instructions this kernel
    // was measured with
    const int w = warp >> 2;
    const int row = (warp & 3) * 32 + lane;
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    const uint32_t tm_o = tmem_base + 2 * BKV + w * HS + lane_off;
    float m_run = -INFINITY, l_run = 0.f;
    for (int j = 0; j < n_kv; ++j) {
      const int kv0 = j * BKV, buf = j & 1, sb = w * 2 + buf;
      const uint32_t tm_s = tmem_base + sb * BKV + lane_off;
      if ((warp & 3) == 0) TRACE(w, j, 0);
      mbar_wait(s_full + 8 * sb, (j >> 1) & 1);
      if ((warp & 3) == 0) TRACE(w, j, 1);
      tc_fence_after();
      uint32_t r0[32], r1[32];
      tmem_ld32(tm_s, r0);
      tmem_ld32(tm_s + 32, r1);
      tmem_wait_ld();
      if ((warp & 3) == 0) TRACE(w, j, 2);
      float p_max = -INFINITY;
      if (kv0 + BKV <= T) {
        // four independent chains of 3-input maxima (one 32-long dependent chain cost ~250 cycles of every tile's critical path)
        float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
        for (int i = 0; i < 32; ++i) m4[i & 3] = fmaxf(m4[i & 3], fmaxf(__uint_as_float(r0[i]), __uint_as_float(r1[i])));
        p_max = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          if (kv0 + i < T) p_max = fmaxf(p_max, __uint_as_float(r0[i]));
          if (kv0 + 32 + i < T) p_max = fmaxf(p_max, __uint_as_float(r1[i]));
        }
      }
      p_max *= scale_log2;
      // lazy rescale (exact: m only has to bound the exponent).  Measured and NOT kept: taking the exponentials speculatively against the
      // running maximum and tracking the row maximum inside that loop (tile repeated when it moved by > 8) removes this maximum pass
      // but lengthens the exponential loop: +1 .. 2.4 us per launch at every head size (profiles/r02sp_attn_fwd_speculative_tiles.txt).
      const bool need = p_max > m_run + 8.f;
      if (__any_sync(0xffffffffu, need)) {
        const float m_new = need ? p_max : m_run;
        const float alpha = ex2_approx(m_run - m_new);
        if (j > 0) {
          mbar_wait(p_empty + 8 * (w * 2 + ((j - 1) & 1)), ((j - 1) >> 1) & 1);  // P.V(j-1) retired: O is stable
          tc_fence_after();
#pragma unroll 1
          for (int c = 0; c < HS; c += 16) {
            uint32_t o[16];
            tmem_ld16(tm_o + c, o);
            tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < 16; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
            tmem_st16(tm_o + c, o);
          }
          tmem_wait_st();
        }
        l_run *= alpha;
        m_run = m_new;
      }
      if ((warp & 3) == 0) TRACE(w, j, 3);
      // the P buffer is the S tile itself, and s_full(j) already says it is free: S(j) was issued after P.V(j-2) by the same
      // thread, whose MMAs complete in order
      float l_add = 0.f;
      const bool full = kv0 + BKV <= T;
      const int qrow = q0 + 128 * w + row;
      const uint64_t rowid = ((uint64_t)b * nh + h) * T + qrow;
      if (full && !ad.thresh8) {
        // packed fast path: x = s * scale - m as FFMA2, the row sum as FADD2, every POLY-th pair off the MUFU pipe
        const uint64_t sc2 = pack2(scale_log2, scale_log2), nm2 = pack2(-m_run, -m_run);
        uint64_t lsum = pack2(0.f, 0.f);
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          uint32_t pk[16];
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            const uint32_t a0 = half ? r1[i] : r0[i], a1 = half ? r1[i + 1] : r0[i + 1];
            const uint64_t x = fma2(pack2(__uint_as_float(a0), __uint_as_float(a1)), sc2, nm2);
            float p0, p1;
            if ((i / 2) % POLY == POLY - 1) {
              ex2_poly2(x, p0, p1);
            } else {
              float x0, x1;
              unpack2(x, x0, x1);
              p0 = ex2_approx(x0);
              p1 = ex2_approx(x1);
            }
            lsum = add2(lsum, pack2(p0, p1));
            pk[i / 2] = pack_bf16x2(p0, p1);
          }
          tmem_st16(tm_s + half * 16, pk);
        }
        float l0, l1;
        unpack2(lsum, l0, l1);
        l_add = l0 + l1;
      } else
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t keepw = 0xFFFFFFFFu;
        if (ad.thresh8) {  // attn_drop: decide 32 keys, remember the bits for the backward kernels
          keepw = attn_keep_word(ad, rowid, (uint32_t)(kv0 / 32 + half));
          if (qrow < T) ad.bits[rowid * ad.Tw + kv0 / 32 + half] = keepw;
        }
        uint32_t pk[16];
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          const uint32_t a0 = half ? r1[i] : r0[i], a1 = half ? r1[i + 1] : r0[i + 1];
          float p0 = ex2_approx(fmaf(__uint_as_float(a0), scale_log2, -m_run));
          float p1 = ex2_approx(fmaf(__uint_as_float(a1), scale_log2, -m_run));
          if (!full) {
            if (kv0 + half * 32 + i >= T) p0 = 0.f;
            if (kv0 + half * 32 + i + 1 >= T) p1 = 0.f;
          }
          l_add += p0 + p1;  // softmax denominator: un-dropped probabilities (dropout acts on the normalised P)
          if (ad.thresh8) {
            p0 *= (keepw >> i) & 1u ? ad.scale : 0.f;
            p1 *= (keepw >> (i + 1)) & 1u ? ad.scale : 0.f;
          }
          pk[i / 2] = pack_bf16x2(p0, p1);
        }
        tmem_st16(tm_s + half * 16, pk);  // keys 32*half .. +31 -> packed columns 16*half .. +15 of the S tile
      }
      l_run += l_add;
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(p_full + 8 * sb);
      if ((warp & 3) == 0) TRACE(w, j, 5);
    }
    mbar_wait(p_empty + 8 * (w * 2 + ((n_kv - 1) & 1)), ((n_kv - 1) >> 1) & 1);
    tc_fence_after();
    const int q = q0 + 128 * w + row;
    const float inv_l = 1.0f / l_run;
    __nv_bfloat16* yrow = y + ((size_t)b * T + q) * C + h * HS;
#pragma unroll 1
    for (int c = 0; c < HS; c += 16) {
      uint32_t o[16];
      tmem_ld16(tm_o + c, o);
      tmem_wait_ld();
      if (q < T) store_row16_bf16(yrow + c, o, inv_l);
    }
    if (q < T) lse[((size_t)b * nh + h) * T + q] = (m_run + log2f(l_run)) * 0.6931471805599453f;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == MMAW) tmem_dealloc(tmem_base, L::TMEM_COLS);
}

// =============================================================================================== host
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static PFN_encodeTiled get_encode3() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (PFN_encodeTiled)p;
  }
  return fn;
}

// bf16 tensor (B, T, ncols) row-major; box = (box_cols, box_rows, 1); swizzle span = box_cols * 2 bytes
static int make_tmap3(CUtensorMap* m, const void* base, int ncols, int T, int B, int box_cols, int box_rows) {
  PFN_encodeTiled enc = get_encode3();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point not available"); return DSF_ELAUNCH; }
  cuuint64_t gdim[3] = {(cuuint64_t)ncols, (cuuint64_t)T, (cuuint64_t)B};
  cuuint64_t gstr[2] = {(cuuint64_t)ncols * 2, (cuuint64_t)ncols * 2 * (cuuint64_t)T};
  cuuint32_t box[3] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows, 1u};
  cuuint32_t estr[3] = {1u, 1u, 1u};
  CUtensorMapSwizzle sw = box_cols * 2 == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : (box_cols * 2 == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(3d) failed (%d) ncols=%d T=%d B=%d box=%dx%d", (int)r, ncols, T, B, box_cols, box_rows); return DSF_ELAUNCH; }
  return DSF_OK;
}

template <int HS, int KST, int VST>
static int launch_fwd3(const void* qkv, void* y, float* lse, int B, int T, int C, int nh, const AttnDrop& ad, cudaStream_t st) {
  using L = Fwd3<HS, KST, VST>;
  using H = HeadCfg<HS>;
  static bool configured_on[64] = {};
  bool& configured = per_device_flag(configured_on);
  if (!configured) {
    if (cudaFuncSetAttribute(attn_fwd3_kernel<HS, KST, VST>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::DYN) != cudaSuccess)
      return check_launch("attn_fwd3/attr");
    configured = true;
  }
  CUtensorMap tmQ, tmKV;
  if (int e = make_tmap3(&tmQ, qkv, 3 * C, T, B, H::BOXC, 128)) return e;
  if (int e = make_tmap3(&tmKV, qkv, 3 * C, T, B, H::BOXC, L::BKV)) return e;
  const float scale_log2 = (1.0f / sqrtf((float)HS)) * 1.4426950408889634f;
  dim3 grid(cdiv(T, 128), nh, B);
  launch_pdl(attn_fwd3_kernel<HS, KST, VST>, grid, dim3(L::THREADS), L::DYN, st, tmQ, tmKV, (__nv_bfloat16*)y, lse, T, C, nh, scale_log2, ad);
  return check_launch("attn_fwd3");
}

int run_attn_delta(const void* y, const void* dy, float* delta, int B, int T, int C, int nh, cudaStream_t st);  // attn_api.cu

// Backward kernels: measured variants that were removed (scripts/bench_attn_parts.py, B200, batch 12, T = 962, head size
// 16 / 32 / 64 / 128):
// * Four math warpgroups sharing every tile instead of two (profiles/r02aj_attn_pairs.txt): dK/dV 29.1 / 31.9 / 42.0 / 59.7 us
//   against 28.7 / 31.7 / 41.2 / 59.3 us, dQ 25.3 / 27.8 / 33.0 / 44.8 against 25.9 / 27.7 / 32.1 / 44.6 us.  The in-kernel timeline
//   (profiles/r02aj_attn_trace.txt) says why: halving a warp's columns shortens its tile from ~740 to ~670 cycles only — the tile
//   is a fixed latency chain (tcgen05.ld, wait::ld, tcgen05.st, wait::st, fence, mbarrier), not arithmetic.  An earlier variant
//   whose two pairs of warpgroups took alternate tiles (git history) lost as well: with two S^T/dP^T buffers the next tile of a
//   pair cannot be issued before its previous one is consumed.
// * Every 3rd pair of exponentials on the FMA pipe, as in the forward (profiles/r02ai_attn_bwd_poly.txt): dK/dV 30.2 / 32.7 / 41.9 /
//   62.9 us against 28.4 / 31.6 / 41.4 / 60.3 us.  They run 32 exponentials per thread and tile against the forward's 64 and are
//   bound by the per-tile latency chain, not by the MUFU pipe, so every exponential stays on MUFU.EX2.  The packed-pair arithmetic
//   (FFMA2 / FADD2 / FMUL2) stays: -1.3 / -1.8 us at head size 16 / 32.
template <int HS, int BQ, int STA, bool DROP>
static int launch_bwd_kv(const CUtensorMap& tmKV128, const CUtensorMap& tmQs, const CUtensorMap& tmDOs, const float* lse, const float* delta, void* dqkv,
                         dim3 grid, int T, int C, int nh, float scale, const AttnDrop& ad, cudaStream_t st) {
  using LA = BwdKV2<HS, BQ, STA>;
  const int dyn = LA::dyn_bytes(T);
  if (dyn > 232448) { set_error("attn_bwd: T = %d needs %d bytes of shared memory for the per-query statistics (limit 232448)", T, dyn); return DSF_EUNSUPPORTED; }
  static bool configured_on[64] = {};
  bool& configured = per_device_flag(configured_on);
  if (!configured) {
    if (cudaFuncSetAttribute(attn_bwd_kv2_kernel<HS, BQ, STA, DROP>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448) != cudaSuccess)
      return check_launch("attn_bwd2/kv/attr");
    configured = true;
  }
  launch_pdl(attn_bwd_kv2_kernel<HS, BQ, STA, DROP>, grid, dim3(LA::THREADS), dyn, st, tmKV128, tmQs, tmDOs, lse, delta, (__nv_bfloat16*)dqkv, T, C, nh,
             scale, ad);
  return check_launch("attn_bwd2/kv");
}

template <int HS, int STB, bool DROP>
static int launch_bwd_q(const CUtensorMap& tmQ128, const CUtensorMap& tmDO128, const CUtensorMap& tmKV64, const float* lse, const float* delta, void* dqkv,
                        dim3 grid, int T, int C, int nh, float scale, const AttnDrop& ad, const void* qkv, const void* dy, cudaStream_t st) {
  using LB = BwdQ2<HS, STB>;
  static bool configured_on[64] = {};
  bool& configured = per_device_flag(configured_on);
  if (!configured) {
    if (cudaFuncSetAttribute(attn_bwd_q2_kernel<HS, STB, DROP>, cudaFuncAttributeMaxDynamicSharedMemorySize, LB::DYN) != cudaSuccess)
      return check_launch("attn_bwd2/q/attr");
    configured = true;
  }
  launch_pdl(attn_bwd_q2_kernel<HS, STB, DROP>, grid, dim3(256 + 64), LB::DYN, st, tmQ128, tmDO128, tmKV64, lse, delta, (__nv_bfloat16*)dqkv, T, C, nh,
             scale, ad, (const __nv_bfloat16*)qkv, (const __nv_bfloat16*)dy);
  return check_launch("attn_bwd2/q");
}

template <int HS, int BQ, int STA, int STB>
static int launch_bwd2(const void* qkv, const void* y, const void* dy, const float* lse, float* delta, void* dqkv, int B, int T, int C, int nh,
                       const AttnDrop& ad, int parts, cudaStream_t st) {
  using H = HeadCfg<HS>;
  const float scale = 1.0f / sqrtf((float)HS);
  if (parts & 1) {
    if (int e = run_attn_delta(y, dy, delta, B, T, C, nh, st)) return e;
  }
  const dim3 grid(cdiv(T, 128), nh, B);
  const bool drop = ad.thresh8 != 0;
  if (parts & 2) {
    CUtensorMap tmKV128, tmQs, tmDOs;
    if (int e = make_tmap3(&tmKV128, qkv, 3 * C, T, B, H::BOXC, 128)) return e;
    if (int e = make_tmap3(&tmQs, qkv, 3 * C, T, B, H::BOXC, BQ)) return e;
    if (int e = make_tmap3(&tmDOs, dy, C, T, B, H::BOXC, BQ)) return e;
    const int e = drop ? launch_bwd_kv<HS, BQ, STA, true>(tmKV128, tmQs, tmDOs, lse, delta, dqkv, grid, T, C, nh, scale, ad, st)
                       : launch_bwd_kv<HS, BQ, STA, false>(tmKV128, tmQs, tmDOs, lse, delta, dqkv, grid, T, C, nh, scale, ad, st);
    if (e) return e;
  }
  if (parts & 4) {
    CUtensorMap tmQ128, tmDO128, tmKV64;
    if (int e = make_tmap3(&tmQ128, qkv, 3 * C, T, B, H::BOXC, 128)) return e;
    if (int e = make_tmap3(&tmDO128, dy, C, T, B, H::BOXC, 128)) return e;
    if (int e = make_tmap3(&tmKV64, qkv, 3 * C, T, B, H::BOXC, 64)) return e;
    const int e = drop ? launch_bwd_q<HS, STB, true>(tmQ128, tmDO128, tmKV64, lse, delta, dqkv, grid, T, C, nh, scale, ad, qkv, dy, st)
                       : launch_bwd_q<HS, STB, false>(tmQ128, tmDO128, tmKV64, lse, delta, dqkv, grid, T, C, nh, scale, ad, qkv, dy, st);
    if (e) return e;
  }
  return DSF_OK;
}

#ifdef DSF_ATTN_TRACE
}  // namespace dsf
extern "C" int dsf_debug_attn_trace(long long* host_out) {  // 3 x 64 x 6 clock64 stamps of the last traced launch
  return cudaMemcpyFromSymbol(host_out, dsf::g_attn_trace, sizeof(dsf::g_attn_trace)) == cudaSuccess ? 0 : 2;
}
namespace dsf {
#endif

// attn_drop arguments: 8-bit threshold (p quantised to k/256), bitmap of T_words = 2*ceil(T/64) words per (b, h, q) row
static AttnDrop make_attn_drop(const dsf_dropout* d, uint32_t* bits, int T) {
  AttnDrop a{0u, 1.0f, 0u, 0u, 0u, bits, 2 * cdiv(T, 64), nullptr};
  if (d && d->p > 0.f && bits) {
    int k = (int)lrintf(d->p * 256.0f);
    k = std::max(1, std::min(255, k));
    a.thresh8 = (uint32_t)k;
    a.scale = 256.0f / (256.0f - (float)k);
    a.k0 = (uint32_t)(d->seed & 0xFFFFFFFFull) ^ d->step;
    a.k1 = (uint32_t)(d->seed >> 32);
    a.site = d->site;
    a.seed_dev = reinterpret_cast<const unsigned long long*>(d->seed_dev);
  }
  return a;
}

// Forward, measured variants that were removed:
// * CTA shape: 128-row CTAs, two per SM, against 256-row CTAs (two softmax warpgroups sharing every K/V tile), one per SM.  On
//   B200 (scripts/bench_kernels.py attnq, batch 12, T = 962): 42 vs 48 us at hs = 128, 36 vs 43 (hs = 64), 34 vs 41 (hs = 32), 33
//   vs 40 us (hs = 16); T = 3842, batch 2, hs = 128: 68 vs 80 us (891 vs 760 TF/s) — the half-size CTAs win even where the 256-row
//   grid fills the SMs in one round: two independent MMA / TMA / softmax pipelines per SM overlap better than one pipeline with
//   two softmax warpgroups, and the grid is scheduled in finer units.
// * Exponentials (Fwd3::POLY): moving every 3rd pair from MUFU.EX2 to the FMA pipe (ex2_poly2) at head sizes <= 64 and every 4th at
//   128 is kept.  On B200 (scripts/bench_attn_parts.py, batch 12, T = 962; profiles/r02ah_attn_exp_poly.txt), none / every 4th /
//   3rd / 2nd pair: hs 16: 28.1 / 25.2 / 24.4 / 25.3 us, hs 32: 28.6 / 25.5 / 24.8 / 25.5, hs 64: 30.3 / 27.0 / 27.1 / 27.8, hs 128:
//   35.4 / 34.8 / 35.7 / 35.1 us; T = 3842, hs 128: 64.9 / 55.0 / 56.0 / 57.4 us (932 -> 1099 TF/s).
int attn_fwd_run(const void* qkv, void* y, float* lse, int B, int T, int C, int nh, const dsf_dropout* drop, uint32_t* bits, cudaStream_t st) {
  const AttnDrop ad = make_attn_drop(drop, bits, T);
  switch (C / nh) {
    case 16: return launch_fwd3<16, 3, 2>(qkv, y, lse, B, T, C, nh, ad, st);
    case 32: return launch_fwd3<32, 3, 2>(qkv, y, lse, B, T, C, nh, ad, st);
    case 64: return launch_fwd3<64, 3, 2>(qkv, y, lse, B, T, C, nh, ad, st);
    case 128: return launch_fwd3<128, 2, 2>(qkv, y, lse, B, T, C, nh, ad, st);
  }
  set_error("attn_fwd: head size %d not supported (16, 32, 64, 128)", C / nh);
  return DSF_EUNSUPPORTED;
}

int attn_bwd_run(const void* qkv, const void* y, const void* dy, const float* lse, float* delta, void* dqkv, int B, int T, int C, int nh,
                 const dsf_dropout* drop, uint32_t* bits, int parts, cudaStream_t st) {
  const AttnDrop ad = make_attn_drop(drop, bits, T);
  switch (C / nh) {
    case 16: return launch_bwd2<16, 64, 3, 3>(qkv, y, dy, lse, delta, dqkv, B, T, C, nh, ad, parts, st);
    case 32: return launch_bwd2<32, 64, 3, 3>(qkv, y, dy, lse, delta, dqkv, B, T, C, nh, ad, parts, st);
    case 64: return launch_bwd2<64, 64, 3, 3>(qkv, y, dy, lse, delta, dqkv, B, T, C, nh, ad, parts, st);
    case 128: return launch_bwd2<128, 64, 3, 3>(qkv, y, dy, lse, delta, dqkv, B, T, C, nh, ad, parts, st);
  }
  set_error("attn_bwd: head size %d not supported (16, 32, 64, 128)", C / nh);
  return DSF_EUNSUPPORTED;
}

}  // namespace dsf

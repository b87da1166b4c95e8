// K3/K5/K6 (v2): persistent, warp-specialised bf16 GEMMs on tcgen05.
//   NT: C[M,N] = A[M,K] . B[N,K]^T (+bias)(relu)(+residual) — 128 x BN tiles (BN = 256 / 128 / 64), one CTA per SM
//       looping over tiles; the fp32 accumulator is double-buffered in TMEM (2 x BN columns) so the epilogue of
//       tile i (8 warps, TMEM -> registers -> global) overlaps the TMA/MMA main loop of tile i+1.
//   TN: C[N',K'] += A[M,N']^T . B[M,K'] (weight gradient) — 128 x BN tiles, contraction split across CTAs,
//       vectorised fp32 reductions (red.global.add.v4.f32) into the gradient buffer.
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2..9 = epilogue
// (TMEM lane quarter = warp % 4, column half = (warp - 2) / 4).
#include <algorithm>

#include "tc_common.cuh"

namespace dsf {

using namespace tc;

int make_tmap_bf16(CUtensorMap* m, const void* base, int rows, int cols, int ld, int box_rows);  // gemm_tc.cu
int make_tmap_2d(CUtensorMap* m, const void* base, int dtype, int rows, int cols, int ld, int box_cols, int box_rows);

constexpr int G2_BM = 128, G2_BK = 64, G2_THREADS = 320;

struct EpiArgs2 {
  void* C;
  int ldc;
  int c_dtype;
  const float* bias;
  const float* residual;
  int flags;
  int N;          // row length for the dropout element index m*N + n
  const __nv_bfloat16* relu_src;  // nullable: v = relu_src[m,n] > 0 ? v : 0 (ReLU backward fused into the dgrad GEMM)
  DropArgs drop;  // resid_drop (model2_seq.py:109,125): after bias/ReLU, before the residual add
};

// epilogue math on 32 accumulator columns of one row: (+bias)(relu)(+residual); row_ok guards the residual read
__device__ __forceinline__ void epi_math32(const EpiArgs2& e, int row, int n, const uint32_t (&r)[32], float (&v)[32], bool row_ok) {
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
  if (e.flags & DSF_EPI_BIAS) {
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      const float4 b = __ldg(reinterpret_cast<const float4*>(e.bias + n + j));
      v[j] += b.x; v[j + 1] += b.y; v[j + 2] += b.z; v[j + 3] += b.w;
    }
  }
  if (e.flags & DSF_EPI_RELU) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
  }
  if (e.relu_src != nullptr && row_ok) {
    const uint4* hp = reinterpret_cast<const uint4*>(e.relu_src + (size_t)row * e.ldc + n);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint4 h = __ldg(hp + j);
      const uint32_t hw[4] = {h.x, h.y, h.z, h.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {  // bf16 > 0  <=>  sign bit clear and magnitude non-zero
        if (!((hw[k] & 0x8000u) == 0u && (hw[k] & 0x7FFFu) != 0u)) v[8 * j + 2 * k] = 0.f;
        if (!((hw[k] & 0x80000000u) == 0u && (hw[k] & 0x7FFF0000u) != 0u)) v[8 * j + 2 * k + 1] = 0.f;
      }
    }
  }
  if (e.drop.thresh) {
    const uint64_t e8 = ((uint64_t)row * e.N + n) >> 3;  // N and n are multiples of 8
#pragma unroll
    for (int j = 0; j < 32; j += 8) {
      float m[8];
      drop_scale8(e.drop, e8 + (j >> 3), m);
#pragma unroll
      for (int k = 0; k < 8; ++k) v[j + k] *= m[k];
    }
  }
  if ((e.flags & DSF_EPI_RESIDUAL) && row_ok) {
    const float4* rp = reinterpret_cast<const float4*>(e.residual + (size_t)row * e.ldc + n);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 t = rp[j];
      v[4 * j] += t.x; v[4 * j + 1] += t.y; v[4 * j + 2] += t.z; v[4 * j + 3] += t.w;
    }
  }
}

template <int BN, int STAGES, bool STAGED = true>
struct G2Smem {
  static constexpr int A_BYTES = G2_BM * G2_BK * 2;
  static constexpr int B_BYTES = BN * G2_BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGING_OFF = STAGES * STAGE_BYTES;  // 8 epilogue warps x 2 buffers x 4 KB (TMA-store staging)
  static constexpr int STAGING_BYTES = STAGED ? 8 * 2 * 4096 : 0;
  static constexpr int BAR_OFF = STAGING_OFF + STAGING_BYTES;
  static constexpr int DYN = BAR_OFF + (2 * STAGES + 4) * 8 + 16 + 1024;
  static constexpr uint32_t TMEM_COLS = 2 * BN < 32 ? 32 : 2 * BN;
  static_assert(DYN <= 232448, "shared memory budget");
};

// ---------------------------------------------------------------------------------- NT, persistent
template <int BN, int STAGES>
__global__ void __launch_bounds__(G2_THREADS, 1)
gemm_nt2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmC,
                EpiArgs2 epi, int M, int N, int K, int m_tiles, int n_tiles) {
  using L = G2Smem<BN, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_full = base + L::BAR_OFF, bar_empty = bar_full + STAGES * 8, acc_full = bar_empty + STAGES * 8,
                 acc_empty = acc_full + 16, tmem_slot = acc_empty + 16;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;  // warp-uniform for the compiler
  const int num_k = K / G2_BK;
  const int total = m_tiles * n_tiles;
  pdl_trigger();

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < STAGES; ++s) { mbar_init(bar_full + s * 8, 1); mbar_init(bar_empty + s * 8, 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(acc_full + a * 8, 1); mbar_init(acc_empty + a * 8, 8); }
    fence_barrier_init();
  }
  if (warp == 1) { tmem_alloc(tmem_slot, L::TMEM_COLS); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  pdl_wait();  // everything above overlapped the previous kernel's tail

  if (warp == 0) {
    if (lane == 0) {
      int it = 0;  // k-block counter across all tiles of this CTA
      for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const int m0 = (tile % m_tiles) * G2_BM, n0 = (tile / m_tiles) * BN;
        for (int kb = 0; kb < num_k; ++kb, ++it) {
          const int s = it % STAGES;
          mbar_wait(bar_empty + s * 8, ((it / STAGES) & 1) ^ 1);
          mbar_expect_tx(bar_full + s * 8, L::STAGE_BYTES);
          const uint32_t sa = base + s * L::STAGE_BYTES, sb = sa + L::A_BYTES;
          tma_load_2d(sa, &tmA, bar_full + s * 8, kb * G2_BK, m0);
          tma_load_2d(sb, &tmB, bar_full + s * 8, kb * G2_BK, n0);
        }
      }
    }
  } else if (warp == 1) {
    {  // MMA issuer: all 32 lanes walk the schedule (uniform control flow keeps descriptors in uniform registers)
      constexpr uint32_t idesc = make_idesc_bf16(G2_BM, BN, 0, 0);
      int it = 0, i = 0;
      for (int tile = blockIdx.x; tile < total; tile += gridDim.x, ++i) {
        const int ab = i & 1;
        mbar_wait(acc_empty + ab * 8, ((i >> 1) & 1) ^ 1);  // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t acc = tmem_base + ab * BN;
        for (int kb = 0; kb < num_k; ++kb, ++it) {
          const int s = it % STAGES;
          mbar_wait(bar_full + s * 8, (it / STAGES) & 1);
          tc_fence_after();
          const uint32_t sa = base + s * L::STAGE_BYTES, sb = sa + L::A_BYTES;
          const uint64_t da = make_smem_desc(sa, 16, 1024, SWZ_128B);
          const uint64_t db = make_smem_desc(sb, 16, 1024, SWZ_128B);
          const uint32_t first = kb != 0 ? 1u : 0u;
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < G2_BK / 16; ++k) tc_mma_bf16(acc, da + (uint32_t)(k * 2), db + (uint32_t)(k * 2), idesc, k == 0 ? first : 1u);
            tc_commit(bar_empty + s * 8);
          }
          __syncwarp();
        }
        if (elect_one()) tc_commit(acc_full + ab * 8);
        __syncwarp();
      }
    }
  } else {
    const int q = warp & 3;            // TMEM lane quarter this warp may access
    const int ch = (warp - 2) >> 2;    // column half handled by this warp
    epi.drop = resolve_drop(epi.drop);
    constexpr int NSPLIT = BN >= 128 ? 2 : 1;  // BN = 64: warps 2..5 drain the whole tile, warps 6..9 only hand the buffer back
    constexpr int HALF = BN / NSPLIT;
    int i = 0, nbox = 0;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x, ++i) {
      const int ab = i & 1;
      const int m0 = (tile % m_tiles) * G2_BM, n0 = (tile / m_tiles) * BN;
      mbar_wait(acc_full + ab * 8, (i >> 1) & 1);
      tc_fence_after();
      if (ch >= NSPLIT || m0 + q * 32 >= M) {  // nothing to store for this warp
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(acc_empty + ab * 8);
        continue;
      }
      const int row = m0 + q * 32 + lane;
      const uint32_t tacc = tmem_base + ab * BN + ((uint32_t)(q * 32) << 16) + ch * HALF;
      // coalesced epilogue: registers -> this warp's 128B-swizzled staging box [32 rows x 128 B] -> TMA store
      const uint32_t stg = base + L::STAGING_OFF + (warp - 2) * 8192;
      const int CW = epi.c_dtype == DSF_F32 ? 32 : 64;  // columns per 128-byte staged row
#pragma unroll 1
      for (int c = 0; c < HALF; c += CW, ++nbox) {
        const uint32_t sbuf = stg + (nbox & 1) * 4096;
        if (lane == 0) bulk_wait_read<1>();  // the store issued two boxes ago has finished reading this buffer
        __syncwarp();
        const int ncol = n0 + ch * HALF + c;
        uint32_t w[32];  // 128 bytes of this thread's output row
        if (epi.c_dtype == DSF_F32) {
          uint32_t r[32];
          tmem_ld32(tacc + c, r);
          tmem_wait_ld();
          float v[32];
          epi_math32(epi, row, ncol, r, v, row < M);
#pragma unroll
          for (int j = 0; j < 32; ++j) w[j] = __float_as_uint(v[j]);
        } else {
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            uint32_t r[32];
            tmem_ld32(tacc + c + hh * 32, r);
            tmem_wait_ld();
            float v[32];
            epi_math32(epi, row, ncol + hh * 32, r, v, row < M);
#pragma unroll
            for (int j = 0; j < 16; ++j) w[hh * 16 + j] = pack_bf16x2(v[2 * j], v[2 * j + 1]);
          }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint32_t dst = sbuf + lane * 128 + ((j ^ (lane & 7)) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(w[4 * j]), "r"(w[4 * j + 1]), "r"(w[4 * j + 2]), "r"(w[4 * j + 3])
                       : "memory");
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(&tmC, sbuf, ncol, m0 + q * 32);
          bulk_commit();
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty + ab * 8);
    }
    if (lane == 0) bulk_wait<0>();  // all stores complete before shared memory is released
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, L::TMEM_COLS);
}

// ---------------------------------------------------------------------------------- NT, persistent, CTA pairs (cta_group::2)
// v3: two CTAs of one cluster (one TPC) compute a 256 x BN tile with tcgen05.mma.cta_group::2.  CTA r of the pair loads its
// own 128 rows of A and only HALF of the B tile (rows n0 + r*BN/2 ..); the tensor cores of both SMs read both halves.
// Per k-block a CTA therefore pulls 16 KB (A) + BN/2 x 128 B (B) through the L2 -> SM fabric instead of 16 KB + BN x 128 B:
// the NT GEMMs of this path are bound by exactly that traffic (11.4 TB/s measured = the chip's L2 request cap), not by
// the tensor pipe.  Protocol (barrier offsets are identical in both CTAs):
//   full[s]      leader only, count 1 + tx bytes of BOTH CTAs (the peer's TMA completes on the leader's barrier)
//   empty[s]     both CTAs, count 1, arrived by the leader's multicast tcgen05.commit
//   acc_full[a]  both CTAs, count 1, multicast commit after the last k-block of a tile
//   acc_empty[a] leader only, count 16: the 8 epilogue warps of both CTAs
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `addr` (a shared::cta address of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  // relaxed: the arrive only hands a drained TMEM buffer back (ordered by tcgen05.wait::ld + tcgen05.fence::before_thread_sync);
  // a release at cluster scope would cost a MEMBAR.GPU per epilogue warp and tile
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* m, uint32_t bar_cluster, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint32_t bar) {  // arrives on `bar` in BOTH CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void tc_mma_bf16_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

template <int BN, int STAGES, bool RTMA = false>
struct G3Smem {
  static constexpr int A_BYTES = G2_BM * G2_BK * 2;        // this CTA's 128 rows of A
  static constexpr int B_BYTES = (BN / 2) * G2_BK * 2;     // this CTA's half of the B tile
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGING_OFF = STAGES * STAGE_BYTES;
  static constexpr int STAGING_BYTES = 8 * 2 * 4096;
  static constexpr int RES_OFF = STAGING_OFF + STAGING_BYTES;  // RTMA: one 32 x 32 fp32 residual box per epilogue warp
  static constexpr int RES_BYTES = RTMA ? 8 * 4096 : 0;
  static constexpr int BAR_OFF = RES_OFF + RES_BYTES;
  static constexpr int RBAR_OFF = BAR_OFF + (2 * STAGES + 4) * 8 + 16;  // 8 mbarriers (one per epilogue warp) when RTMA
  static constexpr int DYN = RBAR_OFF + (RTMA ? 64 : 0) + 1024;
  static constexpr uint32_t TMEM_COLS = 2 * BN;
  static_assert(DYN <= 232448, "shared memory budget");
  static_assert(TMEM_COLS == 512 || TMEM_COLS == 256, "TMEM columns must be a power of two");
};

// RTMA (fp32 output + residual only): the residual tile is not read by the epilogue threads from global memory (one
// uncoalesced 128-byte row piece per lane and chunk, ~1 us of exposed latency per chunk) but prefetched by TMA, one
// 32 x 32 box per epilogue warp, one chunk ahead — the first box of a tile while its main loop is still running.
template <int BN, int STAGES, bool RTMA = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(G2_THREADS, 1)
gemm_nt3_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmC,
                const __grid_constant__ CUtensorMap tmBt, const __grid_constant__ CUtensorMap tmR, EpiArgs2 epi, int M, int N, int K,
                int m_tiles, int n_tiles, int tail_start, int n_split) {
  using L = G3Smem<BN, STAGES, RTMA>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_full = base + L::BAR_OFF, bar_empty = bar_full + STAGES * 8, acc_full = bar_empty + STAGES * 8,
                 acc_empty = acc_full + 16, tmem_slot = acc_empty + 16;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;  // warp-uniform for the compiler
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  const int num_k = K / G2_BK;
  // Work units: units < tail_start are whole 256 x BN tiles (unit = tile).  n_split > 1: the tiles left over after the
  // last full round of the pairs (tail_start .. ) are each split n_split ways along N — a unit is a 256 x (BN / n_split)
  // sub-tile with its own, narrower MMA shape and B box (tmBt); nothing is reduced across units, so any epilogue works.
  // The short last round costs ~BN/n_split columns of epilogue and a cheaper MMA stream.
  const int total = tail_start + (m_tiles * n_tiles - tail_start) * n_split;
  auto unit_of = [&](int u, int& tile, int& n_off, int& width) {
    if (u < tail_start || n_split == 1) { tile = u; n_off = 0; width = BN; return; }
    const int j = u - tail_start;
    tile = tail_start + j / n_split;
    width = BN / n_split;
    n_off = (j % n_split) * width;
  };
  pdl_trigger();

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < STAGES; ++s) { mbar_init(bar_full + s * 8, 1); mbar_init(bar_empty + s * 8, 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(acc_full + a * 8, 1); mbar_init(acc_empty + a * 8, 16); }
    if (RTMA) {
      for (int w = 0; w < 8; ++w) mbar_init(base + L::RBAR_OFF + w * 8, 1);
    }
    fence_barrier_init();
  }
  if (warp == 1) { tmem_alloc_pair(tmem_slot, L::TMEM_COLS); tmem_relinquish_pair(); }
  tc_fence_before();
  cluster_sync_all();  // barriers of BOTH CTAs are initialised before any remote arrive / TMA completion
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  pdl_wait();

  if (warp == 0) {
    if (lane == 0) {
      const uint32_t full0 = mapa_u32(bar_full, 0);  // the leader's full barriers
      int it = 0;
      for (int u = pair; u < total; u += n_pairs) {
        int tile, n_off, width;
        unit_of(u, tile, n_off, width);
        const bool narrow = width != BN;
        const int m0 = (tile % m_tiles) * 256 + (int)rank * G2_BM, n0 = (tile / m_tiles) * BN + n_off + (int)rank * (width / 2);
        const uint32_t tx = 2u * (uint32_t)(L::A_BYTES + (width / 2) * G2_BK * 2);
        for (int kb = 0; kb < num_k; ++kb, ++it) {
          const int s = it % STAGES;
          mbar_wait(bar_empty + s * 8, ((it / STAGES) & 1) ^ 1);
          if (rank == 0) mbar_expect_tx(bar_full + s * 8, tx);
          const uint32_t sa = base + s * L::STAGE_BYTES, sb = sa + L::A_BYTES;
          tma_load_2d_pair(sa, &tmA, full0 + s * 8, kb * G2_BK, m0);
          tma_load_2d_pair(sb, narrow ? &tmBt : &tmB, full0 + s * 8, kb * G2_BK, n0);
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0) {  // MMA issuer of the pair: all 32 lanes walk the schedule, one elected lane issues
      int it = 0, i = 0;
      for (int u = pair; u < total; u += n_pairs, ++i) {
        int tile, n_off, width;
        unit_of(u, tile, n_off, width);
        const uint32_t idesc = make_idesc_bf16(256, width, 0, 0);
        const int ab = i & 1;
        mbar_wait(acc_empty + ab * 8, ((i >> 1) & 1) ^ 1);  // the epilogues of both CTAs have drained this accumulator
        tc_fence_after();
        const uint32_t acc = tmem_base + ab * BN;
        for (int kb = 0; kb < num_k; ++kb, ++it) {
          const int s = it % STAGES;
          mbar_wait(bar_full + s * 8, (it / STAGES) & 1);
          tc_fence_after();
          const uint32_t sa = base + s * L::STAGE_BYTES, sb = sa + L::A_BYTES;
          const uint64_t da = make_smem_desc(sa, 16, 1024, SWZ_128B);
          const uint64_t db = make_smem_desc(sb, 16, 1024, SWZ_128B);
          const uint32_t first = kb != 0 ? 1u : 0u;
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < G2_BK / 16; ++k) tc_mma_bf16_pair(acc, da + (uint32_t)(k * 2), db + (uint32_t)(k * 2), idesc, k == 0 ? first : 1u);
            tc_commit_pair(bar_empty + s * 8);
          }
          __syncwarp();
        }
        if (elect_one()) tc_commit_pair(acc_full + ab * 8);
        __syncwarp();
      }
    }
  } else {
    const int q = warp & 3;            // TMEM lane quarter this warp may access
    const int ch = (warp - 2) >> 2;    // column half handled by this warp
    epi.drop = resolve_drop(epi.drop);
    const uint32_t acc_empty0 = mapa_u32(acc_empty, 0);
    int i = 0, nbox = 0;
    // RTMA: residual boxes of this warp.  chunks_of() mirrors exactly the conditions under which the chunk loop below
    // runs for a unit (every issued box is consumed, every consumed box was issued); r_inflight is warp-uniform.
    const uint32_t rbuf = base + L::RES_OFF + (warp - 2) * 4096, rbar = base + L::RBAR_OFF + (warp - 2) * 8;
    int nres = 0;
    bool r_inflight = false;
    auto chunks_of = [&](int uu, int& cm0, int& cn0, int& clo, int& chi) -> bool {
      int t2, off2, w2;
      unit_of(uu, t2, off2, w2);
      cm0 = (t2 % m_tiles) * 256 + (int)rank * G2_BM;
      cn0 = (t2 / m_tiles) * BN + off2;
      const int hu = w2 / 2;
      clo = hu >= 32 ? ch * hu : 0;
      chi = hu >= 32 ? clo + hu : (ch == 0 ? w2 : 0);
      return cm0 + q * 32 < M && clo < chi;
    };
    auto issue_res = [&](int ncol, int row0) {
      if (lane == 0) {
        fence_proxy_async();  // the box is re-filled after generic-proxy reads of the previous one
        mbar_expect_tx(rbar, 4096);
        tma_load_2d(rbuf, &tmR, rbar, ncol, row0);
      }
      r_inflight = true;
    };
    if (RTMA && pair < total) {
      int cm0, cn0, clo, chi;
      if (chunks_of(pair, cm0, cn0, clo, chi)) issue_res(cn0 + clo, cm0 + q * 32);
    }
    for (int u = pair; u < total; u += n_pairs, ++i) {
      int tile, n_off, width;
      unit_of(u, tile, n_off, width);
      const int ab = i & 1;
      const int m0 = (tile % m_tiles) * 256 + (int)rank * G2_BM, n0 = (tile / m_tiles) * BN + n_off;
      mbar_wait(acc_full + ab * 8, (i >> 1) & 1);
      tc_fence_after();
      if (m0 + q * 32 < M) {
        const int row = m0 + q * 32 + lane;
        const uint32_t tacc = tmem_base + ab * BN + ((uint32_t)(q * 32) << 16);
        const uint32_t stg = base + L::STAGING_OFF + (warp - 2) * 8192;
        const int CW = epi.c_dtype == DSF_F32 ? 32 : 64;  // columns per 128-byte staged row
        // columns of this unit drained by this warp: its column half, or (narrow unit, half narrower than one staged
        // box) the whole unit for column-half 0 and nothing for column-half 1
        const int half_u = width / 2;
        const int c_lo = half_u >= CW ? ch * half_u : 0;
        const int c_hi = half_u >= CW ? c_lo + half_u : (ch == 0 ? width : 0);
#pragma unroll 1
        for (int c = c_lo; c < c_hi; c += CW, ++nbox) {
          const uint32_t sbuf = stg + (nbox & 1) * 4096;
          if (lane == 0) bulk_wait_read<1>();
          __syncwarp();
          const int ncol = n0 + c;
          uint32_t w[32];
          if (RTMA) {  // fp32 output + residual: the residual box of this chunk was requested one chunk (or one tile) ago
            if (!r_inflight) issue_res(ncol, m0 + q * 32);
            mbar_wait(rbar, nres & 1);
            ++nres;
            float rr[32];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const uint32_t src = rbuf + lane * 128 + ((j ^ (lane & 7)) << 4);
              asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(rr[4 * j]), "=f"(rr[4 * j + 1]), "=f"(rr[4 * j + 2]), "=f"(rr[4 * j + 3]) : "r"(src) : "memory");
            }
            __syncwarp();  // every lane has read the box: it can be re-filled
            r_inflight = false;
            if (c + CW < c_hi) {
              issue_res(ncol + CW, m0 + q * 32);
            } else if (u + n_pairs < total) {
              int cm0, cn0, clo, chi;
              if (chunks_of(u + n_pairs, cm0, cn0, clo, chi)) issue_res(cn0 + clo, cm0 + q * 32);
            }
            uint32_t r[32];
            tmem_ld32(tacc + c, r);
            tmem_wait_ld();
            float v[32];
            EpiArgs2 e2 = epi;
            e2.flags &= ~DSF_EPI_RESIDUAL;
            epi_math32(e2, row, ncol, r, v, row < M);
#pragma unroll
            for (int j = 0; j < 32; ++j) w[j] = __float_as_uint(v[j] + rr[j]);
          } else if (epi.c_dtype == DSF_F32) {
            uint32_t r[32];
            tmem_ld32(tacc + c, r);
            tmem_wait_ld();
            float v[32];
            epi_math32(epi, row, ncol, r, v, row < M);
#pragma unroll
            for (int j = 0; j < 32; ++j) w[j] = __float_as_uint(v[j]);
          } else {
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              uint32_t r[32];
              tmem_ld32(tacc + c + hh * 32, r);
              tmem_wait_ld();
              float v[32];
              epi_math32(epi, row, ncol + hh * 32, r, v, row < M);
#pragma unroll
              for (int j = 0; j < 16; ++j) w[hh * 16 + j] = pack_bf16x2(v[2 * j], v[2 * j + 1]);
            }
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const uint32_t dst = sbuf + lane * 128 + ((j ^ (lane & 7)) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(w[4 * j]), "r"(w[4 * j + 1]), "r"(w[4 * j + 2]), "r"(w[4 * j + 3])
                         : "memory");
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&tmC, sbuf, ncol, m0 + q * 32);
            bulk_commit();
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(acc_empty0 + ab * 8);
    }
    if (lane == 0) bulk_wait<0>();  // all stores complete before shared memory is released
  }
  tc_fence_before();
  cluster_sync_all();  // neither CTA may exit (or free TMEM) while its peer can still touch its barriers / TMEM
  if (warp == 1) tmem_dealloc_pair(tmem_base, L::TMEM_COLS);
}


// ---------------------------------------------------------------------------------- TN (wgrad), split contraction

// colsum (nullable): colsum[n'] += sum_m A[m, n'] — the bias gradient of the Linear whose weight gradient this GEMM computes
// (model2_seq.py:97-99, 122).  It rides on the tensor core: the CTAs of the first K' tile issue one extra 128 x 16 MMA per k-step
// whose B operand is a 2 KB shared-memory tile of ones, so an accumulator column next to the C tile collects the row sums of A^T.
// (The separate column-sum kernel re-read dqkv / da: 16 launches and 0.12 - 0.19 ms of kernel time per stage.)
template <int BN, int STAGES>
struct TnSmem : G2Smem<BN, STAGES, false> {
  using Base = G2Smem<BN, STAGES, false>;
  static constexpr int ONES_OFF = (Base::BAR_OFF + (2 * STAGES + 4) * 8 + 16 + 1023) / 1024 * 1024;
  static constexpr int ONES_BYTES = 16 * 128;  // 16 contraction rows x one 128-byte swizzle row, every element 1.0
  static constexpr int DYN = ONES_OFF + ONES_BYTES + 1024;
  static constexpr uint32_t TMEM_COLS = BN + 32 <= 128 ? 128 : (BN + 32 <= 256 ? 256 : 512);
  static_assert(DYN <= 232448, "shared memory budget");
};

template <int BN, int STAGES>
__global__ void __launch_bounds__(G2_THREADS, 1)
gemm_tn2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, float* __restrict__ C, int ldc, int M, int Nout,
                int Kout, int m_chunk, float* __restrict__ colsum) {
  using L = TnSmem<BN, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_full = base + L::BAR_OFF, bar_empty = bar_full + STAGES * 8, bar_acc = bar_empty + STAGES * 8, tmem_slot = bar_acc + 8 * 4;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;  // warp-uniform for the compiler
  const int n0 = blockIdx.y * G2_BM;  // rows of C (N' index)
  const int k0 = blockIdx.x * BN;     // cols of C (K' index)
  const int m_lo = blockIdx.z * m_chunk, m_hi = min(M, m_lo + m_chunk);
  const int num_it = (m_hi - m_lo + G2_BK - 1) / G2_BK;
  constexpr uint32_t TMEM_COLS = L::TMEM_COLS;
  constexpr int BOX_BYTES = G2_BK * 128;  // 64 rows x 128 B
  const bool do_cs = colsum != nullptr && blockIdx.x == 0;
  pdl_trigger();
  if (do_cs) {  // the ones tile (bf16 1.0 = 0x3F80), visible to the tensor core's operand reads after the barrier below
    uint32_t* ones = reinterpret_cast<uint32_t*>(smem_raw + (base - smem_u32(smem_raw)) + L::ONES_OFF);
    for (int i = threadIdx.x; i < L::ONES_BYTES / 4; i += G2_THREADS) ones[i] = 0x3F803F80u;
    fence_proxy_async();
  }

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < STAGES; ++s) { mbar_init(bar_full + s * 8, 1); mbar_init(bar_empty + s * 8, 1); }
    mbar_init(bar_acc, 1);
    fence_barrier_init();
  }
  if (warp == 1) { tmem_alloc(tmem_slot, TMEM_COLS); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  pdl_wait();

  if (warp == 0) {
    if (lane == 0) {
      for (int it = 0; it < num_it; ++it) {
        const int s = it % STAGES;
        mbar_wait(bar_empty + s * 8, ((it / STAGES) & 1) ^ 1);
        mbar_expect_tx(bar_full + s * 8, L::STAGE_BYTES);
        const uint32_t sa = base + s * L::STAGE_BYTES, sb = sa + L::A_BYTES;
        const int m = m_lo + it * G2_BK;
#pragma unroll
        for (int j = 0; j < G2_BM / 64; ++j) tma_load_2d(sa + j * BOX_BYTES, &tmA, bar_full + s * 8, n0 + j * 64, m);
#pragma unroll
        for (int j = 0; j < BN / 64; ++j) tma_load_2d(sb + j * BOX_BYTES, &tmB, bar_full + s * 8, k0 + j * 64, m);
      }
    }
  } else if (warp == 1) {
    {  // MMA issuer: all 32 lanes walk the schedule (uniform control flow keeps descriptors in uniform registers)
      constexpr uint32_t idesc = make_idesc_bf16(G2_BM, BN, 1, 1);
      constexpr uint32_t idesc_cs = make_idesc_bf16(G2_BM, 16, 1, 1);
      const uint64_t d_ones = make_smem_desc(base + L::ONES_OFF, BOX_BYTES, 1024, SWZ_128B);  // the same 16 rows for every k-step
      for (int it = 0; it < num_it; ++it) {
        const int s = it % STAGES;
        mbar_wait(bar_full + s * 8, (it / STAGES) & 1);
        tc_fence_after();
        const uint32_t sa = base + s * L::STAGE_BYTES, sb = sa + L::A_BYTES;
        const uint64_t da = make_smem_desc(sa, BOX_BYTES, 1024, SWZ_128B);
        const uint64_t db = make_smem_desc(sb, BOX_BYTES, 1024, SWZ_128B);
        const uint32_t first = it != 0 ? 1u : 0u;
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < G2_BK / 16; ++k) tc_mma_bf16(tmem_base, da + (uint32_t)(k * 128), db + (uint32_t)(k * 128), idesc, k == 0 ? first : 1u);
          if (do_cs) {
#pragma unroll
            for (int k = 0; k < G2_BK / 16; ++k) tc_mma_bf16(tmem_base + BN, da + (uint32_t)(k * 128), d_ones, idesc_cs, k == 0 ? first : 1u);
          }
          tc_commit(bar_empty + s * 8);
        }
        __syncwarp();
      }
      if (elect_one()) tc_commit(bar_acc);
      __syncwarp();
    }
  } else {
    mbar_wait(bar_acc, 0);
    tc_fence_after();
    const int q = warp & 3, ch = (warp - 2) >> 2;
    constexpr int HALF = BN / 2;
    const int row = n0 + q * 32 + lane;
    if (do_cs && ch == 0) {  // every one of the 16 columns holds the row sum of A^T over this CTA's contraction chunk
      uint32_t r[16];
      tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + BN, r);
      tmem_wait_ld();
      if (row < Nout) atomicAdd(colsum + row, __uint_as_float(r[0]));
    }
#pragma unroll 1
    for (int c = 0; c < HALF; c += 32) {
      uint32_t r[32];
      tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + ch * HALF + c, r);
      tmem_wait_ld();
      if (row < Nout) {
        float* cp = C + (size_t)row * ldc + k0 + ch * HALF + c;
        if (k0 + ch * HALF + c + 32 <= Kout) {
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            red_add_v4(cp + j, __uint_as_float(r[j]), __uint_as_float(r[j + 1]), __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (k0 + ch * HALF + c + j < Kout) atomicAdd(cp + j, __uint_as_float(r[j]));
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, TMEM_COLS);
}

template <int BN, int STAGES>
static int launch_nt2(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, const EpiArgs2& epi, int M, int N, int K,
                      cudaStream_t st) {
  using L = G2Smem<BN, STAGES>;
  static bool configured_on[64] = {};
  bool& configured = per_device_flag(configured_on);
  if (!configured) {
    if (cudaFuncSetAttribute(gemm_nt2_kernel<BN, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::DYN) != cudaSuccess)
      return check_launch("gemm_nt2/attr");
    configured = true;
  }
  const int m_tiles = cdiv(M, G2_BM), n_tiles = N / BN;
  const int grid = std::min(m_tiles * n_tiles, num_sms());
  launch_pdl(gemm_nt2_kernel<BN, STAGES>, dim3(grid), dim3(G2_THREADS), L::DYN, st, tmA, tmB, tmC, epi, M, N, K, m_tiles, n_tiles);
  return check_launch("gemm_nt2");
}

template <int BN, int STAGES>
static int launch_tn2(const CUtensorMap& tmA, const CUtensorMap& tmB, float* C, int ldc, int M, int Nout, int Kout, float* colsum, cudaStream_t st) {
  using L = TnSmem<BN, STAGES>;
  static bool configured_on[64] = {};
  bool& configured = per_device_flag(configured_on);
  if (!configured) {
    if (cudaFuncSetAttribute(gemm_tn2_kernel<BN, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::DYN) != cudaSuccess)
      return check_launch("gemm_tn2/attr");
    configured = true;
  }
  const int tiles = cdiv(Nout, G2_BM) * cdiv(Kout, BN);
  // one wave of CTAs: split the contraction so that tiles * splits ~ number of SMs (chunks are multiples of 64 rows)
  int splits = std::max(1, std::min(cdiv(M, 2 * G2_BK), num_sms() / std::max(1, tiles)));
  int m_chunk = cdiv(cdiv(M, splits), G2_BK) * G2_BK;
  splits = cdiv(M, m_chunk);
  dim3 grid(cdiv(Kout, BN), cdiv(Nout, G2_BM), splits);
  launch_pdl(gemm_tn2_kernel<BN, STAGES>, grid, dim3(G2_THREADS), L::DYN, st, tmA, tmB, C, ldc, M, Nout, Kout, m_chunk, colsum);
  return check_launch("gemm_tn2");
}

template <int BN, int STAGES, bool RTMA = false>
static int launch_nt3(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, const EpiArgs2& epi, int M, int N, int K,
                      cudaStream_t st, const void* Bptr = nullptr, int ldb = 0) {
  using L = G3Smem<BN, STAGES, RTMA>;
  static bool configured_on[64] = {};
  bool& configured = per_device_flag(configured_on);
  if (!configured) {
    if (cudaFuncSetAttribute(gemm_nt3_kernel<BN, STAGES, RTMA>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::DYN) != cudaSuccess)
      return check_launch("gemm_nt3/attr");
    configured = true;
  }
  CUtensorMap tmR = tmC;
  if (RTMA) {
    if (int e = make_tmap_2d(&tmR, epi.residual, DSF_F32, M, N, epi.ldc, 32, 32)) return e;
  }
  const int m_tiles = cdiv(M, 256), n_tiles = N / BN;
  const int tiles = m_tiles * n_tiles;
  const int pairs = std::min(tiles, num_sms() / 2);
  int tail_start = tiles;
  const int rem = tiles % pairs;
  // Split the leftover tiles along N (256 x 128 or 256 x 64 units, see the kernel): no partial sums, works with every
  // epilogue.  (Splitting them along K, with fp32 reductions into a zero-filled C, was measured slower and removed.)
  int n_split = 1;
  CUtensorMap tmBt = tmB;
  if (BN == 256 && Bptr != nullptr && rem > 0 && tiles > pairs) {
    for (int ns = 4; ns >= 2; ns >>= 1) {
      if (rem * ns <= pairs) { n_split = ns; break; }
    }
    if (n_split > 1) {
      tail_start = tiles - rem;
      if (int e = make_tmap_bf16(&tmBt, Bptr, N, K, ldb, BN / n_split / 2)) return e;
    }
  }
  launch_pdl(gemm_nt3_kernel<BN, STAGES, RTMA>, dim3(2 * pairs), dim3(G2_THREADS), L::DYN, st, tmA, tmB, tmC, tmBt, tmR, epi, M, N, K, m_tiles,
             n_tiles, tail_start, n_split);
  return check_launch("gemm_nt3");
}

// tile-shape choice: fewest "rounds" of 128 x BN tiles over the SMs, weighted by the per-tile efficiency of wider tiles
static int pick_bn_nt(int M, int N) {
  const int sms = num_sms();
  const int m_tiles = cdiv(M, G2_BM);
  int best = 64;
  double best_cost = 1e30;
  const int cands[3] = {256, 128, 64};
  const double tile_eff[3] = {1.0, 0.85, 0.6};
  for (int i = 0; i < 3; ++i) {
    const int bn = cands[i];
    if (N % bn) continue;
    const int tiles = m_tiles * (N / bn);
    const double cost = (double)cdiv(tiles, sms) * bn / tile_eff[i];
    if (cost < best_cost) { best_cost = cost; best = bn; }
  }
  return best;
}

int gemm_nt_run(const void* A, int lda, const void* B, int ldb, void* C, int ldc, int c_dtype, const float* bias, const float* residual, int M,
                int N, int K, int flags, const dsf_dropout* drop, const void* relu_src, bool pairs, cudaStream_t st) {
  CUtensorMap tmA, tmB;
  if (pairs && N % 128 == 0 && M > 128) {
    // CTA-pair kernel: 256 x BN tiles, each CTA loads BN/2 rows of B.  BN = 256 whenever N allows: one tcgen05.mma costs
    // about the same ~85 ns for N = 128 as for N = 256 (operand reads from shared memory bound it), so narrow tiles
    // waste the tensor pipe even when they would balance the 74 pairs better (measured: N = 512, K = 2048 runs 27.0 us
    // with 256-wide and 30.2 us with 128-wide tiles).
    const int BN3 = (N % 256 == 0) ? 256 : 128;
    if (int e = make_tmap_bf16(&tmA, A, M, K, lda, G2_BM)) return e;
    if (int e = make_tmap_bf16(&tmB, B, N, K, ldb, BN3 / 2)) return e;
    CUtensorMap tmC3;
    if (int e = make_tmap_2d(&tmC3, C, c_dtype, M, N, ldc, c_dtype == DSF_F32 ? 32 : 64, 32)) return e;
    EpiArgs2 epi3{C, ldc, c_dtype, bias, residual, flags, N, reinterpret_cast<const __nv_bfloat16*>(relu_src), make_drop(drop)};
    // fp32 output + residual: the residual tile is prefetched by TMA (RTMA, see the kernel)
    const bool res_tma = c_dtype == DSF_F32 && (flags & DSF_EPI_RESIDUAL) && residual != nullptr;
    if (BN3 == 256 && res_tma) return launch_nt3<256, 4, true>(tmA, tmB, tmC3, epi3, M, N, K, st, B, ldb);
    if (BN3 == 256) return launch_nt3<256, 5>(tmA, tmB, tmC3, epi3, M, N, K, st, B, ldb);
    if (res_tma) return launch_nt3<128, 5, true>(tmA, tmB, tmC3, epi3, M, N, K, st);
    return launch_nt3<128, 6>(tmA, tmB, tmC3, epi3, M, N, K, st);
  }
  const int BN = pick_bn_nt(M, N);
  if (int e = make_tmap_bf16(&tmA, A, M, K, lda, G2_BM)) return e;
  if (int e = make_tmap_bf16(&tmB, B, N, K, ldb, BN)) return e;
  CUtensorMap tmC;  // store boxes: 32 rows x 128 bytes
  if (int e = make_tmap_2d(&tmC, C, c_dtype, M, N, ldc, c_dtype == DSF_F32 ? 32 : 64, 32)) return e;
  EpiArgs2 epi{C, ldc, c_dtype, bias, residual, flags, N, reinterpret_cast<const __nv_bfloat16*>(relu_src), make_drop(drop)};
  if (BN == 256) return launch_nt2<256, 3>(tmA, tmB, tmC, epi, M, N, K, st);
  if (BN == 128) return launch_nt2<128, 4>(tmA, tmB, tmC, epi, M, N, K, st);
  return launch_nt2<64, 5>(tmA, tmB, tmC, epi, M, N, K, st);
}

int gemm_tn_run(const void* A, int lda, const void* B, int ldb, float* C, int ldc, int M, int Nout, int Kout, float* colsum, cudaStream_t st) {
  const int BN = (Kout % 256 == 0) ? 256 : ((Kout % 128 == 0) ? 128 : 64);
  CUtensorMap tmA, tmB;
  if (int e = make_tmap_bf16(&tmA, A, M, Nout, lda, G2_BK)) return e;
  if (int e = make_tmap_bf16(&tmB, B, M, Kout, ldb, G2_BK)) return e;
  if (BN == 256) return launch_tn2<256, 4>(tmA, tmB, C, ldc, M, Nout, Kout, colsum, st);
  if (BN == 128) return launch_tn2<128, 6>(tmA, tmB, C, ldc, M, Nout, Kout, colsum, st);
  return launch_tn2<64, 8>(tmA, tmB, C, ldc, M, Nout, Kout, colsum, st);
}

}  // namespace dsf

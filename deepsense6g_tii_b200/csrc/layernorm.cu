// K2: warp-shuffle LayerNorm forward / backward (nn.LayerNorm(C), eps 1e-5; model2_seq.py:118-119,199,
// used :131-132,274).  One warp owns one token row held entirely in registers (C <= 1024), statistics
// with two-pass mean / centred variance in fp32; HBM-bound (reads x, writes y).
//
// Backward: dx = rstd * (g*dy - mean(g*dy) - xhat * mean(g*dy*xhat)) [+ dx_add], and per-CTA partial
// dgamma / dbeta column sums that are folded into the fp32 outputs with one atomicAdd per column per CTA.
// Because dx is the gradient of the residual stream, it is also (a) the dY of the preceding Linear's
// bias (model2_seq.py:109,124) and (b) a tensor-core GEMM operand: the kernel optionally emits the column
// sums of dx (bias gradient) and a bf16 copy in the same pass, saving two more passes over the tensor.
#include <algorithm>
#include <cstdlib>

#include "common.cuh"

namespace dsf {

constexpr int LN_WARPS = 8;

// VPT = float4 vectors per lane; covers C <= 128*VPT
template <typename TY, int VPT>
__global__ void __launch_bounds__(LN_WARPS * 32)
layernorm_fwd_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                     TY* __restrict__ y, float* __restrict__ mean, float* __restrict__ rstd, int M, int C, float eps) {
  pdl_trigger();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nvec = C >> 2;
  const float invC = 1.0f / (float)C;
  for (int row = blockIdx.x * LN_WARPS + warp; row < M; row += gridDim.x * LN_WARPS) {
    const float* xr = x + (size_t)row * C;
    float v[VPT][4];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < VPT; ++i) {
      const int vi = lane + 32 * i;
      if (vi < nvec) {
        Vec4<float>::load(xr + vi * 4, v[i]);
        s += (v[i][0] + v[i][1]) + (v[i][2] + v[i][3]);
      } else {
        v[i][0] = v[i][1] = v[i][2] = v[i][3] = 0.f;
      }
    }
    const float mu = warp_sum(s) * invC;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < VPT; ++i) {
      const int vi = lane + 32 * i;
      if (vi < nvec) {
#pragma unroll
        for (int k = 0; k < 4; ++k) { const float d = v[i][k] - mu; q += d * d; }
      }
    }
    const float rs = rsqrtf(warp_sum(q) * invC + eps);
    if (lane == 0) { mean[row] = mu; rstd[row] = rs; }
    TY* yr = y + (size_t)row * C;
#pragma unroll
    for (int i = 0; i < VPT; ++i) {
      const int vi = lane + 32 * i;
      if (vi < nvec) {
        float g4[4], b4[4], o[4];
        Vec4<float>::load(gamma + vi * 4, g4);
        Vec4<float>::load(beta + vi * 4, b4);
#pragma unroll
        for (int k = 0; k < 4; ++k) o[k] = (v[i][k] - mu) * rs * g4[k] + b4[k];
        Vec4<TY>::store(yr + vi * 4, o);
      }
    }
  }
}

// DROP is a template parameter: the Philox code costs ~13 registers, which would take the common p = 0 instantiation
// from 2 to 1 resident CTAs per SM.
template <typename TY, int VPT, bool EXTRA, bool DROP>
__global__ void __launch_bounds__(LN_WARPS * 32, (VPT <= 4 && !DROP) ? 2 : 1)
layernorm_bwd_kernel(const TY* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ gamma,
                     const float* __restrict__ mean, const float* __restrict__ rstd, const float* dx_add, float* dx,
                     float* __restrict__ dgamma, float* __restrict__ dbeta, __nv_bfloat16* __restrict__ dx_bf16,
                     float* __restrict__ dx_colsum, DropArgs drop, int M, int C) {
  // column partials of the CTA's warps: [quantity (dgamma, dbeta, by-product sums)][warp][column]; quantities are
  // reduced one after another for C > 512 (static shared memory is capped at 48 KB), all at once otherwise
  constexpr int NQ = EXTRA ? 3 : 2;
  constexpr int QPP = VPT <= 4 ? NQ : 1;  // quantities per pass
  __shared__ float red[QPP][LN_WARPS][VPT * 128];
  pdl_trigger();
  pdl_wait();
  if (DROP) drop = resolve_drop(drop);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nvec = C >> 2;
  const float invC = 1.0f / (float)C;
  float g4[VPT][4], dg[VPT][4], db[VPT][4], dc[EXTRA ? VPT : 1][4];
#pragma unroll
  for (int i = 0; i < VPT; ++i) {
    const int vi = lane + 32 * i;
#pragma unroll
    for (int k = 0; k < 4; ++k) { dg[i][k] = 0.f; db[i][k] = 0.f; g4[i][k] = 0.f; }
    if (EXTRA) {
#pragma unroll
      for (int k = 0; k < 4; ++k) dc[EXTRA ? i : 0][k] = 0.f;
    }
    if (vi < nvec) Vec4<float>::load(gamma + vi * 4, g4[i]);
  }
  for (int row = blockIdx.x * LN_WARPS + warp; row < M; row += gridDim.x * LN_WARPS) {
    const float mu = mean[row], rs = rstd[row];
    const float* xr = x + (size_t)row * C;
    const TY* dyr = dy + (size_t)row * C;
    float xh[VPT][4], gy[VPT][4], ad[VPT][4];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < VPT; ++i) {
      const int vi = lane + 32 * i;
      if (vi < nvec) {
        float xv[4], dv[4];
        Vec4<float>::load(xr + vi * 4, xv);
        Vec4<TY>::load(dyr + vi * 4, dv);
        if (dx_add) Vec4<float>::load(dx_add + (size_t)row * C + vi * 4, ad[i]);  // issued early: independent of the reductions
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          xh[i][k] = (xv[k] - mu) * rs;
          gy[i][k] = dv[k] * g4[i][k];
          s1 += gy[i][k];
          s2 += gy[i][k] * xh[i][k];
          dg[i][k] += dv[k] * xh[i][k];
          db[i][k] += dv[k];
        }
      } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) { xh[i][k] = 0.f; gy[i][k] = 0.f; }
      }
    }
    const float m1 = warp_sum(s1) * invC, m2 = warp_sum(s2) * invC;
    float* dxr = dx + (size_t)row * C;
#pragma unroll
    for (int i = 0; i < VPT; ++i) {
      const int vi = lane + 32 * i;
      if (vi < nvec) {
        float o[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) o[k] = rs * (gy[i][k] - m1 - xh[i][k] * m2);
        if (dx_add) {
#pragma unroll
          for (int k = 0; k < 4; ++k) o[k] += ad[i][k];
        }
        Vec4<float>::store(dxr + vi * 4, o);
        if (EXTRA) {
          if (DROP) {  // by-products are the gradient of the preceding Linear's PRE-dropout output
            float m[4];
            drop_scale4(drop, (uint64_t)row * nvec + vi, m);
#pragma unroll
            for (int k = 0; k < 4; ++k) o[k] *= m[k];
          }
          if (dx_bf16) Vec4<__nv_bfloat16>::store(dx_bf16 + (size_t)row * C + vi * 4, o);
#pragma unroll
          for (int k = 0; k < 4; ++k) dc[EXTRA ? i : 0][k] += o[k];
        }
      }
    }
  }
  // CTA reduction of the column partials, then one atomic per column and quantity
#pragma unroll 1
  for (int pass = 0; pass < NQ / QPP; ++pass) {
    if (pass > 0) __syncthreads();
#pragma unroll
    for (int qq = 0; qq < QPP; ++qq) {
      const int qn = pass * QPP + qq;
#pragma unroll
      for (int i = 0; i < VPT; ++i) {
        const int vi = lane + 32 * i;
        const float* src = qn == 0 ? dg[i] : (qn == 1 ? db[i] : dc[EXTRA ? i : 0]);
        *reinterpret_cast<float4*>(&red[qq][warp][vi * 4]) = make_float4(src[0], src[1], src[2], src[3]);
      }
    }
    __syncthreads();
#pragma unroll
    for (int qq = 0; qq < QPP; ++qq) {
      const int qn = pass * QPP + qq;
      float* out = qn == 0 ? dgamma : (qn == 1 ? dbeta : dx_colsum);
      if (out == nullptr) continue;
      for (int c = threadIdx.x; c < C; c += LN_WARPS * 32) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < LN_WARPS; ++w) s += red[qq][w][c];
        atomicAdd(out + c, s);
      }
    }
  }
}


// ------------------------------------------------------------------------------------------ v2: cp.async row rings
// The v1 kernels above keep a row in registers and therefore have one row per warp in flight: every row costs a full
// DRAM round trip and the kernels sit at 3-4 TB/s.  v2 decouples bytes in flight from registers: every warp owns a ring
// of LN2_ST row slots in shared memory that it fills with cp.async (each lane copies exactly the 16-byte chunks it will
// consume, so cp.async.wait_group is the only synchronisation for the data; the two row statistics of the backward ride
// in the slot header and are published with __syncwarp).  One CTA of 8 warps per SM, (ST - 1) rows per warp in flight.
// Requires C == 128 * VPT.
constexpr int LN2_WARPS = 8;

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async8(uint32_t dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async4(uint32_t dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ uint32_t smem_addr_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
template <typename T> __device__ __forceinline__ void lds_vec4(const uint8_t* p, float (&v)[4]);
template <> __device__ __forceinline__ void lds_vec4<float>(const uint8_t* p, float (&v)[4]) {
  const float4 t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
template <> __device__ __forceinline__ void lds_vec4<__nv_bfloat16>(const uint8_t* p, float (&v)[4]) {
  const uint2 t = *reinterpret_cast<const uint2*>(p);
  v[0] = __uint_as_float(t.x << 16); v[1] = __uint_as_float(t.x & 0xFFFF0000u);
  v[2] = __uint_as_float(t.y << 16); v[3] = __uint_as_float(t.y & 0xFFFF0000u);
}

template <typename TY, int VPT, int ST>
__global__ void __launch_bounds__(LN2_WARPS * 32, 1)
layernorm_fwd2_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                      TY* __restrict__ y, float* __restrict__ mean, float* __restrict__ rstd, int M, float eps) {
  constexpr int C = 128 * VPT, ROWB = C * 4;
  extern __shared__ __align__(16) uint8_t ln2_smem[];
  pdl_trigger();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t* ring = ln2_smem + (size_t)warp * ST * ROWB;
  const uint32_t ring_u = smem_addr_u32(ring);
  const int row0 = blockIdx.x * LN2_WARPS + warp, rstep = gridDim.x * LN2_WARPS;
  const int n_rows = row0 < M ? (M - row0 + rstep - 1) / rstep : 0;
  pdl_wait();
  auto issue = [&](int k) {
    if (k < n_rows) {
      const float* xr = x + (size_t)(row0 + k * rstep) * C;
      const uint32_t slot = ring_u + (uint32_t)(k % ST) * ROWB;
#pragma unroll
      for (int i = 0; i < VPT; ++i) cp_async16(slot + (lane + 32 * i) * 16, xr + (lane + 32 * i) * 4);
    }
    cp_async_commit();
  };
#pragma unroll
  for (int k = 0; k < ST - 1; ++k) issue(k);
  float g4[VPT][4], b4[VPT][4];
#pragma unroll
  for (int i = 0; i < VPT; ++i) {
    Vec4<float>::load(gamma + (lane + 32 * i) * 4, g4[i]);
    Vec4<float>::load(beta + (lane + 32 * i) * 4, b4[i]);
  }
  constexpr float invC = 1.0f / (float)C;
  for (int k = 0; k < n_rows; ++k) {
    issue(k + ST - 1);
    cp_async_wait<ST - 1>();
    const int row = row0 + k * rstep;
    const uint8_t* slot = ring + (size_t)(k % ST) * ROWB;
    float v[VPT][4];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < VPT; ++i) {
      lds_vec4<float>(slot + (lane + 32 * i) * 16, v[i]);
      s += (v[i][0] + v[i][1]) + (v[i][2] + v[i][3]);
    }
    const float mu = warp_sum(s) * invC;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < VPT; ++i) {
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) { const float d = v[i][kk] - mu; q += d * d; }
    }
    const float rs = rsqrtf(warp_sum(q) * invC + eps);
    if (lane == 0) { mean[row] = mu; rstd[row] = rs; }
    TY* yr = y + (size_t)row * C;
#pragma unroll
    for (int i = 0; i < VPT; ++i) {
      float o[4];
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) o[kk] = (v[i][kk] - mu) * rs * g4[i][kk] + b4[i][kk];
      Vec4<TY>::store(yr + (lane + 32 * i) * 4, o);
    }
  }
}

template <typename TY, int VPT> struct Ln2Bwd {
  static constexpr int C = 128 * VPT;
  static constexpr int ROWB = C * 4 + C * (int)sizeof(TY) + C * 4 + 16;  // x | dy | dx_add | mean, rstd
  static constexpr int ST = VPT <= 4 ? 4 : 2;
  static constexpr int RING = LN2_WARPS * ST * ROWB;
};

template <typename TY, int VPT, bool EXTRA, bool DROP>
__global__ void __launch_bounds__(LN2_WARPS * 32, 1)
layernorm_bwd2_kernel(const TY* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ gamma,
                      const float* __restrict__ mean, const float* __restrict__ rstd, const float* dx_add, float* dx,
                      float* __restrict__ dgamma, float* __restrict__ dbeta, __nv_bfloat16* __restrict__ dx_bf16,
                      float* __restrict__ dx_colsum, DropArgs drop, int M) {
  using L = Ln2Bwd<TY, VPT>;
  constexpr int C = L::C, ROWB = L::ROWB, ST = L::ST, NQ = EXTRA ? 3 : 2;
  constexpr int X_OFF = 0, DY_OFF = C * 4, AD_OFF = DY_OFF + C * (int)sizeof(TY), ST_OFF = AD_OFF + C * 4;
  static_assert(NQ * LN2_WARPS * C * 4 <= L::RING, "column-partial buffer must fit in the row rings it aliases");
  extern __shared__ __align__(16) uint8_t ln2_smem[];
  pdl_trigger();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t* ring = ln2_smem + (size_t)warp * ST * ROWB;
  const uint32_t ring_u = smem_addr_u32(ring);
  const int row0 = blockIdx.x * LN2_WARPS + warp, rstep = gridDim.x * LN2_WARPS;
  const int n_rows = row0 < M ? (M - row0 + rstep - 1) / rstep : 0;
  const bool has_add = dx_add != nullptr;
  pdl_wait();
  if (DROP) drop = resolve_drop(drop);
  auto issue = [&](int k) {
    if (k < n_rows) {
      const size_t row = (size_t)(row0 + k * rstep);
      const uint32_t slot = ring_u + (uint32_t)(k % ST) * ROWB;
#pragma unroll
      for (int i = 0; i < VPT; ++i) {
        const int vi = lane + 32 * i;
        cp_async16(slot + X_OFF + vi * 16, x + row * C + vi * 4);
        if (sizeof(TY) == 4) cp_async16(slot + DY_OFF + vi * 16, dy + row * C + vi * 4);
        else cp_async8(slot + DY_OFF + vi * 8, dy + row * C + vi * 4);
        if (has_add) cp_async16(slot + AD_OFF + vi * 16, dx_add + row * C + vi * 4);
      }
      if (lane == 0) cp_async4(slot + ST_OFF, mean + row);
      if (lane == 1) cp_async4(slot + ST_OFF + 4, rstd + row);
    }
    cp_async_commit();
  };
#pragma unroll
  for (int k = 0; k < ST - 1; ++k) issue(k);
  float g4[VPT][4], dg[VPT][4], db[VPT][4], dc[EXTRA ? VPT : 1][4];
#pragma unroll
  for (int i = 0; i < VPT; ++i) {
#pragma unroll
    for (int k = 0; k < 4; ++k) { dg[i][k] = 0.f; db[i][k] = 0.f; }
    if (EXTRA) {
#pragma unroll
      for (int k = 0; k < 4; ++k) dc[EXTRA ? i : 0][k] = 0.f;
    }
    Vec4<float>::load(gamma + (lane + 32 * i) * 4, g4[i]);
  }
  constexpr float invC = 1.0f / (float)C;
  constexpr int nvec = C / 4;
  for (int k = 0; k < n_rows; ++k) {
    issue(k + ST - 1);
    cp_async_wait<ST - 1>();
    __syncwarp();  // the statistics were copied by lanes 0 / 1
    const int row = row0 + k * rstep;
    const uint8_t* slot = ring + (size_t)(k % ST) * ROWB;
    const float mu = *reinterpret_cast<const float*>(slot + ST_OFF), rs = *reinterpret_cast<const float*>(slot + ST_OFF + 4);
    float xh[VPT][4], gy[VPT][4];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < VPT; ++i) {
      const int vi = lane + 32 * i;
      float xv[4], dv[4];
      lds_vec4<float>(slot + X_OFF + vi * 16, xv);
      lds_vec4<TY>(slot + DY_OFF + vi * (4 * (int)sizeof(TY)), dv);
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        xh[i][kk] = (xv[kk] - mu) * rs;
        gy[i][kk] = dv[kk] * g4[i][kk];
        s1 += gy[i][kk];
        s2 += gy[i][kk] * xh[i][kk];
        dg[i][kk] += dv[kk] * xh[i][kk];
        db[i][kk] += dv[kk];
      }
    }
    const float m1 = warp_sum(s1) * invC, m2 = warp_sum(s2) * invC;
    float* dxr = dx + (size_t)row * C;
#pragma unroll
    for (int i = 0; i < VPT; ++i) {
      const int vi = lane + 32 * i;
      float o[4];
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) o[kk] = rs * (gy[i][kk] - m1 - xh[i][kk] * m2);
      if (has_add) {
        float ad[4];
        lds_vec4<float>(slot + AD_OFF + vi * 16, ad);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) o[kk] += ad[kk];
      }
      Vec4<float>::store(dxr + vi * 4, o);
      if (EXTRA) {
        if (DROP) {  // by-products are the gradient of the preceding Linear's PRE-dropout output
          float m[4];
          drop_scale4(drop, (uint64_t)row * nvec + vi, m);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) o[kk] *= m[kk];
        }
        if (dx_bf16) Vec4<__nv_bfloat16>::store(dx_bf16 + (size_t)row * C + vi * 4, o);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) dc[EXTRA ? i : 0][kk] += o[kk];
      }
    }
    __syncwarp();  // every lane is done with this slot's header before lanes 0 / 1 refill it
  }
  // CTA reduction of the column partials (the buffer aliases the drained rings), then one atomic per column and quantity
  cp_async_wait<0>();
  __syncthreads();
  float* red = reinterpret_cast<float*>(ln2_smem);  // [quantity][warp][column]
#pragma unroll
  for (int qn = 0; qn < NQ; ++qn) {
#pragma unroll
    for (int i = 0; i < VPT; ++i) {
      const float* src = qn == 0 ? dg[i] : (qn == 1 ? db[i] : dc[EXTRA ? i : 0]);
      *reinterpret_cast<float4*>(&red[(qn * LN2_WARPS + warp) * C + (lane + 32 * i) * 4]) = make_float4(src[0], src[1], src[2], src[3]);
    }
  }
  __syncthreads();
#pragma unroll
  for (int qn = 0; qn < NQ; ++qn) {
    float* out = qn == 0 ? dgamma : (qn == 1 ? dbeta : dx_colsum);
    if (out == nullptr) continue;
    for (int c = threadIdx.x; c < C; c += LN2_WARPS * 32) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < LN2_WARPS; ++w) s += red[(qn * LN2_WARPS + w) * C + c];
      atomicAdd(out + c, s);
    }
  }
}

template <typename K>
static bool ln2_configure(K kernel, int smem) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) == cudaSuccess;
}

template <typename TY, int VPT>
int launch_ln_fwd2(const float* x, const float* gamma, const float* beta, TY* y, float* mean, float* rstd, int M, float eps, cudaStream_t st) {
  constexpr int ST = VPT <= 2 ? 8 : (VPT <= 4 ? 8 : 4);
  constexpr int SMEM = LN2_WARPS * ST * 128 * VPT * 4;
  static bool configured_on[64] = {};
  bool& configured = per_device_flag(configured_on);  // the attribute is per device (common.cuh)
  if (!configured && !(configured = ln2_configure(layernorm_fwd2_kernel<TY, VPT, ST>, SMEM))) return check_launch("layernorm_fwd2/attr");
  const int blocks = std::min(cdiv(M, LN2_WARPS), num_sms());
  launch_pdl(layernorm_fwd2_kernel<TY, VPT, ST>, dim3(blocks), dim3(LN2_WARPS * 32), SMEM, st, x, gamma, beta, y, mean, rstd, M, eps);
  return check_launch("layernorm_fwd2");
}

template <typename TY, int VPT, bool EXTRA>
int launch_ln_bwd2(const TY* dy, const float* x, const float* gamma, const float* mean, const float* rstd, const float* dx_add, float* dx,
                   float* dgamma, float* dbeta, __nv_bfloat16* dx_bf16, float* dx_colsum, DropArgs drop, int M, cudaStream_t st) {
  using L = Ln2Bwd<TY, VPT>;
  const int blocks = std::min(cdiv(M, LN2_WARPS), num_sms());
  if (EXTRA && drop.thresh != 0) {
    static bool configured_on[64] = {};
    bool& configured = per_device_flag(configured_on);
    if (!configured && !(configured = ln2_configure(layernorm_bwd2_kernel<TY, VPT, EXTRA, EXTRA>, L::RING))) return check_launch("layernorm_bwd2/attr");
    launch_pdl(layernorm_bwd2_kernel<TY, VPT, EXTRA, EXTRA>, dim3(blocks), dim3(LN2_WARPS * 32), L::RING, st, dy, x, gamma, mean, rstd, dx_add, dx,
               dgamma, dbeta, dx_bf16, dx_colsum, drop, M);
  } else {
    static bool configured_on[64] = {};
    bool& configured = per_device_flag(configured_on);
    if (!configured && !(configured = ln2_configure(layernorm_bwd2_kernel<TY, VPT, EXTRA, false>, L::RING))) return check_launch("layernorm_bwd2/attr");
    launch_pdl(layernorm_bwd2_kernel<TY, VPT, EXTRA, false>, dim3(blocks), dim3(LN2_WARPS * 32), L::RING, st, dy, x, gamma, mean, rstd, dx_add, dx,
               dgamma, dbeta, dx_bf16, dx_colsum, drop, M);
  }
  return check_launch("layernorm_bwd2");
}

template <typename TY>
int launch_ln_fwd(const float* x, const float* gamma, const float* beta, void* y, float* mean, float* rstd, int M, int C,
                  float eps, cudaStream_t st) {
  TY* yy = reinterpret_cast<TY*>(y);
  if (C % 128 == 0) {  // cp.async row rings (v2) where C / 128 is 1, 2, 4 or 8; register-resident rows (v1) otherwise
    switch (C / 128) {
      case 1: return launch_ln_fwd2<TY, 1>(x, gamma, beta, yy, mean, rstd, M, eps, st);
      case 2: return launch_ln_fwd2<TY, 2>(x, gamma, beta, yy, mean, rstd, M, eps, st);
      case 4: return launch_ln_fwd2<TY, 4>(x, gamma, beta, yy, mean, rstd, M, eps, st);
      case 8: return launch_ln_fwd2<TY, 8>(x, gamma, beta, yy, mean, rstd, M, eps, st);
      default: break;
    }
  }
  const int blocks = std::min(cdiv(M, LN_WARPS), num_sms() * 8);
#define DSF_LN_FWD(V) launch_pdl(layernorm_fwd_kernel<TY, V>, dim3(blocks), dim3(LN_WARPS * 32), 0, st, x, gamma, beta, yy, mean, rstd, M, C, eps)
  if (C <= 128) DSF_LN_FWD(1);
  else if (C <= 256) DSF_LN_FWD(2);
  else if (C <= 512) DSF_LN_FWD(4);
  else DSF_LN_FWD(8);
#undef DSF_LN_FWD
  return check_launch("layernorm_fwd");
}

template <typename TY, bool EXTRA>
int launch_ln_bwd(const void* dy, const float* x, const float* gamma, const float* mean, const float* rstd,
                  const float* dx_add, float* dx, float* dgamma, float* dbeta, void* dx_bf16, float* dx_colsum, DropArgs drop, int M, int C,
                  cudaStream_t st) {
  // few, fat CTAs: every CTA ends with 2-3 x C atomics
  const int blocks = std::min(cdiv(M, LN_WARPS * 2), num_sms() * 4);
  const TY* d = reinterpret_cast<const TY*>(dy);
  __nv_bfloat16* xb = reinterpret_cast<__nv_bfloat16*>(dx_bf16);
  if (C % 128 == 0) {
    switch (C / 128) {
      case 1: return launch_ln_bwd2<TY, 1, EXTRA>(d, x, gamma, mean, rstd, dx_add, dx, dgamma, dbeta, xb, dx_colsum, drop, M, st);
      case 2: return launch_ln_bwd2<TY, 2, EXTRA>(d, x, gamma, mean, rstd, dx_add, dx, dgamma, dbeta, xb, dx_colsum, drop, M, st);
      case 4: return launch_ln_bwd2<TY, 4, EXTRA>(d, x, gamma, mean, rstd, dx_add, dx, dgamma, dbeta, xb, dx_colsum, drop, M, st);
      case 8: return launch_ln_bwd2<TY, 8, EXTRA>(d, x, gamma, mean, rstd, dx_add, dx, dgamma, dbeta, xb, dx_colsum, drop, M, st);
      default: break;
    }
  }
#define DSF_LN_BWD1(V, D) launch_pdl(layernorm_bwd_kernel<TY, V, EXTRA, D>, dim3(blocks), dim3(LN_WARPS * 32), 0, st, d, x, gamma, mean, rstd, dx_add, dx, dgamma, dbeta, xb, dx_colsum, drop, M, C)
#define DSF_LN_BWD(V)                                   \
  do {                                                  \
    if (EXTRA && drop.thresh != 0) DSF_LN_BWD1(V, EXTRA); \
    else DSF_LN_BWD1(V, false);                         \
  } while (0)
  if (C <= 128) DSF_LN_BWD(1);
  else if (C <= 256) DSF_LN_BWD(2);
  else if (C <= 512) DSF_LN_BWD(4);
  else DSF_LN_BWD(8);
#undef DSF_LN_BWD
#undef DSF_LN_BWD1
  return check_launch("layernorm_bwd");
}

}  // namespace dsf

using namespace dsf;

extern "C" int dsf_layernorm_fwd(const float* x, const float* gamma, const float* beta, void* y, int32_t y_dtype,
                                 float* mean, float* rstd, int32_t M, int32_t C, float eps, void* stream) {
  DSF_REQUIRE(x && gamma && beta && y && mean && rstd, "layernorm_fwd: NULL pointer");
  DSF_REQUIRE(M > 0 && C > 0 && C % 4 == 0 && C <= 1024, "layernorm_fwd: need M>0 and C multiple of 4 up to 1024 (got M=%d C=%d)", M, C);
  DSF_REQUIRE(aligned16(x) && aligned16(gamma) && aligned16(beta) && aligned16(y), "layernorm_fwd: 16-byte alignment required");
  DSF_REQUIRE(y_dtype == DSF_F32 || y_dtype == DSF_BF16, "layernorm_fwd: bad y_dtype %d", y_dtype);
  cudaStream_t st = (cudaStream_t)stream;
  if (y_dtype == DSF_F32) return launch_ln_fwd<float>(x, gamma, beta, y, mean, rstd, M, C, eps, st);
  return launch_ln_fwd<__nv_bfloat16>(x, gamma, beta, y, mean, rstd, M, C, eps, st);
}

extern "C" int dsf_layernorm_bwd(const void* dy, int32_t dy_dtype, const float* x, const float* gamma, const float* mean,
                                 const float* rstd, const float* dx_add, float* dx_out, float* dgamma, float* dbeta,
                                 void* dx_bf16, float* dx_colsum, const dsf_dropout* byprod_drop, int32_t M, int32_t C, void* stream) {
  DSF_REQUIRE(dy && x && gamma && mean && rstd && dx_out && dgamma && dbeta, "layernorm_bwd: NULL pointer");
  DSF_REQUIRE(M > 0 && C > 0 && C % 4 == 0 && C <= 1024, "layernorm_bwd: need M>0 and C multiple of 4 up to 1024 (got M=%d C=%d)", M, C);
  DSF_REQUIRE(aligned16(dy) && aligned16(x) && aligned16(gamma) && aligned16(dx_add) && aligned16(dx_out) && aligned16(dx_bf16),
              "layernorm_bwd: 16-byte alignment required");
  DSF_REQUIRE(dy_dtype == DSF_F32 || dy_dtype == DSF_BF16, "layernorm_bwd: bad dy_dtype %d", dy_dtype);
  cudaStream_t st = (cudaStream_t)stream;
  const bool extra = dx_bf16 != nullptr || dx_colsum != nullptr;
  DSF_REQUIRE(!byprod_drop || (byprod_drop->p >= 0.f && byprod_drop->p < 1.f), "layernorm_bwd: dropout p must be in [0, 1)");
  const DropArgs dr = make_drop(byprod_drop);
  if (dy_dtype == DSF_F32) {
    if (extra) return launch_ln_bwd<float, true>(dy, x, gamma, mean, rstd, dx_add, dx_out, dgamma, dbeta, dx_bf16, dx_colsum, dr, M, C, st);
    return launch_ln_bwd<float, false>(dy, x, gamma, mean, rstd, dx_add, dx_out, dgamma, dbeta, nullptr, nullptr, dr, M, C, st);
  }
  if (extra) return launch_ln_bwd<__nv_bfloat16, true>(dy, x, gamma, mean, rstd, dx_add, dx_out, dgamma, dbeta, dx_bf16, dx_colsum, dr, M, C, st);
  return launch_ln_bwd<__nv_bfloat16, false>(dy, x, gamma, mean, rstd, dx_add, dx_out, dgamma, dbeta, nullptr, nullptr, dr, M, C, st);
}

// K4 entry points: fused flash-style multi-head self-attention (no mask) on tcgen05 with S / O accumulators in TMEM.
// Replaces model2_seq.py:102-106 (q@k^T * 1/sqrt(hs), softmax, attn_drop, att@v, transpose+contiguous) and its autograd; the
// (B, nh, T, T) score tensor is never materialised.  The kernels live in attn_tc2.cu; this file holds the C ABI, argument
// checks and the small rowsum(dO * O) kernel of the backward.
#include <algorithm>

#include "tc_common.cuh"

namespace dsf {


// ============================================================================================ backward
// delta[b,h,t] = sum_d dy[b,t,h*hs+d] * y[b,t,h*hs+d]   (rowsum(dO * O)); one warp per token row.
__global__ void __launch_bounds__(256)
attn_delta_kernel(const __nv_bfloat16* __restrict__ y, const __nv_bfloat16* __restrict__ dy, float* __restrict__ delta, int B, int T,
                  int C, int nh) {
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int hs = C / nh, gl = hs / 8;  // lanes per head (power of two, 2..16)
  const int nchunk = C / 8;
  for (int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); row < (int64_t)B * T; row += (int64_t)gridDim.x * 8) {
    const int b = (int)(row / T), t = (int)(row % T);
    for (int c0 = 0; c0 < nchunk; c0 += 32) {
      const int ch = c0 + lane;
      float acc = 0.f;
      if (ch < nchunk) {
        const uint4 a = __ldg(reinterpret_cast<const uint4*>(y + row * C + ch * 8));
        const uint4 d = __ldg(reinterpret_cast<const uint4*>(dy + row * C + ch * 8));
        const __nv_bfloat162* ap = reinterpret_cast<const __nv_bfloat162*>(&a);
        const __nv_bfloat162* dp = reinterpret_cast<const __nv_bfloat162*>(&d);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float2 af = __bfloat1622float2(ap[k]), df = __bfloat1622float2(dp[k]);
          acc += af.x * df.x + af.y * df.y;
        }
      }
      for (int o = gl >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (ch < nchunk && (lane % gl) == 0) delta[((size_t)b * nh + (ch * 8) / hs) * T + t] = acc;
    }
  }
}

// warp-specialised, TMA-fed kernels (attn_tc2.cu)
int attn_fwd_run(const void* qkv, void* y, float* lse, int B, int T, int C, int nh, const dsf_dropout* drop, uint32_t* bits, cudaStream_t st);
int attn_bwd_run(const void* qkv, const void* y, const void* dy, const float* lse, float* delta, void* dqkv, int B, int T, int C, int nh,
                 const dsf_dropout* drop, uint32_t* bits, int parts, cudaStream_t st);

int run_attn_delta(const void* y, const void* dy, float* delta, int B, int T, int C, int nh, cudaStream_t st) {
  launch_pdl(attn_delta_kernel, dim3(std::min(cdiv(B * T, 8), num_sms() * 8)), dim3(256), 0, st, (const __nv_bfloat16*)y, (const __nv_bfloat16*)dy,
             delta, B, T, C, nh);
  return check_launch("attn_bwd/delta");
}

}  // namespace dsf

using namespace dsf;

static int check_attn_drop(const char* who, const dsf_dropout* drop, const uint32_t* bits, bool& on) {
  on = drop && drop->p > 0.f;
  if (!on) return DSF_OK;
  if (!(drop->p < 1.f)) { set_error("%s: dropout p must be in [0, 1)", who); return DSF_EINVAL; }
  if (!bits) { set_error("%s: attention dropout needs the drop_bits buffer", who); return DSF_EINVAL; }
  return DSF_OK;
}

static int check_head_size(const char* who, int hs) {
  if (hs == 16 || hs == 32 || hs == 64 || hs == 128) return DSF_OK;
  set_error("%s: head size %d not supported (16, 32, 64, 128)", who, hs);
  return DSF_EUNSUPPORTED;
}

extern "C" int64_t dsf_attn_drop_words(int32_t B, int32_t T, int32_t nh) {
  if (B <= 0 || T <= 0 || nh <= 0) return 0;
  return (int64_t)B * nh * T * (2 * cdiv(T, 64));
}

extern "C" int dsf_attn_fwd(const void* qkv, void* y, float* lse, int32_t B, int32_t T, int32_t C, int32_t nh, const dsf_dropout* drop,
                            uint32_t* drop_bits, void* stream) {
  DSF_REQUIRE(qkv && y && lse, "attn_fwd: NULL pointer");
  bool drop_on;
  if (int e = check_attn_drop("attn_fwd", drop, drop_bits, drop_on)) return e;
  DSF_REQUIRE(B > 0 && T > 0 && C > 0 && nh > 0 && C % nh == 0, "attn_fwd: bad shape B=%d T=%d C=%d nh=%d", B, T, C, nh);
  DSF_REQUIRE(aligned16(qkv) && aligned16(y), "attn_fwd: 16-byte alignment required");
  DSF_REQUIRE(B <= 65535 && nh <= 65535, "attn_fwd: grid too large");
  if (int e = check_head_size("attn_fwd", C / nh)) return e;
  return attn_fwd_run(qkv, y, lse, B, T, C, nh, drop_on ? drop : nullptr, drop_bits, (cudaStream_t)stream);
}

static int attn_bwd_impl(const void* qkv, const void* y, const void* dy, const float* lse, float* delta, void* dqkv, int32_t B, int32_t T,
                         int32_t C, int32_t nh, const dsf_dropout* drop, const uint32_t* drop_bits, int parts, void* stream) {
  DSF_REQUIRE(qkv && y && dy && lse && delta && dqkv, "attn_bwd: NULL pointer");
  bool drop_on;
  if (int e = check_attn_drop("attn_bwd", drop, drop_bits, drop_on)) return e;
  DSF_REQUIRE(B > 0 && T > 0 && C > 0 && nh > 0 && C % nh == 0, "attn_bwd: bad shape B=%d T=%d C=%d nh=%d", B, T, C, nh);
  DSF_REQUIRE(aligned16(qkv) && aligned16(y) && aligned16(dy) && aligned16(dqkv), "attn_bwd: 16-byte alignment required");
  DSF_REQUIRE(B <= 65535 && nh <= 65535, "attn_bwd: grid too large");
  if (int e = check_head_size("attn_bwd", C / nh)) return e;
  return attn_bwd_run(qkv, y, dy, lse, delta, dqkv, B, T, C, nh, drop_on ? drop : nullptr, const_cast<uint32_t*>(drop_bits), parts, (cudaStream_t)stream);
}

extern "C" int dsf_attn_bwd(const void* qkv, const void* y, const void* dy, const float* lse, float* delta, void* dqkv, int32_t B,
                            int32_t T, int32_t C, int32_t nh, const dsf_dropout* drop, const uint32_t* drop_bits, void* stream) {
  return attn_bwd_impl(qkv, y, dy, lse, delta, dqkv, B, T, C, nh, drop, drop_bits, 7, stream);
}

extern "C" int dsf_attn_bwd_parts(const void* qkv, const void* y, const void* dy, const float* lse, float* delta, void* dqkv, int32_t B,
                                  int32_t T, int32_t C, int32_t nh, const dsf_dropout* drop, const uint32_t* drop_bits, int32_t parts,
                                  void* stream) {
  DSF_REQUIRE(parts > 0 && parts <= 7, "attn_bwd_parts: parts must be a non-empty subset of {1 = delta, 2 = dK/dV, 4 = dQ}");
  return attn_bwd_impl(qkv, y, dy, lse, delta, dqkv, B, T, C, nh, drop, drop_bits, parts, stream);
}

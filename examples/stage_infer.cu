// One GPT fusion stage, inference forward, from C++ through libdsfuse.so alone (no Python, no libtorch):
//   make -C deepsense6g_tii_b200/csrc example && deepsense6g_tii_b200/csrc/build/stage_infer
// The stage is the first of TransFuser's four (n_embd 64 on 64 x 64 maps, 8 x 8 anchors, seq_len 5, one camera view, 4 heads,
// 8 blocks, MLP width 256), at batch 1.  Inputs and parameters come from a fixed integer hash, so the run needs no files and
// Python can rebuild the same tensors (tests/test_gpu_stage_capi.py does, and compares the checksums printed here).
// Call sequence: dsf_check_device -> dsf_stage_workspace_size -> cudaMalloc(workspace) -> dsf_stage_fwd -> cudaStreamSynchronize.
// The caller owns every buffer; the library allocates nothing and keeps no pointer after the call returns.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>

#include <vector>

#include "dsfuse.h"

#define CUDA_OK(x)                                                                       \
  do {                                                                                   \
    cudaError_t e_ = (x);                                                                \
    if (e_ != cudaSuccess) {                                                             \
      fprintf(stderr, "%s:%d: %s: %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_)); \
      exit(1);                                                                           \
    }                                                                                    \
  } while (0)
#define DSF_OK_(x)                                                                       \
  do {                                                                                   \
    int e_ = (x);                                                                        \
    if (e_ != DSF_OK) {                                                                  \
      fprintf(stderr, "%s failed (code %d): %s\n", #x, e_, dsf_last_error());            \
      exit(1);                                                                           \
    }                                                                                    \
  } while (0)

// Input values: uniform in [-0.5, 0.5) on a 2^-24 grid, a pure function of (stream, element index).
static uint32_t mix(uint32_t x) {
  x ^= x >> 16;
  x *= 0x7feb352du;
  x ^= x >> 15;
  x *= 0x846ca68bu;
  x ^= x >> 16;
  return x;
}
static float hval(uint32_t stream, uint32_t i) { return (float)(mix(i ^ mix(stream)) >> 8) * (1.0f / 16777216.0f) - 0.5f; }

// Bit-exact checksum of an fp32 device buffer: sum over its 16-bit words h[i] of h[i] * (2i + 1), modulo 2^64.
static unsigned long long checksum(const float* dev, size_t n, double* fsum) {
  std::vector<float> v(n);
  CUDA_OK(cudaMemcpy(v.data(), dev, n * sizeof(float), cudaMemcpyDeviceToHost));
  const unsigned short* h = reinterpret_cast<const unsigned short*>(v.data());  // little-endian 16-bit words
  unsigned long long s = 0;
  for (size_t i = 0; i < 2 * n; ++i) s += (unsigned long long)h[i] * (2ull * i + 1ull);
  double f = 0.0;
  for (size_t i = 0; i < n; ++i) f += v[i];
  *fsum = f;
  return s;
}

static void* upload(std::vector<float>& v) {
  void* d = nullptr;
  CUDA_OK(cudaMalloc(&d, v.size() * sizeof(float)));
  CUDA_OK(cudaMemcpy(d, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice));
  return d;
}

int main() {
  const int B = 1, S = 5, V = 1, A = 8, C = 64, H = 64, W = 64, NH = 4, L = 8, F = 4 * C;
  const int T = (V + 2) * S * A * A + 2;
  DSF_OK_(dsf_check_device());

  dsf_stage_desc d = {};
  d.geom = dsf_geom{B, S, V, A, A, C, H, W, DSF_F32, DSF_NCHW};
  d.n_head = NH;
  d.n_layer = L;
  d.F = F;
  d.residual = 1;
  d.chain = -1;
  d.prepacked = 0;     // the library packs each block's bf16 weight shadows into the workspace
  d.dropout = nullptr; // eval mode

  // feature maps (streams 0..2) and GPS tokens (stream 3)
  const size_t n_img = (size_t)B * V * S * C * H * W, n_map = (size_t)B * S * C * H * W, n_gps = (size_t)B * 2 * C;
  const size_t n_in[4] = {n_img, n_map, n_map, n_gps};
  void* in[4];
  for (int k = 0; k < 4; ++k) {
    std::vector<float> v(n_in[k]);
    for (size_t i = 0; i < v.size(); ++i) v[i] = hval(k, (uint32_t)i) * (k < 3 ? 2.0f : 1.0f);
    in[k] = upload(v);
  }
  // parameters in state-dict order (stream 100 + index): LayerNorm weights 1 + u/4, LayerNorm biases u/8, Linear weights u/8,
  // Linear biases u/16, pos_emb u/8
  std::vector<const float*> params;
  auto param = [&](size_t n, float scale, float shift) {
    std::vector<float> v(n);
    const uint32_t stream = 100u + (uint32_t)params.size();
    for (size_t i = 0; i < n; ++i) v[i] = shift + hval(stream, (uint32_t)i) * scale;
    params.push_back((const float*)upload(v));
  };
  param((size_t)T * C, 0.125f, 0.f);
  for (int i = 0; i < L; ++i) {
    param(C, 0.25f, 1.f), param(C, 0.125f, 0.f), param(C, 0.25f, 1.f), param(C, 0.125f, 0.f);  // ln1, ln2
    for (int k = 0; k < 4; ++k) param((size_t)C * C, 0.125f, 0.f), param(C, 0.0625f, 0.f);      // key, query, value, proj
    param((size_t)F * C, 0.125f, 0.f), param(F, 0.0625f, 0.f);                                  // mlp.0
    param((size_t)C * F, 0.125f, 0.f), param(C, 0.0625f, 0.f);                                  // mlp.2
  }
  param(C, 0.25f, 1.f), param(C, 0.125f, 0.f);  // ln_f
  dsf_stage_params p = {params.data(), nullptr, nullptr, 0};  // no pre-packed shadows, no ready events, no repack

  void *out_img, *out_lidar, *out_radar, *gps_out, *ws;
  CUDA_OK(cudaMalloc(&out_img, n_img * 4));
  CUDA_OK(cudaMalloc(&out_lidar, n_map * 4));
  CUDA_OK(cudaMalloc(&out_radar, n_map * 4));
  CUDA_OK(cudaMalloc(&gps_out, n_gps * 4));
  size_t ws_bytes = 0;
  DSF_OK_(dsf_stage_workspace_size(&d, &ws_bytes));
  CUDA_OK(cudaMalloc(&ws, ws_bytes));  // cudaMalloc returns 256-byte aligned memory
  cudaStream_t st;
  CUDA_OK(cudaStreamCreate(&st));

  const long long n0 = dsf_launch_count();
  DSF_OK_(dsf_stage_fwd(&d, &p, in[0], in[1], in[2], (const float*)in[3], out_img, out_lidar, out_radar, (float*)gps_out, ws, ws_bytes, st));
  CUDA_OK(cudaStreamSynchronize(st));
  const long long launches = dsf_launch_count() - n0;

  printf("stage_infer: B=%d C=%d H=%d W=%d n_layer=%d T=%d workspace=%zu bytes\n", B, C, H, W, L, T, ws_bytes);
  const char* names[4] = {"img_out", "lidar_out", "radar_out", "gps_out"};
  void* outs[4] = {out_img, out_lidar, out_radar, gps_out};
  for (int k = 0; k < 4; ++k) {
    double fsum;
    const unsigned long long s = checksum((const float*)outs[k], n_in[k], &fsum);
    printf("checksum %s %016llx sum %.9e\n", names[k], s, fsum);
  }
  printf("launches %lld\n", launches);

  CUDA_OK(cudaStreamDestroy(st));
  for (void* q : {out_img, out_lidar, out_radar, gps_out, ws, in[0], in[1], in[2], in[3]}) CUDA_OK(cudaFree(q));
  for (const float* q : params) CUDA_OK(cudaFree((void*)q));
  return 0;
}

// Whole fusion-stage inference forward (dsf_stage_fwd): the launch sequence of the bf16 no-grad path, driven from host code
// through the library's own entry points.  No kernel lives here.
#include <string.h>

#include <utility>

#include "common.cuh"

namespace dsf {

int check_geom(const dsf_geom* g);

namespace {

constexpr size_t kWsAlign = 256;
inline size_t A(size_t n) { return (n + kWsAlign - 1) / kWsAlign * kWsAlign; }

// Everything dsf_stage_fwd derives from the descriptor, after the descriptor checks.
struct Plan {
  int B, T, Tm, C, nh, L, F;
  int M;
  bool chain;       // chain kernel between two attention calls (and in place of ln_f)
  bool attn_drop;   // attention dropout on: the workspace holds keep bits
  int slots;        // shadow slots in the workspace
  // byte offsets into the workspace
  size_t x[2], h1, qkv, y, lse, stats, yf, x_mid, h2, a, bits, shadow0, shadow_bytes, total;
};

float drop_p(const dsf_dropout_cfg* c, int which) { return c == nullptr ? 0.f : which == 0 ? c->embd : which == 1 ? c->attn : c->resid; }

// the dsf_dropout of one site (model2_seq.py:104, 109, 125, 272), or p = 0 when it is off
dsf_dropout site_drop(const dsf_dropout_cfg* c, int which, uint32_t site) {
  dsf_dropout d{};
  d.p = drop_p(c, which) > 0.f ? drop_p(c, which) : 0.f;
  if (d.p > 0.f) {
    d.seed = c->seed;
    d.site = site;
    d.step = c->step;
    d.seed_dev = c->seed_dev;
  }
  return d;
}
inline const dsf_dropout* on(const dsf_dropout& d) { return d.p > 0.f ? &d : nullptr; }

// bf16 weight shadows of one block packed contiguously into a slot: the order and sizes dsf_pack_block_weights writes
void slot_views(char* base, int C, int F, dsf_block_shadows& s) {
  const size_t cc = (size_t)C * C * 2, fc = (size_t)F * C * 2;
  size_t off = 0;
  void** v[8] = {&s.wqkv, &s.wqkv_t, &s.wp, &s.wp_t, &s.w1, &s.w1_t, &s.w2, &s.w2_t};
  const size_t n[8] = {3 * cc, 3 * cc, cc, cc, fc, fc, fc, fc};
  for (int k = 0; k < 8; ++k) {
    *v[k] = base + off;
    off += A(n[k]);
  }
  s.bqkv = reinterpret_cast<float*>(base + off);
}

int make_plan(const dsf_stage_desc* d, Plan& p) {
  DSF_REQUIRE(d != nullptr, "stage: descriptor is NULL");
  if (int e = check_geom(&d->geom)) return e;
  const dsf_geom& g = d->geom;
  p.C = g.C;
  p.nh = d->n_head;
  p.L = d->n_layer;
  p.F = d->F;
  DSF_REQUIRE(p.nh > 0 && p.C % 64 == 0 && p.C <= 1024 && p.C % p.nh == 0 &&
                  (p.C / p.nh == 16 || p.C / p.nh == 32 || p.C / p.nh == 64 || p.C / p.nh == 128),
              "stage: bf16 tensor-core mode needs n_embd %% 64 == 0 (at most 1024) and head size in {16,32,64,128}; got n_embd=%d n_head=%d",
              p.C, p.nh);
  DSF_REQUIRE(p.L >= 0, "stage: n_layer=%d must not be negative", p.L);
  DSF_REQUIRE(p.L == 0 || (p.F > 0 && p.F % 64 == 0), "stage: MLP width F=%d must be a positive multiple of 64", p.F);
  DSF_REQUIRE(d->residual == 0 || d->residual == 1, "stage: residual must be 0 or 1, got %d", d->residual);
  DSF_REQUIRE(d->chain >= -1 && d->chain <= 2, "stage: chain must be -1 (default), 0, 1 or 2, got %d", d->chain);
  DSF_REQUIRE(d->prepacked == 0 || d->prepacked == 1, "stage: prepacked must be 0 or 1, got %d", d->prepacked);
  bool drop_on = false;
  for (int k = 0; k < 3; ++k) {
    const float q = drop_p(d->dropout, k);
    DSF_REQUIRE(q < 1.f, "stage: dropout p must be in [0, 1)");
    drop_on |= q > 0.f;
  }
  p.Tm = (g.V + 2) * g.S * g.A_h * g.A_w;
  p.T = p.Tm + 2;
  p.B = g.B;
  DSF_REQUIRE(p.B <= 65535 && (int64_t)p.B * p.T <= (1 << 30), "stage: B=%d x T=%d token rows is too many", p.B, p.T);
  p.M = p.B * p.T;
  // Default rule (chain = -1, as chain = 2): the row-local chain between two attention calls as one launch at the narrow stages,
  // where it is faster (DESIGN.md §2).  The chain kernel has no dropout and a fixed F = 4C.  functional._forward_bf16, the
  // training forward, applies the same rule.
  const int mode = d->chain < 0 ? 2 : d->chain;
  p.chain = ((mode >= 1 && p.C == 64) || (mode >= 2 && p.C == 128)) && p.F == 4 * p.C && p.L > 0 && !drop_on;
  p.attn_drop = drop_p(d->dropout, 1) > 0.f && p.L > 0;
  p.slots = d->prepacked ? 0 : (p.chain && p.L > 1) ? 2 : (p.L > 0 ? 1 : 0);

  const size_t M = (size_t)p.M, C = (size_t)p.C, F = (size_t)p.F;
  size_t off = 0;
  auto take = [&](size_t n) { const size_t o = off; off += A(n); return o; };
  p.x[0] = take(4 * M * C);
  p.x[1] = take(4 * M * C);
  p.h1 = take(2 * M * C);
  p.qkv = take(6 * M * C);
  p.y = take(2 * M * C);
  p.lse = take(4 * (size_t)p.B * p.nh * p.T);
  p.stats = take(8 * M);
  p.yf = take(4 * M * C);
  p.x_mid = p.h2 = p.a = p.bits = 0;
  if (!p.chain && p.L > 0) {
    p.x_mid = take(4 * M * C);
    p.h2 = take(2 * M * C);
    p.a = take(2 * M * F);
  }
  if (p.attn_drop) p.bits = take(4 * (size_t)dsf_attn_drop_words(p.B, p.T, p.nh));
  p.shadow_bytes = p.slots == 0 ? 0 : 2 * A(6 * C * C) + 2 * A(2 * C * C) + 4 * A(2 * F * C) + A(12 * C);
  p.shadow0 = off;
  off += p.slots * p.shadow_bytes;
  p.total = off;
  return DSF_OK;
}

bool aligned_all(const void* const* ptrs, int n) {
  for (int k = 0; k < n; ++k)
    if (ptrs[k] == nullptr || !aligned16(ptrs[k])) return false;
  return true;
}

}  // namespace
}  // namespace dsf

using namespace dsf;

extern "C" int dsf_stage_workspace_size(const dsf_stage_desc* d, size_t* bytes) {
  DSF_REQUIRE(bytes != nullptr, "stage_workspace_size: bytes is NULL");
  *bytes = 0;
  Plan p;
  if (int e = make_plan(d, p)) return e;
  *bytes = p.total;
  return DSF_OK;
}

#define DSF_TRY(call)                  \
  do {                                 \
    if (int e_ = (call)) return e_;    \
  } while (0)

extern "C" int dsf_stage_fwd(const dsf_stage_desc* d, const dsf_stage_params* prm, const void* img, const void* lidar, const void* radar,
                             const float* gps_emb, void* img_out, void* lidar_out, void* radar_out, float* gps_out, void* workspace,
                             size_t workspace_bytes, void* stream) {
  // ---------------------------------------------------------------- every check before the first launch
  Plan p;
  if (int e = make_plan(d, p)) return e;
  DSF_REQUIRE(prm != nullptr && prm->params != nullptr, "stage_fwd: parameter table is NULL");
  const void* io[8] = {img, lidar, radar, gps_emb, img_out, lidar_out, radar_out, gps_out};
  DSF_REQUIRE(aligned_all(io, 8), "stage_fwd: feature maps, gps_emb and the four outputs must be non-NULL and 16-byte aligned");
  const int n_params = 1 + 16 * p.L + 2;
  DSF_REQUIRE(aligned_all(reinterpret_cast<const void* const*>(prm->params), n_params),
              "stage_fwd: the %d parameter pointers must be non-NULL and 16-byte aligned", n_params);
  DSF_REQUIRE((prm->shadows != nullptr) == (d->prepacked != 0) || p.L == 0,
              "stage_fwd: shadows are %s but the descriptor says prepacked=%d", prm->shadows ? "given" : "NULL", d->prepacked);
  DSF_REQUIRE(prm->repack == 0 || prm->repack == 1, "stage_fwd: repack must be 0 or 1, got %d", prm->repack);
  if (d->prepacked && p.L > 0) {
    for (int i = 0; i < p.L; ++i) {
      const dsf_block_shadows& s = prm->shadows[i];
      const void* v[9] = {s.wqkv, s.wqkv_t, s.wp, s.wp_t, s.w1, s.w1_t, s.w2, s.w2_t, s.bqkv};
      DSF_REQUIRE(aligned_all(v, 9), "stage_fwd: the shadows of block %d must be non-NULL and 16-byte aligned", i);
    }
  }
  DSF_REQUIRE(workspace_bytes >= p.total, "stage_fwd: workspace of %zu bytes is smaller than the %zu bytes this stage needs",
              workspace_bytes, p.total);
  DSF_REQUIRE(workspace != nullptr && (reinterpret_cast<uintptr_t>(workspace) % kWsAlign) == 0,
              "stage_fwd: workspace must be non-NULL and %zu-byte aligned", kWsAlign);

  // ---------------------------------------------------------------- the launches (functional.FusionStageFn's forward, store-free)
  char* ws = static_cast<char*>(workspace);
  const float* const* P = prm->params;
  const int M = p.M, C = p.C, F = p.F, L = p.L;
  const float eps = 1e-5f;
  float* x = reinterpret_cast<float*>(ws + p.x[0]);
  float* x_alt = reinterpret_cast<float*>(ws + p.x[1]);
  void* h1 = ws + p.h1;
  void* qkv = ws + p.qkv;
  void* y = ws + p.y;
  float* lse = reinterpret_cast<float*>(ws + p.lse);
  float* mean = reinterpret_cast<float*>(ws + p.stats);
  float* rstd = mean + M;
  float* yf = reinterpret_cast<float*>(ws + p.yf);
  float* x_mid = reinterpret_cast<float*>(ws + p.x_mid);
  void* h2 = ws + p.h2;
  void* a = ws + p.a;
  uint32_t* bits = p.attn_drop ? reinterpret_cast<uint32_t*>(ws + p.bits) : nullptr;

  DSF_TRY(dsf_tokens_fwd(&d->geom, img, lidar, radar, gps_emb, P[0], x, stream));
  const dsf_dropout embd = site_drop(d->dropout, 0, 0);
  if (on(embd)) DSF_TRY(dsf_dropout_inplace(x, (int64_t)M * C, &embd, stream));

  // Shadows of block i: the caller's (re-packed first when asked), or packed into workspace slot i % slots.  With the chain
  // kernel, block i + 1 is packed while block i's shadows are still read, hence two slots.
  auto take = [&](int i, dsf_block_shadows& s) -> int {
    if (d->prepacked) {
      s = prm->shadows[i];
      if (prm->ready && prm->ready[i] && cudaStreamWaitEvent((cudaStream_t)stream, (cudaEvent_t)prm->ready[i], 0) != cudaSuccess) {
        set_error("stage_fwd: waiting for the shadows of block %d failed: %s", i, cudaGetErrorString(cudaGetLastError()));
        return DSF_ELAUNCH;
      }
      if (!prm->repack) return DSF_OK;
    } else {
      slot_views(ws + p.shadow0 + (size_t)(i % p.slots) * p.shadow_bytes, C, F, s);
    }
    const float* const* b = P + 1 + 16 * i;
    return dsf_pack_block_weights(b[6], b[4], b[8], b[10], b[12], b[14], b[7], b[5], b[9], C, F, s.wqkv, s.wqkv_t, s.wp, s.wp_t, s.w1,
                                  s.w1_t, s.w2, s.w2_t, s.bqkv, stream);
  };

  dsf_block_shadows cur{}, nxt{};
  bool have_qkv = false;  // chain: block i's qkv was written by block i - 1's chain launch
  for (int i = 0; i < L; ++i) {
    // ln1.weight, ln1.bias, ln2.weight, ln2.bias, key, query, value (weight, bias), proj, mlp.0, mlp.2 (weight, bias)
    const float* const* b = P + 1 + 16 * i;
    if (!have_qkv) {
      DSF_TRY(take(i, cur));
      DSF_TRY(dsf_layernorm_fwd(x, b[0], b[1], h1, DSF_BF16, mean, rstd, M, C, eps, stream));
      DSF_TRY(dsf_gemm_bf16_nt(h1, C, cur.wqkv, C, qkv, 3 * C, DSF_BF16, cur.bqkv, nullptr, M, 3 * C, C, DSF_EPI_BIAS, nullptr, nullptr,
                               stream));
    }
    const dsf_dropout attn = site_drop(d->dropout, 1, 1 + 3 * i);
    DSF_TRY(dsf_attn_fwd(qkv, y, lse, p.B, p.T, C, p.nh, on(attn), bits, stream));
    if (p.chain) {
      if (i + 1 < L) {
        DSF_TRY(take(i + 1, nxt));
        const float* const* bn = b + 16;
        DSF_TRY(dsf_chain_fwd(y, x, cur.wp, cur.w1, cur.w2, nxt.wqkv, b[11], b[13], b[15], nxt.bqkv, b[2], b[3], bn[0], bn[1], nullptr,
                              x_alt, nullptr, nullptr, nullptr, qkv, nullptr, nullptr, nullptr, nullptr, nullptr, M, C, eps, stream));
        cur = nxt;
        have_qkv = true;
      } else {  // the last chain launch ends with ln_f
        DSF_TRY(dsf_chain_fwd(y, x, cur.wp, cur.w1, cur.w2, nullptr, b[11], b[13], b[15], nullptr, b[2], b[3], P[n_params - 2],
                              P[n_params - 1], nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, yf, nullptr, nullptr, nullptr, nullptr,
                              M, C, eps, stream));
      }
    } else {
      const dsf_dropout proj = site_drop(d->dropout, 2, 2 + 3 * i), mlp = site_drop(d->dropout, 2, 3 + 3 * i);
      DSF_TRY(dsf_gemm_bf16_nt(y, C, cur.wp, C, x_mid, C, DSF_F32, b[11], x, M, C, C, DSF_EPI_BIAS | DSF_EPI_RESIDUAL, on(proj), nullptr,
                               stream));
      DSF_TRY(dsf_layernorm_fwd(x_mid, b[2], b[3], h2, DSF_BF16, mean, rstd, M, C, eps, stream));
      DSF_TRY(dsf_gemm_bf16_nt(h2, C, cur.w1, C, a, F, DSF_BF16, b[13], nullptr, M, F, C, DSF_EPI_BIAS | DSF_EPI_RELU, nullptr, nullptr,
                               stream));
      DSF_TRY(dsf_gemm_bf16_nt(a, F, cur.w2, F, x_alt, C, DSF_F32, b[15], x_mid, M, C, F, DSF_EPI_BIAS | DSF_EPI_RESIDUAL, on(mlp), nullptr,
                               stream));
    }
    std::swap(x, x_alt);
  }
  if (!p.chain) DSF_TRY(dsf_layernorm_fwd(x, P[n_params - 2], P[n_params - 1], yf, DSF_F32, mean, rstd, M, C, eps, stream));

  const cudaStream_t st = (cudaStream_t)stream;
  const dsf_geom& g = d->geom;
  if (d->residual) {
    DSF_TRY(dsf_upsample_add_fwd(&g, yf, img, lidar, radar, img_out, lidar_out, radar_out, stream));
  } else {
    // out = 0 + up(tokens): the upsample-add kernels read each map element and write it back from the same thread, so the
    // zero-filled outputs can be their own residual input
    const size_t elt = g.feat_dtype == DSF_BF16 ? 2 : 4, plane = (size_t)C * g.H * g.W * elt * g.B * g.S;
    if (cudaMemsetAsync(img_out, 0, plane * g.V, st) != cudaSuccess || cudaMemsetAsync(lidar_out, 0, plane, st) != cudaSuccess ||
        cudaMemsetAsync(radar_out, 0, plane, st) != cudaSuccess) {
      set_error("stage_fwd: zero-filling the outputs failed: %s", cudaGetErrorString(cudaGetLastError()));
      return DSF_ELAUNCH;
    }
    DSF_TRY(dsf_upsample_add_fwd(&g, yf, img_out, lidar_out, radar_out, img_out, lidar_out, radar_out, stream));
  }
  // the two GPS token rows of every sample: gps_out (B, 2, C) = yf[:, Tm:, :]
  if (cudaMemcpy2DAsync(gps_out, (size_t)2 * C * 4, yf + (size_t)p.Tm * C, (size_t)p.T * C * 4, (size_t)2 * C * 4, p.B,
                        cudaMemcpyDeviceToDevice, st) != cudaSuccess) {
    set_error("stage_fwd: GPS token copy failed: %s", cudaGetErrorString(cudaGetLastError()));
    return DSF_ELAUNCH;
  }
  return DSF_OK;
}

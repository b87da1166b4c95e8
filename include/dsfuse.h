/*
 * dsfuse.h — C ABI of the B200-native multimodal fusion stage (libdsfuse.so, sm_100a only).
 *
 * The reference (szy4017/DeepSense6G_TII) is 100 % Python and has no FFI of its own: the boundary it
 * exposes for this path is the Python class API of model2_seq.py (GPT :175-287, Encoder :406-597,
 * TransFuser :850-894).  The drop-in Python modules in deepsense6g_tii_b200/modules.py keep that class
 * API; underneath they call the entry points declared here through ctypes.  Each entry point names
 * the reference lines whose ATen/cuBLAS kernels it replaces.
 *
 * Conventions
 *   - Every pointer is a DEVICE pointer owned by the caller (PyTorch); the library never allocates,
 *     frees or retains device memory.  Pointers must be 16-byte aligned.
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on that stream and
 *     touches only the current device.  Calls are re-entrant.
 *   - Return value: 0 on success, a DSF_E* code otherwise.  Never throws, never exits.
 *     dsf_last_error() returns a thread-local message for the last failing call.
 *   - dtype codes: DSF_F32 = 0, DSF_BF16 = 1.  layout codes: DSF_NCHW = 0, DSF_NHWC = 1.
 *   - "tokens" are (B, T, C) row-major fp32 with T = n_slots*S*A*A + 2; the token order is the
 *     reference's: ((slot*S + t)*A + y)*A + x, slots = V image views, lidar, radar; the last two
 *     tokens are the GPS tokens (model2_seq.py:261-270).
 */
#ifndef DSFUSE_H_
#define DSFUSE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSF_VERSION 100

enum { DSF_F32 = 0, DSF_BF16 = 1 };
enum { DSF_NCHW = 0, DSF_NHWC = 1 };
enum {
  DSF_OK = 0,
  DSF_EINVAL = 1,   /* bad shape / dtype / alignment */
  DSF_ELAUNCH = 2,  /* CUDA launch or runtime error */
  DSF_EARCH = 3,    /* device is not sm_100 */
  DSF_EUNSUPPORTED = 4
};

/* GEMM epilogue flags (bit mask) */
enum {
  DSF_EPI_BIAS = 1,      /* + bias[n]                      (nn.Linear bias, model2_seq.py:83-90,122,124) */
  DSF_EPI_RELU = 2,      /* max(.,0)                       (nn.ReLU(True), :123) */
  DSF_EPI_RESIDUAL = 4,  /* + residual[m,n] (fp32)          (x + attn / x + mlp, :131-132) */
  DSF_EPI_ACCUM = 8      /* C += result: dsf_gemm_f32 only (fp32 parity path); the bf16 NT GEMM rejects it, the TN GEMM always accumulates */
};

int dsf_version(void);
const char* dsf_last_error(void);
/* Number of kernels launched through this library since load (process-wide, monotonically increasing). */
int64_t dsf_launch_count(void);
/* 0 if the current device is sm_100 and the kernels can run on it, DSF_EARCH otherwise. */
int dsf_check_device(void);
/* Programmatic dependent launch of the hot kernels (default on): each kernel's launch latency and set-up overlap
 * the tail of its predecessor in the stream; results are identical either way (process-wide; A/B timing). */
int dsf_set_pdl(int32_t on);
/* Grids of the persistent kernels (one CTA per SM, static tile schedule) are sized for (SM count - margin): a kernel
 * of another stream that occupies SMs at the same time (the NCCL all-reduce of the data-parallel step) would otherwise
 * push some CTAs into a second wave and nearly double those launches.  Even number in [0, 64]; default 0. */
int dsf_set_sm_margin(int32_t sms);

/* One nn.Dropout site (model2_seq.py:104 attn_drop, :109/:125 resid_drop, :272 embd drop).  The keep/drop decision
 * of element e is a pure function of (seed, site, step, e) (Philox4x32, 7 rounds, one call per 8 elements), so forward
 * and backward kernels agree without storing masks.  p is quantised to t/65536 (t/256 for the attention
 * probabilities); kept elements are scaled by 65536/(65536-t).  NULL or p == 0 disables dropout.               */
typedef struct {
  float p;        /* drop probability in [0, 1) */
  uint64_t seed;  /* per-run seed */
  uint32_t site;  /* which dropout layer (unique per site within a step) */
  uint32_t step;  /* training-step / call counter */
  const uint64_t* seed_dev; /* nullable DEVICE pointer: when set, the kernels use seed ^ *seed_dev.  Lets a CUDA-graph-
                             * captured step draw fresh masks at every replay (the caller bumps the word on the device) */
} dsf_dropout;

/* x[e] *= mask(e)/(1-p), e in [0, n), n a multiple of 8: embedding dropout on the token tensor (:272) and its backward. */
int dsf_dropout_inplace(float* x, int64_t n, const dsf_dropout* d, void* stream);

/* Geometry shared by the token kernels. */
typedef struct {
  int32_t B;        /* samples */
  int32_t S;        /* seq_len (frames per modality slot) */
  int32_t V;        /* camera views (config.n_views) */
  int32_t A_h, A_w; /* vert_anchors, horz_anchors */
  int32_t C;        /* n_embd */
  int32_t H, W;     /* feature-map size; H % A_h == 0 and W % A_w == 0 */
  int32_t feat_dtype; /* DSF_F32 / DSF_BF16: dtype of the feature maps */
  int32_t layout;     /* DSF_NCHW / DSF_NHWC: physical layout of the feature maps */
} dsf_geom;

/* K1 forward. Replaces nn.AdaptiveAvgPool2d x3 (model2_seq.py:515-517, 533-535, 552-554, 571-573) +
 * view/cat/permute/contiguous/cat(gps) + pos_emb add (model2_seq.py:256-272).
 *   img   (B*V*S, C, H, W), lidar/radar (B*S, C, H, W)  [feat_dtype, layout]
 *   gps   (B, 2, C) fp32, pos_emb (T, C) fp32  ->  x (B, T, C) fp32                                */
int dsf_tokens_fwd(const dsf_geom* g, const void* img, const void* lidar, const void* radar,
                   const float* gps, const float* pos_emb, float* x, void* stream);

/* K1 backward (autograd of the above, train2_seq.py:127).
 *   dx (B,T,C) fp32 -> dimg/dlidar/dradar = [dres_* +] pool-broadcast(dx)/(kh*kw)  [feat_dtype]
 *                      dgps (B,2,C) fp32, dpos_emb (T,C) fp32 (= sum_b dx, overwritten)
 * dres_* may be NULL; when given it is the gradient that reaches the same feature map through the
 * residual branch (feat + up, model2_seq.py:524-526) and is added in the same pass.               */
int dsf_tokens_bwd(const dsf_geom* g, const float* dx, const void* dres_img, const void* dres_lidar,
                   const void* dres_radar, void* dimg, void* dlidar, void* dradar, float* dgps,
                   float* dpos_emb, void* stream);

/* K2. nn.LayerNorm(C), eps 1e-5 (model2_seq.py:118-119,199; used :131-132,274).
 *   x (M,C) fp32 -> y (M,C) y_dtype; mean, rstd (M) fp32 saved for backward.                        */
int dsf_layernorm_fwd(const float* x, const float* gamma, const float* beta, void* y, int32_t y_dtype,
                      float* mean, float* rstd, int32_t M, int32_t C, float eps, void* stream);
/*   dy (M,C) dy_dtype; dx_out = (dx_add ? dx_add : 0) + LN'(dy); dgamma/dbeta (C) fp32 are
 *   ACCUMULATED into (caller zeroes or passes .grad).  Optional same-pass by-products of dx_out
 *   (the residual-stream gradient): dx_bf16 (M,C) bf16 copy (next GEMM operand) and dx_colsum (C)
 *   fp32 += column sums (= bias gradient of the preceding proj / mlp.2 Linear); either may be NULL. */
/*   `byprod_drop` (nullable): the dropout site of that preceding Linear; its mask (element m*C + c) is applied
 *   to the two by-products only (they are the gradient of the Linear's pre-dropout output), never to dx_out. */
int dsf_layernorm_bwd(const void* dy, int32_t dy_dtype, const float* x, const float* gamma,
                      const float* mean, const float* rstd, const float* dx_add, float* dx_out,
                      float* dgamma, float* dbeta, void* dx_bf16, float* dx_colsum,
                      const dsf_dropout* byprod_drop, int32_t M, int32_t C, void* stream);

/* K3/K5/K6 (bf16 tensor-core path, tcgen05 + TMEM + TMA).  Replaces nn.Linear (model2_seq.py:83-90,
 * 97-99,109,122,124) and its autograd.
 *   NT:  C[M,N] = A[M,K] . B[N,K]^T  (+bias)(relu)(+residual)      A, B bf16 row-major (K contiguous)
 *        C is c_dtype (bf16 or fp32) with leading dimension ldc; residual is fp32 with ldc.
 *   TN:  C[N',K'] += A[M,N']^T . B[M,K']   (weight gradient; contraction over the M rows);  colsum_a (N') fp32, nullable:
 *        colsum_a[n'] += sum_m A[m,n'] in the same launch (the bias gradient of that Linear: one extra 128 x 16 MMA per k-step
 *        against a shared-memory tile of ones)
 *        A, B bf16 row-major; C fp32.  The contraction is split over CTAs and the partial products are ADDED to C with
 *        fp32 vector reductions: C must be zero-filled (or hold a running sum) before the call.   */
/*        `drop` (nullable): dropout applied after bias/ReLU and BEFORE the residual add, element index m*N + n
 *        (resid_drop of the proj / mlp.2 outputs, model2_seq.py:109,125).                              */
/*        `relu_src` (nullable): bf16 (M,N) with leading dimension ldc; the result is zeroed where relu_src <= 0
 *        (backward of nn.ReLU(True), model2_seq.py:123, fused into the mlp.2 data-gradient GEMM).            */
int dsf_gemm_bf16_nt(const void* A, int32_t lda, const void* B, int32_t ldb, void* C, int32_t ldc,
                     int32_t c_dtype, const float* bias, const float* residual, int32_t M, int32_t N,
                     int32_t K, int32_t epi_flags, const dsf_dropout* drop, const void* relu_src,
                     void* stream);
int dsf_gemm_bf16_tn(const void* A, int32_t lda, const void* B, int32_t ldb, float* C, int32_t ldc,
                     int32_t M, int32_t Nout, int32_t Kout, float* colsum_a, void* stream);
/* Selects the NT tile schedule (process-wide, atomic; tests and A/B timing): 0 = default (CTA pairs, tcgen05.mma.cta_group::2 on
 * 256 x 256 / 256 x 128 tiles where N % 128 == 0 and M > 128, single-CTA persistent tiles otherwise), 2 = single-CTA tiles only. */
int dsf_gemm_set_impl(int32_t impl);

/* fp32 parity path: generic strided, two-level batched SIMT GEMM (FFMA).
 *   C[b1,b2][m,n] = alpha * sum_k A[b1,b2][m,k] * B[b1,b2][n,k]  (+bias)(relu)(+residual)(+C)      */
typedef struct {
  int32_t M, N, K;
  int32_t nb1, nb2;                  /* batch extents (1,1 for a plain GEMM) */
  int64_t a_b1, a_b2, a_m, a_k;      /* element strides */
  int64_t b_b1, b_b2, b_n, b_k;
  int64_t c_b1, c_b2, c_m, c_n;
  float alpha;
  int32_t epi_flags;
} dsf_gemm_f32_desc;
int dsf_gemm_f32(const dsf_gemm_f32_desc* d, const float* A, const float* B, float* C,
                 const float* bias, const float* residual, void* stream);

/* Column sums: out[n] (+)= sum_m X[m,n]  (bias gradients).  X dtype x_dtype, out fp32 accumulated. */
int dsf_colsum(const void* X, int32_t x_dtype, int32_t ldx, float* out, int32_t M, int32_t N,
               void* stream);
/* dst = relu-mask: dy * (h > 0), elementwise in place on dy (bf16 or fp32), n elements.           */
int dsf_relu_bwd(void* dy, const void* h, int32_t dtype, int64_t n, void* stream);
/* bf16 (M,N): dy <- dy * (h > 0) in place and out[n] += sum_m dy[m,n] (mlp.0 bias gradient), one pass. */
int dsf_relu_bwd_colsum(void* dy, const void* h, float* out, int32_t M, int32_t N, void* stream);

/* Per transformer block: fp32 master weights (nn.Linear layout [out, in]; model2_seq.py:83-90,122,124)
 * -> bf16 shadows for the tensor-core GEMMs, plain and transposed, query/key/value fused:
 *   wqkv (3C,C) = [query; key; value], wqkv_t (C,3C), wp_b/wp_t (C,C), w1_b (F,C), w1_t (C,F),
 *   w2_b (C,F), w2_t (F,C), bqkv (3C) fp32 = [bq | bk | bv].  F = block_exp * C.  One launch.     */
int dsf_pack_block_weights(const float* wq, const float* wk, const float* wv, const float* wp, const float* w1,
                           const float* w2, const float* bq, const float* bk, const float* bv, int32_t C,
                           int32_t F, void* wqkv, void* wqkv_t, void* wp_b, void* wp_t, void* w1_b, void* w1_t,
                           void* w2_b, void* w2_t, float* bqkv, void* stream);

/* fp32 parity path softmax over the last dim of (rows, T), in place (model2_seq.py:103) and its
 * backward dS = P * (dP - sum(dP*P)), in place on dP.                                             */
int dsf_softmax_fwd(float* s, int64_t rows, int32_t T, void* stream);
int dsf_softmax_bwd(float* dp, const float* p, int64_t rows, int32_t T, void* stream);

/* K4 (bf16 tensor-core path): fused flash-style attention, no mask (model2_seq.py:102-106).
 *   qkv (B, T, 3C) bf16 = [q | k | v] per token, head h at columns h*hs within each third
 *   -> y (B, T, C) bf16 (heads re-assembled side by side), lse (B, nh, T) fp32 (natural log units
 *   of the scaled scores).  hs = C/nh in {16, 32, 64, 128}.                                        */
/*   attn_drop (model2_seq.py:104; `drop` nullable): dropout on the normalised probabilities.  p is
 *   quantised to k/256 (one Philox call decides 16 keys); the forward writes the keep bits of every
 *   (b, h, query) row into drop_bits (dsf_attn_drop_words(B,T,nh) uint32 words, bit j%32 of word
 *   j/32 = key j kept) and the backward reads them back.                                           */
int64_t dsf_attn_drop_words(int32_t B, int32_t T, int32_t nh);
int dsf_attn_fwd(const void* qkv, void* y, float* lse, int32_t B, int32_t T, int32_t C, int32_t nh,
                 const dsf_dropout* drop, uint32_t* drop_bits, void* stream);
/*   dy (B,T,C) bf16 -> dqkv (B,T,3C) bf16.  delta (B,nh,T) fp32 is scratch (rowsum(dy*y)).         */
int dsf_attn_bwd(const void* qkv, const void* y, const void* dy, const float* lse, float* delta,
                 void* dqkv, int32_t B, int32_t T, int32_t C, int32_t nh, const dsf_dropout* drop,
                 const uint32_t* drop_bits, void* stream);
/*   The backward is three launches: 1 = delta (rowsum(dy*y)), 2 = dK/dV kernel, 4 = dQ kernel; 2 and 4 only need 1 and
 *   are independent of each other, so a caller may issue them on two streams (`parts` = bit mask of what to launch). */
int dsf_attn_bwd_parts(const void* qkv, const void* y, const void* dy, const float* lse, float* delta,
                       void* dqkv, int32_t B, int32_t T, int32_t C, int32_t nh, const dsf_dropout* drop,
                       const uint32_t* drop_bits, int32_t parts, void* stream);

/* K7 forward.  Replaces slice/view/permute/contiguous (model2_seq.py:275-286) + F.interpolate
 * (bilinear, align_corners=False; :521-523, 539-541, 558-560) + residual add (:524-526 ...).
 *   y (B,T,C) fp32 (ln_f output), feat_* in -> out_* = feat_* + up(untokenise(y))   [feat_dtype]   */
int dsf_upsample_add_fwd(const dsf_geom* g, const float* y, const void* img, const void* lidar,
                         const void* radar, void* out_img, void* out_lidar, void* out_radar,
                         void* stream);
/* K7 backward: dout_* (N,C,H,W) -> dy (B,T,C) fp32 for the n_slots*S*A*A map tokens; the two GPS
 * rows are copied from dgps_out (B,2,C) (zero when NULL).                                          */
int dsf_upsample_add_bwd(const dsf_geom* g, const void* dout_img, const void* dout_lidar,
                         const void* dout_radar, const float* dgps_out, float* dy, void* stream);

/* Input stem of one trunk (SURVEY.md §8 (f) item 2).  Replaces, in ONE pass over the frames: normalize_imagenet
 * (model2_seq.py:36-45, applied at :481-482), torch.stack(frames, dim=1).view(B*n_frames, C_in, H, W) (:491-493) and the
 * dtype / layout change conv1 wants under autocast with channels_last weights.
 *   frames   HOST array of n_frames (<= 16) DEVICE pointers, each a contiguous fp32 (B, C_in, H, W) tensor, C_in in 1..3
 *   scale, shift   HOST arrays of C_in floats (NULL = 1 / 0): out = x * scale[c] + shift[c]
 *                  (ImageNet: scale = 1 / (255 std), shift = -mean / std)
 *   out      (B*n_frames, C_in, H, W) in out_dtype (DSF_F32 / DSF_BF16); out_layout DSF_NCHW = contiguous, DSF_NHWC =
 *            channels_last storage; stacked frame index = b * n_frames + t                                                */
int dsf_stem_pack(const void* const* frames, int32_t n_frames, int32_t B, int32_t C_in, int32_t H, int32_t W,
                  const float* scale, const float* shift, void* out, int32_t out_dtype, int32_t out_layout, void* stream);

/* Pooled tail of Encoder.forward (model2_seq.py:581-595): AdaptiveAvgPool2d((1,1)) of the three stage-4 maps + flatten + view +
 * cat with the GPS tokens + sum over the rows, and its autograd (train2_seq.py:127).
 *   img (B*frames_img, C, H, W), lidar (B*frames_lidar, ...), radar (B*frames_radar, ...)  [feat_dtype, layout]
 *   gps (B, 2, C) fp32  ->  fused[b, c] = sum_maps sum_frames mean_px f[(b, t), c, :, :] + gps[b, 0, c] + gps[b, 1, c]   (B, C) fp32
 *   backward: d f[(b, t), c, y, x] = dfused[b, c] / (H*W)  [feat_dtype, layout],  dgps[b, j, c] = dfused[b, c]              */
int dsf_tail_fwd(const void* img, const void* lidar, const void* radar, const float* gps, float* fused, int32_t B,
                 int32_t frames_img, int32_t frames_lidar, int32_t frames_radar, int32_t C, int32_t H, int32_t W,
                 int32_t feat_dtype, int32_t layout, void* stream);
int dsf_tail_bwd(const float* dfused, void* dimg, void* dlidar, void* dradar, float* dgps, int32_t B, int32_t frames_img,
                 int32_t frames_lidar, int32_t frames_radar, int32_t C, int32_t H, int32_t W, int32_t feat_dtype,
                 int32_t layout, void* stream);

/* Narrow stages (n_embd = 64 or 128): the row-local chain between two attention calls as ONE launch —
 *   x_mid = x_in + y Wp^T + bp                      proj + residual                (model2_seq.py:109, 131)
 *   h2 = LayerNorm(x_mid; ln2), a = ReLU(h2 W1^T + b1), x_out = x_mid + a W2^T + b2   (:119, 121-126, 132)
 *   then either (wqkv_next != NULL)  h_next = LayerNorm(x_out; ln1 of the next block), qkv_next = h_next Wqkv^T + bqkv  (:118, 97-99)
 *   or     (last block)              yf = LayerNorm(x_out; ln_f) in fp32                                                (:274)
 * y (M,C) bf16; x_in, x_mid, x_out, yf (M,C) fp32; wp (C,C), w1 (4C,C), w2 (C,4C), wqkv_next (3C,C) bf16 weight shadows as packed
 * by dsf_pack_block_weights; h2, h_next (M,C), a (M,4C), qkv_next (M,3C) bf16 and the four statistics vectors (M) are the
 * tensors the backward reads.  No dropout on this path (the caller keeps the separate kernels when p > 0).
 * Store-free variant (inference, no backward follows): x_mid, h2, a, mean2, rstd2, mean_next, rstd_next and, when wqkv_next is
 * given, h_next are one group: all non-NULL runs the kernel above, all NULL a kernel that computes the same values by the same
 * expressions (x_out, qkv_next and yf come out bit-identical) but writes only x_out and qkv_next, or only yf after the last block,
 * where x_out may then be NULL too.  Any other mix is an error. */
int dsf_chain_fwd(const void* y, const float* x_in, const void* wp, const void* w1, const void* w2, const void* wqkv_next,
                  const float* bp, const float* b1, const float* b2, const float* bqkv_next, const float* ln2_g,
                  const float* ln2_b, const float* lnn_g, const float* lnn_b, float* x_mid, float* x_out, void* h2, void* a,
                  void* h_next, void* qkv_next, float* yf, float* mean2, float* rstd2, float* mean_next, float* rstd_next,
                  int32_t M, int32_t C, float eps, void* stream);

/* Optimizer step as one multi-tensor launch: torch.optim.AdamW.step() (train2_seq.py:131, 539: decoupled weight decay,
 * bias-corrected moments, eps added to sqrt(v / bc2)) + EMA.update() (train2_seq.py:133-134, 315-320: shadow = decay * shadow +
 * (1 - decay) * param, taken AFTER the parameter update) + the fp32 -> bf16 repack of GPT weights (what
 * dsf_pack_block_weights does at the start of a forward), in a single pass over the parameters.
 * One dsf_opt_tensor per parameter tensor (a dense blob of rows * cols fp32 elements; all pointers DEVICE pointers):
 *   p, g, m, v : parameter (updated in place), gradient, AdamW first / second moment (updated in place)
 *   ema        : nullable EMA shadow (updated in place)
 *   shadow     : nullable bf16 copy of the updated parameter: element (r, c) at shadow[(row_off + r) * cols + c]
 *   shadow_t   : nullable transposed bf16 copy: element (r, c) at shadow_t[c * ld_t + row_off + r]; needs rows, cols % 32 == 0
 *   copy_f32   : nullable fp32 copy of the updated parameter (q/k/v biases concatenated into one [3C] vector)
 * `tensors_dev` (n_tensors entries) and `tile0_dev` (first CTA of each tensor: prefix sums of dsf_opt_tiles(rows, cols,
 * shadow_t != NULL), n_tiles in total) live in device memory, so one launch covers any number of tensors.
 * `step_dev`: device int64 holding the 1-based step count t (the caller increments it on the device, which keeps the call
 * CUDA-graph capturable); gradients are multiplied by `grad_scale` first (1 = as they are).  Hyper-parameters are doubles, as
 * torch holds them: 1 - beta and 1 - decay are formed in double before rounding to fp32, like torch's own kernels do.  */
typedef struct {
  float* p;
  const float* g;
  float* m;
  float* v;
  float* ema;
  void* shadow;
  void* shadow_t;
  float* copy_f32;
  int32_t rows, cols, row_off, ld_t;
  float weight_decay;
  int32_t reserved;
} dsf_opt_tensor;
int32_t dsf_opt_tiles(int32_t rows, int32_t cols, int32_t transposed_shadow);
/* Copies the tensor table from PINNED host memory (cudaHostAlloc / torch pin_memory: device-accessible under unified addressing)
 * into device memory with a kernel instead of a copy-engine transfer; nbytes a multiple of 16.  Graph-capturable: a replay
 * re-reads the host table. */
int dsf_opt_upload_table(void* dst_dev, const void* src_pinned_host, int64_t nbytes, void* stream);
int dsf_adamw_ema_pack(const dsf_opt_tensor* tensors_dev, const int32_t* tile0_dev, int32_t n_tensors, int32_t n_tiles, double lr,
                       double beta1, double beta2, double eps, double ema_decay, const int64_t* step_dev, double grad_scale,
                       void* stream);

/* fp32 -> bf16 conversion (weight shadow refresh), n elements. */
int dsf_cast_f32_bf16(const float* src, void* dst, int64_t n, void* stream);

/* ---------------------------------------------------------------- whole fusion stage, inference forward (bf16 mode)
 * One GPT fusion stage without a backward to follow (model2_seq.py:515-526: pool -> GPT -> upsample + residual), in one call:
 * the token kernel, the embedding dropout, per block LayerNorm / fused QKV GEMM / flash attention and either the chain kernel
 * (store-free variant) or proj / ln2 / fc1 / fc2, then ln_f unless the chain ended with it, the upsample-add and the copy of the
 * two GPS token rows.  Each of those is one of the entry points above, launched on `stream` in that order; the call launches
 * nothing else (dsf_launch_count advances by exactly their launches), allocates nothing and never synchronises, so it can be
 * captured into a CUDA graph.  Compute mode is bf16 (tensor-core GEMMs and attention, fp32 residual stream). */

/* nn.Dropout probabilities of one GPT in train() mode (model2_seq.py:104, 109/125, 272).  Site ids: 0 = embedding, and per block
 * i 1 + 3i = attention, 2 + 3i = proj output, 3 + 3i = mlp output; see dsf_dropout for seed / step / seed_dev. */
typedef struct {
  float embd, attn, resid;    /* drop probabilities in [0, 1); 0 disables a site */
  uint64_t seed;
  uint32_t step;
  const uint64_t* seed_dev;   /* nullable DEVICE pointer */
} dsf_dropout_cfg;

typedef struct {
  dsf_geom geom;      /* maps and tokens; geom.C = n_embd */
  int32_t n_head;     /* head size C / n_head in {16, 32, 64, 128}; C % 64 == 0 */
  int32_t n_layer;    /* >= 0 */
  int32_t F;          /* MLP width (block_exp * C), a multiple of 64 */
  int32_t residual;   /* 1: out = feat + up(tokens) (Encoder); 0: out = up(tokens) (GPT.forward) */
  int32_t chain;      /* -1: default rule (chain kernel at C = 64 and 128); 0 never, 1 C = 64, 2 C = 64 and 128 (as DSF_CHAIN).
                       * It runs only when also F == 4C, n_layer > 0 and dropout is off. */
  int32_t prepacked;  /* 1: dsf_stage_params.shadows will be given (the workspace then has no room for shadows), 0: it is NULL */
  const dsf_dropout_cfg* dropout;  /* HOST pointer, nullable: NULL (or every p == 0) = no dropout */
} dsf_stage_desc;

/* bf16 weight shadows of one block, as dsf_pack_block_weights writes them (DEVICE pointers, 16-byte aligned). */
typedef struct {
  void *wqkv, *wqkv_t, *wp, *wp_t, *w1, *w1_t, *w2, *w2_t;
  float* bqkv;
} dsf_block_shadows;

typedef struct {
  /* HOST array of 1 + 16 * n_layer + 2 DEVICE pointers to the fp32 parameters in the reference's state-dict order: pos_emb (T, C),
   * per block ln1.weight, ln1.bias, ln2.weight, ln2.bias, attn.{key, query, value}.{weight, bias}, attn.proj.{weight, bias},
   * mlp.0.{weight, bias}, mlp.2.{weight, bias}, then ln_f.weight, ln_f.bias. */
  const float* const* params;
  /* HOST array of n_layer pre-packed shadows, or NULL: each block is then packed into the workspace from params (one
   * dsf_pack_block_weights launch per block).  Given: repack = 1 re-packs each block into them first (one launch per block),
   * repack = 0 uses them as they are. */
  const dsf_block_shadows* shadows;
  /* HOST array of n_layer cudaEvent_t (passed as void*), or NULL; entries may be NULL.  With pre-packed shadows, the call makes
   * `stream` wait for ready[i] just before the first launch that reads block i's shadows, so shadows still being packed on
   * another stream overlap the blocks before i (under CUDA-graph capture, events recorded in the same capture). */
  void* const* ready;
  int32_t repack;
} dsf_stage_params;

/* Workspace bytes dsf_stage_fwd needs for `d`.  With A(n) = n rounded up to a multiple of 256, M = B * T, T = (V + 2) * S * A_h * A_w + 2:
 *     2 A(4MC)                          x (fp32 residual stream, ping-pong)
 *   + A(2MC) + A(6MC) + A(2MC)          h1, qkv, y (bf16)
 *   + A(4 B n_head T) + A(8M)           attention log-sum-exp, LayerNorm mean / rstd (fp32)
 *   + A(4MC)                            yf (ln_f output, fp32)
 *   + [no chain, n_layer > 0]  A(4MC) + A(2MC) + A(2MF)                x_mid (fp32), h2, a (bf16)
 *   + [attention dropout]  A(4 dsf_attn_drop_words(B, T, n_head))     keep bits
 *   + [prepacked == 0]  s (2 A(6C^2) + 2 A(2C^2) + 4 A(2FC) + A(12C))   bf16 shadows + fused QKV bias
 *                       with s = 2 shadow slots if the chain runs and n_layer > 1, else min(n_layer, 1)
 * Returns DSF_EINVAL (and *bytes = 0) for a descriptor dsf_stage_fwd would reject. */
int dsf_stage_workspace_size(const dsf_stage_desc* d, size_t* bytes);

/* img (B*V*S, C, H, W), lidar / radar (B*S, C, H, W) [geom.feat_dtype, geom.layout]; gps_emb (B, 2, C) fp32
 *   -> img_out / lidar_out / radar_out, same shapes, dtype and layout as the maps, gps_out (B, 2, C) fp32.
 * workspace: DEVICE memory of at least dsf_stage_workspace_size(d) bytes, 256-byte aligned, owned by the caller; it may be reused
 * by the next call on the same stream.  Every pointer is checked (NULL, 16-byte alignment, workspace size and alignment) before
 * anything is enqueued.  The outputs must not alias the inputs or the workspace. */
int dsf_stage_fwd(const dsf_stage_desc* d, const dsf_stage_params* p, const void* img, const void* lidar, const void* radar,
                  const float* gps_emb, void* img_out, void* lidar_out, void* radar_out, float* gps_out, void* workspace,
                  size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DSFUSE_H_ */

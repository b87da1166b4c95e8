"""Autograd wiring of one GPT fusion stage onto the dsfuse C ABI.

``fusion_stage(...)`` computes, for one ResNet stage, exactly what ``Encoder.forward`` does at
model2_seq.py:515-526 (and :533-544, :552-563, :571-579):

    pooled_m = AdaptiveAvgPool2d((A, A))(feat_m)                      m in {image, lidar, radar}
    tok_m, gps_out = GPT(pooled_image, pooled_lidar, pooled_radar, gps_emb)
    feat_m' = feat_m + bilinear_upsample(tok_m)

as ONE ``torch.autograd.Function`` whose forward and backward are sequences of hand-written CUDA
kernels (no ATen math on the path).  Two compute modes:

  * ``torch.bfloat16`` (performance mode): tcgen05/TMEM GEMMs + flash attention, fp32 residual
    stream and LayerNorm statistics, bf16 activations / weight shadows.  Needs C % 64 == 0 and
    head size in {16, 32, 64, 128}.
  * ``torch.float32`` (parity mode, <= 1e-3 of the reference): FFMA GEMMs and materialised
    softmax attention, everything fp32.

Dropout (model2_seq.py:104,109,125,272; bf16 mode only): ``cfg["dropout"] = dict(embd=p, attn=p, resid=p,
seed=int, step=int[, seed_dev=int64 device tensor][, capture=dict])``; with ``seed_dev`` the kernels use
``seed ^ seed_dev[0]`` read on the device, so a CUDA-graph replay draws new masks whenever that word was bumped.  Masks are counter-based (Philox4x32, 7 rounds, of (seed, site, step, element)),
recomputed by the backward kernels; sites are numbered ``drop_site(...)``.  torch's own RNG stream cannot be
reproduced bit for bit, so parity with dropout is tested by feeding the oracle the masks the kernels drew
(``capture`` receives the attention keep-bitmaps; the elementwise masks are regenerated with
``dsf_dropout_inplace`` on a tensor of ones).
"""
import math
import os

import torch
from torch.autograd.function import once_differentiable

from . import _capi as K
from ._capi import EPI_ACCUM, EPI_BIAS, EPI_RELU, EPI_RESIDUAL, GemmF32Desc

PER_BLOCK = ("ln1.weight", "ln1.bias", "ln2.weight", "ln2.bias",
             "attn.key.weight", "attn.key.bias", "attn.query.weight", "attn.query.bias",
             "attn.value.weight", "attn.value.bias", "attn.proj.weight", "attn.proj.bias",
             "mlp.0.weight", "mlp.0.bias", "mlp.2.weight", "mlp.2.bias")


def param_names(n_layer):
    """Flat parameter order used by ``FusionStageFn`` (names are the reference state-dict names)."""
    names = ["pos_emb"]
    for i in range(n_layer):
        names += ["blocks.%d.%s" % (i, n) for n in PER_BLOCK]
    return names + ["ln_f.weight", "ln_f.bias"]


def _f32_linear_desc(M, N, Kd, flags, trans=None):
    """Descriptors for y = x W^T (+...), x (M,K) row-major, W (N,K) row-major, fp32 SIMT path."""
    return GemmF32Desc(M, N, Kd, 1, 1, 0, 0, Kd, 1, 0, 0, Kd, 1, 0, 0, N, 1, 1.0, flags)


class _Ctx:
    pass


_SIDE_STREAMS = {}


def _side_stream(device, which=0):
    """Extra streams per device: 0 carries the weight-gradient GEMMs / bias sums of the backward and the weight packs of
    the forward, 1 the dQ attention kernel (see ``_backward_bf16``)."""
    key = (device.type, device.index, which)
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device=device)
    return _SIDE_STREAMS[key]


def _chain_mode(C):
    """Whether the forward chain kernel (csrc/chain.cu) serves n_embd = C: DSF_CHAIN=0 never, 1 n_embd 64, 2 (default) 64 and 128."""
    try:
        m = int(os.environ.get("DSF_CHAIN", 2))
    except ValueError:
        m = 2
    return (m >= 1 and C == 64) or (m >= 2 and C == 128)


def _use_side_stream():
    """Whether the bf16 forward and backward put work on the side streams of ``_side_stream``.
    Default: on while the step is being captured into a CUDA graph (the fork/join events become graph edges, free at replay:
    -0.2 ms per step), off for eager launches (creating and recording ~40 events per step costs more host time than the
    overlap returns).  DSF_WGRAD_STREAM=1 / 0 forces it."""
    env = os.environ.get("DSF_WGRAD_STREAM")
    return (env == "1") if env in ("0", "1") else torch.cuda.is_current_stream_capturing()


def drop_site(kind, block=0):
    """Site id of an nn.Dropout layer inside one GPT: 'embd' (:272), per block 'attn' (:104), 'proj' (:109), 'mlp' (:125)."""
    return 0 if kind == "embd" else 1 + 3 * block + ("attn", "proj", "mlp").index(kind)


class _Runner:
    """Holds shapes + mode and implements forward / backward over raw tensors."""

    def __init__(self, B, S, V, A_h, A_w, C, H, W, n_head, n_layer, feat_dtype, compute_dtype, layout):
        self.B, self.S, self.V, self.A_h, self.A_w, self.C, self.H, self.W = B, S, V, A_h, A_w, C, H, W
        self.nh, self.L = n_head, n_layer
        self.hs = C // n_head
        self.Tm = (V + 2) * S * A_h * A_w
        self.T = self.Tm + 2
        self.M = B * self.T
        self.bf16 = compute_dtype == torch.bfloat16
        self.act = torch.bfloat16 if self.bf16 else torch.float32
        self.grad_hook = None  # optional dist.OverlappedGradReducer (bf16 path)
        self.dropout = None    # cfg["dropout"] dict (bf16 path)
        self.shadows = None    # cfg["shadows"]: persistent bf16 weight shadows owned by the GPT module (modules.GPT._shadow_cfg)
        self.capture = None    # cfg["capture"] dict: receives the mlp.0 outputs ("relu.{i}", the ReLU decisions) of every block
        if self.bf16:
            if C % 64 != 0 or self.hs not in (16, 32, 64, 128):
                raise RuntimeError("bf16 tensor-core mode needs n_embd %% 64 == 0 and head size in {16,32,64,128}; "
                                   "got n_embd=%d n_head=%d" % (C, n_head))
        self.geom = K.make_geom(B, S, V, A_h, A_w, C, H, W, K.DSF_BF16 if feat_dtype == torch.bfloat16 else K.DSF_F32, layout)

    # ------------------------------------------------------------------ linear layers
    def _linear_fwd(self, x, w, b, out_dtype, relu=False, residual=None):
        """fp32 parity mode: y = x W^T + b (ReLU) (+ residual) on the SIMT GEMM."""
        M, Kd = x.shape
        N = w.shape[0]
        out = torch.empty(M, N, device=x.device, dtype=out_dtype)
        flags = EPI_BIAS | (EPI_RELU if relu else 0) | (EPI_RESIDUAL if residual is not None else 0)
        K.gemm_f32(_f32_linear_desc(M, N, Kd, flags), x, w, out, bias=b, residual=residual)
        return out

    def _linear_bwd(self, dy, x, w):
        """fp32 parity mode: dy (M,N), x (M,K), w (N,K) -> dx (M,K), dw (N,K), db (N)."""
        M, N = dy.shape
        Kd = x.shape[1]
        dev = dy.device
        dw = torch.zeros(N, Kd, device=dev, dtype=torch.float32)
        db = torch.zeros(N, device=dev, dtype=torch.float32)
        K.colsum(dy, db)
        # dW[n,k] = sum_m dy[m,n] x[m,k]
        K.gemm_f32(GemmF32Desc(N, Kd, M, 1, 1, 0, 0, 1, N, 0, 0, 1, Kd, 0, 0, Kd, 1, 1.0, 0), dy, x, dw)
        dx = torch.empty(M, Kd, device=dev, dtype=torch.float32)
        # dx[m,k] = sum_n dy[m,n] w[n,k]
        K.gemm_f32(GemmF32Desc(M, Kd, N, 1, 1, 0, 0, N, 1, 0, 0, 1, Kd, 0, 0, Kd, 1, 1.0, 0), dy, w, dx)
        return dx, dw, db

    # ------------------------------------------------------------------ attention
    def _attn_fwd(self, qkv, st):
        B, T, C, nh, hs = self.B, self.T, self.C, self.nh, self.hs
        dev = qkv.device
        y = torch.empty(self.M, C, device=dev, dtype=self.act)
        if self.bf16:
            st.lse = torch.empty(B, nh, T, device=dev, dtype=torch.float32)
            K.attn_fwd(qkv, y, st.lse, B, T, C, nh)
            return y
        # fp32 parity mode: materialised scores (model2_seq.py:102-105)
        P = torch.empty(B, nh, T, T, device=dev, dtype=torch.float32)
        q, k, v = qkv, qkv[:, C:], qkv[:, 2 * C:]
        ld = 3 * C
        K.gemm_f32(GemmF32Desc(T, T, hs, B, nh, T * ld, hs, ld, 1, T * ld, hs, ld, 1, nh * T * T, T * T, T, 1,
                               1.0 / math.sqrt(hs), 0), q, k, P)
        K.softmax_fwd(P, B * nh * T, T)
        # y[b,t,h*hs+d] = sum_j P[b,h,t,j] v[b,j,h,d]
        K.gemm_f32(GemmF32Desc(T, hs, T, B, nh, nh * T * T, T * T, T, 1, T * ld, hs, 1, ld, T * C, hs, C, 1, 1.0, 0), P, v, y)
        st.P = P
        return y

    def _attn_bwd(self, dy, qkv, y, st):
        B, T, C, nh, hs = self.B, self.T, self.C, self.nh, self.hs
        dev = dy.device
        dqkv = torch.empty(self.M, 3 * C, device=dev, dtype=self.act)
        if self.bf16:
            delta = torch.empty(B, nh, T, device=dev, dtype=torch.float32)
            K.attn_bwd(qkv, y, dy, st.lse, delta, dqkv, B, T, C, nh)
            return dqkv
        P = st.P
        q, k, v = qkv, qkv[:, C:], qkv[:, 2 * C:]
        dq, dk, dv = dqkv, dqkv[:, C:], dqkv[:, 2 * C:]
        ld = 3 * C
        sc = 1.0 / math.sqrt(hs)
        dP = torch.empty_like(P)
        # dP[b,h,t,j] = sum_d dy[b,t,h,d] v[b,j,h,d]
        K.gemm_f32(GemmF32Desc(T, T, hs, B, nh, T * C, hs, C, 1, T * ld, hs, ld, 1, nh * T * T, T * T, T, 1, 1.0, 0), dy, v, dP)
        # dv[b,j,h,d] = sum_t P[b,h,t,j] dy[b,t,h,d]
        K.gemm_f32(GemmF32Desc(T, hs, T, B, nh, nh * T * T, T * T, 1, T, T * C, hs, 1, C, T * ld, hs, ld, 1, 1.0, 0), P, dy, dv)
        K.softmax_bwd(dP, P, B * nh * T, T)  # dP <- dS
        # dq[b,t,h,d] = sc * sum_j dS[t,j] k[j,d]
        K.gemm_f32(GemmF32Desc(T, hs, T, B, nh, nh * T * T, T * T, T, 1, T * ld, hs, 1, ld, T * ld, hs, ld, 1, sc, 0), dP, k, dq)
        # dk[b,j,h,d] = sc * sum_t dS[t,j] q[t,d]
        K.gemm_f32(GemmF32Desc(T, hs, T, B, nh, nh * T * T, T * T, 1, T, T * ld, hs, 1, ld, T * ld, hs, ld, 1, sc, 0), dP, q, dk)
        return dqkv

    # ------------------------------------------------------------------ forward
    def forward(self, feats, gps_emb, params, residual=True):
        """feats: 3 tensors (N, C, H, W) [or NHWC storage]; gps_emb (B, 2, C) fp32; params: flat list.
        residual=False returns the upsampled token maps alone (plain ``GPT.forward`` semantics)."""
        if self.bf16:
            return self._forward_bf16(feats, gps_emb, params, residual)
        dev = gps_emb.device
        M, C, L = self.M, self.C, self.L
        f32 = torch.float32
        saved = _Ctx()
        saved.layers = []
        x = torch.empty(M, C, device=dev, dtype=f32)
        K.tokens_fwd(self.geom, feats[0], feats[1], feats[2], gps_emb, params[0], x)
        saved.shadows = []
        for i in range(L):
            (ln1w, ln1b, ln2w, ln2b, kw, kb, qw, qb, vw, vb, pw, pb, w1, b1, w2, b2) = params[1 + 16 * i: 17 + 16 * i]
            st = _Ctx()
            # fused QKV weight [3C, C] in the order [query | key | value]
            wqkv = torch.cat([qw, kw, vw], dim=0)
            bqkv = torch.cat([qb, kb, vb], dim=0)
            st.wqkv = wqkv
            st.x_in = x
            st.mean1 = torch.empty(M, device=dev, dtype=f32)
            st.rstd1 = torch.empty(M, device=dev, dtype=f32)
            st.h1 = torch.empty(M, C, device=dev, dtype=f32)
            K.layernorm_fwd(x, ln1w, ln1b, st.h1, st.mean1, st.rstd1)
            st.qkv = self._linear_fwd(st.h1, wqkv, bqkv, f32)
            st.y = self._attn_fwd(st.qkv, st)
            x_mid = self._linear_fwd(st.y, pw, pb, f32, residual=x)
            st.x_mid = x_mid
            st.mean2 = torch.empty(M, device=dev, dtype=f32)
            st.rstd2 = torch.empty(M, device=dev, dtype=f32)
            st.h2 = torch.empty(M, C, device=dev, dtype=f32)
            K.layernorm_fwd(x_mid, ln2w, ln2b, st.h2, st.mean2, st.rstd2)
            st.a = self._linear_fwd(st.h2, w1, b1, f32, relu=True)
            if self.capture is not None:
                self.capture["relu.%d" % i] = st.a
            x = self._linear_fwd(st.a, w2, b2, f32, residual=x_mid)
            saved.layers.append(st)
        saved.x_last = x
        saved.mean_f = torch.empty(M, device=dev, dtype=f32)
        saved.rstd_f = torch.empty(M, device=dev, dtype=f32)
        yf = torch.empty(M, C, device=dev, dtype=f32)
        K.layernorm_fwd(x, params[-2], params[-1], yf, saved.mean_f, saved.rstd_f)
        outs = [torch.empty_like(f) for f in feats]
        K.upsample_add_fwd(self.geom, yf, feats if residual else [torch.zeros_like(f) for f in feats], outs)
        gps_out = yf.view(self.B, self.T, C)[:, self.Tm:, :].contiguous()
        return outs, gps_out, saved

    # ------------------------------------------------------------------ backward
    # ------------------------------------------------------------------ bf16 tensor-core path
    def _forward_bf16(self, feats, gps_emb, params, residual):
        """Per block: 1 weight-pack launch, LN, QKV GEMM, flash attention, proj GEMM(+residual), LN,
        fc1 GEMM(+ReLU), fc2 GEMM(+residual) = 8 launches."""
        dev = gps_emb.device
        M, C, L = self.M, self.C, self.L
        f32, bf = torch.float32, torch.bfloat16
        F = params[13].shape[0] if L > 0 else 4 * C  # mlp.0.weight rows
        saved = _Ctx()
        saved.layers = []
        # Weight shadows (fp32 -> bf16, plain + transposed, one launch per block) do not depend on the activations: under
        # graph capture they are packed on the side stream while the token kernel and the first blocks run.
        main = torch.cuda.current_stream()
        side = _side_stream(dev) if _use_side_stream() else None
        sizes = [3 * C * C, 3 * C * C, C * C, C * C, F * C, F * C, C * F, C * F]
        packed = []

        def pack(i):
            (ln1w, ln1b, ln2w, ln2b, kw, kb, qw, qb, vw, vb, pw, pb, w1, b1, w2, b2) = params[1 + 16 * i: 17 + 16 * i]
            st = _Ctx()
            if self.shadows is not None:   # persistent shadows: up to date (written by the fused optimizer step), or re-packed in place
                v = self.shadows["views"][i]
                st.wqkv, st.wqkv_t, st.wp, st.wp_t, st.w1, st.w1_t, st.w2, st.w2_t, st.bqkv = (
                    v["wqkv"], v["wqkv_t"], v["wp"], v["wp_t"], v["w1"], v["w1_t"], v["w2"], v["w2_t"], v["bqkv"])
                if not self.shadows["fresh"]:
                    K.pack_block_weights(qw, kw, vw, pw, w1, w2, qb, kb, vb,
                                         (st.wqkv, st.wqkv_t, st.wp, st.wp_t, st.w1, st.w1_t, st.w2, st.w2_t, st.bqkv))
                return st
            # one flat bf16 buffer holds the 8 weight shadows of this block (plain + transposed)
            flat = torch.empty(sum(sizes), device=dev, dtype=bf)
            views, off = [], 0
            for n in sizes:
                views.append(flat[off:off + n])
                off += n
            st.wqkv, st.wqkv_t = views[0].view(3 * C, C), views[1].view(C, 3 * C)
            st.wp, st.wp_t = views[2].view(C, C), views[3].view(C, C)
            st.w1, st.w1_t = views[4].view(F, C), views[5].view(C, F)
            st.w2, st.w2_t = views[6].view(C, F), views[7].view(F, C)
            st.bqkv = torch.empty(3 * C, device=dev, dtype=f32)
            K.pack_block_weights(qw, kw, vw, pw, w1, w2, qb, kb, vb,
                                 (st.wqkv, st.wqkv_t, st.wp, st.wp_t, st.w1, st.w1_t, st.w2, st.w2_t, st.bqkv))
            return st

        if side is not None:
            ev = torch.cuda.Event()
            ev.record(main)
            side.wait_event(ev)
            with torch.cuda.stream(side):
                for i in range(L):
                    st = pack(i)
                    st.packed_ev = torch.cuda.Event()
                    st.packed_ev.record(side)
                    packed.append(st)
        x = torch.empty(M, C, device=dev, dtype=f32)
        K.tokens_fwd(self.geom, feats[0], feats[1], feats[2], gps_emb, params[0], x)
        if self._drop("embd") is not None:
            K.dropout_inplace(x, self._drop("embd"))
        def take(i):
            if side is not None:
                st = packed[i]
                main.wait_event(st.packed_ev)
                st.packed_ev = None
                return st
            return pack(i)

        # Narrow stages (no dropout): everything between two attention calls is row-local and runs as ONE launch (csrc/chain.cu):
        # per block = flash attention + dsf_chain_fwd instead of seven launches.  Measured on B200 (batch 12, graph-replayed stage
        # step, profiles/r02f_*): n_embd 64: 13.6 us per chain launch, step 1.82 -> 1.68 ms; n_embd 128: 34 us, 2.17 -> 2.09 ms.
        # DSF_CHAIN=0: never, 1: n_embd 64 only, 2 (default): n_embd 64 and 128.
        chain = _chain_mode(C) and F == 4 * C and L > 0 and self.dropout is None
        yf = torch.empty(M, C, device=dev, dtype=f32)
        saved.mean_f = torch.empty(M, device=dev, dtype=f32)
        saved.rstd_f = torch.empty(M, device=dev, dtype=f32)
        nxt = None  # chain mode: (st, h1, qkv, mean1, rstd1) of block i, produced by block i-1's chain launch
        for i in range(L):
            (ln1w, ln1b, ln2w, ln2b, kw, kb, qw, qb, vw, vb, pw, pb, w1, b1, w2, b2) = params[1 + 16 * i: 17 + 16 * i]
            st = take(i) if nxt is None else nxt
            nxt = None
            bqkv = st.bqkv
            st.x_in = x
            if not hasattr(st, "h1"):
                stats = torch.empty(2, M, device=dev, dtype=f32)
                st.mean1, st.rstd1 = stats[0], stats[1]
                st.h1 = torch.empty(M, C, device=dev, dtype=bf)
                K.layernorm_fwd(x, ln1w, ln1b, st.h1, st.mean1, st.rstd1)
                st.qkv = torch.empty(M, 3 * C, device=dev, dtype=bf)
                K.gemm_bf16_nt(st.h1, st.wqkv, st.qkv, bias=bqkv)
            stats2 = torch.empty(2, M, device=dev, dtype=f32)
            st.mean2, st.rstd2 = stats2[0], stats2[1]
            st.y = torch.empty(M, C, device=dev, dtype=bf)
            st.lse = torch.empty(self.B, self.nh, self.T, device=dev, dtype=f32)
            st.drop_bits = None
            if self._drop("attn", i) is not None:
                st.drop_bits = torch.empty(K.attn_drop_words(self.B, self.T, self.nh), device=dev, dtype=torch.int32)
                if "capture" in self.dropout:
                    self.dropout["capture"]["attn_bits.%d" % i] = st.drop_bits
            K.attn_fwd(st.qkv, st.y, st.lse, self.B, self.T, C, self.nh, self._drop("attn", i), st.drop_bits)
            st.x_mid = torch.empty(M, C, device=dev, dtype=f32)
            st.h2 = torch.empty(M, C, device=dev, dtype=bf)
            st.a = torch.empty(M, F, device=dev, dtype=bf)
            x_new = torch.empty(M, C, device=dev, dtype=f32)
            if chain:
                if i + 1 < L:
                    sn = take(i + 1)
                    statn = torch.empty(2, M, device=dev, dtype=f32)
                    sn.mean1, sn.rstd1 = statn[0], statn[1]
                    sn.h1 = torch.empty(M, C, device=dev, dtype=bf)
                    sn.qkv = torch.empty(M, 3 * C, device=dev, dtype=bf)
                    K.chain_fwd(st.y, x, st.wp, st.w1, st.w2, sn.wqkv, pb, b1, b2, sn.bqkv, ln2w, ln2b, params[1 + 16 * (i + 1)],
                                params[2 + 16 * (i + 1)], st.x_mid, x_new, st.h2, st.a, sn.h1, sn.qkv, None, st.mean2, st.rstd2, sn.mean1, sn.rstd1)
                    nxt = sn
                else:   # last block: the chain ends with ln_f
                    K.chain_fwd(st.y, x, st.wp, st.w1, st.w2, None, pb, b1, b2, None, ln2w, ln2b, params[-2], params[-1], st.x_mid, x_new,
                                st.h2, st.a, None, None, yf, st.mean2, st.rstd2, saved.mean_f, saved.rstd_f)
            else:
                K.gemm_bf16_nt(st.y, st.wp, st.x_mid, bias=pb, residual=x, drop=self._drop("proj", i))
                K.layernorm_fwd(st.x_mid, ln2w, ln2b, st.h2, st.mean2, st.rstd2)
                K.gemm_bf16_nt(st.h2, st.w1, st.a, bias=b1, relu=True)
                K.gemm_bf16_nt(st.a, st.w2, x_new, bias=b2, residual=st.x_mid, drop=self._drop("mlp", i))
            if self.capture is not None:
                self.capture["relu.%d" % i] = st.a
            x = x_new
            saved.layers.append(st)
        saved.x_last = x
        if not chain:
            K.layernorm_fwd(x, params[-2], params[-1], yf, saved.mean_f, saved.rstd_f)
        outs = [torch.empty_like(f) for f in feats]
        K.upsample_add_fwd(self.geom, yf, feats if residual else [torch.zeros_like(f) for f in feats], outs)
        gps_out = yf.view(self.B, self.T, C)[:, self.Tm:, :].contiguous()
        if self.shadows is not None and not self.shadows["fresh"]:
            self.shadows["owner"].mark_shadows_fresh()
        return outs, gps_out, saved

    def _drop(self, kind, block=0):
        """``_capi.Dropout`` of one site, or None when that probability is 0 / dropout is off."""
        d = self.dropout
        if d is None:
            return None
        p = float(d.get("resid" if kind in ("proj", "mlp") else kind, 0.0))
        if p <= 0.0:
            return None
        sd = d.get("seed_dev")  # int64 device tensor (1 element) or None
        return K.Dropout(p, int(d["seed"]), drop_site(kind, block), int(d.get("step", 0)), None if sd is None else sd.data_ptr())

    def _backward_bf16(self, saved, params, douts, dgps_out, residual):
        """Per block: 4 wgrad + 4 dgrad GEMMs, fused ReLU-mask+bias-grad, 2 LayerNorm backward kernels that also
        emit the bf16 operand copy and the bias gradient of the preceding Linear, flash-attention backward,
        one column-sum for the QKV bias; all gradients of a block live in one zero-filled flat buffer."""
        dev = douts[0].device
        M, C, L = self.M, self.C, self.L
        f32, bf = torch.float32, torch.bfloat16
        grads = [None] * len(params)
        dyf = torch.empty(M, C, device=dev, dtype=f32)
        K.upsample_add_bwd(self.geom, douts, dgps_out, dyf)
        F = params[13].shape[0] if L > 0 else 4 * C
        # flat zero-filled gradient buffer per block: [dWqkv | dWp | dW1 | dW2 | dbqkv | dbp | db1 | db2 | dg1 | db1ln | dg2 | db2ln]
        sizes = [3 * C * C, C * C, F * C, C * F, 3 * C, C, F, C, C, C, C, C]
        per_block = sum(sizes)
        gbuf = torch.zeros(L * per_block + 2 * C + self.T * C, device=dev, dtype=f32)   # blocks | ln_f | pos_emb

        def block_views(i):
            out, off = [], i * per_block
            for n in sizes:
                out.append(gbuf[off:off + n])
                off += n
            return out

        def bucket(i):
            """All-reduce bucket of block i; the last block's bucket carries the ln_f gradients that follow it in the buffer (they
            are final before any block's backward has started, so they must not wait for the tail of the backward)."""
            return gbuf[i * per_block:(i + 1) * per_block + (2 * C if i == L - 1 else 0)]

        # The four weight-gradient GEMMs of a block only feed the optimizer, so they run on a second stream next to the
        # data-gradient chain: their CTAs fill the SMs that chain leaves idle (second, partly filled rounds of the
        # N = n_embd GEMMs and of the attention kernels, tails of the short HBM-bound kernels).  fork() orders a wgrad
        # after everything enqueued so far on the main stream; join() makes the main stream wait for the side stream
        # (before buffers the wgrads read are overwritten or released, and before the block's gradients are handed on).
        use_side = _use_side_stream()
        main = torch.cuda.current_stream()
        side = _side_stream(dev) if use_side else None
        side_q = _side_stream(dev, 1) if use_side else None

        def fork(fn, stream=None):
            stream = stream or side
            if stream is None:
                fn()
                return
            ev = torch.cuda.Event()
            ev.record(main)
            stream.wait_event(ev)
            with torch.cuda.stream(stream):
                fn()

        def join(stream=None):
            stream = stream or side
            if stream is not None:
                ev = torch.cuda.Event()
                ev.record(stream)
                main.wait_event(ev)

        # The weight-gradient work of block i is only joined one block later (before anything it reads can be overwritten
        # or released): the side stream gets a whole block of slack instead of having to finish inside its own block.
        pending = None  # (event recorded on the side stream after block i's last fork, block index, references kept alive)

        def join_pending():
            nonlocal pending
            if pending is not None:
                ev, blk, _keep = pending
                main.wait_event(ev)
                pending = None
                if self.grad_hook is not None:  # data parallel: average this block's bucket while the other blocks compute
                    self.grad_hook.block_ready(blk, bucket(blk))

        dgf, dbf = gbuf[L * per_block:L * per_block + C], gbuf[L * per_block + C:L * per_block + 2 * C]
        # The fc1 / QKV data-gradient GEMMs hand dL/d(LayerNorm output) to the LayerNorm backward kernels in bf16 (what stock
        # autocast does; halves that tensor's traffic, -0.06 ms per step).  DSF_LN_DY_BF16=0 keeps it in fp32: measured on B200 at
        # all four stage shapes it changes no gradient tensor's error beyond the 3rd digit (profiles/r02a_error_tables.txt).
        dh_dt = bf if os.environ.get("DSF_LN_DY_BF16", "1") == "1" else f32
        dx = torch.empty(M, C, device=dev, dtype=f32)
        dxa_bufs = [torch.empty(M, C, device=dev, dtype=bf), torch.empty(M, C, device=dev, dtype=bf)]  # block i reads [i & 1]
        # ln_f backward; by-products: bf16 copy of dx and db2 of the last block
        last = block_views(L - 1) if L > 0 else None
        K.layernorm_bwd(dyf, saved.x_last, params[-2], saved.mean_f, saved.rstd_f, None, dx, dgf, dbf,
                        dx_bf16=dxa_bufs[(L - 1) & 1] if L > 0 else None, dx_colsum=last[7] if L > 0 else None,
                        byprod_drop=self._drop("mlp", L - 1) if L > 0 else None)
        grads[-2], grads[-1] = dgf, dbf
        for i in reversed(range(L)):
            base = 1 + 16 * i
            (ln1w, ln1b, ln2w, ln2b, kw, kb, qw, qb, vw, vb, pw, pb, w1, b1, w2, b2) = params[base: base + 16]
            st = saved.layers[i]
            dxa = dxa_bufs[i & 1]
            dwqkv, dwp, dw1, dw2, dbqkv, dbp, db1, db2, dg1, dbt1, dg2, dbt2 = block_views(i)
            dwqkv, dwp, dw1, dw2 = dwqkv.view(3 * C, C), dwp.view(C, C), dw1.view(F, C), dw2.view(C, F)
            # ---- MLP:  x_out = x_mid + relu(h2 W1^T + b1) W2^T + b2     (model2_seq.py:121-126,132)
            fork(lambda: K.gemm_bf16_tn(dxa, st.a, dw2))
            da = torch.empty(M, F, device=dev, dtype=bf)
            K.gemm_bf16_nt(dxa, st.w2_t, da, relu_src=st.a)  # ReLU backward fused in the epilogue

            fork(lambda: K.gemm_bf16_tn(da, st.h2, dw1, colsum=db1))  # mlp.0 weight and bias gradients in one launch
            dh2 = torch.empty(M, C, device=dev, dtype=dh_dt)  # feeds LayerNorm backward, not a GEMM
            K.gemm_bf16_nt(da, st.w1_t, dh2)
            dx_mid = torch.empty(M, C, device=dev, dtype=f32)
            dxm = torch.empty(M, C, device=dev, dtype=bf)
            K.layernorm_bwd(dh2, st.x_mid, ln2w, st.mean2, st.rstd2, dx, dx_mid, dg2, dbt2, dx_bf16=dxm, dx_colsum=dbp,
                            byprod_drop=self._drop("proj", i))
            # ---- attention:  x_mid = x_in + proj(attn(qkv(ln1(x_in))))   (model2_seq.py:94-110,131)
            fork(lambda: K.gemm_bf16_tn(dxm, st.y, dwp))
            dy = torch.empty(M, C, device=dev, dtype=bf)
            K.gemm_bf16_nt(dxm, st.wp_t, dy)
            dqkv = torch.empty(M, 3 * C, device=dev, dtype=bf)
            delta = torch.empty(self.B, self.nh, self.T, device=dev, dtype=f32)
            if side is None:
                K.attn_bwd(st.qkv, st.y, dy, st.lse, delta, dqkv, self.B, self.T, C, self.nh, self._drop("attn", i), st.drop_bits)
            else:  # the dQ kernel runs next to the dK/dV kernel: together they leave one partly filled round instead of two
                adrop = self._drop("attn", i)
                K.attn_bwd(st.qkv, st.y, dy, st.lse, delta, dqkv, self.B, self.T, C, self.nh, adrop, st.drop_bits, parts=1)
                fork(lambda: K.attn_bwd(st.qkv, st.y, dy, st.lse, delta, dqkv, self.B, self.T, C, self.nh, adrop, st.drop_bits, parts=4), side_q)
                K.attn_bwd(st.qkv, st.y, dy, st.lse, delta, dqkv, self.B, self.T, C, self.nh, adrop, st.drop_bits, parts=2)
                join(side_q)

            fork(lambda: K.gemm_bf16_tn(dqkv, st.h1, dwqkv, colsum=dbqkv))  # fused QKV weight and bias gradients in one launch
            dh1 = torch.empty(M, C, device=dev, dtype=dh_dt)
            K.gemm_bf16_nt(dqkv, st.wqkv_t, dh1)
            # block i+1's weight-gradient work must be complete now: the next kernel overwrites the bf16 buffer its first wgrad
            # read, and its activations / gradient operands are released here
            join_pending()
            if side is not None:
                ev_blk = torch.cuda.Event()
                ev_blk.record(side)
                pending = (ev_blk, i, (st, da, dxm, dqkv))
            dx = torch.empty(M, C, device=dev, dtype=f32)
            prev = block_views(i - 1) if i > 0 else None
            K.layernorm_bwd(dh1, st.x_in, ln1w, st.mean1, st.rstd1, dx_mid, dx, dg1, dbt1,
                            dx_bf16=dxa_bufs[(i - 1) & 1] if i > 0 else None, dx_colsum=prev[7] if i > 0 else None,
                            byprod_drop=self._drop("mlp", i - 1) if i > 0 else None)
            grads[base: base + 16] = [dg1, dbt1, dg2, dbt2,
                                      dwqkv[C:2 * C], dbqkv[C:2 * C], dwqkv[:C], dbqkv[:C], dwqkv[2 * C:], dbqkv[2 * C:],
                                      dwp, dbp, dw1, db1, dw2, db2]
            saved.layers[i] = None  # release this block's activations early (with the side stream: once `pending` lets go)
            if side is None and self.grad_hook is not None:  # data parallel: average this block's bucket while blocks i-1..0 compute
                self.grad_hook.block_ready(i, bucket(i))
        join_pending()
        dfeats = [torch.empty_like(d) for d in douts]
        dgps = torch.empty(self.B, 2, C, device=dev, dtype=f32)
        # pos_emb's gradient lives at the end of the flat buffer, like every other gradient of the stage: autograd adopts such views
        # without copying them, which a deferred all-reduce relies on (a copy would be taken before the collective has run)
        dpos = gbuf[L * per_block + 2 * C:].view(1, self.T, C)
        if self._drop("embd") is not None:
            K.dropout_inplace(dx, self._drop("embd"))
        K.tokens_bwd(self.geom, dx, douts if residual else None, dfeats, dgps, dpos)
        grads[0] = dpos
        if self.grad_hook is not None:
            self.grad_hook.finish([gbuf[L * per_block + 2 * C:]])
        return dfeats, dgps, grads

    def backward(self, saved, params, douts, dgps_out, residual=True):
        if self.bf16:
            return self._backward_bf16(saved, params, douts, dgps_out, residual)
        dev = douts[0].device
        M, C, L = self.M, self.C, self.L
        f32 = torch.float32
        grads = [None] * len(params)
        dyf = torch.empty(M, C, device=dev, dtype=f32)
        K.upsample_add_bwd(self.geom, douts, dgps_out, dyf)
        dg = torch.zeros(C, device=dev, dtype=f32)
        db = torch.zeros(C, device=dev, dtype=f32)
        dx = torch.empty(M, C, device=dev, dtype=f32)
        K.layernorm_bwd(dyf, saved.x_last, params[-2], saved.mean_f, saved.rstd_f, None, dx, dg, db)
        grads[-2], grads[-1] = dg, db
        for i in reversed(range(L)):
            base = 1 + 16 * i
            (ln1w, ln1b, ln2w, ln2b, kw, kb, qw, qb, vw, vb, pw, pb, w1, b1, w2, b2) = params[base: base + 16]
            st = saved.layers[i]
            # ---- MLP:  x_out = x_mid + relu(h2 W1^T + b1) W2^T + b2     (model2_seq.py:121-126,132)
            da, dw2, db2 = self._linear_bwd(dx, st.a, w2)
            K.relu_bwd(da, st.a)
            dh2, dw1, db1 = self._linear_bwd(da, st.h2, w1)
            dg2 = torch.zeros(C, device=dev, dtype=f32)
            dbt2 = torch.zeros(C, device=dev, dtype=f32)
            dx_mid = torch.empty(M, C, device=dev, dtype=f32)
            K.layernorm_bwd(dh2, st.x_mid, ln2w, st.mean2, st.rstd2, dx, dx_mid, dg2, dbt2)
            # ---- attention:  x_mid = x_in + proj(attn(qkv(ln1(x_in))))   (model2_seq.py:94-110,131)
            dy, dwp, dbp = self._linear_bwd(dx_mid, st.y, pw)
            dqkv = self._attn_bwd(dy, st.qkv, st.y, st)
            dh1, dwqkv, dbqkv = self._linear_bwd(dqkv, st.h1, st.wqkv)
            dg1 = torch.zeros(C, device=dev, dtype=f32)
            dbt1 = torch.zeros(C, device=dev, dtype=f32)
            dx = torch.empty(M, C, device=dev, dtype=f32)
            K.layernorm_bwd(dh1, st.x_in, ln1w, st.mean1, st.rstd1, dx_mid, dx, dg1, dbt1)
            grads[base: base + 16] = [dg1, dbt1, dg2, dbt2,
                                      dwqkv[C:2 * C], dbqkv[C:2 * C], dwqkv[:C], dbqkv[:C], dwqkv[2 * C:], dbqkv[2 * C:],
                                      dwp, dbp, dw1, db1, dw2, db2]
            saved.layers[i] = None  # release this layer's activations early
        dfeats = [torch.empty_like(d) for d in douts]
        dgps = torch.empty(self.B, 2, C, device=dev, dtype=f32)
        dpos = torch.empty(1, self.T, C, device=dev, dtype=f32)
        K.tokens_bwd(self.geom, dx, douts if residual else None, dfeats, dgps, dpos)
        grads[0] = dpos
        return dfeats, dgps, grads


def attn_drop_scale(p):
    """Keep scale of attention dropout: p is quantised to k/256 in the kernels (include/dsfuse.h)."""
    k = max(1, min(255, int(round(float(p) * 256.0))))
    return 256.0 / (256.0 - k)


def materialise_dropout_masks(dropout, B, T, C, n_head, n_layer, device):
    """The multiplicative masks (0 or 1/(1-p)) a ``fusion_stage`` call with ``cfg["dropout"] = dropout`` drew, as
    dense tensors keyed like ``oracle.fusion_ref`` expects: ``embd``, ``proj.{i}``, ``mlp.{i}`` (B,T,C) and
    ``attn.{i}`` (B,nh,T,T).  Elementwise masks are regenerated by running ``dsf_dropout_inplace`` on ones; the
    attention masks are unpacked from the keep-bitmaps in ``dropout["capture"]``.  Diagnostic / test helper."""
    out = {}

    def elem(kind, blk=0):
        p = float(dropout.get("resid" if kind in ("proj", "mlp") else kind, 0.0))
        if p <= 0.0:
            return None
        m = torch.ones(B, T, C, device=device, dtype=torch.float32)
        sd = dropout.get("seed_dev")
        K.dropout_inplace(m, K.Dropout(p, int(dropout["seed"]), drop_site(kind, blk), int(dropout.get("step", 0)),
                                       None if sd is None else sd.data_ptr()))
        return m

    m = elem("embd")
    if m is not None:
        out["embd"] = m
    for i in range(n_layer):
        for kind in ("proj", "mlp"):
            m = elem(kind, i)
            if m is not None:
                out["%s.%d" % (kind, i)] = m
        if float(dropout.get("attn", 0.0)) > 0.0:
            bits = dropout["capture"]["attn_bits.%d" % i].view(B, n_head, T, -1, 1)
            sh = torch.arange(32, device=device, dtype=torch.int32)
            keep = ((bits >> sh) & 1).reshape(B, n_head, T, -1)[..., :T]
            out["attn.%d" % i] = keep.to(torch.float32) * attn_drop_scale(dropout["attn"])
    return out


def _layout_of(t):
    """NCHW-contiguous -> DSF_NCHW; channels_last storage -> DSF_NHWC."""
    if t.is_contiguous():
        return K.DSF_NCHW
    if t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last):
        return K.DSF_NHWC
    raise RuntimeError("feature maps must be contiguous or channels_last")


class FusionStageFn(torch.autograd.Function):
    """(image, lidar, radar feature maps, gps_emb, *GPT params) -> (image', lidar', radar', gps_out)."""

    @staticmethod
    def forward(ctx, cfg, img, lidar, radar, gps_emb, *params):
        for t, n in ((img, "image features"), (lidar, "lidar features"), (radar, "radar features")):
            if not t.is_cuda:
                raise RuntimeError("%s must be CUDA tensors (the fusion stage has no CPU path)" % n)
        # Every launch goes to the CURRENT device's stream with raw pointers: all operands must live on one device, and that
        # device is made current for the whole call (tensors on cuda:1 while cuda:0 is current — nn.DataParallel replicas,
        # TransFuser(cfg, 'cuda:1') without set_device — would otherwise fault instead of raising).
        for t in (lidar, radar, gps_emb) + tuple(params):
            if t.device != img.device:
                raise RuntimeError("fusion stage: all inputs and parameters must be on %s, found a tensor on %s" % (img.device, t.device))
        with torch.cuda.device(img.device):
            return FusionStageFn._forward(ctx, cfg, img, lidar, radar, gps_emb, *params)

    @staticmethod
    def _forward(ctx, cfg, img, lidar, radar, gps_emb, *params):
        K.check_device()
        layout = _layout_of(img)
        if _layout_of(lidar) != layout or _layout_of(radar) != layout:
            lidar = lidar.contiguous(memory_format=torch.channels_last if layout == K.DSF_NHWC else torch.contiguous_format)
            radar = radar.contiguous(memory_format=torch.channels_last if layout == K.DSF_NHWC else torch.contiguous_format)
        if img.dtype not in (torch.float32, torch.bfloat16) or lidar.dtype != img.dtype or radar.dtype != img.dtype:
            raise RuntimeError("feature maps must share one dtype (float32 or bfloat16)")
        S, V = cfg["seq_len"], cfg["n_views"]
        N, C, H, W = lidar.shape
        B = N // S
        if img.shape[0] != B * V * S or radar.shape[0] != B * S:
            raise RuntimeError("inconsistent frame counts: image %d lidar %d radar %d (seq_len %d, n_views %d)"
                               % (img.shape[0], N, radar.shape[0], S, V))
        r = _Runner(B, S, V, cfg["vert_anchors"], cfg["horz_anchors"], C, H, W, cfg["n_head"], cfg["n_layer"],
                    img.dtype, cfg["compute_dtype"], layout)
        if params[0].shape[1] != r.T:
            raise RuntimeError("pos_emb has %d tokens, inputs imply %d" % (params[0].shape[1], r.T))
        gps_emb = gps_emb.contiguous().float()
        plist = [p.detach().contiguous().float() for p in params]
        residual = bool(cfg.get("residual", True))
        r.grad_hook = cfg.get("grad_hook")
        r.dropout = cfg.get("dropout")
        r.capture = cfg.get("capture")
        r.shadows = cfg.get("shadows")
        if r.dropout is not None and any(float(r.dropout.get(k, 0.0)) > 0.0 for k in ("embd", "attn", "resid")):
            if not r.bf16:
                raise NotImplementedError("dropout is implemented in the bf16 tensor-core mode only (the fp32 mode is the "
                                          "p = 0 parity path)")
        else:
            r.dropout = None
        outs, gps_out, saved = r.forward([img.detach(), lidar.detach(), radar.detach()], gps_emb.detach(), plist, residual)
        ctx.runner, ctx.saved_state, ctx.plist, ctx.residual = r, saved, plist, residual
        ctx.device = img.device
        ctx.param_versions = [p._version for p in params]
        ctx.params_ref = params
        ctx.feat_mf = torch.channels_last if layout == K.DSF_NHWC else torch.contiguous_format
        ctx.gps_dtype = gps_emb.dtype
        return outs[0], outs[1], outs[2], gps_out

    @staticmethod
    @once_differentiable
    def backward(ctx, d_img, d_lidar, d_radar, d_gps):
        if ctx.saved_state is None:
            raise RuntimeError("fusion stage: backward called a second time — the saved activations are released block by block "
                               "during the first backward (retain_graph is not supported; call forward again)")
        if any(p._version != v for p, v in zip(ctx.params_ref, ctx.param_versions)):
            raise RuntimeError("fusion stage: a GPT parameter was modified in place between forward and backward (the bf16 weight "
                               "shadows saved by the forward would no longer match the parameters)")
        with torch.cuda.device(ctx.device):
            return FusionStageFn._backward(ctx, d_img, d_lidar, d_radar, d_gps)

    @staticmethod
    def _backward(ctx, d_img, d_lidar, d_radar, d_gps):
        r = ctx.runner
        mf = ctx.feat_mf

        def prep(d, like_dtype):
            return d.contiguous(memory_format=mf).to(like_dtype)

        fdt = torch.bfloat16 if r.geom.feat_dtype == K.DSF_BF16 else torch.float32
        douts = [prep(d_img, fdt), prep(d_lidar, fdt), prep(d_radar, fdt)]
        dgps_out = None if d_gps is None else d_gps.contiguous().float()
        dfeats, dgps, grads = r.backward(ctx.saved_state, ctx.plist, douts, dgps_out, ctx.residual)
        ctx.saved_state = None
        return (None, dfeats[0], dfeats[1], dfeats[2], dgps) + tuple(grads)


def fusion_stage(cfg, img, lidar, radar, gps_emb, params):
    """cfg: dict(seq_len, n_views, vert_anchors, horz_anchors, n_head, n_layer, compute_dtype[, residual][, dropout][, grad_hook]
    [, capture]).  ``capture`` (a dict, diagnostics / tests) receives ``relu.{i}``: the (B*T, 4C) mlp.0 output of block i, whose
    sign pattern is the set of ReLU decisions this evaluation took (see tests/tools/bf16_error_model.py)."""
    return FusionStageFn.apply(cfg, img, lidar, radar, gps_emb, *params)


# ------------------------------------------------------------------------------------------------ stem / tail of Encoder.forward
_IMAGENET_MEAN, _IMAGENET_STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)


def stem_pack_supported(frames):
    """The fused stem takes a list of equally shaped, contiguous fp32 CUDA frames (B, C_in <= 3, H, W) that carry no gradient."""
    f0 = frames[0]
    return (0 < len(frames) <= 16 and f0.is_cuda and f0.dim() == 4 and f0.shape[1] <= 3 and (f0.shape[2] * f0.shape[3]) % 4 == 0
            and all(f.is_cuda and f.dtype == torch.float32 and f.shape == f0.shape and f.is_contiguous() and not f.requires_grad
                    and f.device == f0.device for f in frames))


def stem_pack(frames, normalize, dtype, channels_last):
    """``normalize_imagenet`` (model2_seq.py:36-45, 481-482) + ``torch.stack(frames, dim=1).view(B*S, C, H, W)`` (:491-493) + the
    cast / layout change conv1 needs, as one launch (``dsf_stem_pack``).  Returns the stacked (B*S, C, H, W) tensor in ``dtype``,
    channels_last storage when asked for."""
    f0 = frames[0]
    B, Cin, H, W = f0.shape
    with torch.cuda.device(f0.device):
        out = torch.empty((B * len(frames), Cin, H, W), device=f0.device, dtype=dtype,
                          memory_format=torch.channels_last if (channels_last and Cin > 1) else torch.contiguous_format)
        if normalize:
            if Cin != 3:
                raise RuntimeError("normalize_imagenet expects 3-channel frames, got %d channels" % Cin)
            scale = [1.0 / (255.0 * s) for s in _IMAGENET_STD]
            shift = [-m / s for m, s in zip(_IMAGENET_MEAN, _IMAGENET_STD)]
            K.stem_pack(frames, out, scale, shift)
        else:
            K.stem_pack(frames, out)
    return out


class PooledTailFn(torch.autograd.Function):
    """``avgpool -> flatten -> view -> cat(gps) -> sum(dim=1)`` of Encoder.forward (model2_seq.py:581-595) as one launch per direction
    (``dsf_tail_fwd`` / ``dsf_tail_bwd``): fused[b, c] = sum over maps and frames of the pixel mean + the two GPS tokens."""

    @staticmethod
    def forward(ctx, f_img, f_lid, f_rad, gps, B):
        maps = (f_img, f_lid, f_rad)
        ctx.B = B
        ctx.like = maps
        with torch.cuda.device(f_img.device):
            fused = torch.empty((B, f_img.shape[1]), device=f_img.device, dtype=torch.float32)
            K.tail_fwd(maps, gps, fused, B)
        return fused

    @staticmethod
    @once_differentiable
    def backward(ctx, dfused):
        maps = ctx.like
        dfused = dfused.contiguous().float()
        with torch.cuda.device(dfused.device):
            dmaps = [torch.empty_like(m) for m in maps]  # preserves dtype and (channels_last) strides
            dgps = torch.empty((ctx.B, 2, maps[0].shape[1]), device=dfused.device, dtype=torch.float32)
            K.tail_bwd(dfused, dmaps, dgps, ctx.B)
        return dmaps[0], dmaps[1], dmaps[2], dgps, None


def pooled_tail_supported(f_img, f_lid, f_rad, gps):
    maps = (f_img, f_lid, f_rad)
    lay = K._tail_layout(f_img)
    return (all(m.is_cuda and m.dim() == 4 and m.dtype == f_img.dtype and m.dtype in (torch.float32, torch.bfloat16) and m.shape[1:] == f_img.shape[1:]
                and K._tail_layout(m) == lay and (m.is_contiguous() or m.is_contiguous(memory_format=torch.channels_last)) for m in maps)
            and f_img.shape[1] % 4 == 0 and (f_img.shape[2] * f_img.shape[3]) % 4 == 0
            and gps.is_cuda and gps.dtype == torch.float32 and gps.is_contiguous() and gps.dim() == 3 and gps.shape[1] == 2)


def pooled_tail(f_img, f_lid, f_rad, gps, B):
    return PooledTailFn.apply(f_img, f_lid, f_rad, gps, B)

"""ctypes binding of ``libdsfuse.so`` (C ABI declared in ``include/dsfuse.h``).

The library is built in-tree by ``__graft_entry__.build()`` / ``make -C deepsense6g_tii_b200/csrc``.
There is NO fallback: if the shared object is missing or a call fails, a ``RuntimeError`` is raised.
PyTorch is used only for device memory and streams; every pointer handed to the library is a
``tensor.data_ptr()`` and every call runs on ``torch.cuda.current_stream()``.
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int32, c_int64, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DSF_LIB") or os.path.join(_HERE, "libdsfuse.so")  # DSF_LIB: diagnostics builds (make trace)

DSF_F32, DSF_BF16 = 0, 1
DSF_NCHW, DSF_NHWC = 0, 1
EPI_BIAS, EPI_RELU, EPI_RESIDUAL, EPI_ACCUM = 1, 2, 4, 8

# every symbol include/dsfuse.h declares (tests check that the library exports all of them)
SYMBOLS = [
    "dsf_version", "dsf_last_error", "dsf_launch_count", "dsf_check_device", "dsf_set_pdl", "dsf_set_sm_margin", "dsf_dropout_inplace", "dsf_tokens_fwd", "dsf_tokens_bwd",
    "dsf_layernorm_fwd", "dsf_layernorm_bwd", "dsf_gemm_bf16_nt", "dsf_gemm_bf16_tn", "dsf_gemm_set_impl", "dsf_gemm_f32",
    "dsf_colsum", "dsf_relu_bwd", "dsf_relu_bwd_colsum", "dsf_pack_block_weights", "dsf_softmax_fwd", "dsf_softmax_bwd", "dsf_attn_fwd", "dsf_attn_bwd", "dsf_attn_bwd_parts", "dsf_attn_drop_words",
    "dsf_upsample_add_fwd", "dsf_upsample_add_bwd", "dsf_cast_f32_bf16", "dsf_opt_tiles", "dsf_adamw_ema_pack", "dsf_opt_upload_table", "dsf_chain_fwd",
    "dsf_stem_pack", "dsf_tail_fwd", "dsf_tail_bwd", "dsf_stage_workspace_size", "dsf_stage_fwd",
]


class Geom(ctypes.Structure):
    """``dsf_geom`` (include/dsfuse.h)."""
    _fields_ = [(n, c_int32) for n in ("B", "S", "V", "A_h", "A_w", "C", "H", "W", "feat_dtype", "layout")]


class Dropout(ctypes.Structure):
    """``dsf_dropout`` (include/dsfuse.h): one nn.Dropout site; mask = f(seed, site, step, element index)."""
    _fields_ = [("p", c_float), ("seed", ctypes.c_uint64), ("site", ctypes.c_uint32), ("step", ctypes.c_uint32),
                ("seed_dev", c_void_p)]  # nullable device pointer to a uint64 XOR-ed into the seed (graph-safe reseeding)


def _dp(d):
    return None if d is None else ctypes.byref(d)


class GemmF32Desc(ctypes.Structure):
    """``dsf_gemm_f32_desc`` (include/dsfuse.h)."""
    _fields_ = ([(n, c_int32) for n in ("M", "N", "K", "nb1", "nb2")] +
                [(n, c_int64) for n in ("a_b1", "a_b2", "a_m", "a_k", "b_b1", "b_b2", "b_n", "b_k",
                                        "c_b1", "c_b2", "c_m", "c_n")] +
                [("alpha", c_float), ("epi_flags", c_int32)])


class OptTensor(ctypes.Structure):
    """``dsf_opt_tensor`` (include/dsfuse.h): one parameter tensor of the fused AdamW + EMA + bf16-repack step."""
    _fields_ = ([(n, c_void_p) for n in ("p", "g", "m", "v", "ema", "shadow", "shadow_t", "copy_f32")] +
                [(n, c_int32) for n in ("rows", "cols", "row_off", "ld_t")] + [("weight_decay", c_float), ("reserved", c_int32)])


SHADOW_KEYS = ("wqkv", "wqkv_t", "wp", "wp_t", "w1", "w1_t", "w2", "w2_t", "bqkv")


class DropoutCfg(ctypes.Structure):
    """``dsf_dropout_cfg`` (include/dsfuse.h): the dropout probabilities of one GPT in train() mode."""
    _fields_ = [("embd", c_float), ("attn", c_float), ("resid", c_float), ("seed", ctypes.c_uint64), ("step", ctypes.c_uint32),
                ("seed_dev", c_void_p)]


class StageDesc(ctypes.Structure):
    """``dsf_stage_desc`` (include/dsfuse.h): one fusion stage for ``dsf_stage_fwd``."""
    _fields_ = ([("geom", Geom)] + [(n, c_int32) for n in ("n_head", "n_layer", "F", "residual", "chain", "prepacked")] +
                [("dropout", POINTER(DropoutCfg))])


class BlockShadows(ctypes.Structure):
    """``dsf_block_shadows`` (include/dsfuse.h): the bf16 weight shadows of one block."""
    _fields_ = [(n, c_void_p) for n in SHADOW_KEYS]


class StageParams(ctypes.Structure):
    """``dsf_stage_params`` (include/dsfuse.h)."""
    _fields_ = [("params", POINTER(c_void_p)), ("shadows", POINTER(BlockShadows)), ("ready", POINTER(c_void_p)), ("repack", c_int32)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                "libdsfuse.so not found at %s — build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU / PyTorch fallback for the fusion stage)" % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        L.dsf_last_error.restype = c_char_p
        L.dsf_version.restype = c_int32
        L.dsf_launch_count.restype = c_int64
        P = c_void_p
        sig = {
            "dsf_check_device": [],
            "dsf_tokens_fwd": [POINTER(Geom), P, P, P, P, P, P, P],
            "dsf_tokens_bwd": [POINTER(Geom), P, P, P, P, P, P, P, P, P, P],
            "dsf_layernorm_fwd": [P, P, P, P, c_int32, P, P, c_int32, c_int32, c_float, P],
            "dsf_layernorm_bwd": [P, c_int32, P, P, P, P, P, P, P, P, P, P, POINTER(Dropout), c_int32, c_int32, P],
            "dsf_dropout_inplace": [P, c_int64, POINTER(Dropout), P],
            "dsf_relu_bwd_colsum": [P, P, P, c_int32, c_int32, P],
            "dsf_pack_block_weights": [P] * 9 + [c_int32, c_int32] + [P] * 10,
            "dsf_gemm_bf16_nt": [P, c_int32, P, c_int32, P, c_int32, c_int32, P, P, c_int32, c_int32, c_int32, c_int32, POINTER(Dropout), P, P],
            "dsf_gemm_bf16_tn": [P, c_int32, P, c_int32, P, c_int32, c_int32, c_int32, c_int32, P, P],
            "dsf_gemm_f32": [POINTER(GemmF32Desc), P, P, P, P, P, P],
            "dsf_colsum": [P, c_int32, c_int32, P, c_int32, c_int32, P],
            "dsf_relu_bwd": [P, P, c_int32, c_int64, P],
            "dsf_softmax_fwd": [P, c_int64, c_int32, P],
            "dsf_softmax_bwd": [P, P, c_int64, c_int32, P],
            "dsf_attn_fwd": [P, P, P, c_int32, c_int32, c_int32, c_int32, POINTER(Dropout), P, P],
            "dsf_attn_bwd": [P, P, P, P, P, P, c_int32, c_int32, c_int32, c_int32, POINTER(Dropout), P, P],
            "dsf_attn_bwd_parts": [P, P, P, P, P, P, c_int32, c_int32, c_int32, c_int32, POINTER(Dropout), P, c_int32, P],
            "dsf_set_pdl": [c_int32],
            "dsf_set_sm_margin": [c_int32],
            "dsf_gemm_set_impl": [c_int32],
            "dsf_upsample_add_fwd": [POINTER(Geom), P, P, P, P, P, P, P, P],
            "dsf_upsample_add_bwd": [POINTER(Geom), P, P, P, P, P, P],
            "dsf_cast_f32_bf16": [P, P, c_int64, P],
            "dsf_chain_fwd": [P] * 25 + [c_int32, c_int32, c_float, P],
            "dsf_stem_pack": [P, c_int32, c_int32, c_int32, c_int32, c_int32, P, P, P, c_int32, c_int32, P],
            "dsf_tail_fwd": [P, P, P, P, P] + [c_int32] * 9 + [P],
            "dsf_tail_bwd": [P, P, P, P, P] + [c_int32] * 9 + [P],
            "dsf_opt_tiles": [c_int32, c_int32, c_int32],
            "dsf_opt_upload_table": [P, P, c_int64, P],
            "dsf_adamw_ema_pack": [P, P, c_int32, c_int32, c_double, c_double, c_double, c_double, c_double, P, c_double, P],
        }
        for name, argtypes in sig.items():
            fn = getattr(L, name)
            fn.argtypes = argtypes
            fn.restype = c_int32
        L.dsf_stage_workspace_size.argtypes = [POINTER(StageDesc), POINTER(ctypes.c_size_t)]
        L.dsf_stage_workspace_size.restype = c_int32
        L.dsf_stage_fwd.argtypes = [POINTER(StageDesc), POINTER(StageParams)] + [P] * 9 + [ctypes.c_size_t, P]
        L.dsf_stage_fwd.restype = c_int32
        L.dsf_attn_drop_words.argtypes = [c_int32, c_int32, c_int32]
        L.dsf_attn_drop_words.restype = c_int64
        _lib = L
    return _lib


def _chk(code, what):
    if code != 0:
        raise RuntimeError("%s failed (code %d): %s" % (what, code, lib().dsf_last_error().decode()))


def _stream():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return None if t is None else c_void_p(t.data_ptr())


def _dt(t):
    if t.dtype == torch.float32:
        return DSF_F32
    if t.dtype == torch.bfloat16:
        return DSF_BF16
    raise RuntimeError("dsfuse supports float32 and bfloat16 tensors only, got %s" % t.dtype)


def _req(t, dtype=None, name="tensor"):
    if not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor (the fusion stage has no CPU path)" % name)
    if not t.is_contiguous():
        raise RuntimeError("%s must be contiguous" % name)
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError("%s must be %s, got %s" % (name, dtype, t.dtype))


def launch_count():
    """Kernels launched through the C ABI so far (every launch site passes through check_launch)."""
    return int(lib().dsf_launch_count())


def check_device():
    _chk(lib().dsf_check_device(), "dsf_check_device")


def make_geom(B, S, V, A_h, A_w, C, H, W, feat_dtype, layout=DSF_NCHW):
    return Geom(B, S, V, A_h, A_w, C, H, W, feat_dtype, layout)


# ------------------------------------------------------------------------------------------ wrappers
def tokens_fwd(g, img, lidar, radar, gps, pos_emb, x):
    _chk(lib().dsf_tokens_fwd(ctypes.byref(g), _p(img), _p(lidar), _p(radar), _p(gps), _p(pos_emb), _p(x), _stream()), "dsf_tokens_fwd")


def tokens_bwd(g, dx, dres, douts, dgps, dpos_emb):
    dres = dres or (None, None, None)
    _chk(lib().dsf_tokens_bwd(ctypes.byref(g), _p(dx), _p(dres[0]), _p(dres[1]), _p(dres[2]), _p(douts[0]), _p(douts[1]),
                              _p(douts[2]), _p(dgps), _p(dpos_emb), _stream()), "dsf_tokens_bwd")


def layernorm_fwd(x, gamma, beta, y, mean, rstd, eps=1e-5):
    M, C = x.shape
    _chk(lib().dsf_layernorm_fwd(_p(x), _p(gamma), _p(beta), _p(y), _dt(y), _p(mean), _p(rstd), M, C, eps, _stream()), "dsf_layernorm_fwd")


def layernorm_bwd(dy, x, gamma, mean, rstd, dx_add, dx_out, dgamma, dbeta, dx_bf16=None, dx_colsum=None, byprod_drop=None):
    M, C = x.shape
    _chk(lib().dsf_layernorm_bwd(_p(dy), _dt(dy), _p(x), _p(gamma), _p(mean), _p(rstd), _p(dx_add), _p(dx_out), _p(dgamma),
                                 _p(dbeta), _p(dx_bf16), _p(dx_colsum), _dp(byprod_drop), M, C, _stream()), "dsf_layernorm_bwd")


def dropout_inplace(x, drop):
    _chk(lib().dsf_dropout_inplace(_p(x), x.numel(), _dp(drop), _stream()), "dsf_dropout_inplace")


def relu_bwd_colsum(dy, h, out):
    M, N = dy.shape
    _chk(lib().dsf_relu_bwd_colsum(_p(dy), _p(h), _p(out), M, N, _stream()), "dsf_relu_bwd_colsum")


def pack_block_weights(wq, wk, wv, wp, w1, w2, bq, bk, bv, outs):
    """outs = (wqkv, wqkv_t, wp_b, wp_t, w1_b, w1_t, w2_b, w2_t, bqkv) preallocated."""
    C, F = wq.shape[0], w1.shape[0]
    _chk(lib().dsf_pack_block_weights(_p(wq), _p(wk), _p(wv), _p(wp), _p(w1), _p(w2), _p(bq), _p(bk), _p(bv), C, F,
                                      *[_p(t) for t in outs], _stream()), "dsf_pack_block_weights")


def gemm_bf16_nt(A, B, C, bias=None, residual=None, relu=False, drop=None, relu_src=None):
    """C[M,N] = A[M,K] @ B[N,K]^T (+bias)(relu)(* [relu_src > 0])(dropout)(+residual fp32).  A, B bf16 2-D contiguous;
    C bf16 or fp32; relu_src bf16 with C's shape and leading dimension."""
    M, K = A.shape
    N = B.shape[0]
    flags = (EPI_BIAS if bias is not None else 0) | (EPI_RELU if relu else 0) | (EPI_RESIDUAL if residual is not None else 0)
    _chk(lib().dsf_gemm_bf16_nt(_p(A), A.stride(0), _p(B), B.stride(0), _p(C), C.stride(0), _dt(C), _p(bias), _p(residual),
                                M, N, K, flags, _dp(drop), _p(relu_src), _stream()), "dsf_gemm_bf16_nt")


def gemm_bf16_tn(A, B, C, colsum=None):
    """C[N',K'] += A[M,N']^T @ B[M,K'] (fp32 atomics; C must be pre-zeroed or hold a running sum).  colsum (N') fp32, optional:
    colsum[n'] += sum_m A[m, n'] in the same launch (the bias gradient next to the weight gradient)."""
    M, Nout = A.shape
    Kout = B.shape[1]
    _chk(lib().dsf_gemm_bf16_tn(_p(A), A.stride(0), _p(B), B.stride(0), _p(C), C.stride(0), M, Nout, Kout, _p(colsum), _stream()),
         "dsf_gemm_bf16_tn")


def gemm_f32(desc, A, B, C, bias=None, residual=None):
    _chk(lib().dsf_gemm_f32(ctypes.byref(desc), _p(A), _p(B), _p(C), _p(bias), _p(residual), _stream()), "dsf_gemm_f32")


def colsum(X, out):
    M, N = X.shape
    _chk(lib().dsf_colsum(_p(X), _dt(X), X.stride(0), _p(out), M, N, _stream()), "dsf_colsum")


def relu_bwd(dy, h):
    _chk(lib().dsf_relu_bwd(_p(dy), _p(h), _dt(dy), dy.numel(), _stream()), "dsf_relu_bwd")


def softmax_fwd(s, rows, T):
    _chk(lib().dsf_softmax_fwd(_p(s), rows, T, _stream()), "dsf_softmax_fwd")


def softmax_bwd(dp, p, rows, T):
    _chk(lib().dsf_softmax_bwd(_p(dp), _p(p), rows, T, _stream()), "dsf_softmax_bwd")


def attn_drop_words(B, T, nh):
    """int32 words of the attention-dropout keep bitmap for (B, nh, T) query rows."""
    return int(lib().dsf_attn_drop_words(B, T, nh))


def attn_fwd(qkv, y, lse, B, T, C, nh, drop=None, drop_bits=None):
    _chk(lib().dsf_attn_fwd(_p(qkv), _p(y), _p(lse), B, T, C, nh, _dp(drop), _p(drop_bits), _stream()), "dsf_attn_fwd")


def attn_bwd(qkv, y, dy, lse, delta, dqkv, B, T, C, nh, drop=None, drop_bits=None, parts=7):
    """parts: bit mask 1 = delta, 2 = dK/dV kernel, 4 = dQ kernel (2 and 4 are independent once 1 has run)."""
    _chk(lib().dsf_attn_bwd_parts(_p(qkv), _p(y), _p(dy), _p(lse), _p(delta), _p(dqkv), B, T, C, nh, _dp(drop), _p(drop_bits), parts,
                                  _stream()), "dsf_attn_bwd")


def gemm_set_impl(impl):
    """0 = default (NT on CTA pairs, cta_group::2, where the shape allows), 2 = single-CTA persistent tiles only; process-wide."""
    _chk(lib().dsf_gemm_set_impl(impl), "dsf_gemm_set_impl")


def set_pdl(on):
    """Programmatic dependent launch of the hot kernels on/off (default on); results are identical."""
    _chk(lib().dsf_set_pdl(1 if on else 0), "dsf_set_pdl")


def set_sm_margin(sms):
    """Size persistent grids for (SM count - sms): leaves room for concurrently running NCCL kernels (even, 0..64)."""
    _chk(lib().dsf_set_sm_margin(int(sms)), "dsf_set_sm_margin")


def upsample_add_fwd(g, y, feats, outs):
    _chk(lib().dsf_upsample_add_fwd(ctypes.byref(g), _p(y), _p(feats[0]), _p(feats[1]), _p(feats[2]), _p(outs[0]), _p(outs[1]),
                                    _p(outs[2]), _stream()), "dsf_upsample_add_fwd")


def upsample_add_bwd(g, douts, dgps_out, dy):
    _chk(lib().dsf_upsample_add_bwd(ctypes.byref(g), _p(douts[0]), _p(douts[1]), _p(douts[2]), _p(dgps_out), _p(dy), _stream()), "dsf_upsample_add_bwd")


def stem_pack(frames, out, scale=None, shift=None):
    """frames: list of contiguous fp32 (B, C_in, H, W) CUDA tensors -> out (B*len(frames), C_in, H, W), bf16 / fp32, contiguous or
    channels_last (taken from out's dtype and strides); out = x * scale[c] + shift[c]."""
    n = len(frames)
    B, Cin, H, W = frames[0].shape
    ptrs = (c_void_p * n)(*[f.data_ptr() for f in frames])
    sc = None if scale is None else (c_float * Cin)(*[float(v) for v in scale])
    sh = None if shift is None else (c_float * Cin)(*[float(v) for v in shift])
    nhwc = Cin > 1 and out.is_contiguous(memory_format=torch.channels_last) and not out.is_contiguous()
    _chk(lib().dsf_stem_pack(ptrs, n, B, Cin, H, W, sc, sh, _p(out), _dt(out), DSF_NHWC if nhwc else DSF_NCHW, _stream()), "dsf_stem_pack")


def _tail_layout(t):
    return DSF_NHWC if (t.is_contiguous(memory_format=torch.channels_last) and not t.is_contiguous()) else DSF_NCHW


def tail_fwd(maps, gps, fused, B):
    C, H, W = maps[0].shape[1:]
    fr = [m.shape[0] // B for m in maps]
    _chk(lib().dsf_tail_fwd(_p(maps[0]), _p(maps[1]), _p(maps[2]), _p(gps), _p(fused), B, fr[0], fr[1], fr[2], C, H, W, _dt(maps[0]),
                            _tail_layout(maps[0]), _stream()), "dsf_tail_fwd")


def tail_bwd(dfused, dmaps, dgps, B):
    C, H, W = dmaps[0].shape[1:]
    fr = [m.shape[0] // B for m in dmaps]
    _chk(lib().dsf_tail_bwd(_p(dfused), _p(dmaps[0]), _p(dmaps[1]), _p(dmaps[2]), _p(dgps), B, fr[0], fr[1], fr[2], C, H, W, _dt(dmaps[0]),
                            _tail_layout(dmaps[0]), _stream()), "dsf_tail_bwd")


def cast_f32_bf16(src, dst):
    _chk(lib().dsf_cast_f32_bf16(_p(src), _p(dst), src.numel(), _stream()), "dsf_cast_f32_bf16")


def opt_tiles(rows, cols, transposed_shadow):
    """CTAs the fused optimizer kernel spends on one (rows, cols) tensor (32 x 32 tiles with a transposed shadow, else 1024-element chunks)."""
    n = int(lib().dsf_opt_tiles(rows, cols, 1 if transposed_shadow else 0))
    if n < 0:
        raise RuntimeError("dsf_opt_tiles: a tensor with a transposed shadow needs rows and cols that are multiples of 32, got %d x %d" % (rows, cols))
    return n


def adamw_ema_pack(table_dev, tile0_dev, n_tensors, n_tiles, lr, beta1, beta2, eps, ema_decay, step_dev, grad_scale=1.0):
    """One launch: AdamW update + EMA lerp + bf16 repack over every tensor of the device-resident table (see include/dsfuse.h)."""
    _chk(lib().dsf_adamw_ema_pack(_p(table_dev), _p(tile0_dev), n_tensors, n_tiles, lr, beta1, beta2, eps, ema_decay, _p(step_dev),
                                  grad_scale, _stream()), "dsf_adamw_ema_pack")


def chain_fwd(y, x_in, wp, w1, w2, wqkv_next, bp, b1, b2, bqkv_next, ln2_g, ln2_b, lnn_g, lnn_b, x_mid, x_out, h2, a, h_next, qkv_next, yf,
              mean2, rstd2, mean_next, rstd_next, eps=1e-5):
    """n_embd 64 / 128: proj + residual -> ln2 -> mlp.0 -> ReLU -> mlp.2 + residual -> (next block's ln1 -> fused QKV | ln_f) for
    all rows in ONE launch (model2_seq.py:109, 121-126, 131-132 and :97-99 / :274 of what follows).  wqkv_next None = last block.
    x_mid, h2, a, mean2, rstd2, mean_next, rstd_next (and h_next with a next block) all None: the store-free inference variant,
    which writes only x_out / qkv_next, or yf (x_out optional) after the last block (include/dsfuse.h)."""
    M, C = y.shape
    _chk(lib().dsf_chain_fwd(_p(y), _p(x_in), _p(wp), _p(w1), _p(w2), _p(wqkv_next), _p(bp), _p(b1), _p(b2), _p(bqkv_next), _p(ln2_g), _p(ln2_b),
                             _p(lnn_g), _p(lnn_b), _p(x_mid), _p(x_out), _p(h2), _p(a), _p(h_next), _p(qkv_next), _p(yf), _p(mean2), _p(rstd2),
                             _p(mean_next), _p(rstd_next), M, C, eps, _stream()), "dsf_chain_fwd")


def opt_upload_table(dst_dev, src_pinned):
    """Device copy of the (pinned-host) tensor table of the fused optimizer, done by a kernel (no copy-engine transfer)."""
    if not src_pinned.is_pinned():
        raise RuntimeError("opt_upload_table: the host table must be pinned memory")
    _chk(lib().dsf_opt_upload_table(_p(dst_dev), c_void_p(src_pinned.data_ptr()), src_pinned.numel() * src_pinned.element_size(), _stream()),
         "dsf_opt_upload_table")


def make_stage_desc(geom, n_head, n_layer, F, residual=True, chain=-1, prepacked=False, dropout=None):
    """``dsf_stage_desc``; ``dropout`` a ``DropoutCfg`` or None (the descriptor keeps it alive)."""
    d = StageDesc(geom, n_head, n_layer, F, 1 if residual else 0, chain, 1 if prepacked else 0)
    if dropout is not None:
        d.dropout = ctypes.pointer(dropout)
    return d


def stage_workspace_size(desc):
    """Bytes of device workspace ``stage_fwd`` needs for ``desc`` (the formula is in include/dsfuse.h)."""
    n = ctypes.c_size_t(0)
    _chk(lib().dsf_stage_workspace_size(ctypes.byref(desc), ctypes.byref(n)), "dsf_stage_workspace_size")
    return n.value


def stage_fwd(desc, params, feats, gps_emb, outs, gps_out, workspace, workspace_bytes=None, shadows=None, repack=False, ready=None):
    """One whole inference forward of a fusion stage (``dsf_stage_fwd``).  params: the flat fp32 parameter tensors in
    ``functional.param_names`` order; shadows: None or one dict of bf16 shadow views (``SHADOW_KEYS``) per block; ready: None or one
    ``torch.cuda.Event`` per block that block's shadows are waited for; workspace: a uint8 CUDA tensor, or a raw device address with
    ``workspace_bytes``."""
    ptrs = (c_void_p * len(params))(*[p.data_ptr() for p in params])
    sh = None
    if shadows is not None:
        sh = (BlockShadows * len(shadows))(*[BlockShadows(*[v[k].data_ptr() for k in SHADOW_KEYS]) for v in shadows])
    ev = None if ready is None else (c_void_p * len(ready))(*[e.cuda_event for e in ready])
    prm = StageParams(ptrs, sh, ev, 1 if repack else 0)
    if isinstance(workspace, torch.Tensor):
        ws, nbytes = workspace.data_ptr(), workspace.numel() if workspace_bytes is None else workspace_bytes
    else:
        ws, nbytes = workspace, workspace_bytes
    _chk(lib().dsf_stage_fwd(ctypes.byref(desc), ctypes.byref(prm), _p(feats[0]), _p(feats[1]), _p(feats[2]), _p(gps_emb), _p(outs[0]),
                             _p(outs[1]), _p(outs[2]), _p(gps_out), c_void_p(ws), nbytes, _stream()), "dsf_stage_fwd")

"""Per-kernel GPU parity tests: every C-ABI entry point against the oracle restatement
(oracle/fusion_ref.py) or a plain fp32 torch expression of the same reference lines, on the same
seeded inputs.  All calls go through the C ABI (deepsense6g_tii_b200/_capi.py -> libdsfuse.so).

Tolerances: fp32 kernels 1e-5..1e-4 relative (summation order only); bf16 tensor-core kernels are
compared against an fp32 evaluation of the *same bf16-rounded inputs*, 1e-2 relative (north_star
allows 2e-2 end to end).
"""
import math

import pytest
import torch

from conftest import assert_close
from oracle import fusion_ref as R

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def K(cuda_dev):
    from deepsense6g_tii_b200 import _capi
    _capi.check_device()
    return _capi


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _feat(n, c, h, w, g, dev, dtype=torch.float32, nhwc=False):
    t = torch.randn(n, c, h, w, generator=g).to(dev).to(dtype)
    if nhwc:
        t = t.contiguous(memory_format=torch.channels_last)
    return t


# (B, S, V, A_h, A_w, C, H, W): B samples of S frames, V camera views (image frames B*V*S, slots (V+2)*S), an A_h x A_w anchor
# grid on H x W feature maps.  The comments name the NCHW code path each row reaches.  CT is the channel tile of the NCHW
# kernels (nchw_channel_tile: 8 if H*W >= 1024 and C % 8 == 0, else 32); "pool" is the pooling loop of tokens_fwd_nchw_kernel
# (transpose: kh = kw = 1; lanes-W: kw in {4, 8, 16, 32}, W % 4 == 0 and nct*A_h*W/4 % 32 == 0; generic otherwise), "up-bwd"
# the path of upsample_add_bwd_nchw_kernel (transpose: H == A_h and W == A_w; direct: W/4 in {8, 16, 32}, W/A_w % 8 == 0 and
# H/A_h >= 2 * 32/(W/4); narrow: W in {8, 16, 32} and H/A_h % (32/W) == 0; tiny: narrow with H <= 8 * 32/W; generic otherwise).
# A tile with nct < CT channels loads and stores channel by channel.
STAGE_SHAPES = [
    (2, 5, 1, 8, 8, 64, 64, 64),     # stage 1: CT 8, pool lanes-W, up-bwd direct
    (2, 5, 1, 8, 8, 128, 32, 32),    # stage 2: CT 8, pool lanes-W, up-bwd narrow
    (1, 5, 1, 8, 8, 256, 16, 16),    # stage 3: CT 32, pool generic (kw = 2), up-bwd narrow tiny
    (2, 5, 1, 8, 8, 512, 8, 8),      # stage 4: CT 32, pool transpose, up-bwd transpose
    (1, 2, 1, 16, 16, 64, 32, 32),   # scaled config, 16x16 anchors: CT 8, pool generic, up-bwd narrow
    (1, 3, 1, 4, 4, 8, 24, 24),      # odd scale 6, tiny C: CT 32 with one 8-channel tile (nct < CT), pool generic, up-bwd generic
    (1, 2, 1, 2, 2, 8, 8, 8),        # 8-pixel rows: CT 32, nct 8, pool lanes-W, up-bwd narrow tiny (four rows per load)
    # several camera views: image frame b*V*S + sl of slot sl < V*S (B = 2: at B = 1 that is sl whatever the frame stride)
    (2, 2, 2, 8, 8, 64, 64, 64),     # stage-1 plane: CT 8, pool lanes-W, up-bwd direct
    (2, 1, 3, 2, 4, 32, 8, 16),      # V = 3, rectangular: CT 32, pool lanes-W, up-bwd narrow tiny
    # rectangular anchor grids, the same scale on both axes
    (1, 2, 1, 4, 8, 64, 32, 64),     # scale 8: CT 8, pool lanes-W, up-bwd direct
    (1, 2, 1, 2, 4, 32, 8, 16),      # scale 4: CT 32, pool lanes-W, up-bwd narrow tiny
    (1, 2, 1, 8, 16, 128, 8, 16),    # stage-4 width, scale 1: CT 32, pool transpose, up-bwd transpose
    (2, 2, 2, 2, 4, 8, 12, 24),      # scale 6, V = 2: CT 32, nct 8, pool generic, up-bwd generic
    # partial channel tiles
    (1, 2, 1, 4, 8, 40, 16, 32),     # C = 40 on 512 px: CT 32, tiles 32 + 8, pool lanes-W in both, up-bwd narrow
    (1, 2, 1, 4, 4, 36, 32, 32),     # C = 36 on 1024 px (C % 8 != 0): CT 32, tiles 32 + 4, pool lanes-W in both, up-bwd direct
    (1, 2, 1, 2, 2, 4, 8, 8),        # C = 4: CT 32, nct 4, pool generic with 16-byte loads (nct*A_h*W/4 = 16), up-bwd narrow tiny
    # anisotropic: row scale 6, column scale 2 (the reference never builds it, the kernels take separate per-axis scales)
    (1, 2, 1, 4, 8, 8, 24, 16),      # CT 32, nct 8, pool generic, up-bwd narrow (H/A_h = 6 is a multiple of 32/W = 2)
]


def _frames(B, S, V):
    return (B * V * S, B * S, B * S)


@pytest.mark.parametrize("shape", STAGE_SHAPES)
@pytest.mark.parametrize("variant", ["nchw_f32", "nchw_bf16", "nhwc_f32", "nhwc_bf16"])
def test_tokens_fwd_bwd(K, cuda_dev, shape, variant):
    B, S, V, Ah, Aw, C, H, W = shape
    nhwc = variant.startswith("nhwc")
    dt = torch.bfloat16 if variant.endswith("bf16") else torch.float32
    g = _gen(1)
    T = (V + 2) * S * Ah * Aw + 2
    feats = [_feat(n, C, H, W, g, cuda_dev, dt, nhwc) for n in _frames(B, S, V)]
    gps = torch.randn(B, 2, C, generator=g).to(cuda_dev)
    pos = torch.randn(1, T, C, generator=g).to(cuda_dev)
    geom = K.make_geom(B, S, V, Ah, Aw, C, H, W, K.DSF_BF16 if dt == torch.bfloat16 else K.DSF_F32, K.DSF_NHWC if nhwc else K.DSF_NCHW)
    x = torch.empty(B * T, C, device=cuda_dev)
    K.tokens_fwd(geom, feats[0], feats[1], feats[2], gps, pos, x)
    # oracle on the same (possibly bf16-rounded) inputs, fp32 math
    fr = [f.float().contiguous().requires_grad_(True) for f in feats]
    gr, pr = gps.clone().requires_grad_(True), pos.clone().requires_grad_(True)
    ref = R.build_tokens(*[R.anchor_pool(f, Ah, Aw) for f in fr], gr, pr, S, V)
    assert_close(x.view(B, T, C), ref, 2e-6, 1e-6, "tokens_fwd")
    # backward
    dx = torch.randn(B, T, C, generator=g).to(cuda_dev)
    dres = [_feat(n, C, H, W, g, cuda_dev, dt, nhwc) for n in _frames(B, S, V)]
    ref.backward(dx)
    douts = [torch.empty_like(f) for f in feats]
    dgps = torch.empty(B, 2, C, device=cuda_dev)
    dpos = torch.empty(1, T, C, device=cuda_dev)
    K.tokens_bwd(geom, dx.contiguous(), dres, douts, dgps, dpos)
    tol = 1e-2 if dt == torch.bfloat16 else 2e-6
    for d, f, r in zip(douts, fr, dres):
        assert_close(d.float(), f.grad + r.float(), tol, 1e-6, "tokens_bwd dfeat")
    assert_close(dgps, gr.grad, 1e-6, 1e-7, "dgps")
    assert_close(dpos, pr.grad, 2e-6, 1e-6, "dpos_emb")
    # without the residual-branch gradient
    K.tokens_bwd(geom, dx.contiguous(), None, douts, dgps, dpos)
    for d, f in zip(douts, fr):
        assert_close(d.float(), f.grad, tol, 1e-6, "tokens_bwd no-res")


@pytest.mark.parametrize("M,C", [(962, 64), (1924, 128), (300, 256), (11544, 512), (77, 1024), (10, 8)])
@pytest.mark.parametrize("ydt", [torch.float32, torch.bfloat16])
def test_layernorm(K, cuda_dev, M, C, ydt):
    g = _gen(2)
    x = (torch.randn(M, C, generator=g) * 2 + 0.5).to(cuda_dev)
    w = (1 + 0.1 * torch.randn(C, generator=g)).to(cuda_dev)
    b = (0.1 * torch.randn(C, generator=g)).to(cuda_dev)
    y = torch.empty(M, C, device=cuda_dev, dtype=ydt)
    mean = torch.empty(M, device=cuda_dev)
    rstd = torch.empty(M, device=cuda_dev)
    K.layernorm_fwd(x, w, b, y, mean, rstd)
    xr, wr, br = x.clone().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    ref = R.layer_norm(xr, wr, br)
    assert_close(y.float(), ref, 5e-3 if ydt == torch.bfloat16 else 1e-5, 1e-6, "ln fwd")
    assert_close(mean, x.mean(-1), 1e-5, 1e-6, "mean")
    dy = torch.randn(M, C, generator=g).to(cuda_dev).to(ydt)
    add = torch.randn(M, C, generator=g).to(cuda_dev)
    ref.backward(dy.float())
    dx = torch.empty(M, C, device=cuda_dev)
    dg = torch.zeros(C, device=cuda_dev)
    db = torch.zeros(C, device=cuda_dev)
    K.layernorm_bwd(dy, x, w, mean, rstd, add, dx, dg, db)
    assert_close(dx, xr.grad + add, 2e-5, 1e-6, "ln dx")
    assert_close(dg, wr.grad, 1e-4, 1e-5, "ln dgamma")
    assert_close(db, br.grad, 1e-4, 1e-5, "ln dbeta")
    K.layernorm_bwd(dy, x, w, mean, rstd, None, dx, dg, db)  # accumulates into dg/db
    assert_close(dx, xr.grad, 2e-5, 1e-6, "ln dx no-add")
    assert_close(dg, 2 * wr.grad, 1e-4, 1e-5, "ln dgamma accumulate")
    # same-pass by-products: bf16 copy of dx and its column sums (bias gradient of the preceding Linear)
    dxb = torch.empty(M, C, device=cuda_dev, dtype=torch.bfloat16)
    cs = torch.ones(C, device=cuda_dev)
    K.layernorm_bwd(dy, x, w, mean, rstd, add, dx, dg, db, dx_bf16=dxb, dx_colsum=cs)
    assert_close(dx, xr.grad + add, 2e-5, 1e-6, "ln dx (extra)")
    assert torch.equal(dxb, dx.to(torch.bfloat16))
    assert_close(cs, 1 + dx.sum(0), 1e-4, 1e-4, "ln dx colsum")


def test_pack_weights_and_relu_colsum(K, cuda_dev):
    g = _gen(9)
    C, F = 64, 256
    ws = [torch.randn(C, C, generator=g).to(cuda_dev) for _ in range(4)] + [torch.randn(F, C, generator=g).to(cuda_dev),
                                                                             torch.randn(C, F, generator=g).to(cuda_dev)]
    bs = [torch.randn(C, generator=g).to(cuda_dev) for _ in range(3)]
    bf = torch.bfloat16
    outs = [torch.empty(3 * C, C, device=cuda_dev, dtype=bf), torch.empty(C, 3 * C, device=cuda_dev, dtype=bf),
            torch.empty(C, C, device=cuda_dev, dtype=bf), torch.empty(C, C, device=cuda_dev, dtype=bf),
            torch.empty(F, C, device=cuda_dev, dtype=bf), torch.empty(C, F, device=cuda_dev, dtype=bf),
            torch.empty(C, F, device=cuda_dev, dtype=bf), torch.empty(F, C, device=cuda_dev, dtype=bf),
            torch.empty(3 * C, device=cuda_dev)]
    K.pack_block_weights(ws[0], ws[1], ws[2], ws[3], ws[4], ws[5], bs[0], bs[1], bs[2], outs)
    wqkv = torch.cat(ws[:3], 0).to(bf)
    assert torch.equal(outs[0], wqkv) and torch.equal(outs[1], wqkv.t().contiguous())
    assert torch.equal(outs[2], ws[3].to(bf)) and torch.equal(outs[3], ws[3].to(bf).t().contiguous())
    assert torch.equal(outs[4], ws[4].to(bf)) and torch.equal(outs[5], ws[4].to(bf).t().contiguous())
    assert torch.equal(outs[6], ws[5].to(bf)) and torch.equal(outs[7], ws[5].to(bf).t().contiguous())
    assert torch.equal(outs[8], torch.cat(bs, 0))
    M, N = 1001, 192
    h = torch.randn(M, N, generator=g).to(cuda_dev).to(bf)
    d = torch.randn(M, N, generator=g).to(cuda_dev).to(bf)
    ref = torch.where(h > 0, d, torch.zeros_like(d))
    out = torch.ones(N, device=cuda_dev)
    K.relu_bwd_colsum(d, h, out)
    assert torch.equal(d, ref)
    assert_close(out, 1 + ref.float().sum(0), 1e-5, 1e-5, "relu colsum")


@pytest.mark.parametrize("shape", STAGE_SHAPES)
@pytest.mark.parametrize("variant", ["nchw_f32", "nchw_bf16", "nhwc_f32", "nhwc_bf16"])
def test_upsample_add_fwd_bwd(K, cuda_dev, shape, variant):
    import torch.nn.functional as F
    B, S, V, Ah, Aw, C, H, W = shape
    nhwc = variant.startswith("nhwc")
    dt = torch.bfloat16 if variant.endswith("bf16") else torch.float32
    g = _gen(3)
    T = (V + 2) * S * Ah * Aw + 2
    feats = [_feat(n, C, H, W, g, cuda_dev, dt, nhwc) for n in _frames(B, S, V)]
    y = torch.randn(B, T, C, generator=g).to(cuda_dev)
    geom = K.make_geom(B, S, V, Ah, Aw, C, H, W, K.DSF_BF16 if dt == torch.bfloat16 else K.DSF_F32, K.DSF_NHWC if nhwc else K.DSF_NCHW)
    outs = [torch.empty_like(f) for f in feats]
    K.upsample_add_fwd(geom, y.view(B * T, C), feats, outs)
    yr = y.clone().requires_grad_(True)
    maps = yr[:, :T - 2].reshape(B, (V + 2) * S, Ah, Aw, C).permute(0, 1, 4, 2, 3)
    refs = []
    for m, (lo, hi) in enumerate(((0, V * S), (V * S, (V + 1) * S), ((V + 1) * S, (V + 2) * S))):
        tok = maps[:, lo:hi].reshape(-1, C, Ah, Aw)
        # F.interpolate with the output size samples each axis with step A / H; where both axes share one integer scale this is
        # the oracle's restatement of the reference's F.interpolate(scale_factor=s) call
        up = F.interpolate(tok, size=(H, W), mode="bilinear", align_corners=False)
        if H // Ah == W // Aw:
            assert_close(R.bilinear_upsample(tok, H // Ah), up, 1e-6, 1e-7, "oracle vs F.interpolate")
        refs.append(feats[m].float() + up)
    tol = 1e-2 if dt == torch.bfloat16 else 1e-6
    for o, r in zip(outs, refs):
        assert_close(o.float(), r, tol, 1e-6, "upsample_add_fwd")
    douts = [_feat(n, C, H, W, g, cuda_dev, dt, nhwc) for n in _frames(B, S, V)]
    dgps = torch.randn(B, 2, C, generator=g).to(cuda_dev)
    sum((r * d.float()).sum() for r, d in zip(refs, douts)).backward()
    dy = torch.empty(B * T, C, device=cuda_dev)
    K.upsample_add_bwd(geom, douts, dgps, dy)
    dy = dy.view(B, T, C)
    assert_close(dy[:, :T - 2], yr.grad[:, :T - 2], 1e-5, 1e-6, "upsample_add_bwd")
    assert_close(dy[:, T - 2:], dgps, 0, 0, "gps rows")
    K.upsample_add_bwd(geom, douts, None, dy)
    assert float(dy.view(B, T, C)[:, T - 2:].abs().max()) == 0.0


def test_gemm_f32_variants(K, cuda_dev):
    from deepsense6g_tii_b200._capi import GemmF32Desc, EPI_BIAS, EPI_RELU, EPI_RESIDUAL, EPI_ACCUM
    g = _gen(4)
    M, N, Kd = 203, 130, 77
    x = torch.randn(M, Kd, generator=g).to(cuda_dev)
    w = torch.randn(N, Kd, generator=g).to(cuda_dev)
    b = torch.randn(N, generator=g).to(cuda_dev)
    res = torch.randn(M, N, generator=g).to(cuda_dev)
    out = torch.empty(M, N, device=cuda_dev)
    K.gemm_f32(GemmF32Desc(M, N, Kd, 1, 1, 0, 0, Kd, 1, 0, 0, Kd, 1, 0, 0, N, 1, 1.0, EPI_BIAS | EPI_RELU | EPI_RESIDUAL), x, w, out, b, res)
    assert_close(out, torch.relu(x @ w.t() + b) + res, 1e-5, 1e-6, "NT")
    dy = torch.randn(M, N, generator=g).to(cuda_dev)
    dw = torch.ones(N, Kd, device=cuda_dev)
    K.gemm_f32(GemmF32Desc(N, Kd, M, 1, 1, 0, 0, 1, N, 0, 0, 1, Kd, 0, 0, Kd, 1, 0.5, EPI_ACCUM), dy, x, dw)
    assert_close(dw, 1 + 0.5 * dy.t() @ x, 1e-5, 1e-6, "TN accumulate")
    dx = torch.empty(M, Kd, device=cuda_dev)
    K.gemm_f32(GemmF32Desc(M, Kd, N, 1, 1, 0, 0, N, 1, 0, 0, 1, Kd, 0, 0, Kd, 1, 1.0, 0), dy, w, dx)
    assert_close(dx, dy @ w, 1e-5, 1e-6, "NN")
    # batched attention-shaped contraction with head strides
    B, T, C, nh = 2, 70, 24, 3
    hs = C // nh
    qkv = torch.randn(B * T, 3 * C, generator=g).to(cuda_dev)
    P = torch.empty(B, nh, T, T, device=cuda_dev)
    ld = 3 * C
    K.gemm_f32(GemmF32Desc(T, T, hs, B, nh, T * ld, hs, ld, 1, T * ld, hs, ld, 1, nh * T * T, T * T, T, 1, 0.25, 0), qkv, qkv[:, C:], P)
    q = qkv[:, :C].view(B, T, nh, hs).transpose(1, 2)
    k = qkv[:, C:2 * C].view(B, T, nh, hs).transpose(1, 2)
    assert_close(P, 0.25 * q @ k.transpose(-1, -2), 1e-5, 1e-6, "batched QK^T")


def test_softmax_colsum_relu_cast(K, cuda_dev):
    g = _gen(5)
    rows, T = 37, 962
    s = (3 * torch.randn(rows, T, generator=g)).to(cuda_dev)
    p = s.clone()
    K.softmax_fwd(p, rows, T)
    assert_close(p, torch.softmax(s, -1), 1e-5, 1e-8, "softmax")
    dp = torch.randn(rows, T, generator=g).to(cuda_dev)
    ref = p * (dp - (dp * p).sum(-1, keepdim=True))
    K.softmax_bwd(dp, p, rows, T)
    assert_close(dp, ref, 1e-5, 1e-8, "softmax bwd")
    for dt in (torch.float32, torch.bfloat16):
        X = torch.randn(1001, 194, generator=g).to(cuda_dev).to(dt)
        out = torch.ones(194, device=cuda_dev)
        K.colsum(X, out)
        assert_close(out, 1 + X.float().sum(0), 1e-5, 1e-5, "colsum")
        h = torch.randn(64, 96, generator=g).to(cuda_dev).to(dt)
        d = torch.randn(64, 96, generator=g).to(cuda_dev).to(dt)
        ref = torch.where(h > 0, d, torch.zeros_like(d))
        K.relu_bwd(d, h)
        assert torch.equal(d, ref)
    # vectorised column-sum path (16-byte column groups), incl. a strided view, ragged row counts and the bench shape
    for dt in (torch.float32, torch.bfloat16):
        for (M, N, ld) in [(11544, 1536, 1536), (1001, 200, 200), (77, 2048, 2048), (5, 8, 8), (962, 512, 1536)]:
            X = torch.randn(M, ld, generator=g).to(cuda_dev).to(dt)[:, :N]
            out = torch.ones(N, device=cuda_dev)
            K.colsum(X, out)
            assert_close(out, 1 + X.float().sum(0), 2e-5, 1e-4, "colsum vec %s %s" % (dt, (M, N, ld)))
    src = torch.randn(1003, generator=g).to(cuda_dev)
    dst = torch.empty(1003, device=cuda_dev, dtype=torch.bfloat16)
    K.cast_f32_bf16(src, dst)
    assert torch.equal(dst, src.to(torch.bfloat16))


GEMM_SHAPES = [(128, 64, 64), (128, 128, 64), (300, 128, 128), (962, 192, 64), (1000, 256, 512), (11544, 512, 512),
               (2048, 1536, 512), (1924, 512, 2048), (1924, 2048, 512), (130, 64, 256)]


@pytest.fixture(params=[0, 2], ids=["gemm_pairs", "gemm_single_cta"])
def gemm_impl(request, K):
    K.gemm_set_impl(request.param)
    yield request.param
    K.gemm_set_impl(0)


@pytest.mark.parametrize("M,N,Kd", GEMM_SHAPES + [(11544, 2048, 512), (11544, 512, 2048), (300, 1536, 128), (5, 256, 64),
                                                  # leftover tiles of the pair kernel split along N: 4 ways (18 of 92 tiles),
                                                  # 2 ways (36 of 184 tiles)
                                                  (11544, 512, 1536), (11544, 1024, 256)])
def test_gemm_bf16_nt(K, cuda_dev, gemm_impl, M, N, Kd):
    g = _gen(6)
    a = torch.randn(M, Kd, generator=g).to(cuda_dev).to(torch.bfloat16)
    w = (0.05 * torch.randn(N, Kd, generator=g)).to(cuda_dev).to(torch.bfloat16)
    bias = torch.randn(N, generator=g).to(cuda_dev)
    res = torch.randn(M, N, generator=g).to(cuda_dev)
    ref = a.float() @ w.float().t()
    out = torch.empty(M, N, device=cuda_dev, dtype=torch.bfloat16)
    K.gemm_bf16_nt(a, w, out)
    torch.cuda.synchronize()
    assert_close(out.float(), ref, 6e-3, 1e-4, "plain bf16 out")
    K.gemm_bf16_nt(a, w, out, bias=bias, relu=True)
    assert_close(out.float(), torch.relu(ref + bias), 6e-3, 1e-4, "bias+relu")
    out32 = torch.empty(M, N, device=cuda_dev, dtype=torch.float32)
    K.gemm_bf16_nt(a, w, out32, bias=bias, residual=res)
    assert_close(out32, ref + bias + res, 1e-5, 1e-5, "bias+residual fp32 out")
    K.gemm_bf16_nt(a, w, out32, residual=out32.clone())
    assert_close(out32, 2 * ref + bias + res, 1e-5, 1e-5, "residual aliasing a copy")


@pytest.mark.parametrize("M,No,Ko", [(64, 64, 64), (128, 128, 128), (200, 64, 192), (962, 192, 64), (1924, 512, 512),
                                     (11544, 512, 2048), (11544, 2048, 512), (5000, 1536, 512), (77, 128, 64)])
def test_gemm_bf16_tn(K, cuda_dev, gemm_impl, M, No, Ko):
    g = _gen(7)
    dy = (0.1 * torch.randn(M, No, generator=g)).to(cuda_dev).to(torch.bfloat16)
    x = torch.randn(M, Ko, generator=g).to(cuda_dev).to(torch.bfloat16)
    ref = dy.float().t() @ x.float()
    out = torch.zeros(No, Ko, device=cuda_dev)
    K.gemm_bf16_tn(dy, x, out)
    torch.cuda.synchronize()
    assert_close(out, ref, 2e-5, 1e-5, "wgrad")
    K.gemm_bf16_tn(dy, x, out)
    assert_close(out, 2 * ref, 2e-5, 1e-5, "wgrad accumulates")
    # bias gradient in the same launch (ones-tile MMA): colsum += sum_m dy[m, :], the weight gradient unchanged
    out2 = torch.zeros(No, Ko, device=cuda_dev)
    cs = torch.full((No,), 0.5, device=cuda_dev)
    K.gemm_bf16_tn(dy, x, out2, colsum=cs)
    assert_close(out2, ref, 2e-5, 1e-5, "wgrad next to the bias gradient")
    assert_close(cs, 0.5 + dy.float().sum(0), 2e-5, 1e-5, "bias gradient (accumulated)")


def _attn_ref(qkv, B, T, C, nh):
    hs = C // nh
    q, k, v = [t.reshape(B, T, nh, hs).transpose(1, 2) for t in qkv.view(B, T, 3 * C).split(C, dim=-1)]
    att = torch.softmax((q @ k.transpose(-1, -2)) / math.sqrt(hs), dim=-1)
    lse = torch.logsumexp((q @ k.transpose(-1, -2)) / math.sqrt(hs), dim=-1)
    return (att @ v).transpose(1, 2).reshape(B * T, C), lse


@pytest.mark.parametrize("B,T,C,nh", [(1, 128, 64, 4), (2, 64, 128, 4), (2, 130, 256, 4), (1, 962, 512, 4), (2, 962, 64, 4),
                                      (1, 962, 128, 4), (1, 962, 256, 4), (1, 300, 128, 1), (1, 3842, 64, 4),
                                      (3, 257, 512, 4), (2, 1, 64, 4), (1, 513, 64, 1)])
@pytest.mark.parametrize("impl", [0, 2], ids=["fwd_128row_ctas", "fwd_256row_ctas"])
def test_attention_fwd_bwd(K, cuda_dev, B, T, C, nh, impl):
    K.attn_set_impl(impl)
    try:
        _attention_case(K, cuda_dev, B, T, C, nh)
    finally:
        K.attn_set_impl(0)


def _attention_case(K, cuda_dev, B, T, C, nh):
    g = _gen(8)
    qkv = torch.randn(B * T, 3 * C, generator=g).to(cuda_dev).to(torch.bfloat16)
    y = torch.empty(B * T, C, device=cuda_dev, dtype=torch.bfloat16)
    lse = torch.empty(B, nh, T, device=cuda_dev)
    K.attn_fwd(qkv, y, lse, B, T, C, nh)
    torch.cuda.synchronize()
    qr = qkv.float().requires_grad_(True)
    ref, lse_ref = _attn_ref(qr, B, T, C, nh)
    assert_close(lse, lse_ref, 1e-4, 1e-4, "lse")
    assert_close(y.float(), ref, 1e-2, 1e-4, "attn fwd")
    dy = torch.randn(B * T, C, generator=g).to(cuda_dev).to(torch.bfloat16)
    ref.backward(dy.float())
    delta = torch.empty(B, nh, T, device=cuda_dev)
    dqkv = torch.empty(B * T, 3 * C, device=cuda_dev, dtype=torch.bfloat16)
    K.attn_bwd(qkv, y, dy, lse, delta, dqkv, B, T, C, nh)
    torch.cuda.synchronize()
    for nm, sl in (("dq", slice(0, C)), ("dk", slice(C, 2 * C)), ("dv", slice(2 * C, 3 * C))):
        assert_close(dqkv[:, sl].float(), qr.grad[:, sl], 2e-2, 1e-4, nm)


@pytest.mark.parametrize("B,T,C,nh", [(2, 962, 512, 4), (2, 962, 64, 4), (1, 1000, 128, 4), (1, 3842, 256, 4)])
@pytest.mark.parametrize("impl", [0, 2], ids=["fwd_128row_ctas", "fwd_256row_ctas"])
def test_attention_fwd_when_the_running_maximum_keeps_moving(K, cuda_dev, B, T, C, nh, impl):
    """Keys grow along the sequence, so later key tiles raise a row's maximum by far more than the lazy-rescale threshold (2^8):
    the forward kernel's speculative tiles (exponentials taken against the running maximum first) have to be repeated and the
    output accumulator rescaled.  Same softmax, model2_seq.py:94-106."""
    K.attn_set_impl(impl)
    try:
        g = _gen(21)
        qkv = torch.randn(B, T, 3 * C, generator=g)
        ramp = 0.25 + 5.0 * torch.arange(T, dtype=torch.float32).view(1, T, 1) / T
        qkv[:, :, C:2 * C] *= ramp          # logits of key t scale with ramp[t]: standard deviation 0.25 .. 5.25
        qkv = qkv.reshape(B * T, 3 * C).to(cuda_dev).to(torch.bfloat16)
        y = torch.empty(B * T, C, device=cuda_dev, dtype=torch.bfloat16)
        lse = torch.empty(B, nh, T, device=cuda_dev)
        K.attn_fwd(qkv, y, lse, B, T, C, nh)
        torch.cuda.synchronize()
        ref, lse_ref = _attn_ref(qkv.float(), B, T, C, nh)
        assert_close(lse, lse_ref, 1e-4, 1e-4, "lse")
        assert_close(y.float(), ref, 1e-2, 1e-4, "attn fwd")
    finally:
        K.attn_set_impl(0)


def test_error_paths(K, cuda_dev):
    x = torch.zeros(4, 6, device=cuda_dev)
    with pytest.raises(RuntimeError, match="multiple of 4"):
        K.layernorm_fwd(x, x[0], x[0], torch.empty_like(x), x[:, 0].contiguous(), x[:, 0].contiguous())
    a = torch.zeros(128, 48, device=cuda_dev, dtype=torch.bfloat16)
    with pytest.raises(RuntimeError, match="multiple of 64"):
        K.gemm_bf16_nt(a, a, torch.empty(128, 128, device=cuda_dev, dtype=torch.bfloat16))
    with pytest.raises(RuntimeError, match="head size"):
        K.attn_fwd(torch.zeros(8, 3 * 24, device=cuda_dev, dtype=torch.bfloat16), torch.zeros(8, 24, device=cuda_dev, dtype=torch.bfloat16),
                   torch.zeros(1, 1, 8, device=cuda_dev), 1, 8, 24, 1)
    geom = K.make_geom(1, 1, 1, 4, 4, 8, 10, 10, K.DSF_F32)
    with pytest.raises(RuntimeError, match="not a multiple of the anchor grid"):
        K.tokens_fwd(geom, x, x, x, x, x, x)


@pytest.mark.parametrize("M,N,Kd", [(300, 128, 64), (11544, 2048, 512), (962, 256, 128), (130, 64, 256)])
def test_gemm_bf16_nt_relu_mask_epilogue(K, cuda_dev, M, N, Kd):
    """Backward of nn.ReLU(True) (:123) fused into the mlp.2 data-gradient GEMM: out = (A W^T) * [h > 0]."""
    g = _gen(19)
    a = torch.randn(M, Kd, generator=g).to(cuda_dev).to(torch.bfloat16)
    w = (0.05 * torch.randn(N, Kd, generator=g)).to(cuda_dev).to(torch.bfloat16)
    h = torch.relu(torch.randn(M, N, generator=g)).to(cuda_dev).to(torch.bfloat16)  # post-ReLU activations: exact zeros
    h[0, :5] = -0.0
    out = torch.empty(M, N, device=cuda_dev, dtype=torch.bfloat16)
    K.gemm_bf16_nt(a, w, out, relu_src=h)
    ref = (a.float() @ w.float().t()) * (h.float() > 0)
    assert_close(out.float(), ref, 6e-3, 1e-4, "relu-mask epilogue")
    assert torch.all(out[h.float() <= 0] == 0)


# ------------------------------------------------------------------------------------------ dropout (model2_seq.py:104,109,125,272)
def _mask_of(K, cuda_dev, shape, drop):
    m = torch.ones(shape, device=cuda_dev)
    K.dropout_inplace(m, drop)
    return m


def test_dropout_elementwise_mask_properties(K, cuda_dev):
    """Counter-based masks: values are exactly 0 or 65536/(65536 - round(65536 p)) (= 1/(1-p) to 1.5e-5); the keep rate is 1-p within 5 sigma; the mask is a pure
    function of (seed, site, step) and changes with each of them."""
    n = 962 * 512 * 4
    for p in (0.1, 0.5):
        d = K.Dropout(p, 1234, 3, 7)
        m = _mask_of(K, cuda_dev, (n,), d)
        kept = m != 0
        t16 = round(p * 65536)  # p is quantised to t16 / 65536; kept values carry exactly 65536 / (65536 - t16)
        assert torch.all(m[kept] == torch.tensor(65536.0 / (65536.0 - t16), dtype=torch.float32).to(cuda_dev))
        rate = float(kept.float().mean())
        assert abs(rate - (1 - p)) < 5 * math.sqrt(p * (1 - p) / n), rate
        assert torch.equal(m, _mask_of(K, cuda_dev, (n,), K.Dropout(p, 1234, 3, 7)))
        for other in (K.Dropout(p, 1235, 3, 7), K.Dropout(p, 1234, 4, 7), K.Dropout(p, 1234, 3, 8)):
            agree = float((_mask_of(K, cuda_dev, (n,), other) == m).float().mean())
            assert abs(agree - (p * p + (1 - p) * (1 - p))) < 0.01, agree  # independent draws
    x = torch.randn(1024, device=cuda_dev)
    y = x.clone()
    K.dropout_inplace(y, K.Dropout(0.0, 1, 1, 1))
    assert torch.equal(x, y)


@pytest.mark.parametrize("M,N,Kd", [(300, 128, 64), (962, 512, 2048), (11544, 512, 512), (130, 64, 256)])
def test_gemm_bf16_nt_dropout_epilogue(K, cuda_dev, M, N, Kd):
    """resid_drop fused in the GEMM epilogue (:109,125): (A W^T + b) * mask + residual, mask element index m*N + n."""
    g = _gen(16)
    a = torch.randn(M, Kd, generator=g).to(cuda_dev).to(torch.bfloat16)
    w = (0.05 * torch.randn(N, Kd, generator=g)).to(cuda_dev).to(torch.bfloat16)
    bias = torch.randn(N, generator=g).to(cuda_dev)
    res = torch.randn(M, N, generator=g).to(cuda_dev)
    d = K.Dropout(0.1, 99, 5, 2)
    mask = _mask_of(K, cuda_dev, (M, N), d)
    out = torch.empty(M, N, device=cuda_dev)
    K.gemm_bf16_nt(a, w, out, bias=bias, residual=res, drop=d)
    assert_close(out, (a.float() @ w.float().t() + bias) * mask + res, 1e-5, 1e-5, "bias+dropout+residual")
    outb = torch.empty(M, N, device=cuda_dev, dtype=torch.bfloat16)
    K.gemm_bf16_nt(a, w, outb, bias=bias, drop=d)
    assert_close(outb.float(), (a.float() @ w.float().t() + bias) * mask, 6e-3, 1e-4, "bias+dropout bf16")


@pytest.mark.parametrize("M,C", [(962, 64), (300, 256), (1924, 512)])
def test_layernorm_bwd_dropout_byproducts(K, cuda_dev, M, C):
    """The by-products of LayerNorm backward (bf16 copy of dx and its column sums) carry the mask of the preceding
    Linear's dropout; dx itself does not."""
    g = _gen(17)
    x = torch.randn(M, C, generator=g).to(cuda_dev)
    gamma = torch.randn(C, generator=g).to(cuda_dev)
    dy = torch.randn(M, C, generator=g).to(cuda_dev)
    add = torch.randn(M, C, generator=g).to(cuda_dev)
    y = torch.empty_like(x)
    mean, rstd = torch.empty(M, device=cuda_dev), torch.empty(M, device=cuda_dev)
    K.layernorm_fwd(x, gamma, torch.zeros_like(gamma), y, mean, rstd)
    outs = []
    for d in (None, K.Dropout(0.1, 5, 11, 3)):
        dx = torch.empty_like(x)
        dgm, dbt = torch.zeros(C, device=cuda_dev), torch.zeros(C, device=cuda_dev)
        dxb = torch.empty(M, C, device=cuda_dev, dtype=torch.bfloat16)
        cs = torch.zeros(C, device=cuda_dev)
        K.layernorm_bwd(dy, x, gamma, mean, rstd, add, dx, dgm, dbt, dx_bf16=dxb, dx_colsum=cs, byprod_drop=d)
        outs.append((dx, dxb, cs))
    mask = _mask_of(K, cuda_dev, (M, C), K.Dropout(0.1, 5, 11, 3))
    assert torch.equal(outs[0][0], outs[1][0])
    assert_close(outs[1][1].float(), outs[0][0] * mask, 4e-3, 1e-5, "masked bf16 copy")
    assert_close(outs[1][2], (outs[0][0] * mask).sum(0), 1e-4, 1e-4, "masked column sums")


def _unpack_bits(bits, B, nh, T, dev):
    sh = torch.arange(32, device=dev, dtype=torch.int32)
    return ((bits.view(B, nh, T, -1, 1) >> sh) & 1).reshape(B, nh, T, -1)[..., :T].float()


@pytest.mark.parametrize("B,T,C,nh", [(1, 128, 64, 4), (2, 130, 256, 4), (1, 962, 512, 4), (2, 962, 64, 4), (1, 962, 128, 4), (1, 513, 64, 1)])
@pytest.mark.parametrize("impl", [0, 2], ids=["fwd_128row_ctas", "fwd_256row_ctas"])
def test_attention_dropout_fwd_bwd(K, cuda_dev, B, T, C, nh, impl):
    K.attn_set_impl(impl)
    try:
        _attention_dropout_case(K, cuda_dev, B, T, C, nh)
    finally:
        K.attn_set_impl(0)


def _attention_dropout_case(K, cuda_dev, B, T, C, nh):
    """attn_drop (:104): softmax -> dropout -> @v.  The kernel's keep-bitmap is fed to a plain torch evaluation."""
    from deepsense6g_tii_b200.functional import attn_drop_scale
    g = _gen(18)
    hs = C // nh
    p = 0.1
    d = K.Dropout(p, 4242, 1, 1)
    qkv = torch.randn(B * T, 3 * C, generator=g).to(cuda_dev).to(torch.bfloat16)
    y = torch.empty(B * T, C, device=cuda_dev, dtype=torch.bfloat16)
    lse = torch.empty(B, nh, T, device=cuda_dev)
    bits = torch.zeros(K.attn_drop_words(B, T, nh), device=cuda_dev, dtype=torch.int32)
    K.attn_fwd(qkv, y, lse, B, T, C, nh, d, bits)
    torch.cuda.synchronize()
    keep = _unpack_bits(bits, B, nh, T, cuda_dev)
    k256 = round(p * 256)
    rate = float(keep.mean())
    assert abs(rate - (1 - k256 / 256)) < 5 * math.sqrt(p * (1 - p) / keep.numel()) + 1e-4, rate
    mask = keep * attn_drop_scale(p)
    qr = qkv.float().requires_grad_(True)
    q, k, v = [t.reshape(B, T, nh, hs).transpose(1, 2) for t in qr.view(B, T, 3 * C).split(C, dim=-1)]
    s = (q @ k.transpose(-1, -2)) / math.sqrt(hs)
    ref = ((torch.softmax(s, dim=-1) * mask) @ v).transpose(1, 2).reshape(B * T, C)
    assert_close(lse, torch.logsumexp(s, dim=-1), 1e-4, 1e-4, "lse (un-dropped)")
    assert_close(y.float(), ref, 1e-2, 1e-4, "attn fwd with dropout")
    dy = torch.randn(B * T, C, generator=g).to(cuda_dev).to(torch.bfloat16)
    ref.backward(dy.float())
    delta = torch.empty(B, nh, T, device=cuda_dev)
    dqkv = torch.empty(B * T, 3 * C, device=cuda_dev, dtype=torch.bfloat16)
    K.attn_bwd(qkv, y, dy, lse, delta, dqkv, B, T, C, nh, d, bits)
    torch.cuda.synchronize()
    for nm, sl in (("dq", slice(0, C)), ("dk", slice(C, 2 * C)), ("dv", slice(2 * C, 3 * C))):
        assert_close(dqkv[:, sl].float(), qr.grad[:, sl], 2e-2, 1e-4, nm + " with dropout")
    # a different seed draws a different bitmap; the same seed the same one
    bits2 = torch.zeros_like(bits)
    K.attn_fwd(qkv, y, lse, B, T, C, nh, K.Dropout(p, 4243, 1, 1), bits2)
    assert not torch.equal(bits, bits2)
    K.attn_fwd(qkv, y, lse, B, T, C, nh, d, bits2)
    assert torch.equal(bits, bits2)


@pytest.mark.parametrize("M,C,last", [(11544, 64, False), (11544, 128, False), (300, 64, True), (130, 128, True), (5, 64, False), (1924, 128, False)])
def test_chain_fwd_matches_the_separate_operators(K, cuda_dev, M, C, last):
    """dsf_chain_fwd (n_embd 64 / 128): proj + residual -> ln2 -> mlp.0 -> ReLU -> mlp.2 + residual -> next ln1 -> QKV (or ln_f) in one
    launch, against the same operators in plain torch on the same bf16-rounded operands (model2_seq.py:109, 118-126, 131-132, 274)."""
    g = _gen(31)
    F = 4 * C
    bf = torch.bfloat16
    rnd = lambda *s, sc=1.0: (sc * torch.randn(*s, generator=g)).to(cuda_dev)
    y = rnd(M, C).to(bf)
    x_in = rnd(M, C, sc=2.0) + 0.3
    wp, w1, w2, wq = rnd(C, C, sc=0.1).to(bf), rnd(F, C, sc=0.1).to(bf), rnd(C, F, sc=0.1).to(bf), rnd(3 * C, C, sc=0.1).to(bf)
    bp, b1, b2, bq = rnd(C, sc=0.1), rnd(F, sc=0.1), rnd(C, sc=0.1), rnd(3 * C, sc=0.1)
    g2, be2, gn, ben = 1 + rnd(C, sc=0.1), rnd(C, sc=0.1), 1 + rnd(C, sc=0.1), rnd(C, sc=0.1)
    nan = lambda *s, dt=torch.float32: torch.full(s, float("nan"), device=cuda_dev, dtype=dt)
    x_mid, x_out, yf = nan(M, C), nan(M, C), nan(M, C)
    h2, a, hn, qkv = nan(M, C, dt=bf), nan(M, F, dt=bf), nan(M, C, dt=bf), nan(M, 3 * C, dt=bf)
    st = [nan(M) for _ in range(4)]
    K.chain_fwd(y, x_in, wp, w1, w2, None if last else wq, bp, b1, b2, None if last else bq, g2, be2, gn, ben, x_mid, x_out, h2, a,
                None if last else hn, None if last else qkv, yf if last else None, st[0], st[1], st[2], st[3])
    torch.cuda.synchronize()
    r_mid = y.float() @ wp.float().t() + bp + x_in
    assert_close(x_mid, r_mid, 1e-5, 1e-5, "x_mid")
    mu, var = x_mid.mean(-1), x_mid.var(-1, unbiased=False)
    assert_close(st[0], mu, 1e-4, 1e-5, "mean2")
    assert_close(st[1], torch.rsqrt(var + 1e-5), 1e-4, 1e-5, "rstd2")
    r_h2 = R.layer_norm(x_mid, g2, be2)
    assert_close(h2.float(), r_h2, 6e-3, 1e-3, "h2 (bf16)")
    r_a = torch.relu(h2.float() @ w1.float().t() + b1)          # from the kernel's own bf16 h2: isolates this GEMM
    assert_close(a.float(), r_a, 6e-3, 1e-3, "a (bf16)")
    r_out = a.float() @ w2.float().t() + b2 + x_mid
    assert_close(x_out, r_out, 1e-5, 1e-5, "x_out")
    r_n = R.layer_norm(x_out, gn, ben)
    assert_close(st[2], x_out.mean(-1), 1e-4, 1e-5, "mean_next")
    assert_close(st[3], torch.rsqrt(x_out.var(-1, unbiased=False) + 1e-5), 1e-4, 1e-5, "rstd_next")
    if last:
        assert_close(yf, r_n, 1e-5, 1e-5, "ln_f output")
    else:
        assert_close(hn.float(), r_n, 6e-3, 1e-3, "h_next (bf16)")
        assert_close(qkv.float(), hn.float() @ wq.float().t() + bq, 6e-3, 1e-3, "qkv_next (bf16)")


# ---------------------------------------------------------------------------------------------- stem / tail of Encoder.forward
@pytest.mark.parametrize("cin,normalize", [(3, True), (1, False), (2, False), (3, False)])
@pytest.mark.parametrize("out", ["f32_nchw", "f32_nhwc", "bf16_nhwc", "bf16_nchw"])
def test_stem_pack_matches_normalize_stack_view(K, cuda_dev, cin, normalize, out):
    """dsf_stem_pack vs the reference's op sequence (model2_seq.py:36-45, 481-482, 491-493) as restated in oracle/model_ref.py."""
    from deepsense6g_tii_b200 import functional as Fn
    from oracle import model_ref as MR
    B, S, H, W = 3, 5, 24, 20
    g = _gen(7)
    frames = [(torch.rand(B, cin, H, W, generator=g) * 255.0).to(cuda_dev) for _ in range(S)]
    ref_frames = [MR.normalize_imagenet(f) for f in frames] if normalize else frames
    ref = torch.stack(ref_frames, dim=1).view(B * S, cin, H, W)
    dtype = torch.bfloat16 if out.startswith("bf16") else torch.float32
    assert Fn.stem_pack_supported(frames)
    got = Fn.stem_pack(frames, normalize, dtype, out.endswith("nhwc"))
    assert got.shape == ref.shape and got.dtype == dtype
    if out.endswith("nhwc") and cin > 1:
        assert got.is_contiguous(memory_format=torch.channels_last)
    else:
        assert got.is_contiguous()
    if dtype == torch.float32:
        assert_close(got, ref, 2e-6, msg="stem_pack fp32")     # x*a + b against (x/255 - mean)/std: a few ulp
    else:
        assert torch.equal(got, got.float().to(torch.bfloat16))
        assert_close(got.float(), ref, 4e-3, msg="stem_pack bf16")  # one bf16 rounding
    assert not Fn.stem_pack_supported([f.requires_grad_(True) for f in frames[:1]])


@pytest.mark.parametrize("variant", ["nchw_f32", "nhwc_f32", "nchw_bf16", "nhwc_bf16"])
@pytest.mark.parametrize("shape", [(2, 5, 1, 512, 8), (3, 2, 2, 64, 6), (1, 5, 1, 40, 4)])
def test_pooled_tail_fwd_bwd(K, cuda_dev, variant, shape):
    """dsf_tail_fwd / dsf_tail_bwd vs avgpool -> flatten -> view -> cat(gps) -> sum (model2_seq.py:581-595) and its autograd."""
    from deepsense6g_tii_b200 import functional as Fn
    B, S, V, C, H = shape
    g = _gen(11)
    nhwc, dt = variant.startswith("nhwc"), torch.bfloat16 if variant.endswith("bf16") else torch.float32
    maps = [_feat(B * n, C, H, H, g, cuda_dev, dt, nhwc).requires_grad_(True) for n in (V * S, S, S)]
    gps = torch.randn(B, 2, C, generator=g).to(cuda_dev).requires_grad_(True)
    assert Fn.pooled_tail_supported(maps[0], maps[1], maps[2], gps)
    fused = Fn.pooled_tail(maps[0], maps[1], maps[2], gps, B)
    dfused = torch.randn(B, C, generator=g).to(cuda_dev)
    fused.backward(dfused)
    got = [fused.detach()] + [m.grad.float() for m in maps] + [gps.grad]
    for m in maps:
        assert m.grad.dtype == dt and m.grad.stride() == m.stride()
    ref_maps = [m.detach().double().requires_grad_(True) for m in maps]
    ref_gps = gps.detach().double().requires_grad_(True)
    pool = torch.nn.AdaptiveAvgPool2d((1, 1))
    rows = [torch.flatten(pool(m), 1).view(B, -1, C) for m in ref_maps] + [ref_gps]
    ref = torch.cat(rows, dim=1).sum(dim=1)
    ref.backward(dfused.double())
    want = [ref.detach()] + [m.grad for m in ref_maps] + [ref_gps.grad]
    tol = 1e-5 if dt == torch.float32 else 4e-3  # bf16: the gradient maps are rounded to bf16 once
    for name, a, b in zip(["fused", "dimg", "dlidar", "dradar", "dgps"], got, want):
        assert_close(a.double(), b, 1e-5 if name in ("fused", "dgps") else tol, msg="pooled tail %s" % name)

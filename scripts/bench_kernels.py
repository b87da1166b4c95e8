"""Kernel micro-benchmarks (GPU): CUDA-event timing of single C-ABI entry points at the bench shapes.
Usage: python scripts/bench_kernels.py [attn] [gemm] [elem]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from deepsense6g_tii_b200 import _capi as K  # noqa: E402

dev = torch.device("cuda")
K.check_device()
what = sys.argv[1:] or ["attn", "gemm", "elem"]


def timeit(fn, iters=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


if "attn" in what or "attn512" in what or "attnq" in what:
    shapes = [(12, 962, 512, 4), (12, 962, 256, 4), (12, 962, 128, 4), (12, 962, 64, 4), (2, 3842, 512, 4)]
    for (B, T, C, nh) in (shapes if ("attn" in what or "attnq" in what) else shapes[:1]):
        qkv = torch.randn(B * T, 3 * C, device=dev).to(torch.bfloat16)
        y = torch.empty(B * T, C, device=dev, dtype=torch.bfloat16)
        dy = torch.randn(B * T, C, device=dev).to(torch.bfloat16)
        lse = torch.empty(B, nh, T, device=dev)
        delta = torch.empty(B, nh, T, device=dev)
        dqkv = torch.empty_like(qkv)
        fl = 4.0 * T * T * C * B
        tf = timeit(lambda: K.attn_fwd(qkv, y, lse, B, T, C, nh))
        tb = timeit(lambda: K.attn_bwd(qkv, y, dy, lse, delta, dqkv, B, T, C, nh))
        print("attn B=%d T=%d C=%d hs=%d: fwd %.3f ms (%.0f TF/s)  bwd %.3f ms (%.0f TF/s, 2x fwd flops)"
              % (B, T, C, C // nh, tf, fl / tf / 1e9, tb, 2 * fl / tb / 1e9))

if "gemm" in what:
    M = 11544
    for (N, Kd) in [(1536, 512), (512, 512), (2048, 512), (512, 2048), (512, 1536), (768, 256), (1024, 256), (256, 1024), (192, 64)]:
        a = torch.randn(M, Kd, device=dev).to(torch.bfloat16)
        w = torch.randn(N, Kd, device=dev).to(torch.bfloat16)
        out = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
        bias = torch.randn(N, device=dev)
        tt = timeit(lambda: torch.matmul(a, w.t()))
        dy = torch.randn(M, N, device=dev).to(torch.bfloat16)
        dw = torch.zeros(N, Kd, device=dev)
        fl = 2.0 * M * N * Kd
        line = "gemm M=%d N=%d K=%d: cublas %.4f ms (%.0f TF/s)" % (M, N, Kd, tt, fl / tt / 1e9)
        for impl in (2, 0):  # single-CTA tiles / CTA pairs (default)
            K.gemm_set_impl(impl)
            t = timeit(lambda: K.gemm_bf16_nt(a, w, out, bias=bias))
            line += " | v%d nt %.4f ms (%.0f TF/s)" % (impl, t, fl / t / 1e9)
            if impl == 2:
                t2 = timeit(lambda: K.gemm_bf16_tn(dy, a, dw))
                line += " tn %.4f ms (%.0f TF/s)" % (t2, fl / t2 / 1e9)
        K.gemm_set_impl(0)
        if N == 512:  # the residual-stream GEMMs of the step: fp32 output + bias + fp32 residual (tail tiles split along K)
            out32 = torch.empty(M, N, device=dev)
            res = torch.randn(M, N, device=dev)
            t = timeit(lambda: K.gemm_bf16_nt(a, w, out32, bias=bias, residual=res))
            line += " | v3 f32+bias+residual %.4f ms (%.0f TF/s)" % (t, fl / t / 1e9)
        print(line)

if "elem" in what:
    M, C = 11544, 512
    x = torch.randn(M, C, device=dev)
    g = torch.ones(C, device=dev)
    b = torch.zeros(C, device=dev)
    yb = torch.empty(M, C, device=dev, dtype=torch.bfloat16)
    mean = torch.empty(M, device=dev)
    rstd = torch.empty(M, device=dev)
    t = timeit(lambda: K.layernorm_fwd(x, g, b, yb, mean, rstd))
    print("layernorm_fwd M=%d C=%d: %.4f ms (%.0f GB/s)" % (M, C, t, M * C * 6 / t / 1e6))
    dyb = torch.randn(M, C, device=dev).to(torch.bfloat16)
    dx = torch.empty(M, C, device=dev)
    dg = torch.zeros(C, device=dev)
    db = torch.zeros(C, device=dev)
    t = timeit(lambda: K.layernorm_bwd(dyb, x, g, mean, rstd, x, dx, dg, db))
    print("layernorm_bwd: %.4f ms (%.0f GB/s)" % (t, M * C * 14 / t / 1e6))
    big = torch.randn(M, 4 * C, device=dev).to(torch.bfloat16)
    o = torch.zeros(4 * C, device=dev)
    t = timeit(lambda: K.colsum(big, o))
    print("colsum bf16 M x 2048: %.4f ms (%.0f GB/s)" % (t, M * 4 * C * 2 / t / 1e6))
    t = timeit(lambda: K.colsum(x, o))
    print("colsum f32 M x 512: %.4f ms (%.0f GB/s)" % (t, M * C * 4 / t / 1e6))
    t = timeit(lambda: K.cast_f32_bf16(x, yb))
    print("cast M x 512: %.4f ms (%.0f GB/s)" % (t, M * C * 6 / t / 1e6))
    h = torch.randn(M, 4 * C, device=dev).to(torch.bfloat16)
    t = timeit(lambda: K.relu_bwd(big, h))
    print("relu_bwd M x 2048: %.4f ms (%.0f GB/s)" % (t, M * 4 * C * 6 / t / 1e6))

if "ln" in what:
    # LayerNorm backward as the step runs it: fp32 dy, residual-stream add, bf16 copy + column sums; 8 rotating buffer sets
    # (8 x 106 MB) so that the inputs come from HBM like in the step
    M, C = 11544, 512
    sets = []
    for _ in range(8):
        sets.append(dict(dy=torch.randn(M, C, device=dev), x=torch.randn(M, C, device=dev), add=torch.randn(M, C, device=dev),
                         dx=torch.empty(M, C, device=dev), dxb=torch.empty(M, C, device=dev, dtype=torch.bfloat16)))
    g = torch.randn(C, device=dev)
    mean, rstd = torch.zeros(M, device=dev), torch.ones(M, device=dev)
    dg, db, cs = torch.zeros(C, device=dev), torch.zeros(C, device=dev), torch.zeros(C, device=dev)
    it = [0]

    def run():
        s = sets[it[0] % 8]
        it[0] += 1
        K.layernorm_bwd(s["dy"], s["x"], g, mean, rstd, s["add"], s["dx"], dg, db, dx_bf16=s["dxb"], dx_colsum=cs)
    t = timeit(run, iters=40, warm=8)
    print("layernorm_bwd (step form, HBM-resident): %.4f ms (%.0f GB/s of 18 B/elem)" % (t, M * C * 18 / t / 1e6))
    yb = torch.empty(M, C, device=dev, dtype=torch.bfloat16)

    def runf():
        s = sets[it[0] % 8]
        it[0] += 1
        K.layernorm_fwd(s["x"], g, g, yb, mean, rstd)
    t = timeit(runf, iters=40, warm=8)
    print("layernorm_fwd (HBM-resident): %.4f ms (%.0f GB/s of 6 B/elem)" % (t, M * C * 6 / t / 1e6))
    big = [torch.randn(M, 3 * C, device=dev).to(torch.bfloat16) for _ in range(8)]
    o = torch.zeros(3 * C, device=dev)

    def runc():
        it[0] += 1
        K.colsum(big[it[0] % 8], o)
    t = timeit(runc, iters=40, warm=8)
    print("colsum bf16 M x 1536 (HBM-resident): %.4f ms (%.0f GB/s)" % (t, M * 3 * C * 2 / t / 1e6))


"""Attention kernels timed one by one (GPU): forward, dK/dV (part 2), dQ (part 4), delta (part 1) at the four stage shapes and
the 16x16-anchor shape.  CUDA events around back-to-back launches of one kernel; the working set of a shape (<= 75 MB) is
L2-resident, as it is inside the step (qkv / dy were just written by the preceding kernels).
Usage: python scripts/bench_attn_parts.py [tag] [fwd]     (tag: label printed with the results; fwd: forward kernel only)"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from deepsense6g_tii_b200 import _capi as K  # noqa: E402

dev = torch.device("cuda")
K.check_device()
tag = sys.argv[1] if len(sys.argv) > 1 else "default"
fwd_only = len(sys.argv) > 2 and sys.argv[2] == "fwd"


def timeit(fn, iters=30, warm=5):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3  # us


for (B, T, C, nh) in [(12, 962, 64, 4), (12, 962, 128, 4), (12, 962, 256, 4), (12, 962, 512, 4), (2, 3842, 512, 4)]:
    torch.manual_seed(0)
    qkv = (torch.randn(B * T, 3 * C, device=dev) * 0.5).to(torch.bfloat16)
    y = torch.empty(B * T, C, device=dev, dtype=torch.bfloat16)
    dy = torch.randn(B * T, C, device=dev).to(torch.bfloat16)
    lse = torch.empty(B, nh, T, device=dev)
    delta = torch.empty(B, nh, T, device=dev)
    dqkv = torch.zeros_like(qkv)
    K.attn_fwd(qkv, y, lse, B, T, C, nh)
    fl = 4.0 * T * T * C * B
    tf = timeit(lambda: K.attn_fwd(qkv, y, lse, B, T, C, nh), iters=100 if fwd_only else 30)
    if fwd_only:
        print("%s B=%d T=%d C=%d hs=%d: fwd %.1f us (%.0f TF/s)" % (tag, B, T, C, C // nh, tf, fl / tf / 1e6), flush=True)
        continue
    t1 = timeit(lambda: K.attn_bwd(qkv, y, dy, lse, delta, dqkv, B, T, C, nh, parts=1))
    t2 = timeit(lambda: K.attn_bwd(qkv, y, dy, lse, delta, dqkv, B, T, C, nh, parts=2))
    t4 = timeit(lambda: K.attn_bwd(qkv, y, dy, lse, delta, dqkv, B, T, C, nh, parts=4))
    print("%s B=%d T=%d C=%d hs=%d: fwd %.1f us (%.0f TF/s) | delta %.1f | dK/dV %.1f us | dQ %.1f us | bwd sum %.1f us (%.0f TF/s-eq)"
          % (tag, B, T, C, C // nh, tf, fl / tf / 1e6, t1, t2, t4, t1 + t2 + t4, 2 * fl / (t1 + t2 + t4) / 1e6), flush=True)

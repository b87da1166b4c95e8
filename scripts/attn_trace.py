"""In-kernel timeline of the forward and dK/dV attention kernels (diagnostics build):
    make -C deepsense6g_tii_b200/csrc trace && DSF_LIB=deepsense6g_tii_b200/libdsfuse_trace.so python scripts/attn_trace.py
Prints, per K/V iteration of the forward's CTA (0,0,0), how long the MMA warp waited for V and for the P tile and how the
softmax warpgroup split its time between waiting for S, loading it, the rescale check and the exp/store phase; then the
same for the dK/dV kernel.  Rows of the stamp buffer: 0 / 1 = one warp of math warpgroup 0 / 1, 2 = the MMA warp."""
import ctypes
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from deepsense6g_tii_b200 import _capi as K  # noqa: E402

dev = torch.device("cuda")
B, T, C, nh = 12, 962, int(sys.argv[1]) if len(sys.argv) > 1 else 512, 4
qkv = torch.randn(B * T, 3 * C, device=dev).to(torch.bfloat16)
y = torch.empty(B * T, C, device=dev, dtype=torch.bfloat16)
lse = torch.empty(B, nh, T, device=dev)
for _ in range(3):
    K.attn_fwd(qkv, y, lse, B, T, C, nh)
torch.cuda.synchronize()
buf = (ctypes.c_longlong * (3 * 64 * 6))()
fn = K.lib().dsf_debug_attn_trace
fn.argtypes = [ctypes.c_void_p]
assert fn(buf) == 0
t = torch.tensor(list(buf), dtype=torch.int64).view(3, 64, 6)
n_kv = (T + 63) // 64
t0 = int(t[2, 0, 0])
print("head size %d, T=%d: per-iteration cycles of CTA (0,0,0)" % (C // nh, T))
print("iter | MMA warp: wait V, wait P | softmax: wait S, load+max, rescale chk, exp+store | iter total")
for j in range(n_kv):
    m = t[2, j]
    nxt = int(t[2, j + 1, 0]) if j + 1 < n_kv else None
    row = "%4d | %6d %6d |" % (j, int(m[1] - m[0]), int(m[2] - m[1]))
    a = t[0, j]
    row += " %6d %6d %6d %6d |" % (int(a[1] - a[0]), int(a[2] - a[1]), int(a[3] - a[2]), int(a[5] - a[3]))
    row += " %s" % ("%6d" % (nxt - int(m[0])) if nxt else "")
    print(row)
print("whole loop: %d cycles" % (int(t[0, n_kv - 1, 5]) - t0))

# ---- dK/dV backward kernel (CTA (0,0,0) = keys 0..127 of head 0, batch 0): per 64-query iteration
dy = torch.randn(B * T, C, device=dev).to(torch.bfloat16)
delta = torch.empty(B, nh, T, device=dev)
dqkv = torch.empty_like(qkv)
for _ in range(3):
    K.attn_bwd(qkv, y, dy, lse, delta, dqkv, B, T, C, nh, parts=1)
    K.attn_bwd(qkv, y, dy, lse, delta, dqkv, B, T, C, nh, parts=2)
torch.cuda.synchronize()
assert fn(buf) == 0
t = torch.tensor(list(buf), dtype=torch.int64).view(3, 64, 6)
n_q = (T + 63) // 64
print("dK/dV kernel, head size %d: per-iteration cycles of CTA (0,0,0)" % (C // nh))
print("iter | MMA warp: wait Q/dO(i+1), issue S/dP(i+1), wait dS(i), issue dV/dK | math wg0: prefetch, wait S, tcgen05.ld + wait::ld, exp/dS + tcgen05.st issue, wait::st + fence + arrive | wg1 same | iter total")
for i in range(n_q):
    m = t[2, i]
    nxt = int(t[2, i + 1, 0]) if i + 1 < n_q else None
    if i + 1 < n_q:
        row = "%4d | %6d %6d %6d %6d |" % (i, int(m[1] - m[0]), int(m[2] - m[1]), int(m[3] - m[2]), int(m[4] - m[3]))
    else:
        row = "%4d | %6s %6s %6d %6d |" % (i, "-", "-", int(m[3] - m[2]), int(m[4] - m[3]))
    for w in (0, 1):
        a = t[w, i]
        row += " %6d %6d %6d %6d %6d |" % (int(a[1] - a[0]), int(a[2] - a[1]), int(a[3] - a[2]), int(a[4] - a[3]), int(a[5] - a[4]))
    row += " %s" % ("%6d" % (nxt - int(m[0])) if nxt else "")
    print(row)


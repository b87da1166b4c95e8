"""Host enqueue time and device time of one no-grad fusion-stage forward (``functional.fusion_stage`` under ``torch.no_grad``).

  python scripts/bench_stage_capi.py [--root DIR] [--reps N]

The four stage shapes (n_embd 64 / 128 / 256 / 512 on 64 / 32 / 16 / 8-pixel fp32 NCHW maps, 8 layers, T = 962, bf16 fusion) at
batch 1, 12 and 64.  For each: the host time of the call itself (perf_counter around it, the stream idle before it, so this is the
Python + launch cost of enqueueing one stage), and the CUDA-event time of ``reps`` calls back to back divided by ``reps`` (the device
time, or the host time where the host is the bottleneck).  Both are medians over 5 windows.  ``--root`` imports the package from
another checkout, so that two builds can be measured alternately on the same card: the script uses public entry points only.
The card's name and power limit are printed first (a query; nothing is set)."""
import argparse
import os
import statistics
import subprocess
import sys
import time

ap = argparse.ArgumentParser()
ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap.add_argument("--reps", type=int, default=20)
args = ap.parse_args()
sys.path.insert(0, os.path.abspath(args.root))

import torch  # noqa: E402

from deepsense6g_tii_b200.functional import fusion_stage, param_names  # noqa: E402

dev = torch.device("cuda:0")
S, NH, L = 5, 4, 8


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(dev) + ", power limit unknown"


def stage_params(C, T, g):
    ps = []
    for n in param_names(L):
        if n == "pos_emb":
            t = 0.02 * torch.randn(1, T, C, generator=g)
        elif n.endswith("ln1.weight") or n.endswith("ln2.weight") or n == "ln_f.weight":
            t = 1 + 0.1 * torch.randn(C, generator=g)
        elif n.endswith("bias"):
            t = 0.01 * torch.randn(4 * C if "mlp.0" in n else C, generator=g)
        elif "mlp.0" in n:
            t = 0.02 * torch.randn(4 * C, C, generator=g)
        elif "mlp.2" in n:
            t = 0.02 * torch.randn(C, 4 * C, generator=g)
        else:
            t = 0.02 * torch.randn(C, C, generator=g)
        ps.append(t.to(dev))
    return ps


def main():
    print("# %s" % card(), flush=True)
    cfg = dict(seq_len=S, n_views=1, vert_anchors=8, horz_anchors=8, n_head=NH, n_layer=L, compute_dtype=torch.bfloat16)
    for C, H in ((64, 64), (128, 32), (256, 16), (512, 8)):
        g = torch.Generator().manual_seed(C)
        params = stage_params(C, 3 * S * 64 + 2, g)
        for B in (1, 12, 64):
            feats = [torch.randn(B * S, C, H, H, generator=g).to(dev) for _ in range(3)]
            gps = torch.randn(B, 2, C, generator=g).to(dev)

            def fwd():
                with torch.no_grad():
                    return fusion_stage(cfg, feats[0], feats[1], feats[2], gps, params)
            for _ in range(3):
                fwd()
            torch.cuda.synchronize()
            host, dev_ms = [], []
            for _ in range(5):
                for _ in range(args.reps):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    fwd()
                    host.append((time.perf_counter() - t0) * 1e3)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.reps):
                    fwd()
                e1.record()
                torch.cuda.synchronize()
                dev_ms.append(e0.elapsed_time(e1) / args.reps)
            print("n_embd %3d batch %2d: host enqueue %7.3f ms  back-to-back %7.3f ms/call (min %7.3f)"
                  % (C, B, statistics.median(host), statistics.median(dev_ms), min(dev_ms)), flush=True)
            del feats, gps
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()

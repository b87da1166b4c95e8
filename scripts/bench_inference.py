"""Inference (no_grad) against the grad-enabled forward of the fusion stage, the chain kernel alone, and the configs[3] model.

  python scripts/bench_inference.py [stage] [chain] [model]      (default: all three)

stage: the four stage shapes (n_embd 64 / 128 / 256 / 512 on 64 / 32 / 16 / 8-pixel maps, 8 layers, T = 962) at batch 12, 64 and 256,
       fp32 NCHW maps, bf16 fusion: CUDA-event time of one forward and its peak allocated memory above the pre-call baseline, under
       torch.no_grad() and with grad enabled (forward only, the outputs dropped).
chain: one dsf_chain_fwd launch (a middle block) at n_embd 64 / 128, M = batch * 962, with every output (training) and with the
       backward-only outputs NULL (store-free; a build without that variant rejects the call and prints "n/a").
model: the BASELINE.json configs[3] workload (TransFuser eval, lidar and radar missing, bf16 autocast, channels_last) at batch 64,
       256, 1024 and the largest of 4096 / 2048 / 1536 that fits: samples/s and peak allocated memory.
Uses public entry points only, so the same file measures any build of the package.  The card's name and power limit are printed
first (a query; nothing is set)."""
import os
import subprocess
import sys
import types

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from deepsense6g_tii_b200 import _capi as K  # noqa: E402
from deepsense6g_tii_b200.functional import fusion_stage, param_names  # noqa: E402

dev = torch.device("cuda:0")
S, NH, L = 5, 4, 8
MB = 2.0 ** 20


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(dev) + ", power limit unknown"


def timed(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def peak(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return (torch.cuda.max_memory_allocated() - base) / MB


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
        ps.append(t.to(dev).requires_grad_(True))
    return ps


def bench_stage():
    print("== fusion stage, 8 layers, T = 962, bf16 fusion, fp32 NCHW maps: one forward", flush=True)
    for C, H in ((64, 64), (128, 32), (256, 16), (512, 8)):
        g = torch.Generator().manual_seed(C)
        T = 3 * S * 64 + 2
        params = stage_params(C, T, g)
        cfg = dict(seq_len=S, n_views=1, vert_anchors=8, horz_anchors=8, n_head=NH, n_layer=L, compute_dtype=torch.bfloat16)
        for B in (12, 64, 256):
            feats = [torch.randn(B * S, C, H, H, device=dev) for _ in range(3)]
            gps = torch.randn(B, 2, C, device=dev)

            def fwd():
                fusion_stage(cfg, feats[0], feats[1], feats[2], gps, params)

            def fwd_nograd():
                with torch.no_grad():
                    fwd()
            line = "n_embd %3d batch %3d:" % (C, B)
            n = max(3, min(20, 2560 // (B * (C // 64 + 1))))
            res = {}
            for name, fn in (("no_grad", fwd_nograd), ("grad", fwd)):
                fn()
                res[name] = [timed(fn, n), peak(fn)]
            for r in range(2):   # alternate once more: the two timings share the conditions of one window
                for name, fn in (("no_grad", fwd_nograd), ("grad", fwd)):
                    res[name][0] = min(res[name][0], timed(fn, n))
            for name in ("no_grad", "grad"):
                line += "  %s %8.3f ms %9.1f MB" % (name, res[name][0], res[name][1])
            line += "  | time ratio %.3f, memory ratio %.2f" % (res["no_grad"][0] / res["grad"][0], res["grad"][1] / res["no_grad"][1])
            print(line, flush=True)
            del feats, gps
            torch.cuda.empty_cache()


def bench_chain():
    print("== chain kernel alone (middle block), M = batch * 962", flush=True)
    bf = torch.bfloat16
    for C in (64, 128):
        F = 4 * C
        for B in (12, 256):
            M = B * 962
            r = lambda *s, dt=torch.float32: (0.1 * torch.randn(*s, device=dev)).to(dt)
            y, x_in = r(M, C, dt=bf), r(M, C)
            wp, w1, w2, wq = r(C, C, dt=bf), r(F, C, dt=bf), r(C, F, dt=bf), r(3 * C, C, dt=bf)
            bp, b1, b2, bq, g2, be2, gn, ben = r(C), r(F), r(C), r(3 * C), 1 + r(C), r(C), 1 + r(C), r(C)
            x_out, qkv = torch.empty(M, C, device=dev), torch.empty(M, 3 * C, device=dev, dtype=bf)
            full = [torch.empty(M, C, device=dev), torch.empty(M, C, device=dev, dtype=bf), torch.empty(M, F, device=dev, dtype=bf),
                    torch.empty(M, C, device=dev, dtype=bf)] + [torch.empty(M, device=dev) for _ in range(4)]

            def launch(s):
                K.chain_fwd(y, x_in, wp, w1, w2, wq, bp, b1, b2, bq, g2, be2, gn, ben, s[0], x_out, s[1], s[2], s[3], qkv, None,
                            s[4], s[5], s[6], s[7])
            line = "n_embd %3d batch %3d:" % (C, B)
            variants = (("training", full), ("store-free", [None] * 8))
            ok = {}
            for name, s in variants:
                try:
                    launch(s)
                    torch.cuda.synchronize()
                    ok[name] = 1e9
                except RuntimeError:
                    ok[name] = None
            for _ in range(3):   # alternate the two variants, keep the best window of each
                for name, s in variants:
                    if ok[name] is not None:
                        ok[name] = min(ok[name], timed(lambda: launch(s), 200))
            for name, _ in variants:
                line += "  %s %s" % (name, "n/a" if ok[name] is None else "%7.2f us" % (ok[name] * 1e3))
            print(line, flush=True)
            del full
            torch.cuda.empty_cache()


def bench_model():
    from deepsense6g_tii_b200 import TransFuser
    print("== configs[3] model: TransFuser eval, lidar_radar missing, bf16 autocast, channels_last", flush=True)
    torch.backends.cudnn.benchmark = True
    cfg = types.SimpleNamespace(seq_len=5, pred_len=4, n_views=1, vert_anchors=8, horz_anchors=8, n_embd=512, block_exp=4, n_layer=8,
                                n_head=4, embd_pdrop=0.1, attn_pdrop=0.1, resid_pdrop=0.1, add_velocity=1, fusion_dtype=torch.bfloat16,
                                modality_missing="lidar_radar", modality_missing_type="zerolike")
    torch.manual_seed(100)
    model = TransFuser(cfg, dev).to(memory_format=torch.channels_last).eval()

    def run_batch(B):
        # drawn on the device (the host would take minutes at batch 4096); lidar and radar are replaced by zeros inside the model
        g = torch.Generator(device=dev).manual_seed(B)
        imgs = [torch.randint(0, 256, (B, 3, 256, 256), generator=g, device=dev).float().contiguous(memory_format=torch.channels_last)
                for _ in range(5)]
        lids = [(torch.rand(B, 1, 256, 256, generator=g, device=dev) < 0.05).float() for _ in range(5)]
        rads = [torch.rand(B, 2, 256, 256, generator=g, device=dev) for _ in range(5)]
        gps = ((torch.rand(B, 2, 1, generator=g, device=dev) - 0.5) * 3.14159).expand(B, 2, 2).contiguous()

        def run():
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
                return model(imgs, lids, rads, gps)
        try:
            run()
            torch.cuda.synchronize()
            pk = peak(run)
            ms = min(timed(run, max(2, min(10, 1024 // B))) for _ in range(2))
            print("batch %4d: %9.2f ms  %9.1f samples/s  peak %9.1f MB" % (B, ms, B / ms * 1e3, pk), flush=True)
            return True
        except torch.OutOfMemoryError:
            print("batch %4d: out of memory" % B, flush=True)
            return False
        finally:
            del imgs, lids, rads, gps
            torch.cuda.empty_cache()

    for B in (64, 256, 1024):
        run_batch(B)
    for B in (4096, 2048, 1536):
        if run_batch(B):
            break


if __name__ == "__main__":
    torch.cuda.set_device(dev)
    print("device: %s" % card(), flush=True)
    parts = sys.argv[1:] or ["stage", "chain", "model"]
    for p in parts:
        {"stage": bench_stage, "chain": bench_chain, "model": bench_model}[p]()

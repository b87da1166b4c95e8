#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native GPT fusion path of model2_seq.py.

Metric (BASELINE.json): train samples/sec (fwd+bwd).  Default workload (``--workload fusion4``): the WHOLE hot path north_star
names — the four fusion stages of the 256x256 model back to back (Encoder.forward:515-526, 533-544, 552-563, 571-579 + GPT
:175-287; n_embd 64/128/256/512 on 64/32/16/8-pixel feature maps, 8 layers, 4 heads, 8x8 anchors, seq_len 5 -> T = 962
tokens), fwd+bwd, bf16, per-GPU batch 12, synthetic trunk features.  BASELINE.json configs[1] (the n_embd 512 stage alone)
is measured in the same run and reported as the sub-record ``stage4`` (``--workload stage4`` makes it the whole line).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload fusion4|stage4|model] [--anchors 8|16]
                  [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU): every rank runs its own batch-12 shard (weak scaling) and the GPT gradients
are all-reduced over NCCL every step (DDP semantics of train2_seq.py:538 replaced by one-process-per-GPU).  Rank 0 prints
ONE JSON line.

--impl reference times the reference's own implementation of the same path on the host cores, fp32, batch 12: the unmodified
reference ``GPT`` class (oracle/_ref/model2_seq.py, placed there by ``__graft_entry__.build()`` where /root/reference exists)
inside the pool / interpolate / add calls of Encoder.forward; when oracle/_ref is absent, the oracle port (oracle/fusion_ref.py).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

L, NH, S, V, BATCH = 8, 4, 5, 1, 12
A = 8
STAGES4 = ((64, 8), (128, 4), (256, 2), (512, 1))   # (n_embd, feature-map side / anchors) of the four fusion stages
SPEC = STAGES4                                      # stages of the selected workload
PDROP = 0.0  # --dropout: embd/attn/resid probability (the reference trains with 0.1; 0 = the parity configuration)


def n_tokens():
    return (V + 2) * S * A * A + 2


def fwd_flops_per_sample(c):
    """SURVEY.md §8(d): L * (24 T C^2 + 4 T^2 C); backward = 2x (flash-attention recompute not counted)."""
    t = n_tokens()
    return L * (24.0 * t * c * c + 4.0 * t * t * c)


def workload_name():
    t = n_tokens()
    if len(SPEC) == 1:
        return "gpt_fusion_stage n_embd=%d n_layer=8 n_head=4 anchors=%dx%d seq_len=5 T=%d batch=12/GPU fwd+bwd" % (SPEC[0][0], A, A, t)
    return ("gpt_fusion_path: the 4 fusion stages of model2_seq back to back (n_embd %s on %s-pixel feature maps), n_layer=8 n_head=4 "
            "anchors=%dx%d seq_len=5 T=%d batch=12/GPU fwd+bwd" % ("/".join(str(c) for c, _ in SPEC), "/".join(str(A * s) for _, s in SPEC), A, A, t))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tc_burst=d["bf16_tflops"], tc_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tc_burst=1590.0, tc_sust=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def synth_inputs(gen, batch, c, scale, pin=False):
    """Synthetic inputs of one stage: post-ReLU-like trunk features (non-negative, ~unit scale), GPS embeddings, loss probes."""
    h = A * scale
    feats = [torch.randn(batch * S, c, h, h, generator=gen).abs_() for _ in range(3)]
    gps = torch.randn(batch, 2, c, generator=gen)
    probes = [torch.randn(f.shape, generator=gen) * 1e-3 for f in feats] + [torch.randn(batch, 2, c, generator=gen) * 1e-3]
    ts = feats + [gps] + probes
    if pin:
        ts = [t.pin_memory() for t in ts]
    return ts[:3], ts[3], ts[4:]


def dump_outputs(out_dir, named):
    """Writes every (name, tensor) of ``named`` as ``out_dir/<name>.npy`` in float32, 64 MB in all.  Each tensor gets an equal
    share of that; a larger tensor is stored flattened, as the elements at a fixed set of positions (drawn once per element count
    by a generator seeded with 0), so two runs with the same arguments store the same positions and can be compared file by file."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    cap = (64 * 10 ** 6 // len(named) - 4096) // 4   # elements per file; 4 KB of the share is left for the .npy header
    picks = {}
    for name, t in named:
        x = t.detach()
        n = x.numel()
        if n > cap:
            if n not in picks:
                picks[n] = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:cap].sort().values
            x = x.reshape(-1)[picks[n].to(x.device)]
        np.save(os.path.join(out_dir, name + ".npy"), x.float().cpu().numpy())


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


# ----------------------------------------------------------------------------------------- reference arm (CPU) / stock-PyTorch GPU baseline
def _load_reference_gpt():
    """The reference's own GPT class, imported from the git-ignored copy build() places under oracle/_ref (SURVEY §8c shims:
    stub ``mamba_ssm``).  Returns (model2_seq module, GlobalConfig) or None when the copy is absent."""
    ref = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isfile(os.path.join(ref, "model2_seq.py")):
        return None
    os.environ.setdefault("DSF_REFERENCE_ROOT", ref)
    try:
        from oracle import ref_import
        ref_import.REFERENCE_ROOT = ref
        return ref_import.load_reference()
    except Exception as ex:
        sys.stderr.write("bench.py: oracle/_ref present but not importable (%s); using the oracle port\n" % ex)
        return None


def reference_step_fn(device, batch, autocast=False):
    """fwd+bwd of the selected workload through the reference code (stock PyTorch ops) on ``device``.  Returns (step, kind)."""
    ref = _load_reference_gpt()
    dev = torch.device(device)
    gen = torch.Generator().manual_seed(0)
    units = []
    for c, scale in SPEC:
        feats, gps, probes = synth_inputs(gen, batch, c, scale)
        feats = [f.to(dev).requires_grad_(True) for f in feats]
        gps = gps.to(dev).requires_grad_(True)
        probes = [p.to(dev) for p in probes]
        if ref is not None:
            M, GlobalConfig = ref
            torch.manual_seed(100)
            cfg = GlobalConfig(add_velocity=1, embd_pdrop=PDROP, attn_pdrop=PDROP, resid_pdrop=PDROP)
            cfg.vert_anchors = cfg.horz_anchors = A
            gpt = M.GPT(c, NH, 4, L, A, A, S, PDROP, PDROP, PDROP, cfg).to(dev).train()
            pool = torch.nn.AdaptiveAvgPool2d((A, A))
            params = list(gpt.parameters())

            def fwd(feats=feats, gps=gps, gpt=gpt, pool=pool, scale=scale):   # Encoder.forward, model2_seq.py:515-526
                o = gpt(pool(feats[0]), pool(feats[1]), pool(feats[2]), gps)
                ups = [o[k] if scale == 1 else torch.nn.functional.interpolate(o[k], scale_factor=scale, mode="bilinear") for k in range(3)]
                return [f + u for f, u in zip(feats, ups)] + [o[3]]
        else:
            from oracle import fusion_ref as R
            p = R.init_gpt_params(c, NH, 4, L, n_tokens(), generator=gen, pos_std=0.02)
            p = {k: v.to(dev).requires_grad_(True) for k, v in p.items()}
            params = list(p.values())

            def fwd(feats=feats, gps=gps, p=p):
                (a, b, cc), g = R.fusion_stage(p, feats, gps, NH, S, A, A)
                return [a, b, cc, g]
        units.append((fwd, params, feats, gps, probes))

    def step():
        total = 0.0
        for fwd, params, feats, gps, probes in units:
            for t in params + feats + [gps]:
                t.grad = None
            with torch.autocast(dev.type, dtype=torch.bfloat16, enabled=autocast):
                outs = fwd()
            torch.autograd.backward(outs, [pr.to(o.dtype) for o, pr in zip(outs, probes)])   # probes = upstream gradients, as in the GPU arm
            total = total + outs[3].detach().float().sum()
        return total
    return step, ("reference" if ref is not None else "port")


def time_cpu(steps, warmup):
    torch.set_num_threads(os.cpu_count() or 1)
    step, kind = reference_step_fn("cpu", BATCH)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return BATCH * steps / dt, dt / steps * 1e3, kind


def cpu_sample_note(kind, cores, steps, warmup):
    what = ("the reference's own GPT class (oracle/_ref/model2_seq.py, unmodified) inside the pool/interpolate/add of Encoder.forward"
            if kind == "reference" else "oracle port (oracle/fusion_ref.py)")
    return "%s, same workload, fp32, batch %d per step, %d warm-up + %d timed steps, %d threads, %s" % (what, BATCH, warmup, steps, cores, cpu_model())


def run_reference(args, rank):
    if rank != 0:
        return
    steps, warmup = args.steps, max(0, args.warmup)
    v, ms, kind = time_cpu(steps, warmup)
    cores = torch.get_num_threads()
    print(json.dumps({
        "impl": "reference", "metric": "train samples/sec (fwd+bwd)", "value": v, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(args.gpus),
        "cpu_baseline": {"value": v, "unit": "samples/s", "cores": cores, "kind": kind, "sample": cpu_sample_note(kind, cores, steps, warmup)},
        "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def workload_config(world):
    """The part of ``config`` both arms share (the driver compares them)."""
    return {"workload": workload_name(), "global_batch": BATCH * world, "seq_len": S, "parallelism": "dp%d" % world}


# ----------------------------------------------------------------------------------------- GPU arm
def build_gpt(device, c):
    import types
    from deepsense6g_tii_b200 import GPT
    cfg = types.SimpleNamespace(n_views=V, fusion_dtype=torch.bfloat16)
    torch.manual_seed(100)  # the reference's seed (train2_seq.py:430-434)
    m = GPT(c, NH, 4, L, A, A, S, PDROP, PDROP, PDROP, cfg)
    with torch.no_grad():
        m.pos_emb.normal_(0, 0.02)
    return m.to(device)


class StageWork:
    """One fusion stage of the workload: its GPT, its device-resident inputs and the pinned host copies of them."""

    def __init__(self, c, scale, dev, gen, pin=True, optimizer=False):
        self.c, self.scale = c, scale
        self.gpt = build_gpt(dev, c)
        self.opt = self.ema = None
        if optimizer:   # --optimizer: AdamW + EMA + bf16 repack as one dsfuse launch per stage (the forward then packs nothing)
            from deepsense6g_tii_b200.optim import FusedAdamWEMA
            from deepsense6g_tii_b200.train import EMA
            self.ema = EMA(self.gpt, 0.999)
            self.ema.register()
            self.opt = FusedAdamWEMA(self.gpt.parameters(), lr=1e-4, ema=self.ema, gpts=[self.gpt])
        self.feats_h, self.gps_h, probes_h = synth_inputs(gen, BATCH, c, scale, pin=pin)
        self.feats = [f.to(dev).requires_grad_(True) for f in self.feats_h]
        self.gps = self.gps_h.to(dev).requires_grad_(True)
        self.probes = [p.to(dev) for p in probes_h]

    def step(self):
        for p in self.gpt.parameters():
            p.grad = None
        for t in self.feats:
            t.grad = None
        self.gps.grad = None
        outs = self.gpt.fuse(self.feats[0], self.feats[1], self.feats[2], self.gps)
        # kept for --dump-outputs (a replayed CUDA graph rewrites them in place); detached, so that they do not keep this step's
        # autograd graph, and with it the parameters' gradient accumulators, alive into the next step
        self.outs = [o.detach() for o in outs]
        # the probes are the upstream gradients (in the model they come from the ResNet layers that follow the stage); the step's
        # scalar result is the sum of the two GPS output tokens (a 12 x 2 x C reduction: the only non-dsfuse kernel of the step)
        torch.autograd.backward(outs, self.probes)
        if self.opt is not None:
            self.opt.step()
            self.ema.update()
        return outs[3].detach().sum()

    def computed(self):
        """(name, tensor) of what the last step handed back: the four outputs and the gradients of the inputs and parameters."""
        names = ("img", "lidar", "radar", "gps")
        named = [("C%d.out.%s" % (self.c, n), o) for n, o in zip(names, self.outs)]
        named += [("C%d.grad.%s" % (self.c, n), t.grad) for n, t in zip(names, self.feats + [self.gps])]
        return named + [("C%d.grad.%s" % (self.c, n), p.grad) for n, p in self.gpt.named_parameters() if p.grad is not None]


def one_step(works):
    total = None
    for w in works:
        l = w.step()
        total = l if total is None else total + l
    return total


def capture_step(fn, warm=3):
    """Warm ``fn`` up on a side stream, then capture it into ONE CUDA graph (the launch sequence is static: fixed shapes, torch's
    caching allocator keeps the captured addresses alive).  Under capture ``functional`` moves the weight-gradient GEMMs, bias
    sums, weight packs and the dQ attention kernel to side streams (fork/join events = graph edges).  Returns
    (graph, value returned by the captured call, dsfuse launches per replay)."""
    from deepsense6g_tii_b200 import _capi
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(warm):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    n0 = _capi.launch_count()
    with torch.cuda.graph(graph):
        out = fn()
    n = _capi.launch_count() - n0
    torch.cuda.synchronize()
    return graph, out, n


FAMILIES = ["tokens_fwd", "tokens_bwd", "layernorm_fwd", "layernorm_bwd", "gemm_bf16_nt", "gemm_bf16_tn", "colsum", "attn_fwd", "attn_bwd",
            "upsample_add_fwd", "upsample_add_bwd", "pack_block_weights", "dropout_inplace"]


def profile_families_graph(work):
    """Per-call device times of ONE stage INSIDE a CUDA graph: the instrumented step is captured with `external` CUDA events
    (event-record nodes) around every C-ABI call and replayed; the events bracket the kernels exactly as a graph-launched step
    runs them (no host launch latency).  The side streams are switched off for this capture, so every call is timed as an
    isolated launch (an event between two kernels forces a drain): per-family times are conservative and the roofline of a
    family is taken against the BURST peak.  Returns {family: {launch_calls, ms, flops, bytes}} or None."""
    from deepsense6g_tii_b200 import _capi
    import deepsense6g_tii_b200.functional as Fn
    try:
        torch.cuda.Event(enable_timing=True, external=True)
    except TypeError:
        return None
    rec, orig = [], {}
    for n in FAMILIES:
        if not hasattr(_capi, n):
            continue
        f = getattr(_capi, n)
        orig[n] = f

        def wrap(*a, _f=f, _n=n, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True, external=True), torch.cuda.Event(enable_timing=True, external=True)
            e0.record()
            _f(*a, **k)
            e1.record()
            flops = nbytes = 0.0
            if _n == "gemm_bf16_nt":      # a (M,K) bf16, w (N,K) bf16, out (M,N) bf16|fp32 [+ fp32 residual]
                m, kk, nn_ = a[0].shape[0], a[0].shape[1], a[1].shape[0]
                flops = 2.0 * m * nn_ * kk
                nbytes = 2.0 * (m * kk + nn_ * kk) + m * nn_ * a[2].element_size() + (4.0 * m * nn_ if k.get("residual") is not None else 0.0) \
                    + (2.0 * m * nn_ if k.get("relu_src") is not None else 0.0)
            elif _n == "gemm_bf16_tn":    # dy (M,N) bf16, x (M,K) bf16 -> dw (N,K) fp32
                m, nn_, kk = a[0].shape[0], a[0].shape[1], a[1].shape[1]
                flops = 2.0 * m * nn_ * kk
                nbytes = 2.0 * (m * nn_ + m * kk) + 4.0 * nn_ * kk
            rec.append((_n, e0, e1, flops, nbytes))
        setattr(_capi, n, wrap)
    old_env = os.environ.get("DSF_WGRAD_STREAM")
    os.environ["DSF_WGRAD_STREAM"] = "0"
    runs = []
    try:
        Fn.K = _capi
        work.step()
        torch.cuda.synchronize()
        del rec[:]
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            work.step()
        for _ in range(4):
            g.replay()
            torch.cuda.synchronize()
            runs.append([e0.elapsed_time(e1) for _, e0, e1, _, _ in rec])
        runs = runs[1:]
    except Exception as ex:  # keep the bench line alive
        sys.stderr.write("bench.py: graph-instrumented profile failed (%s)\n" % ex)
        return None
    finally:
        for n, f in orig.items():
            setattr(_capi, n, f)
        if old_env is None:
            os.environ.pop("DSF_WGRAD_STREAM", None)
        else:
            os.environ["DSF_WGRAD_STREAM"] = old_env
    fam = {}
    for i, (n, _, _, flops, nbytes) in enumerate(rec):
        d = fam.setdefault(n, {"launch_calls": 0, "ms": 0.0, "flops": 0.0, "bytes": 0.0})
        d["launch_calls"] += 1
        d["ms"] += statistics.median(r[i] for r in runs)
        d["flops"] += flops
        d["bytes"] += nbytes
    c, t = work.c, n_tokens()
    m = BATCH * t
    e_t, e_f, F = m * c, 3 * BATCH * S * c * (A * work.scale) ** 2, 4 * c
    per_block_w = 4 * c * c + 2 * F * c
    # algorithmic work of the non-GEMM families (DESIGN.md §3; elements x dtype size, each operand read / written once)
    extra = {
        "attn_fwd": (L * 4.0 * t * t * c * BATCH, L * (m * 3 * c * 2 + e_t * 2)),
        "attn_bwd": (L * 8.0 * t * t * c * BATCH, L * (m * 3 * c * 2 * 2 + e_t * 2 * 2)),                 # recompute not counted
        "tokens_fwd": (0, e_f * 4 + e_t * 4 + t * c * 4),
        "tokens_bwd": (0, e_t * 4 + 2 * e_f * 4 + t * c * 4),
        "layernorm_fwd": (0, (2 * L) * e_t * (4 + 2) + e_t * (4 + 4)),
        "layernorm_bwd": (0, (2 * L) * e_t * (2 + 4 + 4 + 4 + 2) + e_t * (4 + 4 + 4 + 2)),
        "colsum": (0, L * m * (F + 3 * c) * 2),
        "pack_block_weights": (0, L * per_block_w * (4 + 2 * 2)),
        "upsample_add_fwd": (0, e_t * 4 + 2 * e_f * 4),
        "upsample_add_bwd": (0, e_f * 4 + e_t * 4),
    }
    for k, (fl, by) in extra.items():
        if k in fam:
            fam[k]["flops"], fam[k]["bytes"] = float(fl), float(by)
    return fam


def family_rooflines(fam, pk):
    """Per family: achieved TFLOP/s and GB/s of the algorithmic work, and the fraction of min(TC, HBM) — roof time =
    max(flops / burst bf16 peak, bytes / HBM copy peak) over the measured time (SURVEY §8d: stage 1-2 GEMMs sit below the ridge)."""
    out = {}
    for k, d in fam.items():
        ms = d["ms"]
        if ms <= 0:
            continue
        t_tc = d["flops"] / (pk["tc_burst"] * 1e12) * 1e3
        t_hbm = d["bytes"] / (pk["hbm"] * 1e9) * 1e3
        out[k] = {"ms": round(ms, 4), "calls": d["launch_calls"],
                  "tflops": round(d["flops"] / (ms * 1e-3) / 1e12, 1) if d["flops"] else None,
                  "gbps": round(d["bytes"] / (ms * 1e-3) / 1e9, 1) if d["bytes"] else None,
                  "bound": "tensor" if t_tc >= t_hbm else "hbm", "roof_ms": round(max(t_tc, t_hbm), 4),
                  "frac_of_roof": round(max(t_tc, t_hbm) / ms, 3)}
    return out


def check_grads_synced(works, world, dist):
    """N > 1: the replayed / eager steps really exchanged gradients — every rank holds the same averaged gradient for a sample of
    parameters of the first and the last stage (ranks see different data, so un-reduced gradients would differ).  Returns
    (all identical, names that are not)."""
    if world <= 1:
        return None, []
    bad = []
    for w in (works[0], works[-1]):
        blk = w.gpt.blocks
        named = {"pos_emb": w.gpt.pos_emb, "ln_f.weight": w.gpt.ln_f.weight, "blocks.0.mlp.0.weight": blk[0].mlp[0].weight,
                 "blocks.0.attn.query.bias": blk[0].attn.query.bias, "blocks.%d.attn.proj.weight" % (len(blk) - 1): blk[len(blk) - 1].attn.proj.weight,
                 "blocks.%d.mlp.2.bias" % (len(blk) - 1): blk[len(blk) - 1].mlp[2].bias}
        for n, t in named.items():
            g = t.grad.detach().reshape(-1)[:4096].contiguous()
            gs = [torch.empty_like(g) for _ in range(world)]
            dist.all_gather(gs, g)
            ok = all(torch.equal(gs[0], x) for x in gs[1:]) and bool(torch.isfinite(g).all()) and float(g.abs().sum()) > 0
            if not ok:
                bad.append("C%d.%s (max |diff| %.3e, |g| %.3e)" % (w.c, n, max(float((gs[0] - x).abs().max()) for x in gs[1:]), float(g.abs().max())))
    return len(bad) == 0, bad


def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    from deepsense6g_tii_b200 import _capi
    from deepsense6g_tii_b200 import dist as D
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    _capi.check_device()
    _capi.set_pdl(args.pdl)
    _capi.set_sm_margin(int(os.environ.get("DSF_SM_MARGIN", "0")) if world > 1 else 0)
    gen = torch.Generator().manual_seed(rank)  # data generator seed 0 + rank
    works = [StageWork(c, scale, dev, gen, optimizer=args.optimizer) for c, scale in SPEC]
    n_params = sum(p.numel() for w in works for p in w.gpt.parameters())
    reducer = None
    if world > 1:
        # gradients are averaged bucket-by-bucket (one bucket per transformer block) while the backward is still running; ONE
        # reducer serves all stages and the stream only waits for the outstanding collectives at the end of the step, so a
        # stage's last all-reduce runs behind the next stage's kernels (DSF_DEFER_REDUCE=0: wait at the end of every stage)
        reducer = D.OverlappedGradReducer(defer=os.environ.get("DSF_DEFER_REDUCE", "1") == "1")
        for w in works:
            D.broadcast_params(w.gpt.parameters())   # same initial weights on every rank
            w.gpt.set_grad_reducer(reducer)

    def step_eager():
        out = one_step(works)
        if reducer is not None:
            reducer.wait_all()
        return out

    loss_h = torch.empty((), pin_memory=True)
    graph, graph_loss, graph_launches, graph_note = None, None, 0, "eager launches"
    pdl_note = ", programmatic dependent launch " + ("on" if args.pdl else "off")
    # (N > 1: the bucketed NCCL all-reduces issued from inside the backward are captured too; DSF_GRAPH_DDP=0 opts out)
    if args.graph and (world == 1 or os.environ.get("DSF_GRAPH_DDP", "1") == "1"):
        try:
            graph, graph_loss, graph_launches = capture_step(step_eager)
            graph_note = "whole step captured in one CUDA graph (%d dsfuse kernels per replay)" % graph_launches
        except Exception as ex:  # e.g. a collective that cannot be captured: keep the bench line alive with eager launches
            sys.stderr.write("bench.py: CUDA-graph capture failed on rank %d (%s); falling back to eager launches\n" % (rank, ex))
            graph, graph_note = None, "eager launches (graph capture failed: %s)" % type(ex).__name__
        torch.cuda.synchronize()
        if world > 1:  # all ranks must agree: one eager rank next to replaying ranks would dead-lock the collectives
            ok = torch.tensor([1 if graph is not None else 0], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok.item()) == 0:
                graph, graph_note = None, "eager launches (graph capture failed on some rank)"

    def step_resident():
        if graph is not None:
            graph.replay()
        else:
            step_eager()

    # e2e pipeline: every step copies ONE batch of inputs (all stages' feature maps + GPS embeddings) pinned-host -> device and
    # reads the loss back.  The copy of step k+1's batch runs on a copy stream into a double-buffered staging area while step k
    # computes (what a training data loader with pinned-memory prefetch does); the compute stream then moves the staged batch
    # into the step's input tensors (device-to-device) and runs the step.
    copy_stream = torch.cuda.Stream()
    host_in = [t for w in works for t in w.feats_h + [w.gps_h]]
    dev_in = [t for w in works for t in w.feats + [w.gps]]
    stage = [[torch.empty_like(t, device=dev) for t in host_in] for _ in range(2)]
    ev_ready = [torch.cuda.Event() for _ in range(2)]  # batch landed in stage[i]
    ev_free = [torch.cuda.Event() for _ in range(2)]   # the compute stream has consumed stage[i]
    e2e_k = [0, False]

    def prefetch(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev_free[i])
            for d, h in zip(stage[i], host_in):
                d.copy_(h, non_blocking=True)
            ev_ready[i].record(copy_stream)

    def step_e2e():
        i = e2e_k[0] & 1
        if not e2e_k[1]:  # prime the pipeline (first warm-up step only)
            prefetch(i)
            e2e_k[1] = True
        cur = torch.cuda.current_stream()
        cur.wait_event(ev_ready[i])
        with torch.no_grad():
            for d, st_ in zip(dev_in, stage[i]):
                d.copy_(st_, non_blocking=True)
        ev_free[i].record(cur)
        prefetch(i ^ 1)  # next step's batch: overlaps this step's compute
        e2e_k[0] += 1
        if graph is not None:
            graph.replay()
            loss_h.copy_(graph_loss, non_blocking=True)
        else:
            loss_h.copy_(step_eager(), non_blocking=True)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, sampler=None, finalize=None):
        for _ in range(warmup):
            fn()
        barrier()
        if sampler:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = _capi.launch_count()
        ncu_range = sampler is not None and os.environ.get("DSF_NCU_RANGE") == "1"
        if ncu_range:  # `ncu --profile-from-start off` then captures exactly the timed region
            torch.cuda.profiler.start()
        e0.record()
        for _ in range(steps):
            fn()
        if finalize is not None:
            finalize()
        e1.record()
        if ncu_range:
            torch.cuda.profiler.stop()
        barrier()
        clocks = sampler.stop() if sampler else None
        ms = e0.elapsed_time(e1)
        n1 = _capi.launch_count() + (graph_launches * steps if graph is not None else 0)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, n1 - n0, clocks

    steps, warmup = args.steps, max(3, args.warmup)
    ms, launches, clocks = timed(step_resident, steps, warmup, ClockSampler(local_rank) if rank == 0 else None)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, [nt for w in works for nt in w.computed()])
    value = BATCH * world * steps / (ms * 1e-3)
    if args.quick:
        synced, sync_bad = check_grads_synced(works, world, dist)
        if rank == 0:
            print(json.dumps({"quick": True, "ms_per_step": ms / steps, "value": value, "gpu_launches": launches,
                              "grads_identical_across_ranks": synced, "not_identical": sync_bad}))
        return
    # the K-th prefetch issued inside the region must also complete inside it: K steps <-> K host-to-device batch copies
    ms_e2e, _, _ = timed(step_e2e, steps, 2, finalize=lambda: torch.cuda.current_stream().wait_event(ev_ready[e2e_k[0] & 1]))
    e2e_value = BATCH * world * steps / (ms_e2e * 1e-3)
    # sustained behaviour: the same step replayed back to back for >= 2 s (clocks drop under sustained tensor load)
    sustained = None
    if args.sustained > 0:
        n_s = max(steps, int(args.sustained * 1e3 / (ms / steps)))
        smp = ClockSampler(local_rank) if rank == 0 else None
        ms_s, _, clk_s = timed(step_resident, n_s, 1, smp)
        sustained = {"seconds": round(ms_s * 1e-3, 2), "steps": n_s, "ms_per_step": ms_s / n_s, "value": BATCH * world * n_s / (ms_s * 1e-3), "clocks": clk_s}

    synced, sync_bad = check_grads_synced(works, world, dist)
    if rank != 0:
        return
    pk = peaks()
    for w in works:
        w.gpt.set_grad_reducer(None)  # everything below runs on rank 0 only: no collectives in it
    # ---- per stage: graph-replayed time of the stage alone + instrumented per-family times
    stages = {}
    for w in works:
        rec = {"n_embd": w.c, "feature_map": A * w.scale, "flops_per_step": 3.0 * fwd_flops_per_sample(w.c) * BATCH}
        try:
            g_s, _, n_s = capture_step(w.step, warm=1)
            for _ in range(3):
                g_s.replay()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(steps):
                g_s.replay()
            e1.record()
            torch.cuda.synchronize()
            rec["ms_per_step"] = e0.elapsed_time(e1) / steps
            rec["samples_per_s"] = BATCH / (rec["ms_per_step"] * 1e-3)
            rec["tflops"] = rec["flops_per_step"] / (rec["ms_per_step"] * 1e-3) / 1e12
            rec["dsfuse_launches"] = n_s
            del g_s
        except Exception as ex:
            sys.stderr.write("bench.py: per-stage graph of C=%d failed (%s)\n" % (w.c, ex))
        fam = profile_families_graph(w)
        if fam:
            fr = family_rooflines(fam, pk)
            rec["families"] = fr
            rec["sum_family_ms"] = round(sum(d["ms"] for d in fr.values()), 4)
            rec["roof_ms"] = round(sum(d["roof_ms"] for d in fr.values()), 4)
            if "ms_per_step" in rec:
                rec["frac_of_roof"] = round(rec["roof_ms"] / rec["ms_per_step"], 3)   # min(TC, HBM) roof of the stage / its measured time
        stages["C%d" % w.c] = rec
    # ---- headline roofline: the dominant tensor-core family of the whole workload
    tot = {}
    for rec in stages.values():
        for k, d in rec.get("families", {}).items():
            t = tot.setdefault(k, {"ms": 0.0, "calls": 0, "flops": 0.0, "bytes": 0.0})
            t["ms"] += d["ms"]; t["calls"] += d["calls"]
            t["flops"] += (d["tflops"] or 0.0) * 1e12 * d["ms"] * 1e-3
            t["bytes"] += (d["gbps"] or 0.0) * 1e9 * d["ms"] * 1e-3
    roofline = None
    if tot:
        total_ms = sum(d["ms"] for d in tot.values())
        tcf = {k: d for k, d in tot.items() if d["flops"] > 0}
        dom = max(tcf, key=lambda k: tcf[k]["ms"])
        achieved = tcf[dom]["flops"] / (tcf[dom]["ms"] * 1e-3) / 1e12
        traffic, traffic_src = None, None
        import glob
        for tp in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")), reverse=True):
            tj = json.load(open(tp))
            if tj.get("family", "gemm_bf16_nt") == dom:
                traffic, traffic_src = tj["avg_dram_bytes_per_launch"], tj["source"]
                break
        roofline = {"bound": "tensor", "kernel": dom, "achieved": achieved, "peak": pk["tc_burst"], "unit": "TFLOP/s", "frac": achieved / pk["tc_burst"],
                    "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": pk["src"] + " bf16_tflops (burst: every family is timed as isolated launches)",
                    "launches_per_step": tcf[dom]["calls"], "avg_launch_ms": tcf[dom]["ms"] / tcf[dom]["calls"], "share_of_step": tcf[dom]["ms"] / total_ms,
                    "timing": "external CUDA events captured around every kernel of a graph-replayed step, stage by stage (median of 3 replays, side streams off)",
                    "families": {k: {"ms": round(d["ms"], 4), "calls": d["calls"], "tflops": round(d["flops"] / (d["ms"] * 1e-3) / 1e12, 1) if d["flops"] else None,
                                     "gbps": round(d["bytes"] / (d["ms"] * 1e-3) / 1e9, 1) if d["bytes"] else None} for k, d in tot.items()},
                    "hbm_peak_gbps": pk["hbm"], "tc_peak_sustained": pk["tc_sust"]}
    # ---- baselines
    gpu_base = None
    if args.gpu_baseline:
        try:
            gstep, gkind = reference_step_fn(dev, BATCH, autocast=True)
            for _ in range(2):
                gstep()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(5):
                gstep()
            e1.record()
            torch.cuda.synchronize()
            gms = e0.elapsed_time(e1) / 5
            gpu_base = {"value": BATCH / (gms * 1e-3), "unit": "samples/s", "ms_per_step": gms, "kind": gkind,
                        "what": "stock PyTorch eager, torch.autocast(bf16), same workload and batch on the same GPU (cuBLAS / ATen kernels; 2 warm-up + 5 timed steps)"}
            del gstep
            torch.cuda.empty_cache()
        except Exception as ex:
            sys.stderr.write("bench.py: gpu_baseline skipped (%s)\n" % ex)
    cpu_v, cpu_ms, cpu_kind = time_cpu(2, 1)
    cores = torch.get_num_threads()
    h2d = sum(t.numel() * t.element_size() for t in host_in)
    step_flops = sum(3.0 * fwd_flops_per_sample(c) * BATCH for c, _ in SPEC)
    cfg = workload_config(world)
    cfg.update({"launch": graph_note + pdl_note, "dropout": PDROP, "gpt_parameters": n_params,
                "optimizer": "fused AdamW + EMA + bf16 weight repack in the step (dsf_adamw_ema_pack, one launch per stage; no pack launches in the forward)"
                if args.optimizer else "none (fwd+bwd only; bf16 weight shadows re-packed at the start of every forward)",
                "l2": "per-step working set (saved activations of 8 blocks per stage, > 1 GB) > 126 MB L2; no explicit flush",
                "grad_allreduce": ("NCCL all-reduce (avg) of %.1f M fp32 grads per step, one bucket per transformer block, overlapped with backward" % (n_params / 1e6)) if world > 1 else "none (1 GPU)",
                "grads_identical_across_ranks": synced, "grads_not_identical": sync_bad or None})
    out = {
        "metric": "train samples/sec (fwd+bwd)", "value": value, "unit": "samples/s", "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": cfg, "path_tflops": step_flops * world / (ms / steps * 1e-3) / 1e12,
        "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / steps,
                "pipeline": "one pinned-host -> device batch copy per step on a copy stream (double-buffered), overlapped with the previous step's compute; loss read back every step"},
        "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "stages": stages,
        "stage4": stages.get("C512"), "sustained": sustained, "gpu_baseline": gpu_base,
        "cpu_baseline": {"value": cpu_v, "unit": "samples/s", "cores": cores, "kind": cpu_kind, "sample": cpu_sample_note(cpu_kind, cores, 2, 1)},
    }
    if "C512" in stages and len(SPEC) > 1:
        out["stage4"] = dict(stages["C512"], note="BASELINE.json configs[1] (the n_embd 512 stage alone), same run")
        out["stage4"].pop("families", None)
    print(json.dumps(out))


# ----------------------------------------------------------------------------------------- full-model workload (configs[2])
def run_model(args, rank, world, local_rank):
    """BASELINE.json configs[2]: full model2_seq training step — drop-in TransFuser (ResNet trunks + 4 fusion stages on
    the dsfuse kernels + join MLP), bf16, batch 12 per GPU, seq_len 5, 256x256 inputs, dropout 0.1 (config_seq.py:39-41),
    focal loss + fused AdamW + EMA, synthetic data; N > 1: DistributedDataParallel over NCCL (batch-sharded)."""
    import types
    import torch.distributed as dist
    from deepsense6g_tii_b200 import TransFuser, _capi
    from deepsense6g_tii_b200.train import EMA, FocalLoss, synthetic_batch, train_step
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    _capi.check_device()
    _capi.set_pdl(args.pdl)
    torch.backends.cudnn.benchmark = True  # as the reference (train2_seq.py:16)
    cfg = types.SimpleNamespace(seq_len=S, pred_len=4, n_views=1, vert_anchors=A, horz_anchors=A, n_embd=512, block_exp=4, n_layer=L,
                                n_head=NH, embd_pdrop=0.1, attn_pdrop=0.1, resid_pdrop=0.1, add_velocity=1, fusion_dtype=torch.bfloat16)
    torch.manual_seed(100)
    model = TransFuser(cfg, dev).to(memory_format=torch.channels_last).train()
    net = model
    enc = model.encoder
    gpts = [enc.transformer1, enc.transformer2, enc.transformer3, enc.transformer4]
    grad_sync, ddp_note = None, "none (1 GPU)"
    if world > 1:
        from deepsense6g_tii_b200 import dist as D
        D.broadcast_params(model.parameters())
        for b_ in model.buffers():   # BatchNorm statistics start equal on every rank, then stay per replica (as under nn.DataParallel)
            dist.broadcast(b_, 0)
        if args.ddp:   # stock DistributedDataParallel: its reducer hooks cannot be captured -> eager launches
            net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local_rank], gradient_as_bucket_view=True)
            ddp_note = "torch DistributedDataParallel (NCCL, bucketed, overlapped) of %.1f M fp32 gradients; eager launches"
        else:
            grad_sync = D.DataParallelGrads(model, gpts)
            ddp_note = ("dist.DataParallelGrads: GPT gradients all-reduced per transformer block inside the backward, the other "
                        "parameters through one flat fp32 bucket after it (%.1f M gradients in total), all inside the captured CUDA graph")
    crit = FocalLoss()
    use_graph = args.graph and (world == 1 or not args.ddp)
    ema = EMA(model, 0.999)
    ema.register()
    if args.torch_optimizer:
        opt = torch.optim.AdamW(model.parameters(), lr=1e-4, fused=True, capturable=use_graph)
        opt_note = "torch.optim.AdamW(fused, capturable) + multi-tensor EMA lerp"
    else:   # AdamW + EMA + the bf16 repack of the four GPTs' weights in one dsfuse launch (train2_seq.py:131-134, 315-320, 539)
        from deepsense6g_tii_b200.optim import FusedAdamWEMA
        opt = FusedAdamWEMA(model.parameters(), lr=1e-4, ema=ema, gpts=gpts)
        opt_note = "dsf_adamw_ema_pack: AdamW + EMA + bf16 weight repack of the 4 GPTs in one launch"
    gen = torch.Generator().manual_seed(rank)
    host = synthetic_batch(BATCH, S, 256, generator=gen, pin=True)

    def to_dev(b, stream=None):
        imgs, lids, rads, gps, soft, beam = b
        mv = lambda t: t.to(dev, non_blocking=True)
        return ([mv(t).contiguous(memory_format=torch.channels_last) for t in imgs], [mv(t) for t in lids], [mv(t) for t in rads],
                mv(gps), mv(soft), mv(beam))

    resident = to_dev(host)
    loss_h = torch.empty((), pin_memory=True)

    def step_eager(b=None):
        return train_step(net, resident if b is None else b, crit, opt, ema, autocast_dtype=torch.bfloat16, grad_sync=grad_sync)

    # N = 1: the whole training step (trunks, 4 fusion stages with graph-safe dropout, loss, backward, capturable fused
    # AdamW, multi-tensor EMA) is captured in one CUDA graph on static input tensors and replayed.
    graph, graph_loss, launch_note, graph_launches = None, None, "eager launches", 0
    if use_graph:
        try:
            graph, graph_loss, graph_launches = capture_step(step_eager)
            launch_note = "whole training step captured in one CUDA graph (%d dsfuse kernels per replay)" % graph_launches
        except Exception as ex:
            sys.stderr.write("bench.py: CUDA-graph capture of the model step failed (%s); eager launches\n" % ex)
            graph = None
        torch.cuda.synchronize()

    last_loss = [graph_loss]   # the loss of the last resident step (--dump-outputs)

    def step_resident():
        if graph is not None:
            graph.replay()
            return graph_loss
        last_loss[0] = step_eager().detach()
        return last_loss[0]

    # e2e: one pinned-host -> device batch copy (94 MB) per step into preallocated, double-buffered staging tensors on a
    # copy stream, overlapped with the previous step's compute; the step then reads the staged batch (graph mode: after a
    # device-to-device move into the graph's static input tensors)
    copy_stream = torch.cuda.Stream()
    flat = lambda b: list(b[0]) + list(b[1]) + list(b[2]) + list(b[3:5])
    host_flat = flat(host)
    stage = [[torch.empty_like(t, device=dev) for t in host_flat] for _ in range(2)]
    ev_ready = [torch.cuda.Event() for _ in range(2)]
    ev_free = [torch.cuda.Event() for _ in range(2)]
    e2e_k = [0, False]

    def unflat(ts):
        return ts[0:S], ts[S:2 * S], ts[2 * S:3 * S], ts[3 * S], ts[3 * S + 1], None

    def prefetch(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev_free[i])
            for d, h in zip(stage[i], host_flat):
                d.copy_(h, non_blocking=True)
            ev_ready[i].record(copy_stream)

    def step_e2e():
        i = e2e_k[0] & 1
        if not e2e_k[1]:
            prefetch(i)
            e2e_k[1] = True
        cur = torch.cuda.current_stream()
        cur.wait_event(ev_ready[i])
        if graph is not None:
            with torch.no_grad():
                for dst, src in zip(flat(resident), stage[i]):
                    dst.copy_(src, non_blocking=True)
            ev_free[i].record(cur)
            prefetch(i ^ 1)
            graph.replay()
            loss_h.copy_(graph_loss.detach(), non_blocking=True)
        else:
            prefetch(i ^ 1)
            loss_h.copy_(step_eager(unflat(stage[i])).detach(), non_blocking=True)
            ev_free[i].record(cur)
        e2e_k[0] += 1

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, finalize=None):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = _capi.launch_count()
        e0.record()
        for _ in range(steps):
            fn()
        if finalize is not None:
            finalize()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, (_capi.launch_count() - n0) + (graph_launches * steps if graph is not None else 0)

    steps, warmup = args.steps, max(3, args.warmup)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    ms, launches = timed(step_resident, steps, warmup)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:   # what a caller of train_step holds afterwards: the loss, the updated parameters, the gradients
        params = list(model.named_parameters())
        dump_outputs(args.dump_outputs, [("loss", last_loss[0])] + [("param." + n, p) for n, p in params] +
                     [("grad." + n, p.grad) for n, p in params if p.grad is not None])
    ms_e2e, _ = timed(step_e2e, steps, 2, finalize=lambda: torch.cuda.current_stream().wait_event(ev_ready[e2e_k[0] & 1]))
    loss_val = float(loss_h)
    params_synced = None
    if world > 1:   # same start + averaged gradients every step -> the replicas' parameters stay identical
        params_synced, not_synced = True, []
        for n, t in (("join.0.weight", model.join[0].weight), ("image conv1.weight", enc.image_encoder.features.conv1.weight),
                     ("transformer4.blocks.0.mlp.0.weight", enc.transformer4.blocks[0].mlp[0].weight), ("transformer1.pos_emb", enc.transformer1.pos_emb),
                     ("transformer2.ln_f.weight", enc.transformer2.ln_f.weight), ("vel_emb1.weight", enc.vel_emb1.weight),
                     ("lidar bn1.weight", enc.lidar_encoder._model.bn1.weight)):
            v = t.detach().reshape(-1)[:4096].float().contiguous()
            vs = [torch.empty_like(v) for _ in range(world)]
            dist.all_gather(vs, v)
            ok = all(torch.equal(vs[0], x) for x in vs[1:]) and bool(torch.isfinite(v).all())
            if not ok:
                not_synced.append("%s (max |diff| %.3e)" % (n, max(float((vs[0] - x).abs().max()) for x in vs[1:])))
            params_synced = params_synced and ok
    if rank != 0:
        return
    h2d = sum(t.numel() * t.element_size() for t in host[0] + host[1] + host[2]) + sum(t.numel() * t.element_size() for t in host[3:])
    n_params = sum(p.numel() for p in model.parameters())
    print(json.dumps({
        "metric": "train samples/sec (fwd+bwd)", "value": BATCH * world * steps / (ms * 1e-3), "unit": "samples/s", "n_gpus": world,
        "steps": steps, "warmup": warmup, "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "full model2_seq TransFuser training step: fwd + focal loss + bwd + fused AdamW + EMA, batch 12/GPU, seq_len 5, "
                               "256x256 inputs, dropout 0.1, %d parameters, ResNet trunks in stock PyTorch (channels_last, bf16 autocast), "
                               "4 fusion stages on dsfuse kernels" % n_params,
                   "global_batch": BATCH * world, "seq_len": S, "parallelism": "dp%d" % world, "launch": launch_note + ", PDL " + ("on" if args.pdl else "off"),
                   "optimizer": opt_note,
                   "l2": "per-step working set (activations of 3 ResNets + 4 fusion stages) >> 126 MB L2; no explicit flush",
                   "grad_allreduce": (ddp_note % (n_params / 1e6)) if world > 1 else ddp_note,
                   "params_identical_across_ranks": params_synced, "params_not_identical": (not_synced or None) if world > 1 else None},
        "e2e": {"value": BATCH * world * steps / (ms_e2e * 1e-3), "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / steps, "pipeline": "next batch copied pinned-host -> device on a copy stream during the current step"},
        "gpu_launches": launches, "clocks": clocks, "final_loss": loss_val,
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-graph", dest="graph", action="store_false", help="launch every kernel eagerly instead of replaying a CUDA graph")
    ap.add_argument("--workload", default="fusion4", choices=["fusion4", "stage4", "stage", "model"],
                    help="fusion4 = the four fusion stages back to back (default: the whole hot path); stage4 = BASELINE.json configs[1], the "
                         "n_embd 512 stage alone ('stage' is an alias); model = configs[2], the full training step")
    ap.add_argument("--stage", type=int, default=0, choices=[0, 1, 2, 3, 4], help="bench ONE fusion stage (1-4) alone")
    ap.add_argument("--quick", action="store_true", help="profiling runs: skip the e2e leg, the instrumented steps and the baselines")
    ap.add_argument("--no-pdl", dest="pdl", action="store_false", help="disable programmatic dependent launch of the hot kernels")
    ap.add_argument("--no-gpu-baseline", dest="gpu_baseline", action="store_false", help="skip the stock-PyTorch-autocast leg on the GPU")
    ap.add_argument("--sustained", type=float, default=2.0, help="seconds of back-to-back replays for the `sustained` sub-record (0 = skip)")
    ap.add_argument("--optimizer", action="store_true", help="stage workloads: add the fused AdamW + EMA + weight-repack launch to every step")
    ap.add_argument("--ddp", action="store_true", help="model workload, N > 1: stock DistributedDataParallel (eager launches) instead of dist.DataParallelGrads")
    ap.add_argument("--torch-optimizer", action="store_true", help="model workload: stock torch AdamW(fused) + multi-tensor EMA instead of dsf_adamw_ema_pack")
    ap.add_argument("--dropout", type=float, default=0.0,
                    help="embd/attn/resid dropout probability (default 0 = the parity configuration; the reference trains with 0.1)")
    ap.add_argument("--anchors", type=int, default=8, choices=[8, 16],
                    help="16 = BASELINE.json configs[4], the scaled fusion path: 512x512 inputs, 16x16 anchors -> T = 3842 tokens")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32, 64 MB in all; a larger "
                         "tensor is stored as a fixed, seeded sample of its elements): per stage the outputs and the gradients of the "
                         "inputs and parameters; --workload model: the loss, the updated parameters and their gradients")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU arm computed; --impl reference has no such outputs")
    global PDROP, A, SPEC
    PDROP = args.dropout
    A = args.anchors
    if args.stage:
        SPEC = (STAGES4[args.stage - 1],)
    elif args.workload in ("stage4", "stage"):
        SPEC = (STAGES4[3],)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the fusion stage has no CPU path (use --impl reference for the CPU baseline)")
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        if args.workload == "model":
            run_model(args, rank, world, local_rank)
        else:
            run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()

"""Shared helpers of the GPU parity tests and of tests/tools/diag_bf16_error.py: one fusion-stage problem evaluated by
the dsfuse kernels (through the C ABI) and by the oracle restatement (oracle/fusion_ref.py) in float64 on the same
device, with per-tensor relative L2 errors.

ReLU decisions.  The gradient of the stage is discontinuous where an mlp.0 pre-activation crosses 0 (nn.ReLU,
model2_seq.py:123).  Any evaluation that rounds an operand of mlp.0 lands a few pre-activations with |z| below its rounding
error on the other side: in bf16 about 0.2-0.3 % of the active units flip, each flipped unit is a 100 % error of dL/dz
there, and the relative error of the mlp.0 / ln2 gradients is sqrt(flip fraction) = 4-5e-2 for ANY bf16 evaluation (stock
torch.autocast included; tests/tools/bf16_error_model.py reproduces it on the CPU with nothing but round-to-bf16 inserted
into float64 math).  The oracle can therefore be evaluated a second time WITH the decisions the kernels took
(``relu.{i}`` masks of oracle.fusion_ref.block): against that reference only rounding proper is left, and every gradient
tensor has to meet north_star's 2e-2.
"""
import torch

from oracle import fusion_ref as R

S, NH = 5, 4


def make_problem(B, C, H, L, A, dev, seed=None, wscale=0.01, V=1, A_w=None, W=None, feat_dtype=torch.float32,
                 channels_last=False):
    """One fusion-stage problem: B samples of S frames, V camera views, an A x A_w anchor grid (A_w defaults to A) on H x W
    feature maps (W defaults to H).  ``feat_dtype`` / ``channels_last`` (a bool, or one per map: image, lidar, radar) give the
    dtype and memory format the maps are handed to the kernels in; bf16 maps are rounded once here, so the kernels and the
    float64 oracle see identical values.  The defaults draw the same random numbers as before V / A_w / W existed."""
    A_w = A if A_w is None else A_w
    W = H if W is None else W
    T = (V + 2) * S * A * A_w + 2
    gen = torch.Generator().manual_seed(100 + C if seed is None else seed)
    p0 = R.init_gpt_params(C, NH, 4, L, T, generator=gen, pos_std=0.02)
    p0 = {k: (v + wscale * torch.randn(v.shape, generator=gen)).to(dev) for k, v in p0.items()}
    feats = [torch.randn(n, C, H, W, generator=gen).to(dev).to(feat_dtype) for n in (B * V * S, B * S, B * S)]
    cl = channels_last if isinstance(channels_last, (tuple, list)) else (channels_last,) * 3
    feats = [f.contiguous(memory_format=torch.channels_last) if c else f for f, c in zip(feats, cl)]
    gps = torch.randn(B, 2, C, generator=gen).to(dev)
    probes = [torch.randn(f.shape, generator=gen).to(dev) for f in feats] + [torch.randn(B, 2, C, generator=gen).to(dev)]
    return dict(B=B, C=C, H=H, W=W, L=L, A=A, A_w=A_w, V=V, T=T, p0=p0, feats=feats, gps=gps, probes=probes)


def leafs(pb, dt=None):
    """Fresh leaf tensors of the problem: in ``dt`` throughout, or (dt None) as the kernels take them: fp32 parameters and GPS
    embedding, the maps in their own dtype and memory format."""
    pdt = torch.float32 if dt is None else dt
    return ({k: v.to(pdt).clone().requires_grad_(True) for k, v in pb["p0"].items()},
            [(f if dt is None else f.to(dt)).clone().requires_grad_(True) for f in pb["feats"]]
            + [pb["gps"].to(pdt).clone().requires_grad_(True)])


def run_oracle(pb, dt=torch.float64, autocast=False, relu_masks=None):
    """The oracle restatement; ``relu_masks``: {"relu.i": (B*T, 4C) tensor} whose sign pattern replaces ReLU's own decisions."""
    p, i = leafs(pb, dt)
    masks = None
    if relu_masks is not None:
        masks = {k: (v > 0).to(dt).view(pb["B"], pb["T"], -1) for k, v in relu_masks.items()}
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
        (a, b, c), g = R.fusion_stage(p, i[:3], i[3], NH, S, pb["A"], pb["A_w"], n_views=pb["V"], masks=masks)
    outs = (a, b, c, g)
    sum((o.to(dt) * pr.to(dt)).sum() for o, pr in zip(outs, pb["probes"])).backward()
    return outs, p, i


def run_dsfuse(pb, mode, capture=None, **cfg_extra):
    from deepsense6g_tii_b200.functional import fusion_stage, param_names
    p, i = leafs(pb)
    cfg = dict(seq_len=S, n_views=pb["V"], vert_anchors=pb["A"], horz_anchors=pb["A_w"], n_head=NH, n_layer=pb["L"],
               compute_dtype=mode)
    if capture is not None:
        cfg["capture"] = capture
    cfg.update(cfg_extra)
    outs = fusion_stage(cfg, i[0], i[1], i[2], i[3], [p[n] for n in param_names(pb["L"])])
    sum((o.float() * pr).sum() for o, pr in zip(outs, pb["probes"])).backward()
    torch.cuda.synchronize()
    return outs, p, i


def rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def errors(res, ref, L):
    """{tensor name: relative L2 error}: out0-3, gin0-3, g/<param>; attn.key.bias (mathematically zero gradient) is reported
    relative to the query-bias gradient of the same block."""
    from deepsense6g_tii_b200.functional import param_names
    d = {}
    for j, (x, y) in enumerate(zip(res[0], ref[0])):
        d["out%d" % j] = rel(x, y)
    for j, (x, y) in enumerate(zip(res[2], ref[2])):
        d["gin%d" % j] = rel(x.grad, y.grad)
    for n in param_names(L):
        if n.endswith("attn.key.bias"):
            qn = float(ref[1][n.replace("key", "query")].grad.double().norm())
            d["g/" + n] = float((res[1][n].grad.double() - ref[1][n].grad.double()).norm()) / (qn + 1e-30)
        else:
            d["g/" + n] = rel(res[1][n].grad, ref[1][n].grad)
    return d


def worst(d, prefix=""):
    k = max((k for k in d if k.startswith(prefix)), key=lambda k: d[k])
    return d[k], k


def flip_fraction(capture, ref_capture_or_masks):
    """Worst-block fraction of the active mlp.0 units whose ReLU decision differs between two evaluations."""
    w = 0.0
    for k, a in capture.items():
        m, r = a > 0, ref_capture_or_masks[k].reshape(a.shape) > 0
        w = max(w, float((m != r).sum()) / max(1.0, float(r.sum())))
    return w


def oracle_relu_decisions(pb, dt=torch.float64):
    """The mlp.0 outputs of the float64 oracle, block by block (no autograd), for ``flip_fraction``."""
    p = {k: v.to(dt) for k, v in pb["p0"].items()}
    with torch.no_grad():
        pooled = [R.anchor_pool(f.to(dt), pb["A"], pb["A_w"]) for f in pb["feats"]]
        x = R.build_tokens(pooled[0], pooled[1], pooled[2], pb["gps"].to(dt), p["pos_emb"], S, pb["V"])
        out = {}
        for i in range(pb["L"]):
            pre = "blocks.%d." % i
            xm = x + R.self_attention(R.layer_norm(x, p[pre + "ln1.weight"], p[pre + "ln1.bias"]), p, pre + "attn.", NH)
            h = R.layer_norm(xm, p[pre + "ln2.weight"], p[pre + "ln2.bias"])
            out["relu.%d" % i] = R.linear(h, p[pre + "mlp.0.weight"], p[pre + "mlp.0.bias"]).reshape(-1, 4 * pb["C"])
            x = R.block(x, p, i, NH)
    return out


def check(got, cap, pb, ref, what):
    """The bf16-mode bar: every gradient within 2e-2 of the oracle evaluated with the kernels' own ReLU decisions, every output
    within 1e-2, at most 5e-3 flipped decisions, and the decision-free gradients within the flip model (module docstring)."""
    L = pb["L"]
    plain = errors(got, ref, L)
    matched = errors(got, run_oracle(pb, relu_masks=cap), L)
    flip = flip_fraction(cap, oracle_relu_decisions(pb))
    # attn.key.bias: mathematically zero gradient (softmax shift invariance); errors() reports its rounding noise relative to the
    # query-bias gradient of the same block
    bad = ["%s %s: %.3e > 2e-2" % (what, k, v) for k, v in matched.items() if v > (5e-2 if k.endswith("key.bias") else 2e-2)]
    assert not bad, bad
    w_out = worst(plain, "out")
    assert w_out[0] <= 1e-2, (what, w_out)
    # decision-free comparison: bf16 rounding of the mlp.0 operands flips 1-4e-3 of the active units (CPU model: 1.6e-3 at
    # C = 128); a flipped unit is a 100 % error of dL/dz, so no bf16 evaluation gets below sqrt(flip) on mlp.0 / ln2
    assert flip <= 5e-3, (what, "flipped ReLU decisions", flip)
    w_plain = worst({k: v for k, v in plain.items() if k[0] == "g" and not k.endswith("key.bias")})
    assert w_plain[0] <= 2e-2 + 1.25 * flip ** 0.5, (what, w_plain, flip)
    return plain, matched, flip

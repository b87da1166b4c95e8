"""CPU restatement of the reference's GPT fusion stage in plain PyTorch fp32.

TEST INFRASTRUCTURE ONLY — never imported by the product package.  Each function cites the
reference lines it restates (paths are into ``/root/reference``).  The restatement is *pinned* two
ways (see ``tests/test_oracle.py``):

  * in the authoring container against the reference's own classes imported by
    ``oracle/ref_import.py`` (skipped where ``/root/reference`` is absent), and
  * everywhere against the committed golden vectors ``tests/golden/*.npz`` that
    ``oracle/make_golden.py`` produced *from the reference classes*.

The reference ships no tests/golden vectors of its own for this path (SURVEY.md §4, §8c), so
"pinned" here means "pinned to outputs of the reference code executed with this image's torch".

Parameters are passed as a flat ``dict`` whose keys are the reference ``GPT.state_dict()`` names
(``pos_emb``, ``blocks.{i}.ln1.weight`` ... ``ln_f.bias``).
"""
import math
from typing import Dict, Sequence, Tuple

import torch

Tensor = torch.Tensor
LN_EPS = 1e-5  # nn.LayerNorm default, model2_seq.py:118-119,199


# ----------------------------------------------------------------------------- pooling / tokens
def anchor_pool(feat: Tensor, va: int, ha: int) -> Tensor:
    """``nn.AdaptiveAvgPool2d((va, ha))`` (model2_seq.py:414, used :515-517 etc.).

    Restated with the adaptive-window definition: output cell (i, j) averages rows
    ``floor(i*H/va) .. ceil((i+1)*H/va)-1`` (same for columns).  For H divisible by va this is the
    plain mean over an (H/va)x(W/ha) window; at stage 4 (H == va) it is the identity.
    """
    n, c, h, w = feat.shape
    out = feat.new_empty(n, c, va, ha)
    for i in range(va):
        y0, y1 = (i * h) // va, -((-(i + 1) * h) // va)
        for j in range(ha):
            x0, x1 = (j * w) // ha, -((-(j + 1) * w) // ha)
            out[:, :, i, j] = feat[:, :, y0:y1, x0:x1].mean(dim=(2, 3))
    return out


def build_tokens(img: Tensor, lidar: Tensor, radar: Tensor, gps: Tensor, pos_emb: Tensor,
                 seq_len: int, n_views: int) -> Tensor:
    """Token build of ``GPT.forward`` (model2_seq.py:256-272) without dropout.

    img: (B*V*S, C, va, ha); lidar, radar: (B*S, C, va, ha); gps: (B, 2, C); pos_emb: (1, T, C).
    Token index = ((m*S + t)*va + y)*ha + x for modality slot m (V image slots, then lidar, radar);
    the two GPS tokens come last.
    """
    bz = lidar.shape[0] // seq_len
    c, va, ha = lidar.shape[1:4]
    parts = [img.reshape(bz, n_views * seq_len, c, va, ha),
             lidar.reshape(bz, seq_len, c, va, ha),
             radar.reshape(bz, seq_len, c, va, ha)]
    tok = torch.cat(parts, dim=1)                      # (B, (V+2)S, C, A, A)
    tok = tok.permute(0, 1, 3, 4, 2).reshape(bz, -1, c)  # channels last, flatten (slot, y, x)
    tok = torch.cat([tok, gps], dim=1)                 # + 2 GPS tokens
    return pos_emb + tok


# ----------------------------------------------------------------------------- transformer
def layer_norm(x: Tensor, weight: Tensor, bias: Tensor, eps: float = LN_EPS) -> Tensor:
    """``nn.LayerNorm(C)`` (model2_seq.py:118-119,199): biased variance over the last dim."""
    mu = x.mean(dim=-1, keepdim=True)
    var = ((x - mu) ** 2).mean(dim=-1, keepdim=True)
    return (x - mu) * torch.rsqrt(var + eps) * weight + bias


def linear(x: Tensor, w: Tensor, b: Tensor) -> Tensor:
    return x @ w.t() + b


def self_attention(x: Tensor, p: Dict[str, Tensor], prefix: str, n_head: int, attn_mask: Tensor = None,
                   resid_mask: Tensor = None) -> Tensor:
    """``SelfAttention.forward`` (model2_seq.py:94-110).  No causal mask: every token attends to all T
    tokens (the "masked" in the reference docstring is vestigial).  The two ``nn.Dropout`` sites
    (attn_drop :104 on the probabilities, resid_drop :109 on the projection) are restated as a
    multiplication by a caller-supplied tensor holding 0 or 1/(1-p) (``None`` = dropout off), which is
    what ``nn.Dropout`` computes for a given Bernoulli draw."""
    b, t, c = x.shape
    hs = c // n_head

    def heads(name):
        y = linear(x, p[prefix + name + ".weight"], p[prefix + name + ".bias"])
        return y.reshape(b, t, n_head, hs).transpose(1, 2)  # (B, nh, T, hs)

    k, q, v = heads("key"), heads("query"), heads("value")
    att = (q @ k.transpose(-2, -1)) * (1.0 / math.sqrt(hs))
    att = torch.softmax(att, dim=-1)
    if attn_mask is not None:
        att = att * attn_mask
    y = (att @ v).transpose(1, 2).reshape(b, t, c)
    y = linear(y, p[prefix + "proj.weight"], p[prefix + "proj.bias"])
    return y if resid_mask is None else y * resid_mask


def block(x: Tensor, p: Dict[str, Tensor], i: int, n_head: int, masks: Dict[str, Tensor] = None) -> Tensor:
    """``Block.forward`` (model2_seq.py:128-134): pre-LN attention and ReLU MLP, both residual.
    ``masks``: optional dropout masks ``attn.{i}`` (B,nh,T,T), ``proj.{i}``, ``mlp.{i}`` (B,T,C).
    ``relu.{i}`` (B,T,4C) of 0/1, if present, replaces ``nn.ReLU`` (:123) by a multiplication with THAT decision pattern:
    where it equals ``z > 0`` this is ReLU itself; tests use it to evaluate the reference math with the decisions another
    evaluation took (pre-activations within rounding distance of 0 may land on either side)."""
    pre = "blocks.%d." % i
    m = masks or {}
    x = x + self_attention(layer_norm(x, p[pre + "ln1.weight"], p[pre + "ln1.bias"]), p, pre + "attn.", n_head,
                           m.get("attn.%d" % i), m.get("proj.%d" % i))
    h = layer_norm(x, p[pre + "ln2.weight"], p[pre + "ln2.bias"])
    h = linear(h, p[pre + "mlp.0.weight"], p[pre + "mlp.0.bias"])
    h = torch.relu(h) if ("relu.%d" % i) not in m else h * m["relu.%d" % i]
    h = linear(h, p[pre + "mlp.2.weight"], p[pre + "mlp.2.bias"])
    if ("mlp.%d" % i) in m:  # nn.Dropout(resid_pdrop), model2_seq.py:125
        h = h * m["mlp.%d" % i]
    return x + h


def n_layers_of(p: Dict[str, Tensor]) -> int:
    n = 0
    while ("blocks.%d.ln1.weight" % n) in p:
        n += 1
    return n


def gpt_forward(p: Dict[str, Tensor], img: Tensor, lidar: Tensor, radar: Tensor, gps: Tensor,
                n_head: int, seq_len: int, n_views: int = 1, masks: Dict[str, Tensor] = None
                ) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """``GPT.forward`` (model2_seq.py:248-287).  Dropout is off unless ``masks`` supplies the Bernoulli
    draws as 0 / 1/(1-p) tensors: ``embd`` (B,T,C) for :272 and the per-block entries of ``block``.

    Returns (image_out, lidar_out, radar_out, pos_out) in the reference's shapes:
    3 x (B*slots*S, C, A, A) and (B, 2, C).
    """
    bz = lidar.shape[0] // seq_len
    c, va, ha = lidar.shape[1:4]
    x = build_tokens(img, lidar, radar, gps, p["pos_emb"], seq_len, n_views)
    if masks is not None and "embd" in masks:
        x = x * masks["embd"]
    for i in range(n_layers_of(p)):
        x = block(x, p, i, n_head, masks)
    x = layer_norm(x, p["ln_f.weight"], p["ln_f.bias"])
    n_map = (n_views + 2) * seq_len * va * ha
    pos_out = x[:, n_map:, :]
    maps = x[:, :n_map, :].reshape(bz, (n_views + 2) * seq_len, va, ha, c).permute(0, 1, 4, 2, 3)
    vs = n_views * seq_len
    img_o = maps[:, :vs].reshape(bz * vs, c, va, ha)
    lid_o = maps[:, vs:vs + seq_len].reshape(bz * seq_len, c, va, ha)
    rad_o = maps[:, vs + seq_len:].reshape(bz * seq_len, c, va, ha)
    return img_o, lid_o, rad_o, pos_out


# ----------------------------------------------------------------------------- upsample + add
def bilinear_upsample(x: Tensor, scale: int) -> Tensor:
    """``F.interpolate(x, scale_factor=scale, mode='bilinear')`` with align_corners=False
    (model2_seq.py:521-523, 539-541, 558-560), restated from the sampling formula:
    src = max((i + 0.5)/scale - 0.5, 0); i0 = floor(src); i1 = min(i0 + 1, A - 1); lam = src - i0.
    The taps are computed in x's precision (at least float32), so a float64 call is a float64 reference.
    """
    if scale == 1:
        return x
    n, c, a_h, a_w = x.shape
    tdt = torch.promote_types(x.dtype, torch.float32)

    def taps(a, s):
        dst = torch.arange(a * s, dtype=tdt)
        src = torch.clamp((dst + 0.5) / s - 0.5, min=0.0)
        i0 = src.floor().to(torch.long)
        i1 = torch.clamp(i0 + 1, max=a - 1)
        lam = (src - i0.to(tdt)).to(x.dtype)
        return i0.to(x.device), i1.to(x.device), lam.to(x.device)

    y0, y1, ly = taps(a_h, scale)
    x0, x1, lx = taps(a_w, scale)
    rows = x[:, :, y0, :] * (1 - ly)[None, None, :, None] + x[:, :, y1, :] * ly[None, None, :, None]
    return rows[:, :, :, x0] * (1 - lx) + rows[:, :, :, x1] * lx


def fusion_stage(p: Dict[str, Tensor], feats: Sequence[Tensor], gps_emb: Tensor, n_head: int,
                 seq_len: int, va: int, ha: int, n_views: int = 1, masks: Dict[str, Tensor] = None):
    """One fusion stage of ``Encoder.forward`` (model2_seq.py:515-526; same at :533-544, :552-563,
    :571-579): anchor pool x3 -> GPT -> bilinear upsample x3 -> residual add x3.

    feats = (image, lidar, radar) feature maps (N, C, H, W) with H = va*scale.
    Returns ((image', lidar', radar'), gps_out).
    """
    scale = feats[0].shape[2] // va
    pooled = [anchor_pool(f, va, ha) for f in feats]
    io, lo, ro, gps_out = gpt_forward(p, pooled[0], pooled[1], pooled[2], gps_emb, n_head, seq_len, n_views, masks)
    outs = tuple(f + bilinear_upsample(o, scale) for f, o in zip(feats, (io, lo, ro)))
    return outs, gps_out


# ----------------------------------------------------------------------------- parameter helpers
def init_gpt_params(n_embd: int, n_head: int, block_exp: int, n_layer: int, n_tokens: int,
                    generator: torch.Generator = None, pos_std: float = 0.0) -> Dict[str, Tensor]:
    """Random parameters with the reference's init law (model2_seq.py:189, 207-214): Linear weights
    N(0, 0.02), biases 0, LayerNorm weight 1 / bias 0, pos_emb zeros (``pos_std`` > 0 perturbs it
    so tests exercise the pos-emb path)."""
    g = generator
    c = n_embd
    p = {"pos_emb": torch.zeros(1, n_tokens, c)}
    if pos_std > 0:
        p["pos_emb"] = torch.randn(1, n_tokens, c, generator=g) * pos_std

    def lin(name, n_out, n_in):
        p[name + ".weight"] = torch.randn(n_out, n_in, generator=g) * 0.02
        p[name + ".bias"] = torch.zeros(n_out)

    def ln(name):
        p[name + ".weight"] = torch.ones(c)
        p[name + ".bias"] = torch.zeros(c)

    for i in range(n_layer):
        pre = "blocks.%d." % i
        ln(pre + "ln1")
        ln(pre + "ln2")
        for nm in ("key", "query", "value", "proj"):
            lin(pre + "attn." + nm, c, c)
        lin(pre + "mlp.0", block_exp * c, c)
        lin(pre + "mlp.2", c, block_exp * c)
    ln("ln_f")
    return p


def stage_flops(batch: int, n_tokens: int, c: int, n_layer: int) -> float:
    """Forward FLOPs of one GPT stage: L * (24*T*C^2 + 4*T^2*C) per sample (SURVEY.md §8d)."""
    return float(batch) * n_layer * (24.0 * n_tokens * c * c + 4.0 * n_tokens * n_tokens * c)

"""The fusion stage on the geometry the other parity tests leave out, against the float64 oracle (tests/parity_util.py):

* bf16 channels_last feature maps, which is what the model step under torch.autocast with channels_last trunks hands every
  stage (bench.py --workload model), and a stage whose image maps are channels_last while the lidar / radar maps are not;
* several camera views (n_views = 2: image frame b*V*S + sl of slot sl, model2_seq.py:256-272, 489-493) and rectangular anchor
  grids (vert_anchors != horz_anchors, as a 256x512 camera needs), through ``fusion_stage`` and the drop-in ``GPT``.

bf16 mode is held to the bar of test_gpu_parity.py (``parity_util.check``); fp32 mode to 1e-3 on every tensor once the ReLU
decisions are matched.
"""
from types import SimpleNamespace

import pytest
import torch

import parity_util as U
from conftest import assert_close
from oracle import fusion_ref as R

pytestmark = pytest.mark.gpu

BF16, F32 = torch.bfloat16, torch.float32
CL = torch.channels_last


@pytest.mark.parametrize("B,C,H", [(2, 64, 64), (2, 128, 32), (2, 256, 16), (2, 512, 8)])
def test_stage_bf16_channels_last_maps_vs_oracle(cuda_dev, B, C, H):
    """The four stages of the 256x256 model (8 layers, T = 962) on bf16 channels_last maps, fwd + bwd in bf16 mode: outputs and
    input gradients come back bf16 and channels_last."""
    pb = U.make_problem(B, C, H, 8, 8, cuda_dev, feat_dtype=BF16, channels_last=True)
    cap = {}
    got = U.run_dsfuse(pb, BF16, capture=cap)
    U.check(got, cap, pb, U.run_oracle(pb), "bf16 channels_last C=%d" % C)
    for o in got[0][:3]:
        assert o.dtype == BF16 and o.is_contiguous(memory_format=CL)
    for t in got[2][:3]:
        assert t.grad.dtype == BF16 and t.grad.is_contiguous(memory_format=CL)


def test_stage_bf16_channels_last_image_with_nchw_lidar_radar(cuda_dev):
    """Image maps channels_last, lidar / radar maps contiguous NCHW: the stage brings the latter to the image layout."""
    pb = U.make_problem(2, 128, 32, 8, 8, cuda_dev, feat_dtype=BF16, channels_last=(True, False, False))
    cap = {}
    got = U.run_dsfuse(pb, BF16, capture=cap)
    U.check(got, cap, pb, U.run_oracle(pb), "mixed layouts")
    for t in got[2][:3]:
        assert t.grad.dtype == BF16 and t.grad.shape == t.shape


GEOMETRY = [  # (C, L, V, vert_anchors, horz_anchors, scale); B = 2, seq_len 5, T = (V+2)*S*va*ha + 2 = 642
    (64, 2, 2, 4, 8, 4),    # 16 x 32 maps
    (512, 2, 2, 4, 8, 1),   # stage-4 width: maps are the anchor grid
]
MAPS = [(F32, F32, False), (BF16, F32, False), (BF16, BF16, True)]   # (compute mode, map dtype, channels_last)


@pytest.mark.parametrize("C,L,V,va,ha,scale", GEOMETRY)
@pytest.mark.parametrize("mode,fdt,cl", MAPS, ids=["fp32", "bf16", "bf16-maps-channels_last"])
def test_stage_several_views_rectangular_anchors_vs_oracle(cuda_dev, C, L, V, va, ha, scale, mode, fdt, cl):
    pb = U.make_problem(2, C, va * scale, L, va, cuda_dev, V=V, A_w=ha, W=ha * scale, feat_dtype=fdt, channels_last=cl)
    assert pb["T"] == 642
    cap = {}
    got = U.run_dsfuse(pb, mode, capture=cap)
    if mode == F32:
        matched = U.errors(got, U.run_oracle(pb, relu_masks=cap), L)
        bad = ["%s: %.3e" % (k, v) for k, v in matched.items() if v > 1e-3 and not k.endswith("key.bias")]
        assert not bad, bad
    else:
        U.check(got, cap, pb, U.run_oracle(pb), "V=%d %dx%d anchors C=%d" % (V, va, ha, C))


def test_gpt_module_several_views_rectangular_anchors(cuda_dev):
    """Drop-in GPT with n_views = 2 and 4x8 anchors in fp32 mode: pos_emb sized for (V+2)*S*va*ha + 2 tokens, ``forward`` (anchor
    maps in, model2_seq.py:248-287) and ``fuse`` (full-resolution maps, :515-526) against the float64 oracle."""
    from deepsense6g_tii_b200 import GPT
    B, C, L, V, va, ha, scale = 2, 64, 2, 2, 4, 8, 2
    m = GPT(C, U.NH, 4, L, va, ha, U.S, 0.0, 0.0, 0.0, SimpleNamespace(n_views=V, fusion_dtype=F32))
    assert m.pos_emb.shape == (1, (V + 2) * U.S * va * ha + 2, C)
    pb = U.make_problem(B, C, va * scale, L, va, cuda_dev, V=V, A_w=ha, W=ha * scale)
    res = m.load_state_dict({k: v.cpu() for k, v in pb["p0"].items()}, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    m = m.to(cuda_dev)
    p64 = {k: v.double() for k, v in pb["p0"].items()}

    def compare(run, ref_fn, maps, what):
        xs = [t.clone().requires_grad_(True) for t in maps] + [pb["gps"].clone().requires_grad_(True)]
        outs = run(*xs)
        refs_in = [t.detach().double().requires_grad_(True) for t in xs]
        refs = ref_fn(*refs_in)
        probes = [torch.randn(o.shape, generator=torch.Generator().manual_seed(7 + j)).to(cuda_dev) for j, o in enumerate(outs)]
        sum((o * pr).sum() for o, pr in zip(outs, probes)).backward()
        sum((o * pr.double()).sum() for o, pr in zip(refs, probes)).backward()
        for j, (o, r) in enumerate(zip(outs, refs)):
            assert o.shape == r.shape, (what, j)
            assert_close(o, r, 1e-4, 1e-6, "%s out%d" % (what, j))
        for j, (x, r) in enumerate(zip(xs, refs_in)):
            assert_close(x.grad, r.grad, 1e-3, 1e-6, "%s gin%d" % (what, j))

    pooled = [R.anchor_pool(f, va, ha).contiguous() for f in pb["feats"]]
    compare(m, lambda i, l, r, g: R.gpt_forward(p64, i, l, r, g, U.NH, U.S, n_views=V), pooled, "forward")

    def stage_ref(i, l, r, g):
        (a, b, c), go = R.fusion_stage(p64, (i, l, r), g, U.NH, U.S, va, ha, n_views=V)
        return a, b, c, go

    compare(m.fuse, stage_ref, pb["feats"], "fuse")

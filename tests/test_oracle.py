"""CPU tests that pin the oracle restatement (oracle/fusion_ref.py).

1. against the committed golden vectors generated from the reference classes
   (oracle/make_golden.py; reference model2_seq.py:175-287, :414, :521-526);
2. against the reference's parameter names and shapes, stored in the same vectors.
"""
import numpy as np
import pytest
import torch

from conftest import GPT_CASES, STAGE_CASES, load_golden, rel_err, assert_close, GOLDEN
from oracle import fusion_ref as R

TOL = 2e-5  # fp32 CPU vs fp32 CPU, different op order


def _run_oracle(g):
    cfg = g["cfg"]
    p = {k: v.clone().requires_grad_(True) for k, v in g["param"].items()}
    ins = {k: v.clone().requires_grad_(True) for k, v in g["in"].items()}
    if cfg["scale"] == 0:
        outs = R.gpt_forward(p, ins["img"], ins["lidar"], ins["radar"], ins["gps"], cfg["n_head"], cfg["S"])
    else:
        (a, b, c), gps = R.fusion_stage(p, (ins["img"], ins["lidar"], ins["radar"]), ins["gps"],
                                        cfg["n_head"], cfg["S"], cfg["A"], cfg["A"])
        outs = (a, b, c, gps)
    names = ("img", "lidar", "radar", "gps")
    loss = sum((o * g["probe"][n]).sum() for o, n in zip(outs, names))
    loss.backward()
    return dict(zip(names, outs)), p, ins, loss


@pytest.mark.parametrize("case", GPT_CASES + STAGE_CASES)
def test_oracle_matches_golden(case):
    g = load_golden(case)
    outs, p, ins, loss = _run_oracle(g)
    for n, o in outs.items():
        assert o.shape == g["out"][n].shape
        assert rel_err(o, g["out"][n]) < TOL, n
    for n, t in ins.items():
        assert rel_err(t.grad, g["gin"][n]) < TOL, n
    for n, t in p.items():
        assert_close(t.grad, g["gparam"][n], 5e-5, 1e-7, n)
    assert abs(loss.item() - float(g["loss"])) < 1e-3 * max(1.0, abs(float(g["loss"])))


def test_oracle_dropout_matches_golden_on_the_reference_draws():
    """Reference GPT in train() mode, p = 0.1 at all four nn.Dropout sites: given the Bernoulli draws recorded from
    the reference run, the restatement reproduces outputs and every gradient."""
    g = load_golden("gpt_tiny_dropout")
    cfg = g["cfg"]
    assert set(g["mask"]) == {"embd"} | {"%s.%d" % (k, i) for k in ("attn", "proj", "mlp") for i in range(cfg["L"])}
    for m in g["mask"].values():  # 0 or 1/(1-p), roughly 10 % dropped
        assert set(torch.unique(m).tolist()) <= {0.0, float(torch.tensor(1.0) / torch.tensor(0.9))}
    p = {k: v.clone().requires_grad_(True) for k, v in g["param"].items()}
    ins = {k: v.clone().requires_grad_(True) for k, v in g["in"].items()}
    outs = R.gpt_forward(p, ins["img"], ins["lidar"], ins["radar"], ins["gps"], cfg["n_head"], cfg["S"], masks=g["mask"])
    names = ("img", "lidar", "radar", "gps")
    sum((o * g["probe"][n]).sum() for o, n in zip(outs, names)).backward()
    for o, n in zip(outs, names):
        assert rel_err(o, g["out"][n]) < TOL, n
    for n, t in ins.items():
        assert rel_err(t.grad, g["gin"][n]) < TOL, n
    for n, t in p.items():
        assert_close(t.grad, g["gparam"][n], 5e-5, 1e-7, n)
    # and the masks matter: without them the result is far away
    with torch.no_grad():
        plain = R.gpt_forward(g["param"], *[g["in"][n] for n in names], cfg["n_head"], cfg["S"])
    assert rel_err(plain[0], g["out"]["img"]) > 1e-2


def test_ops_golden():
    z = np.load(GOLDEN + "/ops.npz")
    for s in (1, 2, 4, 8):
        x = torch.from_numpy(z["pool_in/%d" % s])
        assert rel_err(R.anchor_pool(x, 4, 4), torch.from_numpy(z["pool_out/%d" % s])) < 1e-6
        if s > 1:
            y = torch.from_numpy(z["up_in/%d" % s])
            assert rel_err(R.bilinear_upsample(y, s), torch.from_numpy(z["up_out/%d" % s])) < 1e-6
    x = torch.from_numpy(z["pool_in/ragged"])
    assert rel_err(R.anchor_pool(x, 4, 4), torch.from_numpy(z["pool_out/ragged"])) < 1e-6


def test_token_order_and_count():
    # T = (V+2)*S*A*A + 2 (model2_seq.py:189); GPS tokens are the last two (:270)
    B, S, A, C = 2, 5, 8, 8
    img = torch.zeros(B * S, C, A, A); lid = torch.ones(B * S, C, A, A); rad = 2 * torch.ones(B * S, C, A, A)
    gps = 3 * torch.ones(B, 2, C)
    x = R.build_tokens(img, lid, rad, gps, torch.zeros(1, 962, C), S, 1)
    assert x.shape == (B, 962, C)
    assert (x[:, :320] == 0).all() and (x[:, 320:640] == 1).all() and (x[:, 640:960] == 2).all() and (x[:, 960:] == 3).all()
    # channels-last inside a token; (y, x) raster inside a frame
    img = torch.arange(B * S * C * A * A, dtype=torch.float32).reshape(B * S, C, A, A)
    x = R.build_tokens(img, lid, rad, gps, torch.zeros(1, 962, C), S, 1)
    assert x[1, 2 * 64 + 3 * 8 + 5, 4] == img[1 * S + 2, 4, 3, 5]
    # several camera views and a rectangular anchor grid, token by token against the reference's stacking
    # (model2_seq.py:256-272 and 489-493): image_tensor.view(bz, n_views * seq_len, -1, h, w), then lidar, then radar, each
    # slot flattened in (y, x) raster order.  Every element is distinct, so a swapped axis or a wrong frame cannot match.
    B, S, V, va, ha, C = 2, 3, 2, 2, 5, 3
    T = (V + 2) * S * va * ha + 2
    n = [B * V * S, B * S, B * S]
    maps = []
    for j, nf in enumerate(n):
        maps.append(1000 * j + torch.arange(nf * C * va * ha, dtype=torch.float64).reshape(nf, C, va, ha))
    gps = -1 - torch.arange(B * 2 * C, dtype=torch.float64).reshape(B, 2, C)
    x = R.build_tokens(maps[0], maps[1], maps[2], gps, torch.zeros(1, T, C, dtype=torch.float64), S, V)
    assert x.shape == (B, T, C)
    for b in range(B):
        for m in range(V + 2):
            for t in range(S):
                sl = m * S + t
                if sl < V * S:
                    frame = maps[0][b * V * S + sl]
                elif sl < (V + 1) * S:
                    frame = maps[1][b * S + sl - V * S]
                else:
                    frame = maps[2][b * S + sl - (V + 1) * S]
                for y in range(va):
                    for xx in range(ha):
                        assert torch.equal(x[b, ((m * S + t) * va + y) * ha + xx], frame[:, y, xx]), (b, m, t, y, xx)
        assert torch.equal(x[b, T - 2:], gps[b])


@pytest.mark.parametrize("hw,va,ha", [((16, 32), 4, 8), ((8, 32), 2, 4), ((4, 8), 4, 8), ((12, 20), 3, 5),
                                      ((13, 22), 4, 8)], ids=["s4", "s4-wide", "s1", "s4-odd-grid", "ragged"])
def test_anchor_pool_matches_adaptive_avg_pool_on_rectangular_maps(hw, va, ha):
    """nn.AdaptiveAvgPool2d((vert_anchors, horz_anchors)) (model2_seq.py:414), float64; "ragged": the windows of a map that is
    no multiple of the grid overlap and differ in size."""
    x = torch.randn(3, 5, *hw, generator=torch.Generator().manual_seed(41), dtype=torch.float64)
    ref = torch.nn.AdaptiveAvgPool2d((va, ha))(x)
    got = R.anchor_pool(x, va, ha)
    assert got.shape == (3, 5, va, ha)
    assert float((got - ref).abs().max()) < 1e-14


@pytest.mark.parametrize("scale", [1, 2, 4, 6, 8])
@pytest.mark.parametrize("va,ha", [(4, 8), (8, 4), (3, 5)])
def test_bilinear_upsample_matches_interpolate_in_float64(scale, va, ha):
    """F.interpolate(scale_factor=s, mode='bilinear', align_corners=False) (model2_seq.py:521-523) on rectangular grids, in
    float64: the restatement is a float64 reference (taps included), so it agrees to rounding of double."""
    import torch.nn.functional as F
    x = torch.randn(2, 3, va, ha, generator=torch.Generator().manual_seed(43), dtype=torch.float64)
    got = R.bilinear_upsample(x, scale)
    ref = F.interpolate(x, scale_factor=scale, mode="bilinear", align_corners=False)
    assert got.dtype == torch.float64 and got.shape == (2, 3, va * scale, ha * scale)
    assert float((got - ref).abs().max()) < 1e-12
    # the same sampling expressed with the output size, as the fused kernels see it (source step A / H per axis)
    ref_size = F.interpolate(x, size=(va * scale, ha * scale), mode="bilinear", align_corners=False)
    assert float((got - ref_size).abs().max()) < 1e-12


def test_init_law_matches_reference():
    g = load_golden("gpt_c64_t962")   # holds the state_dict of the reference GPT(64, 4, 4, 2, 8, 8, 5)
    assert g["cfg"] == dict(C=64, n_head=4, L=2, A=8, S=5, B=1, scale=0)
    p = R.init_gpt_params(64, 4, 4, 2, 962)
    sd = g["param"]
    assert set(sd.keys()) == set(p.keys())
    for k in sd:
        assert sd[k].shape == p[k].shape, k

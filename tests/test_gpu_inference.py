"""The fusion stage without a backward to follow (``torch.no_grad``, ``torch.inference_mode``, frozen modules on plain inputs):
``functional.fusion_stage`` then runs the same kernels as the training forward but keeps no activation, and the narrow stages'
chain kernel runs its store-free variant.  Outputs must be bit-identical to the training forward's, launches the same, and the
memory peak within a bound computed from the shapes."""
import types

import pytest
import torch

import parity_util as U
from conftest import assert_close

pytestmark = pytest.mark.gpu

STAGES = [(64, 64), (128, 32), (256, 16), (512, 8)]   # (n_embd, feature-map side) of the four stages, 8x8 anchors, T = 962


@pytest.fixture(scope="module")
def K(cuda_dev):
    from deepsense6g_tii_b200 import _capi
    _capi.check_device()
    return _capi


def _cfg(pb, mode, **kw):
    cfg = dict(seq_len=U.S, n_views=pb["V"], vert_anchors=pb["A"], horz_anchors=pb["A_w"], n_head=U.NH, n_layer=pb["L"],
               compute_dtype=mode)
    cfg.update(kw)
    return cfg


def _stage(pb, mode, **kw):
    """fusion_stage on fresh leaves of the problem (inputs and parameters requiring grad) -> (call, leaves)."""
    from deepsense6g_tii_b200.functional import fusion_stage, param_names
    p, i = U.leafs(pb)
    plist = [p[n] for n in param_names(pb["L"])]
    return (lambda: fusion_stage(_cfg(pb, mode, **kw), i[0], i[1], i[2], i[3], plist)), (p, i)


def _counted(K, fn):
    n0 = K.launch_count()
    out = fn()
    torch.cuda.synchronize()
    return out, K.launch_count() - n0


def _same_as_training(K, fn, grad_ctx=torch.enable_grad):
    """fn() with grad enabled (the training forward) and under no_grad: equal outputs bit for bit, equal launch counts."""
    with grad_ctx():
        ref, n_ref = _counted(K, fn)
    with torch.no_grad():
        got, n_got = _counted(K, fn)
    assert any(t.requires_grad for t in ref), "the grad-enabled call must record a node"
    assert not any(t.requires_grad for t in got)
    for j, (a, b) in enumerate(zip(ref, got)):
        assert a.dtype == b.dtype and a.shape == b.shape and a.stride() == b.stride(), j
        assert torch.equal(a.detach(), b), "output %d differs from the training forward" % j
    assert n_got == n_ref, (n_got, n_ref)
    return got


@pytest.mark.parametrize("mode", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("C,H", STAGES)
def test_no_grad_matches_the_training_forward_at_the_stage_shapes(K, cuda_dev, C, H, mode):
    pb = U.make_problem(2, C, H, 8, 8, cuda_dev)
    _same_as_training(K, _stage(pb, mode)[0])


@pytest.mark.parametrize("chain", ["2", "0"])
@pytest.mark.parametrize("C", [64, 128])
def test_no_grad_matches_with_and_without_the_chain_kernel(K, cuda_dev, monkeypatch, C, chain):
    """DSF_CHAIN=2: the store-free chain kernel; DSF_CHAIN=0: the separate kernels.  B = 3: M = 2886 rows, a ragged last tile."""
    monkeypatch.setenv("DSF_CHAIN", chain)
    pb = U.make_problem(3, C, 8, 3, 8, cuda_dev, seed=7)
    _same_as_training(K, _stage(pb, torch.bfloat16)[0])


@pytest.mark.parametrize("C,H", [(64, 64), (512, 8)])
def test_no_grad_matches_on_bf16_channels_last_maps(K, cuda_dev, C, H):
    pb = U.make_problem(2, C, H, 2, 8, cuda_dev, feat_dtype=torch.bfloat16, channels_last=True)
    out = _same_as_training(K, _stage(pb, torch.bfloat16)[0])
    assert all(o.dtype == torch.bfloat16 and o.is_contiguous(memory_format=torch.channels_last) for o in out[:3])


@pytest.mark.parametrize("mode", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("C", [64, 512])
def test_no_grad_matches_with_two_views_and_4x8_anchors(K, cuda_dev, C, mode):
    pb = U.make_problem(2, C, 16, 2, 4, cuda_dev, V=2, A_w=8, W=32)
    _same_as_training(K, _stage(pb, mode)[0])


def _gpt(dev, C=64, n_layer=2, pdrop=0.0):
    from deepsense6g_tii_b200.modules import GPT
    torch.manual_seed(0)
    m = GPT(C, 4, 4, n_layer, 8, 8, 5, pdrop, pdrop, pdrop, types.SimpleNamespace(n_views=1, fusion_dtype=torch.bfloat16)).to(dev)
    with torch.no_grad():
        m.pos_emb.normal_(0, 0.02)
    return m


@pytest.mark.parametrize("C", [64, 256])
def test_gpt_forward_without_residual(K, cuda_dev, C):
    """GPT.forward (residual=False): pooled inputs in, anchor maps out."""
    m = _gpt(cuda_dev, C)
    ins = [torch.randn(10, C, 8, 8, device=cuda_dev) for _ in range(3)] + [torch.randn(2, 2, C, device=cuda_dev)]
    _same_as_training(K, lambda: m(*ins))


def test_no_grad_after_a_fused_optimizer_step_uses_the_persistent_shadows(K, cuda_dev):
    from deepsense6g_tii_b200.optim import FusedAdamWEMA
    m = _gpt(cuda_dev, 64, n_layer=3)
    ins = [torch.randn(10, 64, 16, 16, device=cuda_dev) for _ in range(3)] + [torch.randn(2, 2, 64, device=cuda_dev)]
    opt = FusedAdamWEMA(m.parameters(), lr=1e-3, gpts=[m])
    sum(o.float().square().sum() for o in m.fuse(*ins)).backward()
    opt.step()
    opt.zero_grad(set_to_none=True)
    ref = _same_as_training(K, lambda: m.fuse(*ins))   # both calls read the shadows the optimizer step wrote
    _, n_fresh = _counted(K, lambda: m.fuse(*ins))
    m._shadow_fresh_key = None                          # stale shadows: the no-grad forward re-packs them and marks them fresh
    with torch.no_grad():
        got, n_stale = _counted(K, lambda: m.fuse(*ins))
    assert n_stale == n_fresh + 3 and m._shadow_fresh_key is not None
    for a, b in zip(ref, got):
        assert torch.equal(a, b)


def test_train_mode_dropout_draws_the_same_masks_under_no_grad(K, cuda_dev):
    m = _gpt(cuda_dev, 64, pdrop=0.1).train()
    ins = [torch.randn(10, 64, 16, 16, device=cuda_dev) for _ in range(3)] + [torch.randn(2, 2, 64, device=cuda_dev)]

    def call():
        torch.manual_seed(5)
        return m.fuse(*ins)
    got = _same_as_training(K, call)
    torch.manual_seed(6)
    with torch.no_grad():
        assert not torch.equal(m.fuse(*ins)[0], got[0])


def test_inference_mode_and_no_graph_left_behind(K, cuda_dev):
    pb = U.make_problem(2, 64, 16, 2, 8, cuda_dev)
    fn, _ = _stage(pb, torch.bfloat16)
    with torch.no_grad():
        ref = fn()
    with torch.inference_mode():
        got = fn()
    for a, b in zip(ref, got):
        assert torch.equal(a, b) and not b.requires_grad and b.grad_fn is None
    assert all(t.grad_fn is None and not t.requires_grad for t in ref)
    with pytest.raises(RuntimeError):
        sum(o.float().sum() for o in ref).backward()


@pytest.mark.parametrize("case", ["params", "inputs", "both"])
def test_grad_enabled_calls_still_take_the_training_path(K, cuda_dev, case):
    """Parameters requiring grad on plain inputs, inputs requiring grad with frozen parameters, or both: the call records the
    training node and the gradients it returns are those of the all-requiring-grad call."""
    pb = U.make_problem(2, 64, 16, 2, 8, cuda_dev)
    ref_fn, (rp, ri) = _stage(pb, torch.bfloat16)
    sum((o.float() * pr).sum() for o, pr in zip(ref_fn(), pb["probes"])).backward()
    fn, (p, i) = _stage(pb, torch.bfloat16)
    for t in (list(p.values()) if case == "inputs" else []) + (i if case == "params" else []):
        t.requires_grad_(False)
    outs = fn()
    assert type(outs[0].grad_fn).__name__ == "FusionStageFnBackward"
    sum((o.float() * pr).sum() for o, pr in zip(outs, pb["probes"])).backward()
    if case != "inputs":
        for n, t in p.items():
            assert_close(t.grad, rp[n].grad, 1e-5, 1e-7, n)
    if case != "params":
        for j, (t, r) in enumerate(zip(i, ri)):
            assert_close(t.grad, r.grad, 1e-5, 1e-7, "input %d" % j)


@pytest.mark.parametrize("C,H", [(512, 8), (64, 8)])
def test_no_grad_peak_memory_is_bounded_by_one_block(K, cuda_dev, C, H):
    """B = 48, 8 layers, T = 962.  Above the pre-call baseline, a no-grad call may hold its outputs, two blocks' bf16 weight
    shadows (48 C^2 bytes each; the chain path packs block i + 1 while block i runs), 40 C bytes per token row and 64 MB; and
    less than a third of what the training forward of the same call holds (about 224 C bytes per row)."""
    B, L = 48, 8
    pb = U.make_problem(B, C, H, L, 8, cuda_dev)
    fn, _ = _stage(pb, torch.bfloat16)

    def peak(ctx):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        with ctx():
            out = fn()
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base, sum(o.numel() * o.element_size() for o in out)

    fn()   # first call: library set-up outside the measured window
    p_inf, out_bytes = peak(torch.no_grad)
    p_train, _ = peak(torch.enable_grad)
    rows = B * pb["T"]
    bound = out_bytes + 2 * 48 * C * C + 40 * C * rows + (64 << 20)
    print("C=%d: no-grad peak %.1f MB (bound %.1f MB), training forward peak %.1f MB"
          % (C, p_inf / 2 ** 20, bound / 2 ** 20, p_train / 2 ** 20))
    assert p_inf <= bound, (p_inf, bound)
    assert 3 * p_inf < p_train, (p_inf, p_train)


@pytest.mark.parametrize("M,C,last", [(11544, 64, False), (11544, 128, False), (300, 64, True), (130, 128, True), (5, 64, False), (1924, 128, False)])
def test_store_free_chain_kernel_matches_the_full_kernel(K, cuda_dev, M, C, last):
    """dsf_chain_fwd with x_mid, h2, a, h_next and the statistics NULL: x_out / qkv_next / yf bit-identical to the full call, and
    nothing else written.  After the last block x_out may be NULL as well.  A mixed group is rejected."""
    g = torch.Generator().manual_seed(31)
    F = 4 * C
    bf = torch.bfloat16
    rnd = lambda *s, sc=1.0: (sc * torch.randn(*s, generator=g)).to(cuda_dev)
    y = rnd(M, C).to(bf)
    x_in = rnd(M, C, sc=2.0) + 0.3
    wp, w1, w2, wq = rnd(C, C, sc=0.1).to(bf), rnd(F, C, sc=0.1).to(bf), rnd(C, F, sc=0.1).to(bf), rnd(3 * C, C, sc=0.1).to(bf)
    bp, b1, b2, bq = rnd(C, sc=0.1), rnd(F, sc=0.1), rnd(C, sc=0.1), rnd(3 * C, sc=0.1)
    g2, be2, gn, ben = 1 + rnd(C, sc=0.1), rnd(C, sc=0.1), 1 + rnd(C, sc=0.1), rnd(C, sc=0.1)
    nan = lambda *s, dt=torch.float32: torch.full(s, float("nan"), device=cuda_dev, dtype=dt)
    nxt = (None, None) if last else (wq, bq)

    def run(full, with_x_out=True):
        x_out, yf, hn, qkv = nan(M, C), nan(M, C), nan(M, C, dt=bf), nan(M, 3 * C, dt=bf)
        saved = [nan(M, C), nan(M, C, dt=bf), nan(M, F, dt=bf)] + [nan(M) for _ in range(4)] if full else [None] * 7
        K.chain_fwd(y, x_in, wp, w1, w2, nxt[0], bp, b1, b2, nxt[1], g2, be2, gn, ben, saved[0], x_out if with_x_out else None,
                    saved[1], saved[2], None if last else (hn if full else None), None if last else qkv, yf if last else None,
                    saved[3], saved[4], saved[5], saved[6])
        torch.cuda.synchronize()
        return x_out, yf, hn, qkv

    ref = run(True)
    got = run(False)
    assert torch.equal(got[0], ref[0]), "x_out"
    if last:
        assert torch.equal(got[1], ref[1]), "yf"
        x_out, yf, _, _ = run(False, with_x_out=False)
        assert torch.equal(yf, ref[1]) and torch.isnan(x_out).all()
    else:
        assert torch.equal(got[3], ref[3]), "qkv_next"
        assert torch.isnan(got[2].float()).all(), "the store-free kernel wrote h_next"
        with pytest.raises(RuntimeError):   # a middle block needs x_out
            K.chain_fwd(y, x_in, wp, w1, w2, wq, bp, b1, b2, bq, g2, be2, gn, ben, None, None, None, None, None, nan(M, 3 * C, dt=bf),
                        None, None, None, None, None)
    # mixed groups: one saved-only pointer given, or one left out
    x_out, yf, hn, qkv = nan(M, C), nan(M, C), nan(M, C, dt=bf), nan(M, 3 * C, dt=bf)
    with pytest.raises(RuntimeError, match="all given or all NULL"):
        K.chain_fwd(y, x_in, wp, w1, w2, nxt[0], bp, b1, b2, nxt[1], g2, be2, gn, ben, None, x_out, None, nan(M, F, dt=bf), None,
                    None if last else qkv, yf if last else None, None, None, None, None)
    with pytest.raises(RuntimeError, match="all given or all NULL"):
        K.chain_fwd(y, x_in, wp, w1, w2, nxt[0], bp, b1, b2, nxt[1], g2, be2, gn, ben, nan(M, C), x_out, nan(M, C, dt=bf),
                    nan(M, F, dt=bf), None if last else hn, None if last else qkv, yf if last else None, nan(M), nan(M), nan(M), None)
    if not last:   # h_next is part of the group when there is a next block
        with pytest.raises(RuntimeError, match="all given or all NULL"):
            K.chain_fwd(y, x_in, wp, w1, w2, wq, bp, b1, b2, bq, g2, be2, gn, ben, nan(M, C), x_out, nan(M, C, dt=bf), nan(M, F, dt=bf),
                        None, qkv, None, nan(M), nan(M), nan(M), nan(M))


@pytest.mark.parametrize("C", [64, 512])
def test_eval_no_grad_forward_replays_as_a_cuda_graph(K, cuda_dev, C):
    m = _gpt(cuda_dev, C, n_layer=3).eval()
    H = 64 if C == 64 else 8
    make = lambda: [torch.randn(10, C, H, H, device=cuda_dev) for _ in range(3)] + [torch.randn(2, 2, C, device=cuda_dev)]
    static = make()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side), torch.no_grad():
        m.fuse(*static)   # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.no_grad(), torch.cuda.graph(graph):
        out = m.fuse(*static)
    for _ in range(2):
        new = make()
        for s, t in zip(static, new):
            s.copy_(t)
        graph.replay()
        torch.cuda.synchronize()
        with torch.no_grad():
            ref = m.fuse(*new)
        for a, b in zip(out, ref):
            assert torch.equal(a, b)


@pytest.mark.parametrize("missing", [None, "lidar_radar"])
def test_transfuser_eval_logits_equal_under_no_grad(K, cuda_dev, missing):
    """The drop-in model in eval mode (configs[3] of BASELINE.json when lidar and radar are missing: bf16 autocast trunks)."""
    from deepsense6g_tii_b200 import TransFuser
    cfg = types.SimpleNamespace(seq_len=5, pred_len=4, n_views=1, vert_anchors=8, horz_anchors=8, n_embd=512, block_exp=4, n_layer=8,
                                n_head=4, embd_pdrop=0.1, attn_pdrop=0.1, resid_pdrop=0.1, add_velocity=1, fusion_dtype=torch.bfloat16,
                                modality_missing=missing, modality_missing_type="zerolike")
    torch.manual_seed(100)
    m = TransFuser(cfg, cuda_dev).eval()
    g = torch.Generator().manual_seed(1)
    B = 2
    imgs = [(torch.rand(B, 3, 256, 256, generator=g) * 255).to(cuda_dev) for _ in range(5)]
    lids = [(torch.rand(B, 1, 256, 256, generator=g) < 0.05).float().to(cuda_dev) for _ in range(5)]
    rads = [torch.rand(B, 2, 256, 256, generator=g).to(cuda_dev) for _ in range(5)]
    gps = torch.rand(B, 2, 2, generator=g).to(cuda_dev)
    old = torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    try:
        def call():
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=missing is not None):
                return (m(imgs, lids, rads, gps),)
        _same_as_training(K, call)
    finally:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = old

"""``dsf_stage_fwd`` (include/dsfuse.h), called directly through the ctypes bindings with torch-allocated buffers: one whole fusion-stage
inference forward in one C call.  Its outputs must be bit-identical to the grad-enabled ``FusionStageFn`` forward on the same inputs,
with the same launches; it allocates nothing, rejects bad input before launching anything, and replays as a CUDA graph."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
S = 5
STAGES = [(64, 64), (128, 32), (256, 16), (512, 8)]   # (n_embd, feature-map side) of the four stages


@pytest.fixture(scope="module")
def K(cuda_dev):
    from deepsense6g_tii_b200 import _capi
    _capi.check_device()
    return _capi


def _problem(dev, B, C, H, L, F=None, V=1, A=8, A_w=None, W=None, feat_dtype=torch.float32, channels_last=False, nh=4, seed=0):
    from deepsense6g_tii_b200.functional import param_names
    F = 4 * C if F is None else F
    A_w = A if A_w is None else A_w
    W = H if W is None else W
    T = (V + 2) * S * A * A_w + 2
    g = torch.Generator().manual_seed(seed)
    rnd = lambda *s: torch.randn(*s, generator=g)
    params = []
    for n in param_names(L):
        if n == "pos_emb":
            t = 0.02 * rnd(1, T, C)
        elif "ln" in n:
            t = (1.0 + 0.1 * rnd(C)) if n.endswith("weight") else 0.1 * rnd(C)
        elif n.endswith("mlp.0.weight"):
            t = rnd(F, C) * C ** -0.5
        elif n.endswith("mlp.0.bias"):
            t = 0.02 * rnd(F)
        elif n.endswith("mlp.2.weight"):
            t = rnd(C, F) * F ** -0.5
        elif n.endswith("weight"):
            t = rnd(C, C) * C ** -0.5
        else:
            t = 0.02 * rnd(C)
        params.append(t.to(dev))
    feats = [rnd(n, C, H, W).to(dev).to(feat_dtype) for n in (B * V * S, B * S, B * S)]
    if channels_last:
        feats = [f.contiguous(memory_format=torch.channels_last) for f in feats]
    return dict(B=B, C=C, H=H, W=W, L=L, F=F, V=V, A=A, A_w=A_w, nh=nh, T=T, params=params, feats=feats, gps=rnd(B, 2, C).to(dev),
                feat_dtype=feat_dtype, channels_last=channels_last)


def _counted(K, fn):
    torch.cuda.synchronize()
    n0 = K.launch_count()
    out = fn()
    torch.cuda.synchronize()
    return out, K.launch_count() - n0


def _training_forward(K, pb, residual=True, dropout=None):
    """The grad-enabled FusionStageFn forward on leaves requiring grad -> (outputs, launches)."""
    from deepsense6g_tii_b200.functional import fusion_stage
    cfg = dict(seq_len=S, n_views=pb["V"], vert_anchors=pb["A"], horz_anchors=pb["A_w"], n_head=pb["nh"], n_layer=pb["L"],
               compute_dtype=torch.bfloat16, residual=residual)
    if dropout is not None:
        cfg["dropout"] = dropout
    leaves = [t.clone().requires_grad_(True) for t in pb["feats"] + [pb["gps"]] + pb["params"]]
    with torch.enable_grad():
        outs, n = _counted(K, lambda: fusion_stage(cfg, *leaves[:4], leaves[4:]))
    assert outs[0].requires_grad
    return [o.detach() for o in outs], n


def _desc(K, pb, residual=True, chain=-1, prepacked=False, dropout=None, **geom_over):
    g = dict(B=pb["B"], S=S, V=pb["V"], A_h=pb["A"], A_w=pb["A_w"], C=pb["C"], H=pb["H"], W=pb["W"],
             feat_dtype=K.DSF_BF16 if pb["feat_dtype"] == torch.bfloat16 else K.DSF_F32,
             layout=K.DSF_NHWC if pb["channels_last"] else K.DSF_NCHW)
    g.update(geom_over)
    return K.make_stage_desc(K.make_geom(**g), pb["nh"], pb["L"], pb["F"], residual, chain, prepacked, dropout)


def _buffers(K, pb, desc):
    ws = torch.empty(K.stage_workspace_size(desc), device=pb["gps"].device, dtype=torch.uint8)
    outs = [torch.empty_like(f) for f in pb["feats"]] + [torch.empty(pb["B"], 2, pb["C"], device=pb["gps"].device)]
    return ws, outs


def _pack_shadows(K, pb):
    C, F, dev = pb["C"], pb["F"], pb["gps"].device
    shapes = dict(wqkv=(3 * C, C), wqkv_t=(C, 3 * C), wp=(C, C), wp_t=(C, C), w1=(F, C), w1_t=(C, F), w2=(C, F), w2_t=(F, C))
    out = []
    for i in range(pb["L"]):
        v = {k: torch.empty(s, device=dev, dtype=torch.bfloat16) for k, s in shapes.items()}
        v["bqkv"] = torch.empty(3 * C, device=dev)
        (_, _, _, _, kw, kb, qw, qb, vw, vb, pw, _, w1, _, w2, _) = pb["params"][1 + 16 * i: 17 + 16 * i]
        K.pack_block_weights(qw, kw, vw, pw, w1, w2, qb, kb, vb, tuple(v[k] for k in K.SHADOW_KEYS))
        out.append(v)
    torch.cuda.synchronize()
    return out


def _stage_fwd(K, pb, desc, ws, outs, shadows=None, repack=False):
    K.stage_fwd(desc, pb["params"], pb["feats"], pb["gps"], outs[:3], outs[3], ws, shadows=shadows, repack=repack)


def _check(K, pb, residual=True, chain=-1, dropout=None, shadows=None):
    """dsf_stage_fwd against the training forward: equal bits, equal launches (one pack launch per block fewer with pre-packed
    shadows used as they are)."""
    ref, n_ref = _training_forward(K, pb, residual, dropout)
    drop = None
    if dropout is not None:
        sd = dropout.get("seed_dev")
        drop = K.DropoutCfg(dropout["embd"], dropout["attn"], dropout["resid"], dropout["seed"], dropout["step"],
                            None if sd is None else sd.data_ptr())
    for repack in ((False, True) if shadows else (False,)):
        sh = _pack_shadows(K, pb) if shadows else None
        desc = _desc(K, pb, residual, chain, sh is not None, drop)
        ws, outs = _buffers(K, pb, desc)
        _, n = _counted(K, lambda: _stage_fwd(K, pb, desc, ws, outs, sh, repack))
        for j, (a, b) in enumerate(zip(ref, outs)):
            # the stride of a size-1 dimension carries no layout (at B = 1 the training forward's gps_out is a slice of yf)
            strides = lambda t: [s for s, n in zip(t.stride(), t.shape) if n > 1]
            assert a.dtype == b.dtype and a.shape == b.shape and strides(a) == strides(b), j
            assert torch.equal(a, b), "output %d differs from the training forward (repack=%s)" % (j, repack)
        assert n == n_ref - (pb["L"] if sh is not None and not repack else 0), (n, n_ref, repack)


@pytest.mark.parametrize("B,L", [(1, 8), (12, 1)])
@pytest.mark.parametrize("C,H", STAGES)
def test_matches_the_training_forward_at_the_stage_shapes(K, cuda_dev, C, H, B, L):
    _check(K, _problem(cuda_dev, B, C, H, L, seed=C + B))


@pytest.mark.parametrize("feat_dtype,channels_last", [(torch.bfloat16, True), (torch.bfloat16, False), (torch.float32, True)],
                         ids=["bf16-cl", "bf16-nchw", "fp32-cl"])
@pytest.mark.parametrize("C,H", [(64, 64), (512, 8)])
def test_matches_on_map_dtypes_and_layouts(K, cuda_dev, C, H, feat_dtype, channels_last):
    _check(K, _problem(cuda_dev, 2, C, H, 2, feat_dtype=feat_dtype, channels_last=channels_last))


@pytest.mark.parametrize("C", [64, 512])
def test_matches_with_two_views_and_4x8_anchors(K, cuda_dev, C):
    _check(K, _problem(cuda_dev, 2, C, 16, 2, V=2, A=4, A_w=8, W=32))


@pytest.mark.parametrize("C", [64, 256])
def test_matches_without_residual(K, cuda_dev, C):
    _check(K, _problem(cuda_dev, 2, C, 16, 2), residual=False)


@pytest.mark.parametrize("C", [64, 128])
def test_matches_with_block_exp_2(K, cuda_dev, C):
    """F = 2C: the separate kernels at the narrow stages, where F = 4C would run the chain kernel."""
    _check(K, _problem(cuda_dev, 3, C, 16, 3, F=2 * C))


@pytest.mark.parametrize("C", [64, 128])
def test_matches_with_the_chain_kernel_off(K, cuda_dev, monkeypatch, C):
    monkeypatch.setenv("DSF_CHAIN", "0")   # the training forward's switch; chain = 0 is the descriptor's
    _check(K, _problem(cuda_dev, 3, C, 8, 3), chain=0)


@pytest.mark.parametrize("C,L", [(64, 3), (256, 2), (128, 1)])
def test_matches_with_prepacked_shadows(K, cuda_dev, C, L):
    _check(K, _problem(cuda_dev, 2, C, 16, L), shadows=True)


@pytest.mark.parametrize("C,seed_dev", [(64, True), (256, False)])
def test_matches_with_train_mode_dropout(K, cuda_dev, C, seed_dev):
    dropout = dict(embd=0.1, attn=0.1, resid=0.1, seed=1234567, step=3)
    if seed_dev:
        dropout["seed_dev"] = torch.tensor([987654321], device=cuda_dev, dtype=torch.int64)
    _check(K, _problem(cuda_dev, 2, C, 16, 2), dropout=dropout)


@pytest.mark.parametrize("C", [64, 256])
def test_side_stream_packs_with_ready_events_match_the_training_forward(K, cuda_dev, monkeypatch, C):
    """With the side streams on (as under graph capture; DSF_WGRAD_STREAM=1 forces them), the no-grad forward packs the weight shadows
    on the side stream and dsf_stage_fwd waits for block i's ready event only before block i: outputs and launches unchanged."""
    from deepsense6g_tii_b200.functional import fusion_stage
    monkeypatch.setenv("DSF_WGRAD_STREAM", "1")
    pb = _problem(cuda_dev, 2, C, 16, 3)
    ref, n_ref = _training_forward(K, pb)
    cfg = dict(seq_len=S, n_views=1, vert_anchors=8, horz_anchors=8, n_head=pb["nh"], n_layer=pb["L"], compute_dtype=torch.bfloat16)
    with torch.no_grad():
        got, n = _counted(K, lambda: fusion_stage(cfg, *pb["feats"], pb["gps"], pb["params"]))
    assert n == n_ref
    for a, b in zip(ref, got):
        assert torch.equal(a, b)


@pytest.mark.parametrize("C,H", [(512, 8), (64, 8)])
def test_workspace_is_within_the_no_grad_peak_bound(K, cuda_dev, C, H):
    """The bound tests/test_gpu_inference.py puts on a no-grad call's peak above its outputs (B = 48, 8 layers): two blocks' shadows +
    40 C bytes per token row + 64 MB."""
    pb = _problem(cuda_dev, 48, C, H, 8)
    desc = _desc(K, pb)
    rows = 48 * pb["T"]
    ws = K.stage_workspace_size(desc)
    assert ws <= 2 * 48 * C * C + 40 * C * rows + (64 << 20), ws


def test_a_call_allocates_nothing_and_short_or_misaligned_workspaces_are_rejected(K, cuda_dev):
    pb = _problem(cuda_dev, 2, 64, 16, 2)
    desc = _desc(K, pb)
    need = K.stage_workspace_size(desc)
    ws = torch.empty(need + 512, device=cuda_dev, dtype=torch.uint8)
    outs = _buffers(K, pb, desc)[1]
    _stage_fwd(K, pb, desc, ws, outs)   # first call: library set-up
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    _, n = _counted(K, lambda: K.stage_fwd(desc, pb["params"], pb["feats"], pb["gps"], outs[:3], outs[3], ws.data_ptr(), need))
    assert n > 0 and torch.cuda.memory_allocated() == before
    for ptr, nbytes, pattern in ((ws.data_ptr(), need - 1, r"workspace of %d bytes is smaller than the %d bytes" % (need - 1, need)),
                                 (ws.data_ptr() + 16, need, "256-byte aligned")):
        n0 = K.launch_count()
        with pytest.raises(RuntimeError, match=pattern):
            K.stage_fwd(desc, pb["params"], pb["feats"], pb["gps"], outs[:3], outs[3], ptr, nbytes)
        torch.cuda.synchronize()
        assert K.launch_count() == n0


@pytest.mark.parametrize("case", ["geometry", "head_size_24", "null_map"])
def test_rejected_input_launches_nothing(K, cuda_dev, case):
    """Each is reported with an error code and a message before anything is enqueued."""
    pb = _problem(cuda_dev, 2, 192, 16, 2, nh=8) if case == "head_size_24" else _problem(cuda_dev, 2, 64, 16, 2)
    ws, outs = _buffers(K, pb, _desc(K, _problem(cuda_dev, 2, 64, 16, 2)))
    feats = pb["feats"]
    if case == "geometry":
        desc, expect = _desc(K, pb, H=15), "not a multiple of the anchor grid"   # 15 x 16 maps on an 8 x 8 anchor grid
    elif case == "head_size_24":
        desc, expect = _desc(K, pb), "head size"
    else:
        desc, expect = _desc(K, pb), "must be non-NULL"
        feats = [None] + feats[1:]
    if case != "null_map":
        with pytest.raises(RuntimeError, match=expect):
            K.stage_workspace_size(desc)
    torch.cuda.synchronize()
    n0 = K.launch_count()
    with pytest.raises(RuntimeError, match=expect):
        K.stage_fwd(desc, pb["params"], feats, pb["gps"], outs[:3], outs[3], ws)
    torch.cuda.synchronize()
    assert K.launch_count() == n0


@pytest.mark.parametrize("C,H", [(64, 64), (512, 8)])
def test_one_call_replays_as_a_cuda_graph(K, cuda_dev, C, H):
    pb = _problem(cuda_dev, 2, C, H, 3)
    desc = _desc(K, pb)
    ws, outs = _buffers(K, pb, desc)
    _stage_fwd(K, pb, desc, ws, outs)   # warm-up outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        _stage_fwd(K, pb, desc, ws, outs)
    for seed in (1, 2):
        new = _problem(cuda_dev, 2, C, H, 3, seed=seed)
        for s, t in zip(pb["feats"] + [pb["gps"]], new["feats"] + [new["gps"]]):
            s.copy_(t)
        graph.replay()
        torch.cuda.synchronize()
        ws2, ref = _buffers(K, pb, desc)
        _stage_fwd(K, pb, desc, ws2, ref)
        torch.cuda.synchronize()
        for a, b in zip(outs, ref):
            assert torch.equal(a, b)


# ------------------------------------------------------------------------------------------ examples/stage_infer.cu
def _mix(x):
    x = x ^ (x >> np.uint32(16))
    x = x * np.uint32(0x7feb352d)
    x = x ^ (x >> np.uint32(15))
    x = x * np.uint32(0x846ca68b)
    return x ^ (x >> np.uint32(16))


def _hval(stream, n):
    """The example's input values: uniform in [-0.5, 0.5) on a 2^-24 grid, a function of (stream, element index)."""
    with np.errstate(over="ignore"):
        h = _mix(np.arange(n, dtype=np.uint32) ^ _mix(np.array([stream], dtype=np.uint32)))
    return (h >> np.uint32(8)).astype(np.float32) * np.float32(1.0 / 16777216.0) - np.float32(0.5)


def _checksum(t):
    h = t.detach().cpu().contiguous().numpy().view(np.uint16).ravel().astype(np.uint64)
    with np.errstate(over="ignore"):
        return int((h * (2 * np.arange(h.size, dtype=np.uint64) + 1)).sum(dtype=np.uint64))


def test_c_example_matches_python_on_the_same_hashed_inputs(K, cuda_dev, tmp_path):
    """Build examples/stage_infer.cu (linked against libdsfuse.so and cudart only), run it, and compare its four output checksums and
    its launch count with the Python no-grad fusion stage on the same hashed inputs."""
    if shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"):
        pytest.skip("nvcc not found")
    exe = str(tmp_path / "stage_infer")
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "deepsense6g_tii_b200", "csrc"), "example", "EXAMPLE=" + exe], check=True)
    res = subprocess.run([exe], check=True, capture_output=True, text=True, timeout=600).stdout
    got = dict(re.findall(r"checksum (\w+) ([0-9a-f]{16})", res))
    launches = int(re.search(r"launches (\d+)", res).group(1))

    from deepsense6g_tii_b200.functional import fusion_stage, param_names
    B, C, H, L = 1, 64, 64, 8
    F, T = 4 * C, 3 * S * 64 + 2
    t = lambda v, *shape: torch.from_numpy(v).view(*shape).to(cuda_dev)
    ins = [t(_hval(0, B * S * C * H * H) * np.float32(2), B * S, C, H, H), t(_hval(1, B * S * C * H * H) * np.float32(2), B * S, C, H, H),
           t(_hval(2, B * S * C * H * H) * np.float32(2), B * S, C, H, H), t(_hval(3, B * 2 * C), B, 2, C)]
    params = []
    for k, n in enumerate(param_names(L)):
        shape = {"pos_emb": (1, T, C)}.get(n) or ((F, C) if n.endswith("mlp.0.weight") else (C, F) if n.endswith("mlp.2.weight") else
                                                  (C, C) if n.endswith("weight") and "ln" not in n else (F,) if n.endswith("mlp.0.bias") else (C,))
        scale, shift = (0.25, 1.0) if ("ln" in n and n.endswith("weight")) else (0.0625, 0.0) if (n.endswith("bias") and "ln" not in n) else (0.125, 0.0)
        v = np.float32(shift) + _hval(100 + k, int(np.prod(shape))) * np.float32(scale)
        params.append(t(v, *shape))
    cfg = dict(seq_len=S, n_views=1, vert_anchors=8, horz_anchors=8, n_head=4, n_layer=L, compute_dtype=torch.bfloat16)
    with torch.no_grad():
        outs, n = _counted(K, lambda: fusion_stage(cfg, *ins, params))
    print(res)
    for name, o in zip(("img_out", "lidar_out", "radar_out", "gps_out"), outs):
        assert int(got[name], 16) == _checksum(o), name
    assert launches == n

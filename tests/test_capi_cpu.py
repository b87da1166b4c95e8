"""CPU-only checks of the drop-in boundary: the C-ABI library loads and exports every symbol that
include/dsfuse.h declares (no compute calls without a GPU), ctypes struct layouts match the header,
and the host-side modules keep the reference's constructor / state_dict contract
(model2_seq.py:175-214, :411-470, :855-873)."""
import os
import re
import types

import pytest
import torch

from conftest import ROOT, load_golden


def _header_symbols():
    txt = open(os.path.join(ROOT, "include", "dsfuse.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(dsf_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    from deepsense6g_tii_b200 import _capi
    lib = _capi.lib()
    syms = _header_symbols()
    assert len(syms) >= 19
    for s in syms:
        assert hasattr(lib, s), "libdsfuse.so does not export %s" % s
    assert sorted(_capi.SYMBOLS) == syms
    assert lib.dsf_version() == 100


def test_ctypes_struct_layouts():
    import ctypes
    from deepsense6g_tii_b200 import _capi
    assert ctypes.sizeof(_capi.Geom) == 10 * 4
    # 5 x int32 (20 B) + 4 B padding + 12 x int64 + float + int32
    assert ctypes.sizeof(_capi.GemmF32Desc) == 24 + 12 * 8 + 8
    assert _capi.GemmF32Desc.a_b1.offset == 24


def test_missing_gpu_fails_loudly():
    """Product path must raise, not fall back, when there is no CUDA device / CPU tensors."""
    from deepsense6g_tii_b200 import GPT
    cfg = types.SimpleNamespace(n_views=1, fusion_dtype=torch.float32)
    m = GPT(32, 4, 4, 1, 2, 2, 2, 0.0, 0.0, 0.0, cfg)
    ins = [torch.zeros(2 * 2, 32, 2, 2) for _ in range(3)] + [torch.zeros(2, 2, 32)]
    with pytest.raises(RuntimeError):
        m(*ins)


def test_param_order_and_names_match_golden_state_dict():
    from deepsense6g_tii_b200 import GPT, param_names
    g = load_golden("gpt_tiny")
    c = g["cfg"]
    names = param_names(c["L"])
    assert sorted(names) == sorted(g["param"].keys())
    cfg = types.SimpleNamespace(n_views=1)
    m = GPT(c["C"], c["n_head"], 4, c["L"], c["A"], c["A"], c["S"], 0.1, 0.1, 0.1, cfg)
    sd = m.state_dict()
    assert list(sd.keys()) == list(g["param"].keys())  # same registration order as the reference
    for k in sd:
        assert sd[k].shape == g["param"][k].shape
    # reference init law (model2_seq.py:207-214): pos_emb zeros, LN (1, 0), Linear bias 0, weight std 0.02
    assert float(sd["pos_emb"].abs().max()) == 0.0
    assert float(sd["ln_f.weight"].min()) == 1.0 and float(sd["blocks.0.attn.proj.bias"].abs().max()) == 0.0
    assert abs(float(sd["blocks.0.mlp.0.weight"].std()) - 0.02) < 0.004


def test_fused_stem_and_tail_are_declined_off_the_gpu():
    """The fused stem / tail (dsf_stem_pack, dsf_tail_fwd) take CUDA tensors only; anything else makes the drop-in Encoder run the
    reference's op sequence (model2_seq.py:481-493, 581-595) — the predicates must say so without touching the library."""
    import torch
    from deepsense6g_tii_b200 import functional as Fn
    frames = [torch.rand(2, 3, 8, 8) for _ in range(5)]
    assert not Fn.stem_pack_supported(frames)
    maps = [torch.rand(10, 512, 8, 8) for _ in range(3)]
    assert not Fn.pooled_tail_supported(maps[0], maps[1], maps[2], torch.rand(2, 2, 512))

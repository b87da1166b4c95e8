"""CPU checks of the whole-stage C entry points (``dsf_stage_workspace_size`` / ``dsf_stage_fwd``, include/dsfuse.h): the header is
valid C, the ctypes structs have the C layout, the workspace size is the formula the header documents, and the C example builds."""
import ctypes
import os
import shutil
import subprocess

import pytest

from conftest import ROOT

HEADER_DIR = os.path.join(ROOT, "include")
NVCC = shutil.which("nvcc") or ("/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else None)


def _cc():
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    return cc


def test_header_parses_as_c(tmp_path):
    src = tmp_path / "h.c"
    src.write_text('#include "dsfuse.h"\nint main(void) { dsf_stage_desc d; dsf_stage_params p; (void)d; (void)p; return 0; }\n')
    subprocess.run([_cc(), "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-I", HEADER_DIR, str(src)], check=True)


def test_ctypes_stage_structs_match_the_c_layout(tmp_path):
    from deepsense6g_tii_b200 import _capi as K
    src = tmp_path / "l.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "dsfuse.h"\nint main(void) {\n'
                   '  printf("%zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(dsf_dropout_cfg), offsetof(dsf_dropout_cfg, seed_dev),\n'
                   '         sizeof(dsf_stage_desc), offsetof(dsf_stage_desc, chain), offsetof(dsf_stage_desc, dropout),\n'
                   '         sizeof(dsf_block_shadows), sizeof(dsf_stage_params), offsetof(dsf_stage_params, repack));\n  return 0;\n}\n')
    exe = tmp_path / "l"
    subprocess.run([_cc(), "-std=c99", "-I", HEADER_DIR, str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    want = [ctypes.sizeof(K.DropoutCfg), K.DropoutCfg.seed_dev.offset, ctypes.sizeof(K.StageDesc), K.StageDesc.chain.offset,
            K.StageDesc.dropout.offset, ctypes.sizeof(K.BlockShadows), ctypes.sizeof(K.StageParams), K.StageParams.repack.offset]
    assert got == want


def _formula(B, S, V, A_h, A_w, C, nh, L, F, chain=-1, prepacked=False, drop=(0.0, 0.0, 0.0)):
    """The workspace formula of include/dsfuse.h, restated."""
    a = lambda n: (n + 255) // 256 * 256
    T = (V + 2) * S * A_h * A_w + 2
    M = B * T
    mode = 2 if chain < 0 else chain
    chained = ((mode >= 1 and C == 64) or (mode >= 2 and C == 128)) and F == 4 * C and L > 0 and max(drop) <= 0
    n = 2 * a(4 * M * C) + a(2 * M * C) + a(6 * M * C) + a(2 * M * C) + a(4 * B * nh * T) + a(8 * M) + a(4 * M * C)
    if not chained and L > 0:
        n += a(4 * M * C) + a(2 * M * C) + a(2 * M * F)
    if drop[1] > 0 and L > 0:
        n += a(4 * B * nh * T * 2 * ((T + 63) // 64))   # dsf_attn_drop_words
    if not prepacked:
        slots = 2 if chained and L > 1 else min(L, 1)
        n += slots * (2 * a(6 * C * C) + 2 * a(2 * C * C) + 4 * a(2 * F * C) + a(12 * C))
    return n


@pytest.mark.parametrize("B,V,A_h,A_w,C,nh,L,F,chain,prepacked,drop", [
    (1, 1, 8, 8, 64, 4, 8, 256, -1, False, (0.0, 0.0, 0.0)),      # chain, two shadow slots
    (12, 1, 8, 8, 128, 4, 1, 512, -1, False, (0.0, 0.0, 0.0)),    # chain, one block: one slot
    (3, 1, 8, 8, 64, 4, 3, 128, -1, False, (0.0, 0.0, 0.0)),      # F = 2C: separate kernels
    (2, 1, 8, 8, 128, 4, 3, 512, 1, False, (0.0, 0.0, 0.0)),      # chain = 1 leaves C = 128 to the separate kernels
    (2, 1, 8, 8, 64, 4, 2, 256, 0, True, (0.0, 0.0, 0.0)),
    (2, 2, 4, 8, 512, 4, 8, 2048, -1, True, (0.0, 0.0, 0.0)),
    (2, 1, 8, 8, 256, 8, 2, 1024, -1, False, (0.1, 0.1, 0.1)),    # attention dropout: keep bits
    (2, 1, 8, 8, 64, 4, 2, 256, -1, False, (0.0, 0.0, 0.1)),      # dropout turns the chain off
    (4, 1, 8, 8, 64, 4, 0, 0, -1, False, (0.0, 0.0, 0.0)),        # no blocks: tokens -> ln_f -> upsample
])
def test_workspace_size_is_the_header_formula(B, V, A_h, A_w, C, nh, L, F, chain, prepacked, drop):
    from deepsense6g_tii_b200 import _capi as K
    g = K.make_geom(B, 5, V, A_h, A_w, C, 8 * A_h, 8 * A_w, K.DSF_F32, K.DSF_NCHW)
    d = K.make_stage_desc(g, nh, L, F, True, chain, prepacked, K.DropoutCfg(*drop, 1, 0, None) if max(drop) > 0 else None)
    assert K.stage_workspace_size(d) == _formula(B, 5, V, A_h, A_w, C, nh, L, F, chain, prepacked, drop)


@pytest.mark.parametrize("field,value,message", [("n_head", 8, "head size"), ("F", 96, "multiple of 64"), ("chain", 3, "chain must be"),
                                                 ("residual", 2, "residual must be")])
def test_workspace_size_rejects_a_bad_descriptor(field, value, message):
    from deepsense6g_tii_b200 import _capi as K
    d = K.make_stage_desc(K.make_geom(1, 5, 1, 8, 8, 192 if field == "n_head" else 64, 64, 64, K.DSF_F32), 4, 2, 256)
    setattr(d, field, value)
    with pytest.raises(RuntimeError, match=message):
        K.stage_workspace_size(d)


@pytest.mark.skipif(NVCC is None, reason="nvcc not found")
def test_example_cross_compiles_for_sm100a(tmp_path):
    exe = tmp_path / "stage_infer"
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "deepsense6g_tii_b200", "csrc"), "example", "EXAMPLE=%s" % exe], check=True)
    assert exe.is_file() and os.access(exe, os.X_OK)

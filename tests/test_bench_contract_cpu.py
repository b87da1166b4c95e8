"""The reference arm of bench.py runs without a GPU: check the JSON contract of its line here (keys the driver reads)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ref_line(*extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"] + list(extra),
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip().startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    """Stage-1 alone keeps this CPU test short; the driver's line is the default workload (all four stages, batch 12)."""
    d = _ref_line("--stage", "1")
    assert d["impl"] == "reference" and d["metric"] == "train samples/sec (fwd+bwd)" and d["unit"] == "samples/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["config"]["workload"].startswith("gpt_fusion_stage n_embd=64") and d["config"]["global_batch"] == 12
    cb = d["cpu_baseline"]
    have_ref = os.path.isfile(os.path.join(ROOT, "oracle", "_ref", "model2_seq.py"))
    assert cb["kind"] == ("reference" if have_ref else "port") and cb["cores"] >= 1 and cb["value"] == d["value"]
    assert ("oracle/_ref/model2_seq.py" in cb["sample"]) == have_ref
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_both_arms_name_the_same_workload():
    """The driver compares the two arms' ``config``: the shared part comes from one function."""
    sys.path.insert(0, ROOT)
    import bench
    assert bench.SPEC == bench.STAGES4 and bench.n_tokens() == 962
    c = bench.workload_config(1)
    assert c["workload"].startswith("gpt_fusion_path: the 4 fusion stages") and "64/128/256/512" in c["workload"] and c["global_batch"] == 12
    # SURVEY.md §8(d): 92.74 GF forward per sample over the four stages, 63.58 GF of it in stage 4
    tot = sum(bench.fwd_flops_per_sample(c) for c, _ in bench.STAGES4)
    assert abs(tot / 1e9 - 92.74) < 0.05 and abs(bench.fwd_flops_per_sample(512) / 1e9 - 63.58) < 0.05


def test_dump_outputs_keeps_64_mb_and_samples_fixed_positions(tmp_path):
    """--dump-outputs: float32 files, 64 MB in all, small tensors whole, large ones sampled at the same positions every run."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    gen = torch.Generator().manual_seed(1)
    named = [("big.%d" % i, torch.randn(4_000_000, generator=gen).to(torch.bfloat16)) for i in range(8)]
    named += [("small", torch.randn(3, 5, generator=gen, dtype=torch.float64))]
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), named)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(n + ".npy" for n, _ in named)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 * 10 ** 6
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float32 and np.array_equal(a, b)
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), named[-1][1].float().numpy())
    big = np.load(tmp_path / "a" / "big.0.npy")
    assert 1_000_000 < big.size < 4_000_000 and np.isin(big, named[0][1].float().numpy()).all()


def test_steps_below_one_are_refused():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"], capture_output=True,
                         text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0 and "--steps" in out.stderr


def test_gpu_arm_refuses_to_run_without_a_gpu():
    """No CPU fallback on the product path: without CUDA the default arm exits with an error instead of timing the oracle."""
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0 and "no CUDA device" in (out.stderr + out.stdout)

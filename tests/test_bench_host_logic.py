"""CPU: the host-side arithmetic of bench.py (what turns per-launch event records into the `roofline`, `breakdown` and
`train.head` objects of the JSON line) on synthetic records, and the guard that keeps a failing side leg from costing the
run its line. No GPU, no oracle."""
import importlib.util
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bench():
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


class _Tick:
    """Stands in for a CUDA event: elapsed_time(end) in milliseconds."""

    def __init__(self, t_ms):
        self.t = t_ms

    def elapsed_time(self, other):
        return other.t - self.t


def _rec(name, kind, ms, nbytes, flops, at=0.0):
    return (name, dict(bytes=nbytes, flops=flops, kind=kind), _Tick(at), _Tick(at + ms))


PEAKS = dict(hbm_gbs=6548.8, tensor_tflops=1401.6, tensor_tflops_burst=1668.7, source="test")


def test_roofline_names_the_dominant_head_kernel_and_recomputes(bench):
    records = []
    for step in range(4):
        records += [_rec("maxpool2d_nhwc[C=64]", "maxpool", 0.180, 1_027_604_480, 0),          # longest, but backbone-side
                    _rec("gram_pool_fwd[C=256]", "gram_fwd", 0.145, 823_132_160, 52_818_870_272),
                    _rec("gram_pool_fwd[C=512]", "gram_fwd", 0.100, 412_090_368, 52_700_000_000),
                    _rec("attn_head_fwd[B=256]", "attn", 0.052, 30_000_000, 5_400_000_000)]
    kernels, roof = bench.summarise_profile(records, PEAKS)
    assert set(kernels) == {"maxpool2d_nhwc[C=64]", "gram_pool_fwd[C=256]", "gram_pool_fwd[C=512]", "attn_head_fwd[B=256]"}
    assert kernels["maxpool2d_nhwc[C=64]"]["launches"] == 4 and kernels["maxpool2d_nhwc[C=64]"]["avg_us"] == 180.0
    assert roof["kernel"] == "gram_pool_fwd[C=256]" and roof["bound"] == "hbm" and roof["unit"] == "GB/s"
    assert roof["achieved"] == pytest.approx(823_132_160 / 0.145e-3 / 1e9, rel=1e-3)
    assert roof["frac"] == pytest.approx(roof["achieved"] / 6548.8, abs=1e-4) and roof["peak"] == 6548.8
    assert roof["algorithmic_bytes"] == 823_132_160 and roof["avg_launch_us"] == 145.0
    total = 4 * (0.180 + 0.145 + 0.100 + 0.052)
    assert roof["share_of_library_time"] == pytest.approx(4 * 0.145 / total, abs=1e-3)


def test_roofline_switches_to_the_tensor_bound_and_is_none_without_head_kernels(bench):
    rec = [_rec("gram_pool_bwd[C=1024]", "gram_bwd", 0.150, 400_000_000, 2 * 256 * 1024 * 1024 * 196)]
    _, roof = bench.summarise_profile(rec, PEAKS)
    assert roof["bound"] == "tensor" and roof["unit"] == "TFLOP/s" and roof["peak"] == 1401.6
    assert roof["achieved"] == pytest.approx(2 * 256 * 1024 * 1024 * 196 / 0.150e-3 / 1e12, rel=1e-3)
    kernels, none = bench.summarise_profile([_rec("maxpool2d_nhwc", "maxpool", 0.2, 10, 0)], PEAKS)
    assert none is None and list(kernels) == ["maxpool2d_nhwc"]


def test_head_totals_sum_the_head_kernels_per_step(bench):
    steps = 2
    per_step = [_rec("gram_pool_fwd[a]", "gram_fwd", 0.6, 1, 300e9), _rec("gram_pool_bwd[a]", "gram_bwd", 1.2, 1, 600e9),
                _rec("split_bf16[n=1]", "split", 0.02, 1, 0), _rec("attn_head_fwd[B=512]", "attn", 0.06, 1, 30e9),
                _rec("attn_head_bwd[B=512]", "attn", 0.09, 1, 50e9), _rec("nchw_to_nhwc", "transpose", 5.0, 1, 0)]
    h = bench.head_totals(per_step * steps, steps, PEAKS)
    assert h["gram_fwd_us"] == 600.0 and h["gram_bwd_us"] == 1200.0
    assert h["attn_fwd_us"] == 80.0 and h["attn_bwd_us"] == 90.0                    # the plane split counts as attention forward
    assert h["head_us"] == 1970.0 and h["algorithmic_gflop_per_step"] == 980.0      # the transpose is not head time
    tf = 980e9 / 1970e-6 / 1e12
    assert h["TFLOPs"] == pytest.approx(tf, abs=0.06)
    assert h["frac_of_bf16_peak_burst"] == pytest.approx(tf / 1668.7, abs=1e-4)
    assert h["frac_of_bf16_peak_sustained"] == pytest.approx(tf / 1401.6, abs=1e-4)
    assert bench.head_totals([_rec("maxpool", "maxpool", 1.0, 1, 0)], 1, PEAKS) is None


def test_a_failing_side_leg_is_reported_in_its_place(bench, capsys):
    assert bench.guarded("leg", lambda a, b=0: a + b, 2, b=3) == 5

    def boom():
        raise RuntimeError("no such kernel")

    out = bench.guarded("patchgan_head", boom)
    assert out == {"error": "patchgan_head: RuntimeError: no such kernel"}
    assert "no such kernel" in capsys.readouterr().err                              # the traceback goes to stderr


def test_peaks_and_clock_sampler_degrade_without_a_gpu(bench):
    p = bench.load_peaks()
    assert p["hbm_gbs"] > 1000 and p["tensor_tflops_burst"] >= p["tensor_tflops"] > 100 and p["source"]
    import torch
    if torch.cuda.is_available():
        pytest.skip("covers the no-GPU path")
    with bench.ClockSampler(torch.device("cpu")) as c:
        pass
    assert c.summary() == {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}


def test_dump_outputs_writes_float32_and_samples_the_same_rows_above_the_limit(bench, tmp_path, monkeypatch):
    import numpy as np
    import torch
    emb, logits = torch.randn(10, 6, dtype=torch.float64), torch.randn(10, 2)
    bench.dump_outputs(str(tmp_path / "all"), {"embeddings": emb, "logits": logits})
    got = {n: np.load(tmp_path / "all" / f"{n}.npy") for n in ("embeddings", "logits")}
    assert got["embeddings"].dtype == np.float32 and np.array_equal(got["embeddings"], emb.float().numpy())
    assert np.array_equal(got["logits"], logits.numpy())
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4 * 8 * 4)                    # room for 4 rows of 6 + 2 floats
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"embeddings": emb, "logits": logits})
    a = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in ("embeddings", "logits")}
    assert a["embeddings"].shape == (4, 6) and a["logits"].shape == (4, 2)
    rows = [int(np.flatnonzero((got["embeddings"] == r).all(1))[0]) for r in a["embeddings"]]
    assert rows == sorted(rows) and np.array_equal(a["logits"], got["logits"][rows])      # the same rows of every array
    assert all(np.array_equal(a[n], np.load(tmp_path / "b" / f"{n}.npy")) for n in a)      # and the same from run to run
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 8 * 4 - 1)                    # not even one row fits
    with pytest.raises(ValueError, match="limit"):
        bench.dump_outputs(str(tmp_path / "c"), {"embeddings": emb, "logits": logits})


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_rejects_arguments_it_cannot_honour(argv, tmp_path):
    import subprocess
    import sys
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], cwd=str(tmp_path), capture_output=True,
                         text=True, timeout=300)
    assert res.returncode == 2 and "error:" in res.stderr and not (tmp_path / "out").exists()

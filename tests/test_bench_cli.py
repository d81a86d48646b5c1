"""CPU tests of bench.py's contract pieces that do not need a GPU: the reference (CPU) arm prints ONE
JSON line with the keys the driver reads, the clock sampler degrades gracefully without NVML / a GPU,
and the engine arm refuses to run without CUDA instead of falling back."""

import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


def _run(*args, timeout=300):
    return subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, timeout=timeout, cwd=ROOT)


def test_reference_arm_prints_one_json_line():
    r = _run("--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "1", "--cpu-rows", "2048")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "nsf_log_prob_samples_per_sec" and d["unit"] == "samples/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_engine_arm_refuses_without_cuda():
    import torch

    if torch.cuda.is_available():
        pytest.skip("this check is for the CPU-only build container")
    r = _run("--steps", "1")
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)


def test_clock_sampler_without_gpu_is_harmless():
    sys.path.insert(0, str(ROOT))
    import bench

    clk = bench.ClockSampler(0).prepare()
    with clk:
        pass
    s = clk.summary()
    assert set(s) >= {"sm_mhz", "sm_max_mhz", "reasons", "samples"} and isinstance(s["reasons"], list)


def test_tensor_roofline_denominator_follows_the_clock():
    """bench.tensor_peak: the cuBLAS burst figure when the run held >= 98 % of the maximum SM clock, else that figure
    scaled to the clock actually held (a power-capped run is measured against the pipe's capacity at its clock, not
    against a 'sustained' number taken at some other clock) — never a fraction that the kind string does not explain."""
    sys.path.insert(0, str(ROOT))
    import bench

    peaks = {"bf16_tflops": 1640.0, "bf16_tflops_sustained": 1368.6}
    assert bench.tensor_peak(peaks, {"sm_mhz": 1965.0, "sm_max_mhz": 1965.0, "reasons": []}) == (1640.0, "burst")
    assert bench.tensor_peak(peaks, {"sm_mhz": 1935.0, "sm_max_mhz": 1965.0, "reasons": ["sw_power_cap"]}) == (1640.0, "burst")
    peak, kind = bench.tensor_peak(peaks, {"sm_mhz": 1680.0, "sm_max_mhz": 1965.0, "reasons": ["sw_power_cap"]})
    assert abs(peak - 1640.0 * 1680.0 / 1965.0) < 1e-9 and "1680" in kind and "burst" in kind
    assert bench.tensor_peak(peaks, {}) == (1640.0, "burst")  # no NVML: nothing to scale by


def test_dump_outputs_keeps_dtypes_and_a_fixed_sample(tmp_path, monkeypatch):
    import numpy as np
    import torch

    sys.path.insert(0, str(ROOT))
    import bench

    monkeypatch.setattr(bench, "DUMP_ROWS", 8)
    outputs = {"log_prob": torch.arange(20, dtype=torch.float32), "log_prob_sum": torch.tensor([190.0], dtype=torch.float64)}
    bench.dump_outputs(str(tmp_path / "a"), outputs)
    bench.dump_outputs(str(tmp_path / "b"), outputs)
    lp, total = np.load(tmp_path / "a" / "log_prob.npy"), np.load(tmp_path / "a" / "log_prob_sum.npy")
    assert lp.dtype == np.float32 and lp.shape == (8,) and np.all(np.diff(lp) > 0) and set(lp) <= set(range(20))
    assert total.dtype == np.float64 and total.tolist() == [190.0]
    assert np.array_equal(lp, np.load(tmp_path / "b" / "log_prob.npy"))


def test_bench_rejects_bad_arguments():
    assert "--steps" in _run("--steps", "0").stderr
    assert "--dump-outputs" in _run("--impl", "reference", "--dump-outputs", "x").stderr


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(device, tmp_path):
    """The dumped log-densities are those of the seeded input buffer the last timed step used (the fp64
    oracle on the same rows), and two runs dump identical outputs."""
    import numpy as np
    import torch

    sys.path.insert(0, str(ROOT))
    import bench
    from oracle import oracle

    B, steps = 4096, 3
    for run in ("a", "b"):
        r = _run("--batch", str(B), "--steps", str(steps), "--warmup", "1", "--no-configs", "--no-training-step",
                 "--no-cpu-baseline", "--dump-outputs", str(tmp_path / run))  # fmt: skip
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.splitlines()[-1])["steps"] == steps
    lp = np.load(tmp_path / "a" / "log_prob.npy")
    assert lp.dtype == np.float32 and lp.shape == (B,)
    g = torch.Generator().manual_seed(1234)
    xs = [torch.randn(B, bench.D, generator=g) for _ in range(4)]  # bench.run_ours: x buffers, then c buffers
    cs = [torch.randn(B, bench.C, generator=g) for _ in range(4)]
    x, c = xs[(steps - 1) % 4], cs[(steps - 1) % 4]
    ref = oracle.flowspec_from_module(bench.build_model()).log_prob(x.numpy(), c.numpy())
    assert np.max(np.abs(lp - ref) / np.maximum(np.abs(ref), 1.0)) < 1e-5
    total = np.load(tmp_path / "a" / "log_prob_sum.npy")
    assert total.dtype == np.float64 and abs(total[0] - lp.astype(np.float64).sum()) < 1e-6 * np.abs(lp).sum()
    assert np.array_equal(lp, np.load(tmp_path / "b" / "log_prob.npy"))
    assert np.array_equal(total, np.load(tmp_path / "b" / "log_prob_sum.npy"))
    assert np.load(tmp_path / "a" / "mean_nll.npy").tolist() == [-total[0] / B]

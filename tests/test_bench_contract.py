"""bench.py's output contract, checked without a GPU through the `--impl reference` arm and the pure helpers."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load_bench():
    # bench.py points fd 1 at stderr when it is imported (only the JSON line may reach stdout): keep pytest's capture intact
    saved = os.dup(1)
    try:
        spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        os.dup2(saved, 1)
        os.close(saved)
    return mod


def test_reference_arm_prints_exactly_one_json_line(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["steps"] == 1
    out = np.load(tmp_path / "sample.npy")
    assert out.dtype == np.float32 and out.shape == (64, 263, 1, 196) and np.isfinite(out).all()


def test_dump_outputs_keeps_a_fixed_choice_of_rows_under_the_size_limit(tmp_path):
    b = _load_bench()
    rows = torch.arange(520, dtype=torch.float32)[:, None].expand(520, 32768)   # 128 KiB a row, 65 MiB in all
    b.dump_outputs(str(tmp_path / "a"), {"sample": rows})
    b.dump_outputs(str(tmp_path / "b"), {"sample": rows})
    a, again = np.load(tmp_path / "a" / "sample.npy"), np.load(tmp_path / "b" / "sample.npy")
    assert a.nbytes <= b.DUMP_LIMIT_BYTES and a.shape == (512, 32768) and np.array_equal(a, again)
    kept = a[:, 0]
    assert (np.diff(kept) > 0).all() and (a == kept[:, None]).all()


def test_flop_model_matches_the_survey():
    b = _load_bench()
    assert abs(b.flops_per_pass(64) / 1e9 - 470.57) < 0.01          # SURVEY.md 8(d)
    assert abs(b.KERNEL_FLOPS["qkv"](64) / 1e9 - 19.83) < 0.01
    assert b.usable_cpus() >= 1


def test_clock_summary_windows():
    b = _load_bench()
    c = b.ClockSampler(0)
    row = lambda mhz, cap: [str(mhz), "1965", "Not Active", "Not Active", "Not Active", cap]  # noqa: E731
    c.rows = [(10.05, row(1965, "Not Active")), (10.15, row(1900, "Active")), (10.25, row(1890, "Active")),
              (11.05, row(1965, "Not Active"))]
    c.window("timed", 10.0, 10.3)
    c.window("e2e", 11.0, 11.1)
    s = c.summary()
    assert s["window"] == "timed" and s["samples"] == 3 and s["sm_mhz"] == 1900.0 and s["reasons"] == ["sw_power_cap"]
    short = b.ClockSampler(0)
    short.rows = c.rows
    short.window("timed", 10.0, 10.1)      # one sample only: the end-to-end region is added
    short.window("e2e", 11.0, 11.1)
    assert short.summary()["window"] == "timed+e2e" and short.summary()["samples"] == 2


def test_peak_choice_and_chain_flops():
    b = _load_bench()
    short, long_ = b.measured_peaks(0.04), b.measured_peaks(2.1)
    assert "burst" in short["source"] and "sustained" in long_["source"] and short["bf16_tflops"] >= long_["bf16_tflops"]
    # one chained launch = out-proj + FFN1 + FFN2 + next QKV
    k = b.KERNEL_FLOPS
    assert abs(k["chain"](64) - (k["out_proj"](64) + k["ffn1"](64) + k["ffn2"](64) + k["qkv"](64))) < 1.0


def test_nvml_sampler_summary_without_nvml():
    b = _load_bench()
    s = b.NvmlSampler(0)
    s.max_mhz = 1965.0
    s.rows = [(10.001, 1965.0, 0), (10.006, 1950.0, 0x4), (10.011, 1950.0, 0x4), (10.5, 1200.0, 0x8)]
    s.window("timed", 10.0, 10.04)
    out = s.summary()
    assert out["samples"] == 3 and out["sm_mhz"] == 1950.0 and out["reasons"] == ["sw_power_cap"] and out["window"] == "timed"

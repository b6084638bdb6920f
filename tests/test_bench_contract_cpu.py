"""CPU: the pieces of bench.py that do not need a GPU -- the roofline arithmetic, the workload description and the
reference arm's JSON line (contract keys), on a tiny sample so the whole file runs in seconds."""
import json
import subprocess
import sys
import types
from pathlib import Path

import numpy as np
import pytest
import torch

import bench

ROOT = Path(__file__).resolve().parents[1]


def _eng(mode, **kw):
    d = dict(fp64_slices=7, fp64_slices_kinv=6, fp64_min_dim=512, rns_moduli=16, rns_moduli_kinv=14, rns_moduli_f32=10, fp64_slices_f32=4)
    d.update(kw)
    e = types.SimpleNamespace(**d)
    e.emulation_mode = lambda: mode
    return e


def test_roofline_entry_digit_planes_use_the_flop_weighted_product_count():
    r = bench.roofline_entry(_eng("digits"), 75.0, 37.0, {"bf16_tflops_sustained": 1408.0}, "MEASURED_PEAKS.json", 1e12,
                             100, 1000.0, 1)
    pairs_eff = (28 + 2 * 21) / 3.0
    assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s"
    assert abs(r["peak"] - 2 * 1408.0 / pairs_eff) < 1e-9            # no live INT8 figure: derived from bf16
    assert abs(r["frac"] - 75.0 / r["peak"]) < 1e-12
    assert r["vs_fp64_dmma_peak"] == 75.0 / 37.0


def test_roofline_entry_residue_scheme_uses_the_measured_int8_peak():
    r = bench.roofline_entry(_eng("rns"), 110.0, 37.0, {"bf16_tflops_sustained": 1408.0}, "MEASURED_PEAKS.json", 1e12,
                             100, 1000.0, 1, i8_peak=4300.0)
    prods = (16 + 2 * 14) / 3.0
    assert abs(r["int8_products_per_fp64_product"] - prods) < 1e-12
    assert abs(r["peak"] - 4300.0 / prods) < 1e-9 and abs(r["frac"] - 110.0 / r["peak"]) < 1e-12
    assert abs(r["peak_derived_from_measured_bf16"] - 2 * 1408.0 / prods) < 1e-9
    assert "rns_gemm_kernel" in r["kernel"] and "plmc_peak_i8" in r["peak_source"]


def test_roofline_entry_of_a_long_step_uses_the_sustained_int8_rate_and_keeps_the_burst_beside_it():
    r = bench.roofline_entry(_eng("rns", rns_moduli=15, rns_moduli_kinv=12), 120.0, 37.0, {"bf16_tflops_sustained": 1408.0},
                             "MEASURED_PEAKS.json", 1e12, 100, 1000.0, 1, i8_peak=4300.0, i8_sustained=3700.0)
    assert r["int8_products_per_fp64_product"] == 13.0
    assert abs(r["peak"] - 3700.0 / 13.0) < 1e-9 and abs(r["frac"] - 120.0 / r["peak"]) < 1e-12
    assert abs(r["peak_burst"] - 4300.0 / 13.0) < 1e-9 and abs(r["frac_of_burst_peak"] - 120.0 / r["peak_burst"]) < 1e-12
    assert "sustained" in r["peak_source"] and r["traffic"] > 0


def test_roofline_entry_pure_fp64_mode_is_measured_against_the_dmma_peak():
    r = bench.roofline_entry(_eng("fp64"), 32.0, 37.0, {}, "fallback", 1e12, 100, 1000.0, 1)
    assert r["peak"] == 37.0 and abs(r["frac"] - 32.0 / 37.0) < 1e-12


def test_model_shapes_of_the_named_configs():
    W = bench.WORKLOADS
    assert bench.model_shape(W["c2"], 1, "weak") == (7, 4) and bench.model_shape(W["c2"], 8, "weak") == (56, 32)
    assert bench.model_shape(W["c2"], 4, "strong") == (7, 4)              # the fixed 4-latent model, 1 latent per GPU
    assert bench.model_shape(W["c4"], 8, "weak") == (500, 32)             # the named config: 4 latents per GPU
    assert bench.model_shape(W["c4"], 1, "weak") == (63, 4)               # its per-GPU share
    assert bench.model_shape(W["c5"], 8, "weak") == (20, 8) and bench.model_shape(W["c5"], 1, "weak") == (3, 1)


def test_scaling_fit_recovers_the_exponent(monkeypatch):
    monkeypatch.setattr(bench, "oracle_iteration_time", lambda cfg, p, q, n, reps, warm, device="cpu": 2e-9 * n ** 2.7)
    t, e, samples, cores = bench.oracle_scaling_fit(bench.WORKLOADS["c2"], 7, 4, (1000, 2000, 4000), 44484, budget_s=0.0)
    assert abs(e - 2.7) < 1e-9 and abs(t - 2e-9 * 44484 ** 2.7) < 1e-6 * t and len(samples) == 3 and cores >= 1


def test_workload_config_names_the_baseline_configuration():
    args = types.SimpleNamespace(n=0, workload="c2", gpus=1, scaling="weak")
    cfg = bench.workload_config(args, bench.WORKLOADS["c2"], 1)
    assert cfg["n"] == 44484 and cfg["d"] == 21 and cfg["latents_per_gpu"] == 4 and "model" not in cfg
    assert "AdamW" in cfg["step"]


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--points", "300"], capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["cpu_baseline"]["kind"] == "port"
    assert "fitted_exponent" in line["cpu_baseline"] and line["cpu_baseline"]["samples_n_seconds"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0


def test_steps_must_be_positive_and_set_the_count(monkeypatch, capsys):
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "5", "--warmup", "0"])
    assert bench.parse().steps == 5
    monkeypatch.setattr(sys, "argv", ["bench.py"])
    assert bench.parse().steps is None                                    # the workload's own count
    for bad in ("0", "-2"):
        monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", bad])
        with pytest.raises(SystemExit):
            bench.parse()
    assert "must be at least 1" in capsys.readouterr().err


def test_dump_sample_is_fixed_sorted_and_fits_the_budget():
    assert bench.sample_rows(1000, 80, 80 * 1000) is None                 # everything fits: no sampling
    rows = bench.sample_rows(1000, 80, 8000)
    assert rows.numel() == 100 and torch.equal(rows, bench.sample_rows(1000, 80, 8000))
    assert torch.equal(rows, rows.unique()) and 0 <= rows.min() and rows.max() < 1000
    assert bench.sample_rows(1000, 80, -5).numel() == 0


def test_dump_writes_float_arrays_and_refuses_more_than_the_cap(tmp_path, monkeypatch):
    arrays = bench.host_outputs({"loss": torch.tensor(1.5, dtype=torch.float64),
                                 "param.a": torch.arange(6, dtype=torch.float32).reshape(2, 3),
                                 "grad.b": torch.arange(4, dtype=torch.int64)})
    bench.write_outputs(str(tmp_path / "out"), arrays)
    loss, a, b = (np.load(tmp_path / "out" / f"{k}.npy") for k in ("loss", "param.a", "grad.b"))
    assert loss.dtype == np.float64 and loss == 1.5
    assert a.dtype == np.float32 and a.shape == (2, 3) and a[1, 2] == 5
    assert b.dtype == np.float64 and b.tolist() == [0, 1, 2, 3]
    monkeypatch.setattr(bench, "DUMP_BYTES", 16)
    with pytest.raises(ValueError, match="cap"):
        bench.write_outputs(str(tmp_path / "big"), arrays)
    assert not (tmp_path / "big").exists()


def test_reference_arm_refuses_to_dump_outputs(monkeypatch, tmp_path):
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--dump-outputs", str(tmp_path)])
    with pytest.raises(SystemExit, match="--impl ours"):
        bench.main()

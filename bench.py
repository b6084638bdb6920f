#!/usr/bin/env python
"""Benchmark of the projected-LMC hot path (contract: see the repo brief / DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c1|c2|c3|c4|c5]
                    [--scaling weak|strong] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Default workload (BASELINE.json configs[1], "C2"): synthetic SARCOS-shaped projected LMC, n = 44,484 points, d = 21,
Matern-5/2 ARD, fp64, PLMC variant; 4 latents and 7 tasks PER GPU (weak scaling: at N GPUs the model has 4N latents /
7N tasks, each rank owns 4 latents, one NCCL all-reduce of the loss + gradients per step).  One step = one training
iteration of the reference's loop (experiments.py:263-273): zero_grad, MLL forward, full backward to every raw
parameter, AdamW step, learning-rate scheduler step.  `value` counts 4-latent SARCOS-shaped model iterations per
second (N per step at N GPUs).  --scaling strong keeps the NAMED model fixed and splits its latents over the ranks
(C2: 4 latents -> at most 4 GPUs; C4: 32 latents; C5: 8 latents).  c3 is the prediction config (metric: predictive
mean/variance points per second; test points are sharded over the ranks, every rank holds all factors).

--dump-outputs DIR writes, after the timed steps, what the timed path handed its caller in its last step as
DIR/<name>.npy (float32 or float64, at most 64 MB in all; larger outputs as a fixed, seeded sample of their rows).
Training workloads: `loss`, `grad.<parameter>` and `param.<parameter>` (after the optimiser step), and, with the
prediction section on, `predict.mean` / `predict.variance`; c3: `predict.mean` / `predict.variance`.  Inputs depend
only on the arguments, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time
import warnings

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

# per-GPU share (p, q), and the totals / GPU count the BASELINE.json config is quoted on
WORKLOADS = {
    "c1": dict(n=1000, d=6, p=50, q=10, kernel="rbf", named_gpus=1, named_p=50, named_q=10, steps=50,
               label="C1 experiments.py-style projected LMC"),
    "c2": dict(n=44484, d=21, p=7, q=4, kernel="matern52", named_gpus=1, named_p=7, named_q=4, steps=3,
               label="C2 SARCOS-shaped projected LMC"),
    "c3": dict(n=20000, d=8, p=100, q=16, kernel="rbf", named_gpus=8, named_p=100, named_q=16, steps=1,
               n_test=1000000, label="C3 batched predictive mean/variance"),
    "c4": dict(n=20000, d=8, p=63, q=4, kernel="rbf", named_gpus=8, named_p=500, named_q=32, steps=3,
               label="C4 many-task projected LMC"),
    "c5": dict(n=100000, d=4, p=3, q=1, kernel="rbf", named_gpus=8, named_p=20, named_q=8, steps=2,
               label="C5 large-n projected LMC"),
}
CPU_FIT_NS = (1000, 2000, 4000)          # in-line cpu_baseline of the default run (~10 s of host work)
REFERENCE_FIT_NS = (2000, 4000, 8000)    # --impl reference (~1-2 min of host work)
LIBRARY_N = 8192                         # torch -> cuSOLVER restatement on the same GPU
DUMP_BYTES = 64 << 20                    # cap of everything --dump-outputs writes


def positive_int(text):
    v = int(text)
    if v < 1:
        raise argparse.ArgumentTypeError(f"must be at least 1, got {v}")
    return v


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=None, help="timed steps (default: per workload)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=list(WORKLOADS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--points", dest="n", type=int, default=0, help="override n (debug only; reported in config)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-predict", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--test-points", type=int, default=0)
    ap.add_argument("--dtype", default="f64", choices=["f64", "f32"],
                    help="f32: float32 model -> fp32-grade arithmetic (32-bit operands on the INT8 path, FP64 storage)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy")
    return ap.parse_args()


def sample_rows(n_rows, row_bytes, budget, seed=0):
    """Sorted row indices of a fixed, seeded sample of an [n_rows, ...] output that fits `budget` bytes
    (None: every row fits)."""
    k = min(n_rows, max(0, int(budget // max(row_bytes, 1))))
    if k == n_rows:
        return None
    g = torch.Generator().manual_seed(seed)
    return torch.randperm(n_rows, generator=g)[:k].sort().values


def host_outputs(named):
    """name -> detached host copy (float32 stays float32, everything else becomes float64)."""
    out = {}
    for name, t in named.items():
        t = t.detach().cpu()
        out[name] = t.clone() if t.dtype in (torch.float32, torch.float64) else t.to(torch.float64)
    return out


def write_outputs(path, arrays):
    """Writes name -> host tensor as path/<name>.npy; refuses to write more than DUMP_BYTES in all."""
    import numpy as np

    total = sum(a.numel() * a.element_size() for a in arrays.values())
    if total > DUMP_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_BYTES}-byte cap")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a.numpy())


def model_shape(cfg, world, scaling):
    """(p_total, q_total) of the model run on `world` GPUs."""
    if scaling == "strong" or world == cfg["named_gpus"]:
        return cfg["named_p"], cfg["named_q"]
    return cfg["p"] * world, cfg["q"] * world


def make_data(n, d, p, q, seed=0):
    g = torch.Generator().manual_seed(seed)
    X = torch.rand(n, d, generator=g, dtype=torch.float64) * 2 - 1
    W = torch.randn(d, q, generator=g, dtype=torch.float64)
    ph = torch.rand(q, generator=g, dtype=torch.float64) * 6.28
    Fl = torch.sin(X @ W + ph)
    Hm = torch.randn(q, p, generator=g, dtype=torch.float64)
    Y = Fl @ Hm + 0.1 * torch.randn(n, p, generator=g, dtype=torch.float64)
    Y = (Y - Y.mean(0)) / Y.std(0)
    return X.contiguous(), Y.contiguous()


def build_model(X, Y, q, kernel):
    from projected_lmc_b200 import ProjectedGPModel, gp

    ktype = gp.kernels.RBFKernel if kernel == "rbf" else gp.kernels.MaternKernel
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return ProjectedGPModel(X, Y, Y.shape[1], q, mean_type=gp.means.ZeroMean, kernel_type=ktype,
                                init_lmc_coeffs=True, BDN=False, diagonal_B=False, scalar_B=False)


class ClockSampler:
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md clocks line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i",
                 str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0=None, t1=None):
        """Summary of the samples that arrived inside the timed window [t0, t1] (host clock)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lines = [(ts, ln) for ts, ln in self.lines if t0 is None or (t0 <= ts <= t1)]
        window = "timed region"
        if not lines and self.lines and t0 is not None:  # region shorter than the 200 ms sampling period
            mid = 0.5 * (t0 + t1)
            lines = sorted(self.lines, key=lambda x: abs(x[0] - mid))[:3]
            window = "nearest samples (timed region shorter than the sampling period)"
        for _, ln in lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                pw.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_median": statistics.median(pw) if pw else None,
                "samples": len(sm), "reasons": sorted(reasons), "window": window}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "MEASURED_PEAKS.json"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


def dmma_peak_tflops():
    """Live FP64 tensor (DMMA.8x8x4) peak of this GPU: register-resident mma.sync loop on all SMs."""
    from projected_lmc_b200 import ops

    scratch = torch.zeros(16, dtype=torch.float64, device="cuda")
    best = 0.0
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fl = ops.peak_dmma(148 * 2, 512, 20000, scratch)
        e1.record()
        torch.cuda.synchronize()
        best = max(best, fl / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    return best


def i8_peak_tops():
    """Live INT8 tensor-pipe peak: shared-memory-resident tcgen05.mma.kind::i8 loop on every SM (plmc_peak_i8)."""
    from projected_lmc_b200 import ops

    scratch = torch.zeros(16, dtype=torch.float64, device="cuda")
    best = 0.0
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        n_ops = ops.peak_i8(20000, scratch, 2)
        e1.record()
        torch.cuda.synchronize()
        best = max(best, n_ops / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    return best


def products_per_fp64_product(eng):
    """INT8 products per FP64 product, flop-weighted over one training iteration: the factorisation (1/3 of the
    q n^3 FLOP) runs at the main precision, the explicit inverse (2/3; K^-1 feeds only the gradients) at the
    reduced one.  (main, inverse, weighted, description)"""
    mode = eng.emulation_mode() if hasattr(eng, "emulation_mode") else ("digits" if getattr(eng, "fp64_slices", 0) else "fp64")
    f32 = getattr(eng, "grade", "fp64") == "fp32"
    if mode == "rns":
        m = min(eng.rns_moduli_f32, eng.rns_moduli) if f32 else eng.rns_moduli
        mk = m if f32 else min(getattr(eng, "rns_moduli_kinv", 0) or m, m)
        return m, mk, (m + 2.0 * mk) / 3.0, f"{m} moduli in potrf, {mk} in trtri/lauum"
    if mode == "digits":
        s = min(eng.fp64_slices_f32, eng.fp64_slices) if f32 else eng.fp64_slices
        sk = s if f32 else min(getattr(eng, "fp64_slices_kinv", 0) or s, s)
        a, b = s * (s + 1) // 2, sk * (sk + 1) // 2
        return a, b, (a + 2.0 * b) / 3.0, f"{s} digit planes in potrf, {sk} in trtri/lauum"
    return 0, 0, 0.0, "pure FP64"


def i8_peak_sustained_tops(seconds=3.0):
    """The same loop back to back for `seconds` (the chip reaches its power cap after a few hundred ms): INT8 TOPS
    over the last two thirds of the window -- the denominator for a kernel timed inside a long, power-capped step."""
    from projected_lmc_b200 import ops

    scratch = torch.zeros(16, dtype=torch.float64, device="cuda")
    evs, tot = [], []
    t_end = time.time() + seconds
    torch.cuda.synchronize()
    while time.time() < t_end:
        for _ in range(8):                       # ~5 ms per launch: keep the queue a few launches deep
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            evs.append(e)
            tot.append(ops.peak_i8(20000, scratch, 2))
        evs[-8].synchronize()
    e = torch.cuda.Event(enable_timing=True)
    e.record()
    evs.append(e)
    torch.cuda.synchronize()
    k0 = len(tot) // 3
    ms = evs[k0].elapsed_time(evs[-1])
    return sum(tot[k0:]) / (ms * 1e-3) / 1e12 if ms > 0 else None


def roofline_entry(eng, achieved, dmma_peak, peaks, peak_src, gemm_flops, gemm_launches, fact_ms, steps, i8_peak=None,
                   i8_sustained=None):
    """Roofline of the dominant kernel of the step (the O(n^3) factorisation layer).

    achieved = algorithmic q*n^3 FLOP per step / CUDA-event time of the potrf + solve + potri phases.
    With the FP64-via-INT8 path on (default), the large GEMMs run on the tcgen05 INT8 tensor path: one FP64
    product = P INT8 products (P = moduli of the residue scheme, or s(s+1)/2 digit-plane pairs), so the tensor
    roofline is (INT8 dense rate) / P.  `peak` uses the INT8 rate MEASURED on this GPU by plmc_peak_i8 (a
    shared-memory-resident tcgen05.mma.kind::i8 loop on every SM pair); the figure derived from
    MEASURED_PEAKS.json (2 x sustained bf16) is kept beside it.  The FP64 DMMA peak (live) is reported as well."""
    main, kinv, pairs_eff, desc = products_per_fp64_product(eng)
    common = {
        "bound": "tensor", "achieved": achieved, "unit": "TFLOP/s", "traffic": None,
        "fp64_dmma_peak": dmma_peak, "vs_fp64_dmma_peak": (achieved / dmma_peak) if achieved else None,
        "executed_dmma_gemm_tflops": gemm_flops / steps / (fact_ms * 1e-3) / 1e12 if fact_ms > 0 else None,
        "dmma_gemm_launches_per_step": gemm_launches / steps,
        "how": "algorithmic q*n^3 FLOP per step / CUDA-event time of the potrf+solve+potri phases",
    }
    if pairs_eff > 0:
        bf16 = peaks.get("bf16_tflops_sustained") or peaks.get("bf16_tflops")
        derived = 2.0 * bf16 / pairs_eff
        # the step is long and power-capped: its denominator is the SUSTAINED INT8 rate (a kernel timed alone would
        # use the burst figure, kept beside it)
        burst = (i8_peak / pairs_eff) if i8_peak else None
        peak = (i8_sustained / pairs_eff) if i8_sustained else (burst or derived)
        mode = eng.emulation_mode() if hasattr(eng, "emulation_mode") else "digits"
        common.update({
            "kernel": ("rns_gemm_kernel (FP64 GEMM as %d INT8 tcgen05.mma products modulo coprime moduli, CTA pairs, "
                       "TMEM, bulk async copies) + crt_kernel for GEMMs >= %d; gemm_dmma_kernel (DMMA.8x8x4) below"
                       % (main, eng.fp64_min_dim)) if mode == "rns" else
                      ("ozaki_gemm_kernel (FP64 GEMM as %d INT8 tcgen05.mma digit-plane products, TMEM, bulk async "
                       "copies) for GEMMs >= %d; gemm_dmma_kernel (DMMA.8x8x4) below" % (main, eng.fp64_min_dim)),
            "peak": peak, "frac": (achieved / peak) if achieved else None,
            "peak_source": ("live plmc_peak_i8 run back to back for 3 s (%.0f INT8 TOPS sustained at the power cap; "
                            "%.0f in a 5 ms burst; tcgen05.mma.kind::i8 on shared-memory-resident operands, every "
                            "SM pair) / %.2f INT8 products per FP64 product (%s, flop-weighted)"
                            % (i8_sustained, i8_peak, pairs_eff, desc)) if (i8_peak and i8_sustained) else
                           ("live plmc_peak_i8 (%.0f INT8 TOPS, tcgen05.mma.kind::i8 on shared-memory-resident "
                            "operands, every SM) / %.2f INT8 products per FP64 product (%s, flop-weighted)"
                            % (i8_peak, pairs_eff, desc)) if i8_peak else
                           ("2 x %s bf16 sustained (%.0f TFLOP/s) / %.2f INT8 products per FP64 product (%s)"
                            % (peak_src, bf16, pairs_eff, desc)),
            "peak_burst": burst, "frac_of_burst_peak": (achieved / burst) if (achieved and burst) else None,
            "peak_derived_from_measured_bf16": derived,
            "frac_of_derived_peak": (achieved / derived) if achieved else None,
            "int8_products_per_fp64_product": pairs_eff,
        })
        if mode == "rns":
            # one ncu --set full capture of rns_gemm_kernel<2> (8192^3 FP64 product at 16 moduli; profiles/
            # r02_ncu_summary.md): dram read 16.72 GB + write 1.07 GB per launch against 2.15 GB of operand planes +
            # 1.07 GB of residues (algorithmic): each wave of 74 tile pairs re-streams its 8 + 9 operand panels from
            # HBM; 35 % of DRAM peak, tensor pipe 85.5 % active: not traffic bound
            common["traffic"] = 17.79e9
            common["traffic_reference"] = ("ncu --set full, one 8192^3 rns_gemm_kernel<2> launch: 16.72 GB read + 1.07 GB "
                                           "written, 3.2 GB algorithmic, tensor pipe 85.5 % active, DRAM 35 % "
                                           "(profiles/r02_ncu_summary.md)")
        else:
            common["traffic"] = 8.50e9
            common["traffic_reference"] = ("ncu --set full, one 8192^3 ozaki_gemm_kernel launch: 7.91 GB read + 0.60 GB "
                                           "written, 1.47 GB algorithmic (profiles/r01_ozaki_gemm_v2_ncu_summary.md)")
    else:
        common.update({
            "kernel": "gemm_dmma_kernel (FP64 DMMA.8x8x4; potrf/trsm/trtri/lauum)",
            "peak": dmma_peak, "frac": (achieved / dmma_peak) if achieved else None,
            "peak_source": "live register-resident DMMA microbenchmark on this GPU (FP64 is absent from "
                           "MEASURED_PEAKS.json)",
        })
    return common


# --------------------------------------------------------------------------------------------------------------------
# CPU baseline (oracle port) and the library path on the same GPU
# --------------------------------------------------------------------------------------------------------------------
def oracle_iteration_time(cfg, p, q, n_s, reps, warmup, device="cpu"):
    """One training iteration (fwd + bwd + AdamW) of the reference's algorithm (Cholesky-forced gpytorch semantics,
    restated in oracle/) on `device`; returns mean seconds per iteration."""
    from oracle import plmc_oracle as O
    from tests.helpers import oracle_params

    X, Y = make_data(n_s, cfg["d"], p, q, seed=1)
    m = build_model(X, Y, q, cfg["kernel"])
    if device != "cpu":
        m = m.to(device)
        X, Y = X.to(device), Y.to(device)
    times = []
    opt = torch.optim.AdamW(m.parameters(), lr=1e-2)
    for it in range(warmup + reps):
        if device != "cpu":
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none=True)
        loss = -O.mll(oracle_params(m), X, Y)
        loss.backward()
        opt.step()
        if device != "cpu":
            torch.cuda.synchronize()
        t1 = time.perf_counter()
        if it >= warmup:
            times.append(t1 - t0)
    return sum(times) / len(times)


def oracle_scaling_fit(cfg, p, q, ns, n_target, budget_s=60.0):
    """Times the oracle at several n on all host threads, fits t = c n^e by least squares in log-log and evaluates
    the fit at n_target.  Returns (seconds at n_target, exponent, samples [(n, s/iter)], cores)."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ns = [n for n in ns if n <= n_target] or [n_target]
    samples = []
    for i, n_s in enumerate(ns):
        t = oracle_iteration_time(cfg, p, q, n_s, 1, 1 if i == 0 else 0)
        if t < budget_s / 20:      # cheap sample: average a few more
            reps = int(min(4, max(1, (budget_s / 20) / t)))
            t = oracle_iteration_time(cfg, p, q, n_s, reps, 0)
        samples.append((n_s, t))
    if len(samples) >= 2:
        lx = [math.log(n) for n, _ in samples]
        ly = [math.log(t) for _, t in samples]
        mx, my = sum(lx) / len(lx), sum(ly) / len(ly)
        e = sum((a - mx) * (b - my) for a, b in zip(lx, ly)) / sum((a - mx) ** 2 for a in lx)
        # anchor the extrapolation at the largest measured n (the asymptotic regime), exponent from the fit
        n_l, t_l = samples[-1]
        t_target = t_l * (n_target / n_l) ** e
    else:
        e = None
        t_target = samples[0][1]
    return t_target, e, samples, cores


def baseline_sample_text(cfg, p, q, samples, e, n, t_target, cores):
    pts = ", ".join(f"n={a}: {b:.3f} s/iter" for a, b in samples)
    if e is None:
        return (f"oracle (pure-torch restatement of the reference's Cholesky-forced path) fwd+bwd+AdamW measured at the "
                f"full n={n} (d={cfg['d']}, p={p}, q={q}, {cfg['kernel']}) on {cores} host threads: {pts}")
    return (f"oracle (pure-torch restatement of the reference's Cholesky-forced path; gpytorch is not installable) "
            f"fwd+bwd+AdamW at d={cfg['d']}, p={p}, q={q}, {cfg['kernel']} on {cores} host threads: {pts}; fitted "
            f"t ~ n^{e:.2f}; EXTRAPOLATED from the largest sample with that exponent to n={n}: {t_target:.1f} s/iter "
            f"(a full-size CPU iteration would take hours and ~4x the Gram storage in autograd temporaries)")


def run_reference(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.n or cfg["n"]
    # the reference arm times ONE model of the per-GPU shape on this host, whatever N is: a CPU box does not grow
    # with the GPU count, and the GPU arm's `value` counts models of exactly this shape
    p, q = (cfg["named_p"], cfg["named_q"]) if args.scaling == "strong" else (cfg["p"], cfg["q"])
    steps = args.steps or cfg["steps"]
    t, e, samples, cores = oracle_scaling_fit(cfg, p, q, REFERENCE_FIT_NS, n, budget_s=90.0)
    value = 1.0 / t
    sample = baseline_sample_text(cfg, p, q, samples, e, n, t, cores)
    line = {
        "impl": "reference", "metric": "train_iters_per_sec", "value": value, "unit": "it/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 / value, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, cfg, args.gpus),
        "cpu_baseline": {"value": value, "unit": "it/s", "cores": cores, "kind": "port", "sample": sample,
                         "fitted_exponent": e, "samples_n_seconds": samples, "extrapolated": e is not None},
        "e2e": {"value": value, "unit": "it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "value is for ONE model of the per-GPU shape on the host cores (not multiplied by the GPU count)",
    }
    print(json.dumps(line), flush=True)


def workload_config(args, cfg, world):
    n = args.n or cfg["n"]
    scaling = getattr(args, "scaling", "weak")
    p_tot, q_tot = model_shape(cfg, world, scaling)
    q_loc = -(-q_tot // world)
    out = {
        "workload": f"{cfg['label']}: n={n}, d={cfg['d']}, {cfg['kernel']} ARD, "
                    f"{'float32 model (fp32-grade arithmetic)' if getattr(args, 'dtype', 'f64') == 'f32' else 'fp64'}, PLMC variant (BDN=False), "
                    f"{q_tot} latents and {p_tot} tasks on {world} GPU(s) ({q_loc} latents per GPU)",
        "n": n, "d": cfg["d"], "tasks_total": p_tot, "latents_total": q_tot,
        "latents_per_gpu": q_loc, "parallelism": f"latent-parallel x{world}",
        "step": "zero_grad + MLL forward + full backward + AdamW step + LR scheduler step (experiments.py:263-273)",
        "value_definition": ("iterations/s of the named model (fixed size, latents split over the GPUs)"
                             if scaling == "strong" else
                             f"iterations/s of a {cfg['q']}-latent / {cfg['p']}-task model of this shape; one step at N "
                             f"GPUs = N of them"),
        "l2_policy": "inputs larger than L2 (K is %.1f GB per GPU)" % (q_loc * n * n * 8 / 1e9),
    }
    if n * n * 8 * q_loc < 200e6:
        out["l2_policy"] = "L2 flushed between timed iterations (a 256 MB buffer is rewritten; K is %.0f MB)" % (
            q_loc * n * n * 8 / 1e6)
    return out


def timed_calls(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e-3


def secondary_kernels(model, cfg, n, q_loc, phases, steps, peaks, peak_src):
    """HBM-bound kernels of the step against the measured copy bandwidth: Gram build and gradient sweep from the
    phase events of the timed steps, the projection kernels timed alone (workload shape, and a shape large enough
    to leave L2)."""
    from projected_lmc_b200 import ops

    hbm = peaks.get("hbm_gbs")
    np_ = ((n + 127) // 128) * 128
    gram_bytes = 8.0 * q_loc * np_ * (np_ + 128) / 2
    out = []

    def entry(kernel, nbytes, seconds, note=None):
        ach = nbytes / seconds / 1e9 if seconds and seconds > 0 else None
        e = {"kernel": kernel, "bound": "hbm", "achieved": ach, "peak": hbm, "peak_source": peak_src, "unit": "GB/s",
             "frac": (ach / hbm) if (ach and hbm) else None, "bytes": nbytes, "seconds": seconds}
        if note:
            e["note"] = note
        out.append(e)

    in_step = ("inside the power-capped step (phase events): the FP64 pipe that bounds this kernel runs at the SM clock "
               "the preceding O(n^3) phases left (~0.8-1.0 GHz of 1.965)")
    entry("gram_kernel (fused ARD Gram build, lower tiles written once), in the step", gram_bytes,
          phases.get("gram", 0.0) / steps * 1e-3, in_step)
    entry("grad_sweep2_kernel (fused backward sweep over the lower tiles of K^-1, GEMM form), in the step", gram_bytes,
          phases.get("grad_sweep", 0.0) / steps * 1e-3, in_step)
    # the same two kernels timed alone on the workload's own buffers (burst clocks, as the HBM peak was measured)
    try:
        eng = model._engine
        ws = eng.workspace(model.train_y.device, q_loc, n)
        X64 = model.train_inputs[0].to(torch.float64)
        kid = 0 if cfg["kernel"] == "rbf" else 1
        ell = torch.full((q_loc, cfg["d"]), 0.7, dtype=torch.float64, device=X64.device)
        noise = torch.full((q_loc,), 0.5, dtype=torch.float64, device=X64.device)
        Z, zn = ops.scale_inputs(X64, ops.col_mean(X64), ell, np_)
        alpha = torch.randn(q_loc, np_, dtype=torch.float64, device=X64.device)
        entry("gram_kernel, timed alone (same shape, workspace of the step)", gram_bytes,
              timed_calls(lambda: ops.gram(Z, zn, kid, None, noise, ws["K"], n), 3),
              "FP64-datapath bound, not HBM bound: ncu (profiles/r02_ncu_summary_final.md) FP64 + DMMA pipes 65 % "
              "busy, top stall math_pipe_throttle; 24 DMMA-FMA + ~29 FP64 instructions per entry against 23 FMA "
              "slots per entry at the HBM rate")
        entry("grad_sweep2_kernel, timed alone (same shape; the Gram just written stands in for K^-1)", gram_bytes,
              timed_calls(lambda: ops.grad_sweep(ws["K"], alpha, Z, zn, ell, kid, None, n), 3),
              "FP64-datapath bound: two DMMA contractions (48 FMA per entry) + ~40 FP64 instructions per entry")
        eng.generation += 1
    except Exception as ex:  # noqa: BLE001
        out.append({"kernel": "gram / sweep timed alone", "error": repr(ex)[:200]})
    Y = model.train_y.to(torch.float64)          # float32 models: the projection kernels read an FP64 copy
    p = Y.shape[1]
    q = model.n_latents
    dev = Y.device
    T = torch.randn(p, q, dtype=torch.float64, device=dev)
    G = torch.randn(q, n, dtype=torch.float64, device=dev)
    pj = 8.0 * n * (p + q)
    entry("project_fwd kernel (workload shape)", pj, timed_calls(lambda: ops.project_fwd(Y, T), 20),
          "Y is %.1f MB: L2-resident and launch-latency bound at this size" % (Y.numel() * 8 / 1e6))
    entry("project_bwd kernel + reduce (workload shape)", pj, timed_calls(lambda: ops.project_bwd(Y, G), 20))
    nb, pb, qb = 4000000, 32, 8                                   # 1.28 GB: streams from HBM
    Yb = torch.randn(nb, pb, dtype=torch.float64, device=dev)
    Tb = torch.randn(pb, qb, dtype=torch.float64, device=dev)
    Gb = torch.randn(qb, nb, dtype=torch.float64, device=dev)
    entry("project_fwd_mma_kernel (n=4e6, p=32, q=8: DMMA, cp.async double-buffered slabs)", 8.0 * nb * (pb + qb),
          timed_calls(lambda: ops.project_fwd(Yb, Tb), 5))
    entry("project_bwd_mma_kernel + reduce (n=4e6, p=32, q=8)", 8.0 * nb * (pb + qb),
          timed_calls(lambda: ops.project_bwd(Yb, Gb), 5))
    return out


def library_baseline(cfg, n_lib):
    """The same restatement the CPU arm times, on THIS GPU through torch -> cuSOLVER/cuBLAS (cholesky_ex,
    solve_triangular, autograd): the "library path on the same box" of SURVEY section 2."""
    try:
        t = oracle_iteration_time(cfg, cfg["p"], cfg["q"], n_lib, 2, 1, device="cuda")
        return {"n": n_lib, "seconds_per_iter": t, "it_per_s": 1.0 / t,
                "what": "oracle restatement on cuda: torch.linalg.cholesky_ex / solve_triangular / autograd "
                        "(cuSOLVER + cuBLAS), same d, p, q, kernel"}
    except Exception as ex:  # noqa: BLE001
        return {"n": n_lib, "error": repr(ex)[:300]}


# --------------------------------------------------------------------------------------------------------------------
def main():
    args = parse()
    cfg = WORKLOADS[args.workload]
    torch.set_default_dtype(torch.float64)
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes the outputs of the GPU path (--impl ours)")
        run_reference(args, cfg)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    import torch.distributed as dist

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.workload == "c3":
        run_predict_workload(args, cfg, world, rank, dev)
    else:
        run_train_workload(args, cfg, world, rank, dev)
    if world > 1:
        dist.destroy_process_group()


def run_train_workload(args, cfg, world, rank, dev):
    import torch.distributed as dist

    from projected_lmc_b200 import ProjectedLMCmll, distributed as pdist, ops

    n = args.n or cfg["n"]
    steps = args.steps or cfg["steps"]
    p_tot, q_tot = model_shape(cfg, world, args.scaling)
    if q_tot < world:
        raise SystemExit(f"{args.workload}: {q_tot} latents cannot be split over {world} GPUs (DESIGN.md section 4)")
    Xh, Yh = make_data(n, cfg["d"], p_tot, q_tot, seed=0)
    Xh, Yh = Xh.pin_memory(), Yh.pin_memory()
    model = build_model(Xh.clone(), Yh.clone(), q_tot, cfg["kernel"]).to(dev)
    if args.dtype == "f32":
        model = model.float()
        Xh, Yh = Xh.float().pin_memory(), Yh.float().pin_memory()
    if world > 1:
        pdist.shard_latents(model, rank, world)
    lo, hi = model._latent_range
    q_loc = hi - lo
    model.train()
    mll = ProjectedLMCmll(model.likelihood, model)
    Xd, Yd = model.train_inputs[0], model.train_y
    params = [prm for prm in model.parameters() if prm.requires_grad]

    # optimiser and schedule of the reference's training loop (experiments.py:79-86, 240, 251, 263-273)
    small = n * n * 8 * q_loc < 200e6
    gamma = math.exp(math.log(1e-3 / 1e-2) / 10000)
    # launch-bound workloads on one GPU: the whole iteration as two replayed CUDA graphs, exactly as
    # projected_lmc_b200.fit runs it (training._GraphedStep); PLMC_BENCH_GRAPH=0 times the eager loop instead
    use_graph = small and world == 1 and os.environ.get("PLMC_BENCH_GRAPH", "1") != "0"
    if use_graph:
        lr_t = torch.tensor(1e-2, dtype=torch.float64, device=dev)
        opt = torch.optim.AdamW(params, lr=lr_t, capturable=True)
        sched = None
    else:
        lr_t = None
        opt = torch.optim.AdamW(params, lr=1e-2)
        sched = torch.optim.lr_scheduler.ExponentialLR(opt, gamma=gamma)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if small else None
    graphed = {"step": None, "it": 0, "hist": torch.zeros(1 << 16, dtype=torch.float64, device=dev)}

    def step():
        if graphed["step"] is not None:
            it = graphed["it"] % graphed["hist"].numel()
            graphed["step"].set_iteration(it)
            graphed["step"].run(it)
            graphed["it"] += 1
            return graphed["step"].loss
        opt.zero_grad(set_to_none=True)
        loss = -mll(model(Xd), Yd)
        loss.backward()
        loss = pdist.allreduce_loss_and_grads(loss, params) if world > 1 else loss.detach()
        opt.step()
        if sched is not None:
            sched.step()
        else:
            lr_t.mul_(gamma)
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(dev.index)
    sampler.start()
    for _ in range(max(args.warmup, 3)):
        step()
    if use_graph:
        from projected_lmc_b200.training import _GraphedStep

        graphed["step"] = _GraphedStep(model, mll, Xd, Yd, opt, lr_t, gamma, graphed["hist"], 3)
        step()                                   # one untimed replay
    peak = dmma_peak_tflops()
    i8_peak = i8_peak_tops()

    # ---- timed region: device-resident inputs --------------------------------------
    eng = model._engine
    barrier()
    t_wall0 = time.time()
    ops.stats_reset()
    if small:
        # launch-bound regime: per-step events, L2 flushed (untimed) between the steps
        eng.profile = None
        per = []
        for _ in range(steps):
            flush_buf.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            loss = step()
            e1.record()
            per.append((e0, e1))
        barrier()
        total_ms = sum(a.elapsed_time(b) for a, b in per)
        phases = {}
    else:
        eng.profile = []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            loss = step()
        e1.record()
        barrier()
        total_ms = e0.elapsed_time(e1)
        phases = eng.phase_ms()
        eng.profile = None
    clocks = sampler.stop(t_wall0, time.time())
    launches, gemm_launches, gemm_flops = ops.stats_get()
    ms = torch.tensor([total_ms / steps], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(ms.item())
    models_per_step = 1 if args.scaling == "strong" else world
    value = models_per_step / (ms_per_step * 1e-3)
    dump = None
    if args.dump_outputs and rank == 0:
        # the last timed step's loss and gradients, and the parameters its optimiser step left (the e2e steps below
        # move them on)
        named = {"loss": loss}
        for name, prm in model.named_parameters():
            if prm.requires_grad:
                named["param." + name] = prm
                if prm.grad is not None:
                    named["grad." + name] = prm.grad
        dump = host_outputs(named)

    # ---- end to end: host buffers in, loss out, every step -------------------------
    e2e = None
    if not args.no_e2e:
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            Xd.copy_(Xh, non_blocking=True)
            Yd.copy_(Yh, non_blocking=True)
            lv = step()
            _ = float(lv.item())
        e1.record()
        barrier()
        ms2 = torch.tensor([e0.elapsed_time(e1) / steps], device=dev)
        if world > 1:
            dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
        e2e = {"value": models_per_step / (float(ms2.item()) * 1e-3), "unit": "it/s",
               "h2d_bytes_per_step": (Xh.numel() + Yh.numel()) * Xh.element_size(),
               "d2h_bytes_per_step": Xh.element_size()}

    # ---- prediction: batched predictive mean/variance on the same model (secondary metric) -------
    predict = None
    if not args.no_predict:
        n_test = args.test_points or (8192 if not small else 4096)
        gt = torch.Generator().manual_seed(7)
        Xs = (torch.rand(n_test, cfg["d"], generator=gt, dtype=torch.float64) * 2 - 1).to(dev).to(Xd.dtype)
        model.eval()
        if "PLMC_PREDICT_INVERSE" not in os.environ:
            eng.predict_inverse = True               # factor inverted once, inside the excluded factorisation call
        with torch.no_grad(), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            barrier()
            e0.record()
            _ = model(Xs[:128])                      # factorise + invert (cached afterwards) + one small tile
            e1.record()
            barrier()
            fact_s = e0.elapsed_time(e1) * 1e-3
            full_lik = model.full_likelihood()
            _ = full_lik(model(Xs))                  # untimed: allocates the [q, npad, n_test] cross-Gram tile
            pred_reps = 2
            barrier()
            e0.record()
            for _ in range(pred_reps):
                pred = full_lik(model(Xs))
                chk = float(pred.variance.sum().item() + pred.mean.sum().item())
            e1.record()
            barrier()
        ms3 = torch.tensor([e0.elapsed_time(e1) / pred_reps], device=dev)
        if world > 1:
            dist.all_reduce(ms3, op=dist.ReduceOp.MAX)
        pred_s = float(ms3.item()) * 1e-3
        if dump is not None:
            out = host_outputs({"predict.mean": pred.mean, "predict.variance": pred.variance})
            used = sum(a.numel() * a.element_size() for a in dump.values())
            rows = sample_rows(n_test, sum(a[0].numel() * a.element_size() for a in out.values()), DUMP_BYTES - used)
            dump.update(out if rows is None else {k: a[rows] for k, a in out.items()})
        predict = {"points_per_sec": n_test / pred_s, "n_test": n_test, "seconds": pred_s,
                   "factorisation_seconds_excluded": fact_s, "checksum": chk,
                   "variance_path": "explicit inverse of the factor (once, in the excluded call) + triangular multiply",
                   "algorithmic_tflops": q_loc * float(n) ** 2 * n_test / pred_s / 1e12,
                   "note": "mean + variance [n_test, tasks] through model.eval(); full_likelihood(model(X*)); "
                           "FLOP = q*n^2*n* (triangular solve), per GPU"}
        model.train()

    if rank == 0:
        peaks, peak_src = measured_peaks()
        i8_sus = i8_peak_sustained_tops() if (eng.emulation_mode() != "fp64" and not small) else None
        fact_ms = sum(phases.get(k, 0.0) for k in ("potrf", "retry", "solve_logdet", "potri")) / steps
        alg_flops = q_loc * float(n) ** 3                       # n^3/3 potrf + 2n^3/3 inverse, per GPU
        achieved = alg_flops / (fact_ms * 1e-3) / 1e12 if fact_ms > 0 else None
        line = {
            "metric": "train_iters_per_sec", "value": value, "unit": "it/s", "n_gpus": world, "steps": steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "config": workload_config(args, cfg, world),
            "loss": float(loss.item()),
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
            "arithmetic": {"gemm_mode": eng.emulation_mode(), "min_dim": eng.fp64_min_dim,
                           "int8_products": products_per_fp64_product(eng)[3]},
            "roofline": roofline_entry(eng, achieved, peak, peaks, peak_src, gemm_flops, gemm_launches, fact_ms,
                                       steps, i8_peak, i8_sus),
            "phase_ms_per_step": {k: v / steps for k, v in phases.items()},
            "predict": predict,
        }
        if small:
            line["config"]["cuda_graph"] = ("whole iteration replayed as two CUDA graphs (projected_lmc_b200.fit / "
                                            "training._GraphedStep); the factorisation status is read between them"
                                            if use_graph else "eager launches")
            line["roofline"]["note"] = ("launch-bound configuration: n=%d gives a %.0f MFLOP factorisation per latent; "
                                        "the step time is kernel-launch latency, not tensor throughput" % (n, n ** 3 / 1e6))
        if not args.no_secondary and not small:
            line["roofline_secondary"] = secondary_kernels(model, cfg, n, q_loc, phases, steps, peaks, peak_src)
            if predict:
                line["roofline_secondary"].append({
                    "kernel": "prediction: cross-Gram + V = L^-1 K* (triangular multiply with the explicit inverse) on the INT8 tensor path + column reductions",
                    "bound": "tensor", "achieved": predict["algorithmic_tflops"], "unit": "TFLOP/s",
                    "peak": line["roofline"].get("peak") and (i8_sus or i8_peak) / products_per_fp64_product(eng)[0]
                    if products_per_fp64_product(eng)[0] else peak,
                    "how": "q*n^2*n* FLOP / CUDA-event time of model(X*) + full_likelihood, n* = %d" % predict["n_test"]})
                r = line["roofline_secondary"][-1]
                r["frac"] = (r["achieved"] / r["peak"]) if r.get("peak") else None
        if world == 1:
            del model, mll, opt
            eng.release()
            torch.cuda.empty_cache()
            if not args.no_library_baseline and not small:
                line["library_baseline"] = library_baseline(cfg, min(LIBRARY_N, n))
            if not args.no_cpu_baseline:
                t, e, samples, cores = oracle_scaling_fit(cfg, cfg["p"], cfg["q"], CPU_FIT_NS, n, budget_s=20.0)
                line["cpu_baseline"] = {
                    "value": 1.0 / t, "unit": "it/s", "cores": cores, "kind": "port",
                    "sample": baseline_sample_text(cfg, cfg["p"], cfg["q"], samples, e, n, t, cores),
                    "fitted_exponent": e, "samples_n_seconds": samples, "extrapolated": e is not None,
                }
        if dump is not None:
            write_outputs(args.dump_outputs, dump)
        print(json.dumps(line), flush=True)


def run_predict_workload(args, cfg, world, rank, dev):
    """C3: batched predictive mean / variance for n_test points.  Test points are sharded over the ranks (no
    per-point communication); every rank factorises all q latents once (not timed in `value`, reported beside it)."""
    import torch.distributed as dist

    from projected_lmc_b200 import ops

    n = args.n or cfg["n"]
    n_test = args.test_points or cfg["n_test"]
    steps = args.steps or cfg["steps"]
    p, q = cfg["named_p"], cfg["named_q"]
    Xh, Yh = make_data(n, cfg["d"], p, q, seed=0)
    model = build_model(Xh, Yh, q, cfg["kernel"]).to(dev)
    model.eval()
    # n* >> n: the factor is inverted once (inside the untimed, separately reported factorisation call) and the
    # variance term becomes a triangular multiply (engine.predict_inverse; "auto" would decide the same after n/2 points)
    if "PLMC_PREDICT_INVERSE" not in os.environ:
        model._engine.predict_inverse = True
    lo = rank * n_test // world
    hi = (rank + 1) * n_test // world
    gt = torch.Generator().manual_seed(7)
    Xs_h = (torch.rand(n_test, cfg["d"], generator=gt, dtype=torch.float64) * 2 - 1)[lo:hi].contiguous().pin_memory()
    mean_h = torch.empty((hi - lo, p), dtype=torch.float64).pin_memory()
    var_h = torch.empty((hi - lo, p), dtype=torch.float64).pin_memory()
    chunk = 65536

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(dev.index)
    sampler.start()
    with torch.no_grad(), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        _ = model(Xs_h[:128].to(dev))                # factorisation of all q latents (cached)
        e1.record()
        barrier()
        fact_s = e0.elapsed_time(e1) * 1e-3
        full_lik = model.full_likelihood()
        Xs_d = Xs_h.to(dev)
        for _ in range(max(1, min(args.warmup, 2))):
            _ = full_lik(model(Xs_d[:8192]))
        i8_peak = i8_peak_tops()
        peak = dmma_peak_tflops()
        eng = model._engine
        keep = None
        if args.dump_outputs:
            # this rank's rows of a fixed sample of the [n_test, p] outputs, per chunk, gathered in the last timed step
            rows = sample_rows(n_test, 2 * p * 8, DUMP_BYTES)
            rows = torch.arange(n_test) if rows is None else rows
            rows = rows[(rows >= lo) & (rows < hi)] - lo
            keep = {"rows": {s0: (rows[(rows >= s0) & (rows < s0 + chunk)] - s0).to(dev)
                             for s0 in range(0, hi - lo, chunk)}, "mean": [], "variance": []}

        def run(from_host, keep=None):
            chk = torch.zeros((), dtype=torch.float64, device=dev)
            for s0 in range(0, hi - lo, chunk):
                s1 = min(hi - lo, s0 + chunk)
                xs = Xs_h[s0:s1].to(dev, non_blocking=True) if from_host else Xs_d[s0:s1]
                pred = full_lik(model(xs))
                if from_host:
                    mean_h[s0:s1].copy_(pred.mean, non_blocking=True)
                    var_h[s0:s1].copy_(pred.variance, non_blocking=True)
                if keep is not None:
                    keep["mean"].append(pred.mean[keep["rows"][s0]])
                    keep["variance"].append(pred.variance[keep["rows"][s0]])
                chk = chk + pred.mean.sum() + pred.variance.sum()
            return chk

        barrier()
        t_wall0 = time.time()
        ops.stats_reset()
        e0.record()
        for it in range(steps):
            chk = run(False, keep if it == steps - 1 else None)
        e1.record()
        barrier()
        clocks = sampler.stop(t_wall0, time.time())
        launches, gemm_launches, gemm_flops = ops.stats_get()
        ms = torch.tensor([e0.elapsed_time(e1) / steps], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        sec = float(ms.item()) * 1e-3
        e2e = None
        if not args.no_e2e:
            barrier()
            e0.record()
            for _ in range(steps):
                chk2 = run(True)
                _ = float(chk2.item())
            e1.record()
            barrier()
            ms2 = torch.tensor([e0.elapsed_time(e1) / steps], device=dev)
            if world > 1:
                dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
            e2e = {"value": n_test / (float(ms2.item()) * 1e-3), "unit": "points/s",
                   "h2d_bytes_per_step": n_test * cfg["d"] * 8, "d2h_bytes_per_step": 2 * n_test * p * 8 + 8 * world}
    dump = None
    if keep is not None:
        dump = host_outputs({"predict.mean": torch.cat(keep["mean"]), "predict.variance": torch.cat(keep["variance"])})
        if world > 1:                                # the shards are contiguous and in rank order
            shards = [None] * world
            dist.all_gather_object(shards, dump)
            dump = {k: torch.cat([s[k] for s in shards]) for k in dump}
    if rank == 0:
        peaks, peak_src = measured_peaks()
        main = products_per_fp64_product(eng)[0]
        alg = q * float(n) ** 2 * (hi - lo) / sec / 1e12
        i8_sus = i8_peak_sustained_tops() if main else None
        rpeak = (i8_sus / main) if main else peak
        line = {
            "metric": "predict_points_per_sec", "value": n_test / sec, "unit": "points/s", "n_gpus": world,
            "steps": steps, "warmup": max(1, min(args.warmup, 2)), "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{cfg['label']}: n_test={n_test} points sharded over {world} GPU(s), train n={n}, "
                                   f"d={cfg['d']}, {p} tasks, {q} latents, {cfg['kernel']} ARD, fp64; every rank holds "
                                   f"all {q} Cholesky factors ({q * n * n * 8 / 1e9:.1f} GB)",
                       "n": n, "n_test": n_test, "d": cfg["d"], "tasks_total": p, "latents_total": q,
                       "parallelism": f"test-point-parallel x{world} (no collective on the data path)",
                       "step": "predictive mean + variance [n_test, tasks] through model.eval(); full_likelihood(model(X*))",
                       "l2_policy": "inputs larger than L2 (the factors are %.1f GB per GPU)" % (q * n * n * 8 / 1e9)},
            "factorisation_seconds_excluded": fact_s, "checksum": float(chk.item()),
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
            "arithmetic": {"gemm_mode": eng.emulation_mode(), "min_dim": eng.fp64_min_dim,
                           "int8_products": products_per_fp64_product(eng)[3]},
            "roofline": {"bound": "tensor", "achieved": alg, "peak": rpeak, "unit": "TFLOP/s",
                         "frac": alg / rpeak if rpeak else None, "traffic": None,
                         "kernel": "V = L^-1 K* of the predictive variance (q n^2 n* FLOP per rank) as a triangular "
                                   "multiply with the explicit inverse (dense 512-leaves) on the INT8 tensor path",
                         "peak_burst": (i8_peak / main) if main else None,
                         "peak_source": "live plmc_peak_i8 back to back for 3 s (%.0f INT8 TOPS sustained at the power cap; "
                                        "%.0f in a 5 ms burst) / %d INT8 products per FP64 product"
                                        % (i8_sus, i8_peak, main) if main else "live DMMA microbenchmark",
                         "fp64_dmma_peak": peak},
        }
        if dump is not None:
            write_outputs(args.dump_outputs, dump)
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
